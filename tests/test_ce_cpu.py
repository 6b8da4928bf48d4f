"""CPU tests of the frame-level cross-entropy pieces that need no GPU: the restatement the GPU tests hold the kernel
to (tests/ce_util.py), checked against a literal transcription of CE::EvalParallel's matrix arithmetic
(src/net/ce-loss.cc:94-169), and the public declarations."""
import os
import re

import numpy as np

import ce_util
from util import ROOT


def _reference_formulation(y, frames, packed):
    """ce-loss.cc:113-142 as written: AddMat(-1, onehot), MulRowsVec(mask), FindRowMaxId, -Sum(log(y) .* onehot .* mask)"""
    N, K = y.shape
    mask = ce_util.valid_rows(frames, N // len(frames)).astype(y.dtype)
    onehot = np.zeros_like(y)
    onehot[np.arange(N), packed] = 1          # padded rows carry target 0 (train-ce-parallel.cc:154)
    diff = (y + np.asarray(-1.0, y.dtype) * onehot) * mask[:, None]
    correct = int(((np.argmax(y, axis=1) == packed) & (mask == 1)).sum())
    with np.errstate(divide="ignore", invalid="ignore"):
        obj = -float((np.log(y) * onehot * mask[:, None]).astype(np.float64).sum())
    return diff, obj, correct


def _case(seed, S=6, T=20, K=46):
    rng = np.random.default_rng(seed)
    frames = np.sort(rng.integers(5, T + 1, size=S))[::-1].astype(np.int32)
    frames[0] = T
    logits = rng.standard_normal((T * S, K)) * 3
    y = np.exp(logits - logits.max(1, keepdims=True))
    y = (y / y.sum(1, keepdims=True)).astype(np.float32)
    targets = ce_util.random_targets(frames, K, seed + 1)
    return frames, ce_util.pack_targets(targets, frames, T), y


def test_restatement_matches_the_reference_arithmetic():
    for seed in range(3):
        frames, packed, y = _case(seed)
        diff, obj, correct, valid = ce_util.ce_eval(y, frames, packed, np.float32)
        rdiff, robj, rcorrect = _reference_formulation(y, frames, packed)
        assert np.array_equal(diff, rdiff)     # -0 == +0 in padded rows
        assert correct == rcorrect and valid == frames.sum()
        assert abs(obj - robj) <= 1e-6 * abs(robj)
        _, obj64, correct64, _ = ce_util.ce_eval(y, frames, packed, np.float64)
        assert abs(obj - obj64) <= 1e-6 * abs(obj64) and correct64 == correct


def test_objective_reads_the_target_column_only():
    frames, packed, y = _case(7)
    r = 3 * len(frames)                      # a valid row
    y[r, (packed[r] + 1) % y.shape[1]] = 0.0
    _, robj, _ = _reference_formulation(y, frames, packed)
    _, obj, _, _ = ce_util.ce_eval(y, frames, packed, np.float32)
    assert np.isnan(robj) and np.isfinite(obj)
    y[r, packed[r]] = 0.0                    # the target's own posterior 0: +inf, as documented
    assert ce_util.ce_eval(y, frames, packed, np.float32)[1] == np.inf


def test_pack_targets_ignores_extra_targets_and_zero_fills_padding():
    frames = np.array([3, 1], np.int32)
    packed = ce_util.pack_targets([np.array([4, 5, 6, 9]), np.array([7])], frames, 3)
    assert packed.tolist() == [4, 7, 5, 0, 6, 0]


def test_header_and_binding_declare_the_ce_entry_points():
    hdr = open(os.path.join(ROOT, "include", "eesen_b200.h")).read()
    for name in ("eesen_b200_ce_eval", "eesen_b200_net_train_step_ce", "eesen_b200_net_train_step_ce_device"):
        assert re.search(r"\bint " + name + r"\(", hdr), name
    from eesen_b200 import binding
    assert callable(binding.Context.ce_eval)
    for m in ("train_step_ce", "train_step_ce_device"):
        assert callable(getattr(binding.Net, m))
