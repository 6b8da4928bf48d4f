"""GPU tests of frame-level cross-entropy training (run with -m gpu on the B200 box): the fused ce_eval kernel and the
CE train step of the Net mirror, against the restatement in tests/ce_util.py and the oracle's forward / backward.

Tolerances: the kernel is checked bit for bit where the arithmetic is one IEEE operation (diff = y - onehot) or an
integer count; the objective, a sum of fp32 logs in double, to rel 1e-6.  The train step uses the bounds of
tests/test_gpu_parity.py: layer outputs (and obj_diff = y - onehot) abs 2e-5, momentum buffers abs 2e-3 + rel 2e-3,
parameters abs 2e-6 after one SGD step (Adagrad: the adaptive bounds used there).
"""
import numpy as np
import pytest

import ce_util
from util import assert_close, case, model_file
from eesen_b200 import binding
from oracle import oracle

pytestmark = pytest.mark.gpu


def torch_():
    import torch
    return torch


def _ce_case(seed, S, T, K):
    rng = np.random.default_rng(seed)
    frames = np.sort(rng.integers(max(1, T // 3), T + 1, size=S))[::-1].astype(np.int32)
    frames[0] = T
    if S >= 3:
        frames[-1] = 0                       # an utterance without frames: every row of it is padding
    targets = ce_util.random_targets(frames, K, seed + 1)
    y = oracle.softmax((rng.standard_normal((T * S, K)) * 3).astype(np.float32), np.float32)
    # tied maxima: the first index wins (FindRowMaxId); the target is the first one on even rows, the second on odd
    packed = ce_util.pack_targets(targets, frames, T)
    valid = np.nonzero(ce_util.valid_rows(frames, T))[0]
    for i, r in enumerate(valid[: 2 * S]):
        a, b = (1, K - 1) if K > 2 else (0, 1)
        y[r] = 0.5 / K
        y[r, a] = y[r, b] = 0.25
        packed[r] = a if i % 2 == 0 else b
    # a non-target posterior of exactly 0: the reference's objective would be NaN, ours stays finite
    r = valid[-1]
    y[r, (packed[r] + 1) % K] = 0.0
    return frames, packed, y


@pytest.mark.parametrize("seed,S,T,K", [(0, 3, 7, 5), (1, 16, 50, 46), (2, 5, 33, 4000), (3, 64, 120, 46)])
def test_ce_eval_vs_restatement(ctx, seed, S, T, K):
    torch = torch_()
    frames, packed, y = _ce_case(seed, S, T, K)
    ldp = (K + 3) // 4 * 4
    yp = np.zeros((T * S, ldp), np.float32); yp[:, :K] = y
    yp[:, K:] = np.nan                       # padding columns are never read
    d_y = torch.from_numpy(yp).cuda()
    d_len = torch.from_numpy(frames).cuda()
    d_tgt = torch.from_numpy(packed).cuda()
    outs = []
    for _ in range(2):
        d_diff = torch.full((T * S, ldp), 3.0, dtype=torch.float32, device="cuda")
        d_st = torch.full((3,), -1.0, dtype=torch.float64, device="cuda")
        torch.cuda.synchronize()
        ctx.ce_eval(T, S, K, d_len, d_y, ldp, d_tgt, d_diff, ldp, d_st)
        ctx.synchronize()
        outs.append((d_diff.cpu().numpy(), d_st.cpu().numpy()))
    (diff, st), (diff2, st2) = outs
    assert np.array_equal(diff, diff2) and np.array_equal(st, st2), "two runs differ"
    ref_diff, ref_obj, ref_correct, ref_valid = ce_util.ce_eval(y, frames, packed, np.float32)
    assert np.array_equal(diff[:, :K], ref_diff), "diff is not y - onehot bit for bit"
    pad = ~ce_util.valid_rows(frames, T)
    assert np.all(diff[pad, :K] == 0)
    assert np.all(diff[:, K:] == 3.0), "columns [K, ldd) were written"
    _, obj64, _, _ = ce_util.ce_eval(y, frames, packed, np.float64)
    assert np.isfinite(st[0])
    assert abs(st[0] - obj64) <= 1e-6 * abs(obj64)
    assert abs(st[0] - ref_obj) <= 1e-6 * abs(ref_obj)
    assert (st[1], st[2]) == (ref_correct, ref_valid)


def _net(ctx, net, lr, mom, algorithm):
    n = binding.Net(ctx, model_file(net))
    n.set_train_options(lr, mom)
    n.set_optimizer(algorithm)
    n.get(102)   # keep in_diff from the next step on
    return n


@pytest.mark.parametrize("wl", ["small", "mid"])
@pytest.mark.parametrize("bidirectional", [True, False])
@pytest.mark.parametrize("algorithm", ["SGD", "Adagrad"])
def test_train_step_ce_vs_oracle(ctx, wl, bidirectional, algorithm):
    w, net, b = case(wl, bidirectional=bidirectional)
    lr, mom = 1e-3, 0.9
    targets = ce_util.random_targets(b.frames, w.classes, 11)
    packed = ce_util.pack_targets(targets, b.frames, b.T)
    n = _net(ctx, net, lr, mom, algorithm)
    st = n.train_step_ce(b.feats, b.frames, targets, True)
    on = oracle.OracleNet(net, np.float64)
    on.set_optimizer(algorithm)
    y = on.forward(b.feats, b.frames)
    diff, obj, _, valid = ce_util.ce_eval(y, b.frames, packed, np.float64)
    on.backward_update(diff, b.frames, lr, mom)
    L = len(net.layers)
    for i in range(1, L + 1):
        assert_close(f"out_l{i}", n.get(i), on.acts[i], atol=2e-5)
    assert_close("obj_diff", n.get(100), diff, atol=2e-5)
    assert_close("in_diff", n.get(102), on.in_diffs[0], atol=2e-5, rtol=1e-3)
    assert_close("corr", n.corr(), on.flat_corr(), atol=2e-3, rtol=2e-3)
    if algorithm == "SGD":
        assert_close("params", n.params(), on.flat_params(), atol=2e-6)
    else:   # the bounds of the adaptive tests in test_gpu_parity.py: lr*c/sqrt(accu+eps) amplifies corr differences
        assert_close("accu", n.accu(), on.flat_accu(), atol=1e-7, rtol=5e-3)
        assert_close("params", n.params(), on.flat_params(), atol=0.02 * lr)
    assert abs(st["obj"] - obj) <= 2e-5 * abs(obj)
    # the count is exact against the step's own posteriors (near-ties may flip between fp32 and fp64 forwards)
    _, _, correct, _ = ce_util.ce_eval(n.get(L), b.frames, packed, np.float32)
    assert (st["correct"], st["frames"], st["padded"]) == (correct, valid, b.T * b.S)
    n.close()


def test_ce_step_device_matches_host_and_test_mode_keeps_params(ctx):
    torch = torch_()
    w, net, b = case("small")
    targets = ce_util.random_targets(b.frames, w.classes, 12)
    packed = ce_util.pack_targets(targets, b.frames, b.T)
    host = _net(ctx, net, 1e-3, 0.9, "SGD")
    dev = _net(ctx, net, 1e-3, 0.9, "SGD")
    d_feats = torch.from_numpy(np.ascontiguousarray(b.feats)).cuda()
    d_tgt = torch.from_numpy(packed).cuda()
    torch.cuda.synchronize()
    for _ in range(2):
        sh = host.train_step_ce(b.feats, b.frames, targets, True)
        dev.train_step_ce_device(d_feats, b.T, b.S, b.frames, d_tgt, True)
    sd = dev.read_stats(ce=True)
    assert sh == sd
    assert np.array_equal(host.params(), dev.params())
    assert np.array_equal(host.get(100), dev.get(100))
    p0 = host.params()
    se = host.train_step_ce(b.feats, b.frames, targets, False)
    assert np.array_equal(host.params(), p0)
    assert se["frames"] == b.valid_frames
    host.close()
    dev.close()


def test_ce_and_ctc_steps_share_a_net(ctx):
    """read_stats reports the loss of the last step; CTC and CE steps can alternate on one model."""
    w, net, b = case("small")
    targets = ce_util.random_targets(b.frames, w.classes, 13)
    n = _net(ctx, net, 1e-3, 0.9, "SGD")
    st_ctc = n.train_step(b.feats, b.frames, b.labels, True)
    st_ce = n.train_step_ce(b.feats, b.frames, targets, True)
    assert n.read_stats(ce=True) == st_ce
    st_ctc2 = n.train_step(b.feats, b.frames, b.labels, True)
    assert st_ctc["frames"] == st_ctc2["frames"] == st_ce["frames"] == b.valid_frames
    assert st_ctc2["ref_tokens"] == st_ctc["ref_tokens"]
    n.close()


def test_ce_step_rejects_out_of_range_targets(ctx):
    w, net, b = case("small")
    targets = ce_util.random_targets(b.frames, w.classes, 14)
    targets[1][3] = w.classes
    n = _net(ctx, net, 1e-3, 0.9, "SGD")
    p0 = n.params()
    with pytest.raises(binding.EesenB200Error, match="Class id out of network output dimension"):
        n.train_step_ce(b.feats, b.frames, targets, True)
    assert np.array_equal(n.params(), p0)
    n.close()
