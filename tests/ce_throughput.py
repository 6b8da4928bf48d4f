"""Measurement (run on a GPU box): valid frames/s of the device-resident frame-level cross-entropy step against the
CTC step of the same network, in one process, for C2 (4x320 BiLSTM, K = 46) and for C2's body with a K = 4000
output layer (a senone-sized output); plus the time of the fused CE kernel alone (eesen_b200_profile, category
softmax/argmax) and its share of the 6.56 TB/s HBM bandwidth measured in DESIGN.md section 4.1b, from 2*K*4 bytes
per row.  Prints the card name and power limit with the numbers.

    python tests/ce_throughput.py [steps]      -> one JSON line per configuration
"""
import dataclasses
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from eesen_b200 import binding, kaldi_io, synth  # noqa: E402

HBM_TBS = 6.56   # DESIGN.md section 4.1b, measured streaming bandwidth of this card


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except OSError:
        out = "nvidia-smi unavailable"
    return out


def step_rate(ctx, run, sync, steps, warmup):
    for _ in range(warmup):
        run()
    sync()
    t0 = time.perf_counter()
    for _ in range(steps):
        run()
    sync()
    return (time.perf_counter() - t0) / steps


def measure(ctx, torch, w, steps, warmup):
    net = synth.make_model(w, seed=0)
    b = synth.make_batch(w, seed=1)
    d = tempfile.mkdtemp(prefix="eesen_b200_ce_")
    kaldi_io.write_model(os.path.join(d, "model"), net)
    rng = np.random.default_rng(2)
    targets = [rng.integers(0, w.classes, size=int(f)).astype(np.int32) for f in b.frames]
    packed = np.zeros(b.T * b.S, np.int32)
    for s in range(b.S):
        packed[np.arange(int(b.frames[s])) * b.S + s] = targets[s]
    d_feats = torch.from_numpy(np.ascontiguousarray(b.feats)).cuda()
    d_tgt = torch.from_numpy(packed).cuda()
    flat = np.ascontiguousarray(np.concatenate(b.labels), np.int32)
    lab_len = np.array([len(l) for l in b.labels], np.int32)
    n_ctc = binding.Net(ctx, os.path.join(d, "model"))
    n_ctc.set_train_options(w.learn_rate, w.momentum)
    n_ce = binding.Net(ctx, os.path.join(d, "model"))
    n_ce.set_train_options(w.learn_rate, w.momentum)
    torch.cuda.synchronize()
    run_ctc = lambda: n_ctc.train_step_device(d_feats, b.T, b.S, b.frames, flat, lab_len, True)
    run_ce = lambda: n_ce.train_step_ce_device(d_feats, b.T, b.S, b.frames, d_tgt, True)
    # alternate the two, twice, so that drift of the shared host shows in both
    t_ctc, t_ce = [], []
    for _ in range(2):
        t_ctc.append(step_rate(ctx, run_ctc, ctx.synchronize, steps, warmup))
        t_ce.append(step_rate(ctx, run_ce, ctx.synchronize, steps, warmup))
    st = n_ce.read_stats(ce=True)
    # the CE kernel alone on this step's posteriors, timed by the library's per-category events
    N, K = b.T * b.S, w.classes
    ld = (K + 3) // 4 * 4
    probs = torch.rand((N, ld), dtype=torch.float32, device="cuda")
    diff = torch.empty_like(probs)
    d_len = torch.from_numpy(b.frames).cuda()
    d_st = torch.zeros(3, dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()
    for _ in range(warmup):
        ctx.ce_eval(b.T, b.S, K, d_len, probs, ld, d_tgt, diff, ld, d_st)
    ctx.profile(1)
    reps = 200
    for _ in range(reps):
        ctx.ce_eval(b.T, b.S, K, d_len, probs, ld, d_tgt, diff, ld, d_st)
    ms, cnt = ctx.profile(-1)
    ctx.profile(0)
    kern_ms = ms["softmax"] / reps
    bytes_ = 2.0 * K * 4 * N
    n_ctc.close()
    n_ce.close()
    return {
        "config": w.name, "K": K, "S": b.S, "T": b.T, "valid_frames": b.valid_frames,
        "ctc_step_ms": [1e3 * t for t in t_ctc], "ce_step_ms": [1e3 * t for t in t_ce],
        "ctc_valid_fps": b.valid_frames / min(t_ctc), "ce_valid_fps": b.valid_frames / min(t_ce),
        "ce_minus_ctc_ms": 1e3 * (min(t_ce) - min(t_ctc)),
        "ce_kernel_ms": kern_ms, "ce_kernel_bytes": bytes_, "ce_kernel_tbs": bytes_ / (kern_ms * 1e-3) / 1e12,
        "ce_kernel_share_of_hbm": bytes_ / (kern_ms * 1e-3) / 1e12 / HBM_TBS,
        "ce_obj_per_frame": st["obj"] / st["frames"],
        "note": "probs for the kernel-only timing are [T*S x K] fp32 (%.1f MB), the step's working set" % (N * ld * 4 / 1e6),
    }


def main():
    import torch
    steps = int(sys.argv[1]) if len(sys.argv) > 1 else 20
    ctx = binding.Context(0)
    print(json.dumps({"card": card(), "torch_device": torch.cuda.get_device_name(0)}))
    c2 = synth.WORKLOADS["c2"]
    for w in (c2, dataclasses.replace(c2, name="c2_body_k4000", classes=4000)):
        print(json.dumps(measure(ctx, torch, w, steps, 3)))
    ctx.close()


if __name__ == "__main__":
    main()
