#!/usr/bin/env python
"""bench.py -- CTC training frames/sec of the B200-native Eesen hot path (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W [--workload c2] [--impl ours|reference]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

One "step" = one pass of the hot path (Net::Propagate -> Ctc::EvalParallel -> ErrorRateMSeq ->
Net::Backpropagate incl. the gradient all-reduce and the SGD update) over one packed synthetic
minibatch of BASELINE.json configs[1]: 4x320 BiLSTM phone-CTC, 40-dim fbank, 64 utterances per GPU,
T ~ U{400..600}.  Weak scaling: every rank processes its own 64-utterance shard; the only data-path
collective is the per-step NCCL all-reduce of the 8.3 M-float gradient arena.

Rank 0 prints ONE JSON line:
  value      valid frames/s, whole job, inputs resident in HBM, CUDA events on the library's stream,
             max over ranks
  e2e        same metric through the public C-ABI call with HOST buffers (page-locked host memory; H2D of
             the packed features and D2H of the statistics inside the timed region)
  roofline   dominant kernel category of the step, measured live with CUDA events
  roofline_step  the whole step against the HBM roof (SURVEY.md 8d bytes per valid frame)
  cpu_baseline  the reference's own cpucompute path (oracle/_ref/ref_dump_cpu = unmodified reference
             objects) + the restated CTC (the reference has no CPU CTC) on a bounded sample, N=1 only
  gpu_reference  the reference's own gpucompute kernels (oracle/_ref/ref_dump_gpu) on the same GPU and batch, N=1 only
  replicas_identical  (N > 1) sha256 of every rank's parameters after the timed steps agree
--dump-outputs DIR writes what the last timed step returned on rank 0 as DIR/<name>.npy (see dump_outputs); the inputs
are seeded, so two builds run with the same arguments can be compared output for output.
--impl reference times the CPU arm as the main line, on the full minibatch (tens of seconds per step on the host).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from eesen_b200 import kaldi_io, synth  # noqa: E402

METRIC = "ctc_train_frames_per_sec"
UNIT = "frames/s"
REF_SAMPLE_UTTS = 8  # bounded CPU sample inside the GPU arm's line: this many utterances of the same workload per step


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm_gbs": d["hbm_gbs"], "bf16_tflops": d["bf16_tflops"],
                "bf16_tflops_sustained": d.get("bf16_tflops_sustained", d["bf16_tflops"]), "source": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, pw, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1])); pw.append(float(f[2]))
            except ValueError:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "power_w_max": float(max(pw)),
                "samples": len(sm), "reasons": sorted(reasons)}


# --------------------------------------------------------------------------------------- CPU arm
def cpu_reference_arm(w, steps: int, warmup: int, tmp: str, sample_utts: int = REF_SAMPLE_UTTS):
    """Times the reference's CPU implementation of the path on this box's host cores.

    oracle/_ref/ref_dump_cpu = UNMODIFIED reference objects (Net fwd/bwd/update on cpucompute with
    OpenBLAS, all host threads).  The reference has no CPU CTC ("not implemented for CPU yet",
    cuda-matrix.cc:862-864...), so the restated CTC (oracle/cpu_ref.c, fp32, 1 thread) is timed on the
    same sample and added: "reference-CPU BiLSTM + restated-CPU CTC" (BASELINE.md section 3.4)."""
    from oracle import oracle  # test/bench-only import: the checker as the CPU baseline
    cores = os.cpu_count() or 1
    net = synth.make_model(w, seed=0)
    b = synth.make_batch(w, seed=1, S=sample_utts)
    model = os.path.join(tmp, "ref_model")
    batch = os.path.join(tmp, "ref_batch.bin")
    kaldi_io.write_model(model, net)
    kaldi_io.write_batch_file(batch, b)
    # thread-count probe on a small sample (one untimed step each), the timing itself on `b`
    probe = batch
    if sample_utts > REF_SAMPLE_UTTS:
        probe = os.path.join(tmp, "ref_probe.bin")
        kaldi_io.write_batch_file(probe, synth.make_batch(w, seed=1, S=REF_SAMPLE_UTTS))
    sample = (f"{b.S} utterances of the {w.name} workload per step ({b.valid_frames} valid / "
              f"{b.feats.shape[0]} padded frames)")
    # CTC restatement on the sample (fp32 port, single thread)
    rng = np.random.default_rng(0)
    y = oracle.softmax(rng.standard_normal((b.feats.shape[0], w.classes)).astype(np.float32), np.float32)
    t0 = time.perf_counter()
    oracle.ctc_eval(y, b.frames, b.labels, b.S, np.float32)
    t_ctc = time.perf_counter() - t0
    if oracle.have_reference("cpu"):
        # "all the host threads it can use": OpenBLAS stops scaling (and then collapses) well below the
        # core count on the per-timestep [S x C]*[C x 4C] products, so probe a few thread counts with
        # one untimed step each and keep the fastest
        best = None
        for th in sorted({min(cores, c) for c in (8, 16, 32)}):
            try:
                info = oracle.run_reference("cpu", model, probe, os.path.join(tmp, "ref_out"), w.learn_rate,
                                            w.momentum, steps=1, time_only=True, threads=th, timeout=120)
            except Exception:
                continue
            if best is None or info["step_seconds"][0] < best[1]:
                best = (th, info["step_seconds"][0])
        threads = best[0] if best else min(cores, 8)
        info = oracle.run_reference("cpu", model, batch, os.path.join(tmp, "ref_out"), w.learn_rate, w.momentum,
                                    steps=steps + warmup, time_only=True, threads=threads)
        st = info["step_seconds"][warmup:]
        kind = "reference"
        cores = threads
    else:
        on = oracle.OracleNet(net, np.float32)
        st = []
        for i in range(steps + warmup):
            t0 = time.perf_counter()
            on.train_step(b, w.learn_rate, w.momentum)
            if i >= warmup:
                st.append(time.perf_counter() - t0 - t_ctc)
        kind = "port"
    sec = float(np.mean(st)) + t_ctc
    return {"value": b.valid_frames / sec, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample,
            "seconds_per_step": sec, "ctc_restated_seconds": t_ctc,
            "note": "reference cpucompute BiLSTM/affine/softmax/SGD + restated CPU CTC (reference has none)"}


def run_reference_impl(args, w):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    # the SAME configuration as the GPU arm: the full w.S-utterance minibatch per step.  One such step takes the
    # host cores tens of seconds, so at most one warm-up step is executed whatever --warmup asks for; `sample` says
    # how many were.  --steps timed steps are executed.
    run_steps, run_warm = args.steps, min(args.warmup, 1)
    with tempfile.TemporaryDirectory() as tmp:
        cb = cpu_reference_arm(w, run_steps, run_warm, tmp, sample_utts=args.ref_utts or w.S)
    cb["sample"] += f"; {run_steps} timed step(s) after {run_warm} warm-up executed of --steps {args.steps} --warmup {args.warmup}"
    line = {"impl": "reference", "metric": METRIC, "value": cb["value"], "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": cb["seconds_per_step"] * 1e3,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": w.name, "layers": w.layers, "cells_per_direction": w.cells, "input_dim": w.in_dim,
                       "classes": w.classes, "utts_per_gpu": args.ref_utts or w.S, "frames_per_utt": [w.t_lo, w.t_hi],
                       "parallelism": "cpu host cores", "storage": "fp32", "learn_rate": w.learn_rate,
                       "momentum": w.momentum, "frames_counted": "valid (unpadded) frames"},
            "cpu_baseline": {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample", "note")},
            "e2e": {"value": cb["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)
    return 0


def gpu_reference_leg(w, tmp: str, steps: int = 2):
    """The reference's OWN kernels (src/gpucompute, unmodified, compiled for sm_100a: oracle/_ref/ref_dump_gpu)
    on the same B200 and the same full minibatch: one warm-up + `steps` timed train steps (BASELINE.md 3.6)."""
    from oracle import oracle  # bench-only: the reference as a timed comparator, never on the product path
    if not oracle.have_reference("gpu"):
        return {"value": None, "unit": UNIT, "unavailable": "oracle/_ref/ref_dump_gpu not built"}
    net = synth.make_model(w, seed=0)
    b = synth.make_batch(w, seed=1)
    model, batch = os.path.join(tmp, "gref_model"), os.path.join(tmp, "gref_batch.bin")
    kaldi_io.write_model(model, net)
    kaldi_io.write_batch_file(batch, b)
    try:
        info = oracle.run_reference("gpu", model, batch, os.path.join(tmp, "gref_out"), w.learn_rate, w.momentum,
                                    steps=steps + 1, time_only=True, timeout=300)
    except Exception as e:
        return {"value": None, "unit": UNIT, "unavailable": str(e)[-300:]}
    st = info["step_seconds"][1:]
    sec = float(np.mean(st))
    return {"value": b.valid_frames / sec, "unit": UNIT, "seconds_per_step": sec, "steps": len(st), "kind": "reference gpucompute",
            "sample": f"{b.S} utterances of the {w.name} workload ({b.valid_frames} valid / {b.feats.shape[0]} padded frames)",
            "note": "unmodified reference src/gpucompute + src/net built for sm_100a, its own cuBLAS calls and per-kernel device syncs"}


# --------------------------------------------------------------------------------------- GPU arm
DUMP_SAMPLE = 1 << 20   # momentum buffers: this many entries at fixed, seeded positions
DUMP_LIMIT = 63_000_000  # bytes of all dumped arrays together: with the .npy headers under 64 MB however counted


def seeded_sample(a, n, seed):
    """n entries of a (flattened) at fixed positions drawn from `seed`, in order; all of a if it has no more."""
    a = a.ravel()
    if a.size <= n:
        return a
    return a[np.sort(np.random.default_rng(seed).choice(a.size, n, replace=False))]


def last_step_outputs(net, n_layers, stats):
    """What a caller of the timed path holds after its last step: the statistics, log p(z|x) per utterance, the
    posteriors and the CTC gradient [T*S x K], the updated parameters and a fixed, seeded sample of the momentum
    buffers.  When the parameters, posteriors and gradient together would take the dump past DUMP_LIMIT (C4: 27.5 M
    parameters), each of the three is replaced by a fixed, seeded sample of its share of what is left (names
    <name>_sample); C2 is dumped whole, about 50 MB."""
    out = {"stats": np.array([stats[k] for k in ("obj", "token_err", "ref_tokens", "frames")], np.float64),
           "pzx": net.get(101).ravel(), "momentum_sample": seeded_sample(net.corr(), DUMP_SAMPLE, 0)}
    big = {"posteriors": net.get(n_layers), "obj_diff": net.get(100), "params": net.params()}
    room = DUMP_LIMIT - sum(v.nbytes for v in out.values())
    total = sum(v.nbytes for v in big.values())
    for seed, (k, v) in enumerate(big.items(), 1):
        if total <= room:
            out[k] = v
        else:
            out[k + "_sample"] = seeded_sample(v, room * v.size // total, seed)
    return out


def dump_outputs(outdir: str, outputs) -> None:
    os.makedirs(outdir, exist_ok=True)
    for k, v in outputs.items():
        np.save(os.path.join(outdir, k + ".npy"), np.ascontiguousarray(v))


def rooflines_from_profile(ms, counts, w, batches, peaks, steps, prec, wall_ms, engines=(1, 1)):
    """Per-kernel rooflines from the library's per-launch CUDA events (eesen_b200_profile).
    Algorithmic figures (DESIGN.md section 4; SURVEY.md section 8d split by kernel):
      recurrent forward  : 20*C floats per valid frame and layer (read pre-acts 8C, write g,i,f,o,c,m 12C)
                           + 2*C floats' worth for the fp16 hi/lo planes of m the tcgen05 kernel writes
      recurrent backward : 22*C floats per valid frame and layer (read saved 12C + dout 2C, write DGIFO 8C)
      dense GEMMs        : 48*C*I + 16*C*C per layer + 12*C*K flops per PADDED frame (all rows are multiplied)
    `traffic` = dram__bytes_read+write per launch from the committed ncu --set full capture
    (profiles/traffic.json), or null.  engines = (forward, backward): 1 = tcgen05 recurrent kernels, 0 = warp-level."""
    # shares are taken against the measured wall time of the timed steps: the weight-gradient products and the
    # per-layer all-reduces run on a side stream concurrently with the recurrent kernels, so the per-category
    # CUDA-event sums may add up to more than the step
    tot = wall_ms or sum(ms.values()) or 1.0
    valid = float(np.mean([b.valid_frames for b in batches]))
    padded = float(np.mean([b.feats.shape[0] for b in batches]))
    traffic = {}
    tp = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tp):
        try:
            traffic = json.load(open(tp)).get(w.name, {})
        except Exception:
            traffic = {}
    out = {}
    for k in ("lstm_fwd", "lstm_bwd"):
        if counts.get(k, 0) == 0:
            continue
        # bytes per launch (one layer); the tcgen05 forward kernel also writes the two fp16 planes of m (2C x 2 x 2 bytes)
        by = ((22.0 if engines[0] == 1 else 20.0) if k == "lstm_fwd" else 22.0) * w.cells * 4.0 * valid
        dur = ms[k] / counts[k] * 1e-3
        ach = by / dur / 1e9
        eng = engines[0 if k == "lstm_fwd" else 1]
        kname = ("lstm_tc_" if eng == 1 else "lstm_") + ("fwd" if k == "lstm_fwd" else "bwd") + "_kernel"
        out[k] = {"kernel": kname, "bound": "hbm", "achieved": ach, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                  "frac": ach / peaks["hbm_gbs"], "traffic": traffic.get(kname), "peak_source": peaks["source"],
                  "algorithmic_bytes_per_launch": by, "avg_launch_ms": dur * 1e3, "launches_per_step": counts[k] / steps,
                  "share_of_step": ms[k] / tot,
                  "note": "latency-bound at 64 utterances/GPU: T dependent steps per launch (SURVEY.md 7.1)"}
    g_ms = ms.get("gemm", 0.0) + ms.get("gemm_side", 0.0)
    g_cnt = counts.get("gemm", 0) + counts.get("gemm_side", 0)
    if g_cnt:
        d = w.in_dim
        fl = 0.0
        for _ in range(w.layers):
            fl += 48.0 * w.cells * d + 16.0 * w.cells * w.cells
            d = 2 * w.cells
        fl += 12.0 * w.cells * w.classes
        flops = fl * padded
        dur = g_ms / steps * 1e-3
        ach = flops / dur / 1e12
        tf32x3 = os.environ.get("EESEN_B200_GEMM_FP32X3") == "tf32"
        mult = {"fp32x3": 6.0 if tf32x3 else 3.0, "tf32": 2.0, "bf16": 1.0}[prec]   # tensor-pipe work per algorithmic flop, in bf16 units
        gnote = {"fp32x3": "arithmetic fp32x3: 3 tcgen05 kind::f16 MMAs per product on fp16 hi/lo planes (3 bf16-equivalent flops per algorithmic flop)",
                 "tf32": "arithmetic tf32: 1 tcgen05 kind::tf32 MMA per product (tf32 runs at half the bf16 rate)",
                 "bf16": "arithmetic bf16: 1 tcgen05 kind::f16 MMA per product"}[prec]
        if os.environ.get("EESEN_B200_GEMM_FP32X3") == "tf32" and prec == "fp32x3":
            gnote = "arithmetic fp32x3 on kind::tf32 (3 MMAs per product at half the bf16 rate)"
        out["gemm"] = {"kernel": "gemm_tc16_kernel (all dense contractions of a step, operand conversions included)", "bound": "tensor", "achieved": ach,
                       "peak": peaks["bf16_tflops_sustained"], "unit": "TFLOP/s",
                       "frac": ach / peaks["bf16_tflops_sustained"], "traffic": traffic.get("gemm"),
                       "peak_source": peaks["source"], "algorithmic_flops_per_step": flops,
                       "launches_per_step": g_cnt / steps, "share_of_step": ms.get("gemm", 0.0) / tot,
                       "share_note": "share_of_step counts the launches of the main stream only; the side stream's products (gemm_side in per_category_ms_per_step) overlap the recurrent kernels",
                       "tensor_pipe_frac_bf16_equiv": ach * mult / peaks["bf16_tflops_sustained"],
                       "note": gnote}
    return out


def run_ours(args, w):
    import torch
    import torch.distributed as dist
    from eesen_b200 import binding

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- eesen_b200 has no CPU path (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    ctx = binding.Context(local, args.gemm_precision, args.recurrent_precision)
    if world > 1:
        obj = [ctx.nccl_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(obj, src=0)
        ctx.nccl_init(rank, world, obj[0])

    tmp = tempfile.mkdtemp(prefix="eesen_b200_bench_")
    model_path = os.path.join(tmp, f"model_{rank}")
    spec = synth.make_model(w, seed=0)
    kaldi_io.write_model(model_path, spec)  # identical weights on every rank
    net = binding.Net(ctx, model_path)
    net.set_train_options(w.learn_rate, w.momentum)

    # a small pool of distinct batches per rank (weak scaling: per-GPU work fixed)
    pool = [synth.make_batch(w, seed=1000 * rank + 1 + i) for i in range(args.pool)]
    stream = torch.cuda.ExternalStream(ctx.stream)
    dev = []
    for b in pool:
        flat, lab_len = binding.Net._labels(b.labels)
        dev.append((torch.from_numpy(b.feats).cuda(), b.T, b.S, np.ascontiguousarray(b.frames, np.int32), flat, lab_len))
    torch.cuda.synchronize()

    def step_dev(i):
        d = dev[i % len(dev)]
        net.train_step_device(d[0], d[1], d[2], d[3], d[4], d[5], True)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for i in range(args.warmup):
        step_dev(i)
    net.read_stats()
    barrier()

    # ---- timed region 1: device-resident inputs, CUDA events on the library's stream
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    l0 = ctx.launches
    ctx.profile(1)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record(stream)
    for i in range(args.steps):
        step_dev(i)
    e1.record(stream)
    stats = net.read_stats()
    barrier()
    ms_dev = e0.elapsed_time(e1)
    prof_ms, prof_cnt = ctx.profile(0)
    launches = ctx.launches - l0
    clocks = sampler.stop() if rank == 0 else None
    frames_dev = sum(pool[i % len(pool)].valid_frames for i in range(args.steps))
    # read before the e2e and TF32 passes below train the model further
    outputs = last_step_outputs(net, len(spec.layers), stats) if args.dump_outputs and rank == 0 else None
    padded_dev = sum(pool[i % len(pool)].feats.shape[0] for i in range(args.steps))

    # ---- timed region 2: end to end through the public call with HOST buffers.  The packed features of every
    # minibatch sit in page-locked host memory (what a data loader hands over); each timed step copies them to
    # the device and reads the statistics back inside the call.
    pinned = [torch.from_numpy(b.feats).pin_memory() for b in pool]
    host_feats = [t.numpy() for t in pinned]
    for i in range(min(2, args.warmup)):
        b = pool[i % len(pool)]
        net.train_step(host_feats[i % len(pool)], b.frames, b.labels, True)
    barrier()
    t0 = time.perf_counter()
    for i in range(args.steps):
        b = pool[i % len(pool)]
        net.train_step(host_feats[i % len(pool)], b.frames, b.labels, True)   # blocks until the statistics are back
    torch.cuda.synchronize()
    t_e2e = time.perf_counter() - t0
    barrier()

    # ---- informational: the same device-resident loop in single-pass TF32 arithmetic (looser stated
    # tolerance: log p rel 1e-4, per-frame gradient abs 5e-3; tests/test_gpu_parity.py) -- never the headline
    ms_alt = None
    if args.gemm_precision == "fp32x3" and args.recurrent_precision == "fp32x3" and not args.no_alt:
        ctx.set_precision("tf32", "tf32")
        for i in range(2):
            step_dev(i)
        net.read_stats()
        barrier()
        a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a0.record(stream)
        for i in range(args.steps):
            step_dev(i)
        a1.record(stream)
        net.read_stats()
        barrier()
        ms_alt = a0.elapsed_time(a1)
        ctx.set_precision(args.gemm_precision, args.recurrent_precision)

    # correctness next to speed: every replica must hold bit-identical parameters after the timed steps
    replicas_identical = None
    if world > 1:
        import hashlib
        digest = hashlib.sha256(np.ascontiguousarray(net.params()).tobytes()).hexdigest()
        digests = [None] * world
        dist.all_gather_object(digests, digest)
        replicas_identical = all(d == digests[0] for d in digests)

    t = torch.tensor([ms_dev, t_e2e * 1e3, float(frames_dev), float(padded_dev), ms_alt or 0.0], dtype=torch.float64, device="cuda")
    if world > 1:
        mx = t.clone()
        dist.all_reduce(mx, op=dist.ReduceOp.MAX)
        sm = t.clone()
        dist.all_reduce(sm, op=dist.ReduceOp.SUM)
        ms_dev, ms_e2e = mx[0].item(), mx[1].item()
        frames_all, padded_all = sm[2].item(), sm[3].item()
        ms_alt = mx[4].item() if ms_alt else None
    else:
        ms_e2e = t_e2e * 1e3
        frames_all, padded_all = float(frames_dev), float(padded_dev)

    if rank == 0:
        peaks = load_peaks()
        value = frames_all / (ms_dev * 1e-3)
        h2d = int(np.mean([b.feats.nbytes + b.frames.nbytes * 5 + sum(l.nbytes for l in b.labels) + 8 * b.S for b in pool]))
        d2h = int(np.mean([4 * b.S + 4 * b.feats.shape[0] for b in pool]))   # pzx[S] + argmax[T*S]
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_dev / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": w.name, "layers": w.layers, "cells_per_direction": w.cells, "input_dim": w.in_dim,
                       "classes": w.classes, "utts_per_gpu": w.S, "frames_per_utt": [w.t_lo, w.t_hi],
                       "global_utts": w.S * world, "parallelism": f"dp{world}",
                       "gemm_arithmetic": args.gemm_precision, "recurrent_arithmetic": args.recurrent_precision,
                       "storage": "fp32", "learn_rate": w.learn_rate, "momentum": w.momentum,
                       "l2": "inputs larger than L2: ~2 GB of activations are streamed per step, no flush needed",
                       "frames_counted": "valid (unpadded) frames"},
            "padded_frames_per_sec": padded_all / (ms_dev * 1e-3),
            "e2e": {"value": frames_all / (ms_e2e * 1e-3), "unit": UNIT, "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": d2h, "ms_per_step": ms_e2e / args.steps},
            "gpu_launches": int(launches),
            "alt_arithmetic": None if not ms_alt else {
                "gemm": "tf32", "recurrent": "tf32", "value": frames_all / (ms_alt * 1e-3), "unit": UNIT,
                "ms_per_step": ms_alt / args.steps,
                "tolerance": "log p(z|x) rel 1e-4, per-frame gradient abs 5e-3 (not the headline; fp32x3 is)"},
            "clocks": clocks,
            "per_category_ms_per_step": {k: v / args.steps for k, v in prof_ms.items() if v > 0},
            "per_category_note": "CUDA-event time of each launch on its own stream; gemm = dense products and conversions of the "
                                 "main stream, gemm_side (weight gradients, streamed chunks) and allreduce run on the side stream "
                                 "and overlap the recurrent kernels, so the sum can exceed ms_per_step",
            "last_step_stats": stats,
        }
        engines = (ctx.lstm_engine(w.S, w.cells, 2, False), ctx.lstm_engine(w.S, w.cells, 2, True))
        allr = rooflines_from_profile(prof_ms, prof_cnt, w, pool, peaks, args.steps, args.gemm_precision, ms_dev, engines)
        # dominant kernel = the single kernel function with the largest share of the step; the dense
        # contractions are one kernel template launched ~25x per step and are reported next to it
        dom = max((k for k in allr if k != "gemm"), key=lambda k: allr[k]["share_of_step"], default="gemm")
        if "gemm" in allr and allr["gemm"]["share_of_step"] > 1.5 * allr.get(dom, {"share_of_step": 0})["share_of_step"]:
            dom = "gemm"
        line["roofline"] = allr[dom]
        line["rooflines_other"] = {k: v for k, v in allr.items() if k != dom}
        # whole step against the HBM roof: SURVEY.md 8(d) algorithmic bytes per valid frame (374.7 KB for C2,
        # 753 KB for C4; weights excluded) x valid frames / step time -- the figure north_star's 70 % refers to
        max_lab = int(np.mean([max(len(l) for l in b.labels) for b in pool]))
        by_frame = synth.hbm_bytes_per_frame(w, max_lab)
        ach = by_frame * (frames_all / world) / (ms_dev * 1e-3) / 1e9      # per GPU
        line["roofline_step"] = {"bound": "hbm", "achieved": ach, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                                 "frac": ach / peaks["hbm_gbs"], "peak_source": peaks["source"],
                                 "algorithmic_bytes_per_valid_frame": by_frame,
                                 "note": "per GPU; the recurrence is latency-bound at 64 utterances per GPU (T dependent steps per layer and pass)"}
        if world > 1:
            line["replicas_identical"] = replicas_identical
        if world == 1 and not args.no_cpu_baseline:
            try:
                line["cpu_baseline"] = cpu_reference_arm(w, 1, 0, tmp)
            except Exception as e:  # the checker is optional for the measurement itself
                line["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": os.cpu_count(), "kind": "port",
                                        "sample": f"failed: {e}"}
        if world == 1 and not args.no_gpu_reference:
            # the context must not hold the GPU's memory hostage while the reference allocates its ~3 GB
            line["gpu_reference"] = gpu_reference_leg(w, tmp)
        if outputs is not None:
            dump_outputs(args.dump_outputs, outputs)
        print(json.dumps(line), flush=True)
    net.close()
    ctx.close()
    if world > 1:
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c2", choices=sorted(synth.WORKLOADS))
    ap.add_argument("--gemm-precision", default="fp32x3", choices=["fp32x3", "tf32", "bf16"])
    ap.add_argument("--recurrent-precision", default="fp32x3", choices=["fp32x3", "tf32"])
    ap.add_argument("--pool", type=int, default=4, help="distinct synthetic batches per rank")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-alt", action="store_true", help="skip the informational TF32 pass")
    ap.add_argument("--no-gpu-reference", action="store_true", help="skip timing the reference's own gpucompute kernels")
    ap.add_argument("--ref-utts", type=int, default=0, help="--impl reference: utterances per step (default: the full minibatch)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step as DIR/<name>.npy (rank 0)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to --impl ours (the CPU arm returns no device outputs)")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    w = synth.WORKLOADS[args.workload]
    if args.impl == "reference":
        return run_reference_impl(args, w)
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.gpus > 1 and world == 1:
        # convenience: relaunch under torchrun (the driver launches torchrun itself)
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
               "--master-addr", "127.0.0.1", "--master-port", "29517", os.path.abspath(__file__)] + sys.argv[1:]
        return subprocess.call(cmd)
    return run_ours(args, w)


if __name__ == "__main__":
    sys.exit(main())
