#!/usr/bin/env python
"""Generates the committed golden vectors from the UNMODIFIED reference (oracle/_ref binaries).

    python tests/golden/make_golden.py cpu     # here (no GPU): reference cpucompute build
    python tests/golden/make_golden.py gpu     # on the B200 box: reference gpucompute build (sm_100a)

The reference ships no tests / golden vectors for this path (SURVEY.md section 4), so the pins are
minted from runs of the reference itself on seeded synthetic inputs:

* ``<wl>_refcpu.npz``  Net::Propagate / Backpropagate / Update of the reference's CPU path.  CTC is a
  no-op on CPU in the reference (cuda-matrix.cc:862-864 ...), so ``obj_diff`` is supplied by the fp32
  restatement and stored in the fixture; everything else (layer outputs, in_diff, momentum buffers
  after clipping, updated parameters) is the reference's own output.
* ``<wl>_refgpu.npz``  the same plus the reference's own CUDA CTC (alpha, beta, pzx, obj_diff):
  the only place the reference computes CTC at all.

* ``<wl>_refgpu_{adagrad,rmsprop}.npz``  three steps of the reference's GPU build with
  --opt-algorithm Adagrad / RMSProp (GPU-only in the reference: the CPU branches of ApplySqrt /
  AddMatMatElements exit, cuda-matrix.cc:572-573,658-659): updated parameters and the accumulators the
  reference writes into the model (<BiLstmAccus>/<AffineAccus>).

Inputs are regenerated from (workload, seeds) by eesen_b200.synth, so only outputs are stored.

``runs/<name>.npz`` hold the runs of the reference binaries the tests make themselves (tests/util.py:stored_runs).
The tests write them, with the reference built under oracle/_ref; these two commands select exactly those tests:

    EESEN_B200_RECORD_RUNS=1 python -m pytest tests -m "not gpu" \
        -k "reference_reads_and_rewrites or net_initialize or reference_driver_reads or live or token_error_count"
    EESEN_B200_RECORD_RUNS=1 python -m pytest tests -m gpu -k "gpucompute or format_to_nonparallel_and_extract"  # B200

The dropout fixtures (runs/tiny_drop_*) change with every recording: the reference draws its masks from a
random_device-seeded generator, and the fixture stores the masks it drew.  So does runs/net_initialize (unseeded
initialisation); the stored stdout / stderr carry timings.  Everything else records bit for bit the same.
"""
import os
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from eesen_b200 import kaldi_io, synth  # noqa: E402
from oracle import oracle  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))
CASES = [("tiny", 3, 5, 1e-3, 0.9), ("small", 3, 5, 1e-3, 0.9), ("c1", 0, 0, 4e-5, 0.9)]  # workload, model seed, batch seed, lr, momentum
# the same workloads with <LstmParallel> (uni-directional) layers: "<wl>_uni_ref{cpu,gpu}.npz"
UNI_CASES = [("tiny", 3, 5, 1e-3, 0.9), ("small", 3, 5, 1e-3, 0.9)]


def run(kind: str, outdir: str = HERE, uni: bool = False):
    for wl, mseed, bseed, lr, mom in (UNI_CASES if uni else CASES):
        w = synth.WORKLOADS[wl]
        net = synth.make_model(w, seed=mseed, bidirectional=not uni)
        b = synth.make_batch(w, seed=bseed)
        d = tempfile.mkdtemp()
        kaldi_io.write_model(d + "/model", net)
        kaldi_io.write_batch_file(d + "/batch.bin", b)
        diff_in = None
        if kind == "cpu":
            on = oracle.OracleNet(net, np.float32)
            r = on.train_step(b, lr, mom)
            np.save(d + "/diff.npy", r["obj_diff"].astype(np.float32))
            diff_in = d + "/diff.npy"
        oracle.run_reference(kind, d + "/model", d + "/batch.bin", d + "/out", lr, mom, steps=2, diff_in=diff_in)
        dump = oracle.load_dump(d + "/out")
        m2 = kaldi_io.read_model(d + "/out/model_out")
        keep = {k: v for k, v in dump.items() if not k.startswith("out_l0")}
        keep["params_out"] = m2.flat_params()
        keep["meta"] = np.array([mseed, bseed, 2], np.int64)      # seeds, number of steps run
        keep["hyper"] = np.array([lr, mom], np.float64)
        if diff_in:
            keep["diff_in"] = np.load(diff_in)
        path = os.path.join(outdir, f"{wl}{'_uni' if uni else ''}_ref{kind}.npz")
        np.savez_compressed(path, **keep)
        print("wrote", path, os.path.getsize(path), "bytes")


ADAPTIVE = [("tiny", 3, 5, 1e-3, 0.9, "Adagrad"), ("tiny", 3, 5, 1e-3, 0.9, "RMSProp"),
            ("small", 3, 5, 2e-3, 0.5, "Adagrad"), ("small", 3, 5, 2e-3, 0.5, "RMSProp")]


def run_adaptive(outdir: str = HERE, steps: int = 3):
    for wl, mseed, bseed, lr, mom, opt in ADAPTIVE:
        w = synth.WORKLOADS[wl]
        net = synth.make_model(w, seed=mseed)
        b = synth.make_batch(w, seed=bseed)
        d = tempfile.mkdtemp()
        kaldi_io.write_model(d + "/model", net)
        kaldi_io.write_batch_file(d + "/batch.bin", b)
        oracle.run_reference("gpu", d + "/model", d + "/batch.bin", d + "/out", lr, mom, steps=steps, opt=opt)
        dump = oracle.load_dump(d + "/out")
        m2 = kaldi_io.read_model(d + "/out/model_out")
        keep = {"pzx": dump["pzx"], "params_out": m2.flat_params(), "accus_out": m2.flat_accus(),
                "meta": np.array([mseed, bseed, steps], np.int64), "hyper": np.array([lr, mom], np.float64)}
        path = os.path.join(outdir, f"{wl}_refgpu_{opt.lower()}.npz")
        np.savez_compressed(path, **keep)
        print("wrote", path, os.path.getsize(path), "bytes")


def run_infer(outdir: str = HERE):
    """small_netout_refcpu.npz: the reference's own net-output-extract (CPU build, utterance by utterance)
    with --apply-log, class priors, prior scale and blank scale."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from test_inference_cpu import infer_case
    w, net, b, utts, counts = infer_case()
    d = tempfile.mkdtemp()
    kaldi_io.write_model(d + "/model", net)
    keys = [f"utt{i:02d}" for i in range(len(utts))]
    kaldi_io.write_feature_ark(d + "/feats.ark", keys, utts)
    open(d + "/counts", "w").write("[ " + " ".join(repr(float(c)) for c in counts) + " ]\n")
    oracle.run_reference_tool("ref_net_output_extract",
                              ["--apply-log=true", f"--class-frame-counts={d}/counts", "--prior-scale=0.8",
                               "--blank-scale=0.5", d + "/model", f"ark:{d}/feats.ark", f"ark:{d}/out.ark"], threads=4)
    rk, rm = kaldi_io.read_feature_ark(d + "/out.ark")
    keep = {k: m for k, m in zip(rk, rm)}
    keep.update(counts=counts, prior_scale=np.float64(0.8), blank_scale=np.float64(0.5))
    path = os.path.join(outdir, "small_netout_refcpu.npz")
    np.savez_compressed(path, **keep)
    print("wrote", path, os.path.getsize(path), "bytes")


def run_dropout(outdir: str = HERE):
    """<wl>_drop_<variant>_refcpu.npz: one training step of the reference's CPU build with each dropout variant of
    BiLstmParallel; the fixture stores the masks the reference drew (they are random_device-seeded), the obj_diff
    that drove the backward pass and the reference's outputs."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from test_dropout_cpu import VARIANTS, drop_case, masks_from_dump
    for wl, variants in (("tiny", sorted(VARIANTS)), ("small", ["fwd+nml", "rnndropstep"])):
        for variant in variants:
            w, net, b = drop_case(wl, variant)
            lr, mom = 1e-3, 0.9
            d = tempfile.mkdtemp()
            kaldi_io.write_model(d + "/model", net)
            kaldi_io.write_batch_file(d + "/batch.bin", b)
            diff = (np.random.default_rng(1).standard_normal((b.feats.shape[0], w.classes)) * 0.1).astype(np.float32)
            rows_pad = np.concatenate([np.arange(b.frames[s], b.T) * b.S + s for s in range(b.S)]).astype(np.int64)
            diff[rows_pad] = 0.0
            np.save(d + "/diff.npy", diff)
            oracle.run_reference("cpu", d + "/model", d + "/batch.bin", d + "/out", lr, mom, steps=1, diff_in=d + "/diff.npy")
            dump = oracle.load_dump(d + "/out")
            m2 = kaldi_io.read_model(d + "/out/model_out")
            keep = {k: v for k, v in dump.items() if k.startswith(("grad_", "in_diff")) or k == f"out_l{len(net.layers)}"
                    or k == f"out_l{w.layers}"}
            for li, m in enumerate(masks_from_dump(dump, net, b)):
                if m:
                    for k, v in m.items():
                        keep[f"{k}_{li}"] = (v != 0).astype(np.uint8)    # 0/1 pattern; the scale 1/(1-p) is in the model
            keep.update(params_out=m2.flat_params(), diff_in=diff, hyper=np.array([lr, mom], np.float64),
                        meta=np.array([3, 5, 1], np.int64))
            path = os.path.join(outdir, f"{wl}_drop_{variant.replace('+', '_')}_refcpu.npz")
            np.savez_compressed(path, **keep)
            print("wrote", path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    if len(sys.argv) > 1 and sys.argv[1] == "dropcpu":
        run_dropout(sys.argv[2] if len(sys.argv) > 2 else HERE)
        sys.exit(0)
    if len(sys.argv) > 1 and sys.argv[1] == "infer":
        run_infer(sys.argv[2] if len(sys.argv) > 2 else HERE)
        sys.exit(0)
    if len(sys.argv) > 1 and sys.argv[1] == "adaptive":
        run_adaptive(sys.argv[2] if len(sys.argv) > 2 else HERE)
        sys.exit(0)
    kind = sys.argv[1] if len(sys.argv) > 1 else "cpu"
    if kind in ("unicpu", "unigpu"):
        run(kind[3:], sys.argv[2] if len(sys.argv) > 2 else HERE, uni=True)
        sys.exit(0)
    run(kind, sys.argv[2] if len(sys.argv) > 2 else HERE)
