"""CPU tests: the C-ABI library loads and exports every symbol include/eesen_b200.h declares, the
product fails loudly without a GPU (no CPU fallback), and the host-side formats/batching logic."""
import ctypes as C
import os
import re
import subprocess
import tempfile

import numpy as np
import pytest

from util import ROOT, case, stored_runs
from eesen_b200 import binding, kaldi_io, synth

HEADER = os.path.join(ROOT, "include", "eesen_b200.h")


def _declared_symbols():
    src = open(HEADER).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(eesen_b200_[a-z0-9_]+)\s*\(", src)))


def _has_gpu():
    try:
        import torch
        return torch.cuda.is_available()
    except Exception:
        return False


def test_library_exports_every_declared_symbol():
    if not os.path.exists(binding.LIB_PATH):
        import __graft_entry__
        __graft_entry__.build()
    lib = C.CDLL(binding.LIB_PATH)
    syms = _declared_symbols()
    assert len(syms) >= 25
    missing = [s for s in syms if not hasattr(lib, s)]
    assert not missing, f"declared in include/eesen_b200.h but not exported: {missing}"


def test_no_cpu_fallback_create_fails_without_gpu():
    if _has_gpu():
        pytest.skip("GPU present")
    lib = binding.load_library()
    h = C.c_void_p()
    rc = lib.eesen_b200_create(C.byref(h), 0)
    assert rc != 0 and not h.value
    msg = lib.eesen_b200_last_error(None).decode()
    assert "no CPU fallback" in msg
    with pytest.raises(binding.EesenB200Error):
        binding.Context(0)


def test_product_does_not_import_oracle():
    """Only tests/, __graft_entry__.smoke() and bench.py's CPU arm may touch oracle/."""
    pkg = os.path.join(ROOT, "eesen_b200")
    for dp, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cc", ".cu", ".h", ".cuh")):
                txt = open(os.path.join(dp, f), errors="ignore").read()
                assert "from oracle" not in txt and "import oracle" not in txt and "cpu_ref" not in txt, f
    mk = open(os.path.join(ROOT, "Makefile")).read()
    assert "cpu_ref" not in mk


def test_model_roundtrip_and_layout():
    w, net, b = case("tiny")
    with tempfile.TemporaryDirectory() as d:
        p = os.path.join(d, "m")
        kaldi_io.write_model(p, net)
        raw = open(p, "rb").read()
        assert raw.startswith(b"\0B<Nnet> <BiLstmParallel> <InputDim> \x04")
        assert raw.rstrip().endswith(b"</Nnet>")
        net2 = kaldi_io.read_model(p)
    assert [l.kind for l in net2.layers] == [l.kind for l in net.layers]
    assert np.array_equal(net.flat_params(), net2.flat_params())
    assert net.num_params() == sum(int(np.prod(s)) for l in net.layers for s in l.param_shapes().values())
    # WriteData order (bilstm-layer.h:478-492)
    assert net.layers[0].param_names() == ["wx_fw", "wm_fw", "b_fw", "pi_fw", "pf_fw", "po_fw",
                                           "wx_bw", "wm_bw", "b_bw", "pi_bw", "pf_bw", "po_bw"]


def test_model_accumulators_roundtrip():
    """<BiLstmAccus>/<AffineAccus> sit between the option tokens and the weights (bilstm-layer.h:375-395,458-475)."""
    w, net, b = case("tiny")
    rng = np.random.default_rng(1)
    for l in net.layers:
        for n, shp in l.param_shapes().items():
            l.accus[n] = rng.random(shp).astype(np.float32)
    with tempfile.TemporaryDirectory() as d:
        p = os.path.join(d, "m")
        kaldi_io.write_model(p, net)
        raw = open(p, "rb").read()
        assert raw.index(b"<TwiddleForward>") < raw.index(b"<BiLstmAccus>") < raw.index(b"<AffineTransform>")
        assert raw.count(b"<BiLstmAccus>") == sum(l.kind == "bilstm" for l in net.layers)
        assert raw.count(b"<AffineAccus>") == 1
        net2 = kaldi_io.read_model(p)
    assert np.array_equal(net.flat_params(), net2.flat_params())
    assert np.array_equal(net.flat_accus(), net2.flat_accus())


def test_reference_reads_and_rewrites_our_accumulators():
    """The reference's Net::Read accepts the accumulator blocks we write and its Net::Write puts them back
    byte for byte (SGD leaves them alone), so the two writers agree on the format."""
    from oracle import oracle
    w, net, b = case("tiny")
    rng = np.random.default_rng(2)
    for l in net.layers:
        for n, shp in l.param_shapes().items():
            l.accus[n] = rng.random(shp).astype(np.float32)
    with tempfile.TemporaryDirectory() as d:
        kaldi_io.write_model(d + "/model", net)
        kaldi_io.write_batch_file(d + "/batch.bin", b)
        diff = np.zeros((b.feats.shape[0], w.classes), np.float32)
        np.save(d + "/diff.npy", diff)
        with stored_runs("tiny_accus_rewrite", d, keep=("out/model_out",)):
            oracle.run_reference("cpu", d + "/model", d + "/batch.bin", d + "/out", 0.0, 0.0, steps=1,
                                 diff_in=d + "/diff.npy")
        assert open(d + "/out/model_out", "rb").read() == open(d + "/model", "rb").read()


def test_reads_model_written_by_reference_net_initialize():
    """Byte-compatibility with the reference's own model factory (src/netbin/net-initialize.cc)."""
    from oracle import oracle
    with tempfile.TemporaryDirectory() as d:
        proto = os.path.join(d, "proto")
        with open(proto, "w") as f:
            f.write("<Nnet>\n<BiLstmParallel> <InputDim> 40 <CellDim> 32 <ParamRange> 0.1 <LearnRateCoef> 1.0 <MaxGrad> 50.0\n"
                    "<AffineTransform> <InputDim> 32 <OutputDim> 6 <ParamRange> 0.1\n"
                    "<Softmax> <InputDim> 6 <OutputDim> 6\n</Nnet>\n")
        out = os.path.join(d, "nnet.init")
        with stored_runs("net_initialize", d, sample=False):
            r = oracle.run_reference_tool("ref_net_initialize", ["--binary=true", proto, out])
        assert r.returncode == 0, r.stderr[-2000:]
        net = kaldi_io.read_model(out)
        assert [l.kind for l in net.layers] == ["bilstm", "affine", "softmax"]
        assert net.layers[0].cells == 16 and net.layers[0].max_grad == 50.0
        assert net.layers[0].params["wx_fw"].shape == (64, 40)
        assert np.abs(net.flat_params()).max() <= 0.1 + 1e-6
        # and our writer reproduces the file byte for byte
        again = os.path.join(d, "again")
        kaldi_io.write_model(again, net)
        assert open(again, "rb").read() == open(out, "rb").read()


def test_pack_utterances_time_major_interleaved():
    rng = np.random.default_rng(0)
    utts = [rng.standard_normal((5, 3)).astype(np.float32), rng.standard_normal((3, 3)).astype(np.float32)]
    feats, frames = kaldi_io.pack_utterances(utts)
    assert feats.shape == (10, 3) and list(frames) == [5, 3]
    for s, u in enumerate(utts):
        for t in range(u.shape[0]):
            assert np.array_equal(feats[t * 2 + s], u[t])     # row r = t*S + s
    assert np.all(feats[3 * 2 + 1] == 0) and np.all(feats[4 * 2 + 1] == 0)   # zero padding


def test_workload_shapes_match_baseline_configs():
    c2 = synth.WORKLOADS["c2"]
    assert (c2.layers, c2.cells, c2.in_dim, c2.classes, c2.S) == (4, 320, 40, 46, 64)
    net = synth.make_model(c2)
    assert net.num_params() == 8341806            # SURVEY.md section 8e
    assert abs(synth.flops_per_frame(c2) / 1e6 - 49.94) < 0.01
    assert abs(synth.hbm_bytes_per_frame(c2, 60) / 1e3 - 374.7) < 0.1
    b = synth.make_batch(synth.WORKLOADS["c1"], seed=0)
    assert list(b.frames) == [50, 37] and b.S == 2


def test_feature_and_label_archives(tmp_path):
    keys = ["utt1", "utt2"]
    utts = [np.arange(6, dtype=np.float32).reshape(2, 3), np.ones((1, 3), np.float32)]
    kaldi_io.write_feature_ark(str(tmp_path / "f.ark"), keys, utts)
    raw = open(tmp_path / "f.ark", "rb").read()
    assert raw.startswith(b"utt1 \0BFM \x04\x02\x00\x00\x00\x04\x03\x00\x00\x00")
    kaldi_io.write_label_ark(str(tmp_path / "l.ark"), keys, [[1, 2], [3]])
    assert open(tmp_path / "l.ark").read() == "utt1 1 2\nutt2 3\n"


def test_reference_driver_reads_our_archives_and_reports_the_same_accuracy():
    """The reference's own driver (CPU build, --cross-validate: forward + ErrorRateMSeq only) on the feature / label
    archives and the model our writers produce: it must read them, skip what it skips (an utterance without
    targets, one above --frame-limit) and print the TOKEN_ACCURACY the restatement computes for the rest."""
    import re
    from oracle import oracle
    w, net, b = case("small", 5, 6)
    for l in net.layers:
        for k in l.params:
            l.params[k] = (l.params[k] * 8).astype(np.float32)
    utts = [b.feats[np.arange(b.frames[s]) * b.S + s] for s in range(b.S)]
    labels = [list(map(int, l)) for l in b.labels]
    keys = [f"utt{i:02d}" for i in range(b.S)]
    limit = int(sorted(b.frames)[-2])                   # the longest utterance alone exceeds --frame-limit
    longest = int(np.argmax(b.frames))
    no_target = (longest + 1) % b.S
    with tempfile.TemporaryDirectory() as d:
        kaldi_io.write_model(d + "/model", net)
        kaldi_io.write_feature_ark(d + "/feats.ark", keys, utts)
        kaldi_io.write_label_ark(d + "/labels.ark", [k for i, k in enumerate(keys) if i != no_target],
                                 [l for i, l in enumerate(labels) if i != no_target])
        with stored_runs("small_reference_driver_cross_validate", d):
            r = oracle.run_reference_tool("ref_train_ctc_parallel",
                                          ["--cross-validate=true", "--num-sequence=3", f"--frame-limit={limit}",
                                           "--report-step=1000", f"ark:{d}/feats.ark", f"ark,t:{d}/labels.ark", d + "/model"],
                                          timeout=600, threads=4)
    assert r.returncode == 0, r.stderr[-3000:]
    log = r.stdout + r.stderr
    acc = float(re.search(r"TOKEN_ACCURACY >> ([-0-9.e+]+)% <<", log).group(1))
    assert "missing targets" in log and "has too many frames" in log
    used = [i for i in range(b.S) if i not in (no_target, longest)]
    assert re.search(rf"Done {len(used)} files, 1 with no targets", log), log[-1500:]
    on = oracle.OracleNet(net, np.float32)
    err = ref = 0
    for i in used:                                       # utterance by utterance: results do not depend on the packing
        y = on.forward(utts[i], np.array([utts[i].shape[0]], np.int32))
        e, n = oracle.greedy_token_errors(y, [utts[i].shape[0]], [np.asarray(labels[i])], 1)
        err += e; ref += n
    assert abs(acc - 100.0 * (1.0 - err / ref)) < 1e-3


def test_profile_categories_agree_between_header_and_binding():
    """include/eesen_b200.h and the ctypes stub must size the eesen_b200_profile arrays alike (9 categories: index 8 is
    the dense work of the side stream)."""
    src = open(HEADER).read()
    n = int(re.search(r"#define\s+EESEN_B200_NUM_PROFILE_CATEGORIES\s+(\d+)", src).group(1))
    assert n == len(binding.Context.PROFILE_CATEGORIES) == 9
    assert binding.Context.PROFILE_CATEGORIES[0] == "gemm" and binding.Context.PROFILE_CATEGORIES[8] == "gemm_side"


def test_trace_summary_reads_a_launch_trace(tmp_path):
    """tests/trace_summary.py on a hand-written EESEN_B200_TRACE_FILE block (host/context.h:prof_collect format:
    stream, category, start ms, duration ms): busy time per stream and category, idle time of the main stream."""
    import sys
    p = tmp_path / "trace.txt"
    p.write_text("# collect: 2 launches\n0 0 0.0 0.1\n1 8 0.0 0.5\n"
                 "# collect: 4 launches\n0 0 0.000 0.100\n0 1 0.150 1.000\n1 8 0.120 0.700\n0 2 1.200 1.500\n")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "trace_summary.py"), str(p)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    out = r.stdout
    assert "4 launches, span 2.700 ms" in out                      # only the LAST block counts
    assert "'gemm': 0.1" in out and "'lstm_fwd': 1.0" in out and "'lstm_bwd': 1.5" in out
    assert "side busy: {'gemm_side': 0.7}" in out
    assert "idle between launches 0.100 ms" in out                 # 0.05 before lstm_fwd + 0.05 before lstm_bwd
