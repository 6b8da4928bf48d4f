"""GPU parity of the forward-only path (SURVEY.md 8f N2) through the C ABI and the command-line tools:
net-output-extract (Net::Feedforward + ApplyLog + ClassPrior::SubtractOnLogpost) and format-to-nonparallel."""
import os
import subprocess
import tempfile

import numpy as np
import pytest

from util import GOLDEN, ROOT, assert_close, model_file, stored_runs
from test_inference_cpu import infer_case
from eesen_b200 import binding, kaldi_io
from oracle import oracle

pytestmark = pytest.mark.gpu
BIN = os.path.join(ROOT, "eesen_b200", "bin")


@pytest.fixture(scope="module")
def ctx():
    c = binding.Context(0)
    yield c
    c.close()


def _rows(y, b, s):
    return y[np.arange(b.frames[s]) * b.S + s]


def test_feedforward_vs_oracle_and_reference_fixture(ctx):
    w, net, b, utts, counts = infer_case()
    lp = binding.class_log_priors(counts, 1e-10, 0.5)
    n = binding.Net(ctx, model_file(net))
    y = n.feedforward(b.feats, b.frames, True, lp, 0.8)
    on = oracle.OracleNet(net, np.float64)
    ref = oracle.net_output(on, b.feats, b.frames, True, oracle.class_log_priors(counts, 1e-10, 0.5), 0.8)
    masked = lp > 1e30
    assert masked.sum() == 1
    for s in range(b.S):
        got = _rows(y, b, s)
        assert np.all(got[:, masked] < -1e37)
        assert_close(f"loglik utt{s} vs fp64", got[:, ~masked], _rows(ref, b, s)[:, ~masked], atol=2e-5, rtol=1e-5)
    g = np.load(os.path.join(GOLDEN, "small_netout_refcpu.npz"))     # the reference's own tool, CPU build
    for s in range(b.S):
        assert_close(f"loglik utt{s} vs reference", _rows(y, b, s)[:, ~masked], g[f"utt{s:02d}"][:, ~masked],
                     atol=3e-5, rtol=1e-5)
    # plain posteriors (no log, no prior) are what Net::Feedforward returns
    p = n.feedforward(b.feats, b.frames)
    for s in range(b.S):
        assert_close("posteriors", _rows(p, b, s), _rows(on.forward(b.feats, b.frames), b, s), atol=2e-6)
    n.close()


def test_feedforward_packing_independence(ctx):
    """One utterance at a time (the reference's call pattern) == the packed batch, on valid frames."""
    w, net, b, utts, counts = infer_case()
    n = binding.Net(ctx, model_file(net))
    y = n.feedforward(b.feats, b.frames, True)
    for s in (0, 3, b.S - 1):
        one = n.feedforward(utts[s], np.array([utts[s].shape[0]], np.int32), True)
        assert_close(f"utt{s} alone vs packed", one, _rows(y, b, s), atol=2e-5, rtol=1e-5)
    n.close()


def _run(cmd):
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr[-3000:]
    return r


def test_format_to_nonparallel_and_extract_tools(ctx, tmp_path):
    w, net, b, utts, counts = infer_case()
    d = str(tmp_path)
    kaldi_io.write_model(d + "/model", net)
    keys = [f"utt{i:02d}" for i in range(len(utts))]
    kaldi_io.write_feature_ark(d + "/feats.ark", keys, utts)
    open(d + "/counts", "w").write("[ " + " ".join(repr(float(c)) for c in counts) + " ]\n")
    # marker rewrite: bytes equal to the parallel model with the marker replaced
    _run([BIN + "/format-to-nonparallel", d + "/model", d + "/model.np"])
    raw, rnp = open(d + "/model", "rb").read(), open(d + "/model.np", "rb").read()
    assert rnp == raw.replace(b"<BiLstmParallel>", b"<BiLstm>")
    with stored_runs("small_format_to_nonparallel", d):
        oracle.run_reference_tool("ref_format_to_nonparallel", [d + "/model", d + "/model.ref"])
    assert rnp == open(d + "/model.ref", "rb").read()
    # the tool on both model flavours, small batches so that several packed passes happen
    outs = {}
    for tag, model in (("par", d + "/model"), ("np", d + "/model.np")):
        _run([BIN + "/net-output-extract", "--apply-log=true", f"--class-frame-counts={d}/counts", "--prior-scale=0.8",
              "--blank-scale=0.5", "--num-sequence=3", model, f"ark:{d}/feats.ark", f"ark,scp:{d}/{tag}.ark,{d}/{tag}.scp"])
        k, m = kaldi_io.read_feature_ark(f"{d}/{tag}.ark")
        assert k == keys
        outs[tag] = m
        scp = [l.split() for l in open(f"{d}/{tag}.scp")]
        assert [x[0] for x in scp] == keys
        data = open(f"{d}/{tag}.ark", "rb").read()
        for key, loc in scp:                       # scp offsets point at the "\0B" header of each entry
            off = int(loc.rsplit(":", 1)[1])
            assert data[off:off + 2] == b"\0B" and data[off - len(key) - 1:off - 1] == key.encode()
    g = np.load(os.path.join(GOLDEN, "small_netout_refcpu.npz"))
    lp = binding.class_log_priors(counts, 1e-10, 0.5)
    ok = ~(lp > 1e30)
    for s, key in enumerate(keys):
        assert np.array_equal(outs["par"][s], outs["np"][s])
        assert_close(f"tool {key} vs reference", outs["par"][s][:, ok], g[key][:, ok], atol=3e-5, rtol=1e-5)
    # --num-sequence=1 is the reference's own call pattern
    _run([BIN + "/net-output-extract", "--apply-log=true", "--num-sequence=1", d + "/model.np", f"ark:{d}/feats.ark",
          f"ark:{d}/one.ark"])
    _run([BIN + "/net-output-extract", "--apply-log=true", d + "/model.np", f"ark:{d}/feats.ark", f"ark:{d}/all.ark"])
    k1, m1 = kaldi_io.read_feature_ark(d + "/one.ark")
    k2, m2 = kaldi_io.read_feature_ark(d + "/all.ark")
    assert k1 == k2 == keys
    for a, c in zip(m1, m2):
        assert_close("one-by-one vs packed", a, c, atol=2e-5, rtol=1e-5)


def test_nonparallel_model_without_lengths_is_one_sequence(ctx):
    """<BiLstm> + Net::Propagate without SetSeqLengths: the whole matrix is ONE sequence (bilstm-layer.h:548)."""
    w, net, b, utts, counts = infer_case()
    p = model_file(net)
    n = binding.Net(ctx, p)
    n.write_nonparallel(p + ".np")
    n2 = binding.Net(ctx, p + ".np")
    assert np.array_equal(n.params(), n2.params())
    u = utts[1]
    n2.feedforward(b.feats, b.frames)                       # leave packed lengths behind ...
    a = n2.feedforward(u, None)                             # ... which a length-less call must not reuse
    on = oracle.OracleNet(net, np.float64)
    assert_close("single sequence", a, on.forward(u, np.array([u.shape[0]], np.int32)), atol=2e-6)
    with pytest.raises(binding.EesenB200Error):             # the parallel layer needs its lengths, as in the reference
        n.feedforward(u, None)
    n.close(); n2.close()
