"""CPU tests of the forward-only path (SURVEY.md 8f N2): pin the restatement of
net-output-extract (Net::Feedforward + ApplyLog + ClassPrior) against the reference's own CPU tool,
through stored runs of that tool and through the committed fixture."""
import os
import tempfile

import numpy as np
import pytest

from util import GOLDEN, assert_close, case, stored_runs
from eesen_b200 import binding, kaldi_io, synth
from oracle import oracle

def infer_case(wl="small", mseed=3, bseed=9):
    """Model + ragged utterances + class counts (one class below the cutoff) for the inference tests."""
    w, net, b = case(wl, mseed, bseed)
    utts = [b.feats[np.arange(b.frames[s]) * b.S + s] for s in range(b.S)]
    rng = np.random.default_rng(7)
    counts = rng.integers(50, 5000, size=w.classes).astype(np.float64)
    counts[0] *= 20          # blanks dominate
    counts[-1] = 0.0         # never seen: masked with FLT_MAX/2
    return w, net, b, utts, counts


def test_class_log_priors_restatement_vs_abi():
    rng = np.random.default_rng(0)
    for cutoff, bs in ((1e-10, 1.0), (100.0, 0.5), (1e-10, 0.25)):
        counts = rng.integers(0, 3000, size=46).astype(np.float64)
        a = oracle.class_log_priors(counts, cutoff, bs)
        got = binding.class_log_priors(counts, cutoff, bs)
        big = a > 1e30
        assert np.array_equal(big, got > 1e30) and big.sum() == (counts < cutoff).sum()
        assert_close("log priors", got[~big], a[~big], atol=1e-6)


@pytest.mark.parametrize("nonparallel", [False, True])
def test_oracle_matches_reference_net_output_extract_live(nonparallel):
    w, net, b, utts, counts = infer_case()
    with tempfile.TemporaryDirectory() as d, \
            stored_runs(f"small_net_output_extract{'_nonparallel' if nonparallel else ''}", d, sample=False):
        kaldi_io.write_model(d + "/model", net)
        model = d + "/model"
        if nonparallel:
            oracle.run_reference_tool("ref_format_to_nonparallel", [model, d + "/model.np"])
            raw = open(d + "/model.np", "rb").read()
            assert b"<BiLstmParallel>" not in raw and raw.count(b"<BiLstm>") == w.layers
            assert len(raw) == len(open(model, "rb").read()) - len("Parallel") * w.layers
            model = d + "/model.np"
        keys = [f"utt{i:02d}" for i in range(len(utts))]
        kaldi_io.write_feature_ark(d + "/feats.ark", keys, utts)
        open(d + "/counts", "w").write("[ " + " ".join(repr(float(c)) for c in counts) + " ]\n")
        oracle.run_reference_tool("ref_net_output_extract",
                                  ["--apply-log=true", f"--class-frame-counts={d}/counts", "--prior-scale=0.8",
                                   "--blank-scale=0.5", model, f"ark:{d}/feats.ark", f"ark:{d}/out.ark"], threads=4)
        rk, rm = kaldi_io.read_feature_ark(d + "/out.ark")
    assert rk == keys
    lp = oracle.class_log_priors(counts, 1e-10, 0.5)
    on = oracle.OracleNet(net, np.float32)
    y = oracle.net_output(on, b.feats, b.frames, True, lp, 0.8)      # ONE packed batch
    for s, m in enumerate(rm):
        mine = y[np.arange(b.frames[s]) * b.S + s]
        assert m.shape == mine.shape
        masked = lp > 1e30
        assert np.all(m[:, masked] < -1e37) and np.all(mine[:, masked] < -1e37)
        assert_close(f"loglik {keys[s]}", mine[:, ~masked], m[:, ~masked], atol=2e-5, rtol=1e-5)


def test_oracle_matches_reference_net_output_extract_golden():
    path = os.path.join(GOLDEN, "small_netout_refcpu.npz")
    if not os.path.exists(path):
        pytest.skip("fixture not generated (tests/golden/make_golden.py infer)")
    g = np.load(path)
    w, net, b, utts, counts = infer_case()
    assert np.array_equal(counts, g["counts"])
    lp = oracle.class_log_priors(counts, 1e-10, float(g["blank_scale"]))
    on = oracle.OracleNet(net, np.float32)
    y = oracle.net_output(on, b.feats, b.frames, True, lp, float(g["prior_scale"]))
    masked = lp > 1e30
    for s in range(b.S):
        mine = y[np.arange(b.frames[s]) * b.S + s]
        assert_close(f"loglik utt{s}", mine[:, ~masked], g[f"utt{s:02d}"][:, ~masked], atol=2e-5, rtol=1e-5)
