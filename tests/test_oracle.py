"""CPU tests: pin the oracle (oracle/cpu_ref.c) before it is trusted as the checker.

1. against the committed golden vectors minted from the UNMODIFIED reference (tests/golden, see
   make_golden.py) -- CPU build for BiLSTM/affine/softmax/SGD, GPU build (when the fixture exists)
   for the CTC alpha/beta/pzx/diff the reference only computes on a GPU;
2. against stored runs of oracle/_ref/ref_dump_cpu (tests/util.py:stored_runs);
3. CTC against torch.nn.functional.ctc_loss in fp64 (independent third opinion, SURVEY.md 8c);
4. structural properties of the restatement itself.
"""
import os
import tempfile

import numpy as np
import pytest

from util import GOLDEN, assert_close, case, golden_arrays, stored_runs
from eesen_b200 import kaldi_io, synth
from oracle import oracle


def _oracle_two_steps(net, b, lr, mom, diff_override=None, dtype=np.float32):
    on = oracle.OracleNet(net, dtype)
    r = None
    for _ in range(2):
        r = on.train_step(b, lr, mom, diff_override=diff_override)
    return on, r


@pytest.mark.parametrize("wl", ["tiny", "small", "c1"])
def test_oracle_matches_reference_cpu_golden(wl):
    g = np.load(os.path.join(GOLDEN, f"{wl}_refcpu.npz"))
    mseed, bseed, steps = [int(v) for v in g["meta"]]
    lr, mom = [float(v) for v in g["hyper"]]
    assert steps == 2
    w, net, b = case(wl, mseed, bseed)
    on, r = _oracle_two_steps(net, b, lr, mom, diff_override=g["diff_in"])
    for i in range(1, len(net.layers) + 1):
        assert_close(f"out_l{i}", on.acts[i], g[f"out_l{i}"], atol=2e-6)
    assert_close("net_out", r["net_out"], g["net_out"], atol=2e-6)
    assert_close("in_diff", r["in_diff"], g["in_diff"], atol=1e-6, rtol=1e-4)
    assert_close("corr", on.flat_corr(), golden_arrays(g, net), atol=2e-5, rtol=1e-4)
    assert_close("params", on.flat_params(), g["params_out"], atol=1e-6)


@pytest.mark.parametrize("wl", ["tiny", "small", "c1"])
def test_oracle_matches_reference_gpu_golden(wl):
    """The reference's own CUDA CTC (and everything else) run on the B200 box."""
    path = os.path.join(GOLDEN, f"{wl}_refgpu.npz")
    if not os.path.exists(path):
        pytest.skip("GPU-minted golden not generated yet (tests/golden/make_golden.py gpu)")
    g = np.load(path)
    mseed, bseed, steps = [int(v) for v in g["meta"]]
    lr, mom = [float(v) for v in g["hyper"]]
    w, net, b = case(wl, mseed, bseed)
    on, r = _oracle_two_steps(net, b, lr, mom)
    # CTC outputs: fp32 alpha-beta sums carry ~1e-5 abs error in either implementation
    assert_close("pzx", r["pzx"], g["pzx"], atol=0, rtol=1e-5)
    assert_close("obj_diff", r["obj_diff"], g["obj_diff"], atol=1e-4)
    assert_close("net_out", r["net_out"], g["net_out"], atol=5e-6)
    assert_close("corr", on.flat_corr(), golden_arrays(g, net), atol=2e-3, rtol=2e-3)
    assert_close("params", on.flat_params(), g["params_out"], atol=5e-6)
    # alpha/beta lattices of the last step (valid cells only; log-zero cells are sentinels)
    y = r["net_out"]
    _, _, a, bt = oracle.ctc_eval(y, b.frames, b.labels, b.S, np.float32, want_ab=True)
    mask = (g["alpha"] > -1e29) & (a > -1e29)
    assert_close("alpha", a[mask], g["alpha"][mask], atol=1e-3, rtol=1e-5)
    mask = (g["beta"] > -1e29) & (bt > -1e29)
    assert_close("beta", bt[mask], g["beta"][mask], atol=1e-3, rtol=1e-5)
    assert np.array_equal(g["alpha"] > -1e29, a > -1e29)


@pytest.mark.parametrize("wl", ["tiny", "small"])
def test_oracle_lstm_parallel_matches_reference_cpu_golden(wl):
    """<LstmParallel> (uni-directional) stack against the reference's CPU build."""
    g = np.load(os.path.join(GOLDEN, f"{wl}_uni_refcpu.npz"))
    mseed, bseed, steps = [int(v) for v in g["meta"]]
    lr, mom = [float(v) for v in g["hyper"]]
    w, net, b = case(wl, mseed, bseed, bidirectional=False)
    assert [l.kind for l in net.layers][:w.layers] == ["lstm"] * w.layers
    on, r = _oracle_two_steps(net, b, lr, mom, diff_override=g["diff_in"])
    for i in range(1, len(net.layers) + 1):
        assert_close(f"out_l{i}", on.acts[i], g[f"out_l{i}"], atol=2e-6)
    assert_close("in_diff", r["in_diff"], g["in_diff"], atol=1e-6, rtol=1e-4)
    assert_close("corr", on.flat_corr(), golden_arrays(g, net), atol=2e-5, rtol=1e-4)
    assert_close("params", on.flat_params(), g["params_out"], atol=1e-6)


@pytest.mark.parametrize("wl", ["tiny", "small"])
def test_oracle_lstm_parallel_matches_reference_gpu_golden(wl):
    path = os.path.join(GOLDEN, f"{wl}_uni_refgpu.npz")
    if not os.path.exists(path):
        pytest.skip("GPU-minted golden not generated yet (tests/golden/make_golden.py unigpu)")
    g = np.load(path)
    mseed, bseed, steps = [int(v) for v in g["meta"]]
    lr, mom = [float(v) for v in g["hyper"]]
    w, net, b = case(wl, mseed, bseed, bidirectional=False)
    on, r = _oracle_two_steps(net, b, lr, mom)
    assert_close("pzx", r["pzx"], g["pzx"], atol=0, rtol=1e-5)
    assert_close("net_out", r["net_out"], g["net_out"], atol=5e-6)
    assert_close("corr", on.flat_corr(), golden_arrays(g, net), atol=2e-3, rtol=2e-3)
    assert_close("params", on.flat_params(), g["params_out"], atol=5e-6)


@pytest.mark.parametrize("opt", ["Adagrad", "RMSProp"])
@pytest.mark.parametrize("wl", ["tiny", "small"])
def test_oracle_adaptive_matches_reference_gpu_golden(wl, opt):
    """Adagrad/RMSProp exist only in the reference's GPU build: pinned on its output from the B200 box."""
    path = os.path.join(GOLDEN, f"{wl}_refgpu_{opt.lower()}.npz")
    if not os.path.exists(path):
        pytest.skip("GPU-minted golden not generated yet (tests/golden/make_golden.py adaptive)")
    g = np.load(path)
    mseed, bseed, steps = [int(v) for v in g["meta"]]
    lr, mom = [float(v) for v in g["hyper"]]
    w, net, b = case(wl, mseed, bseed)
    on = oracle.OracleNet(net, np.float32)
    on.set_optimizer(opt)
    for _ in range(steps):
        r = on.train_step(b, lr, mom)
    assert_close("pzx", r["pzx"], g["pzx"], atol=0, rtol=5e-5)
    assert_close("accu", on.flat_accu(), g["accus_out"], atol=1e-7, rtol=5e-3)
    assert_close("params", on.flat_params(), g["params_out"], atol=0.02 * lr)   # 2% of one adaptive step


def test_oracle_adaptive_rules_closed_form():
    """trainable-layer.h:65-114 on one tensor, against the formulas written out in numpy fp64."""
    rng = np.random.default_rng(4)
    L = oracle.lib(np.float64)
    import ctypes as C
    for mode, rho, omr in ((1, 0.9, 0.1), (2, 0.9, 0.1), (2, 0.7, 0.1)):
        w = rng.standard_normal(257); c = rng.standard_normal(257) * 3; a = rng.random(257)
        w0, c0, a0 = w.copy(), c.copy(), a.copy()
        L.lib.oracle_ada_update(C.c_long(257), L.p(w), L.p(c), L.p(a), L.real(0.01), L.real(2.0), L.real(1e-6),
                                L.real(rho), L.real(omr), mode)
        cc = np.clip(c0, -2.0, 2.0)
        aa = a0 + cc * cc if mode == 1 else rho * a0 + omr * cc * cc
        assert np.allclose(c, cc, rtol=0, atol=0) and np.allclose(a, aa, rtol=1e-15)
        assert np.allclose(w, w0 - 0.01 * cc / np.sqrt(aa + 1e-6), rtol=1e-14)


def onehot_argmax(y):
    """what the greedy token count reads of the posteriors: each row's argmax"""
    return np.eye(y.shape[1], dtype=y.dtype)[y.argmax(1)]


def test_oracle_matches_reference_cpu_live():
    w, net, b = case("small", 11, 12)
    lr, mom = 2e-3, 0.5
    on = oracle.OracleNet(net, np.float32)
    r = on.train_step(b, lr, mom)
    d = tempfile.mkdtemp()
    kaldi_io.write_model(d + "/model", net)
    kaldi_io.write_batch_file(d + "/batch.bin", b)
    np.save(d + "/diff.npy", r["obj_diff"].astype(np.float32))
    with stored_runs("small_cpu_step", d, keep=("out/out_l[1-9].npy", "out/in_diff.npy", "out/grad_*", "out/net_out.npy",
                                                "out/model_out"), transform={"out/net_out.npy": onehot_argmax}):
        info = oracle.run_reference("cpu", d + "/model", d + "/batch.bin", d + "/out", lr, mom, diff_in=d + "/diff.npy")
    ref = oracle.load_dump(d + "/out")
    # Ctc::ErrorRateMSeq (greedy path, collapse, Levenshtein: ctc-loss.cc:235-298) runs on the CPU build too
    err, nref = oracle.greedy_token_errors(ref["net_out"], b.frames, b.labels, b.S)
    assert (float(info["token_err"]), int(info["ref_tokens"])) == (float(err), int(nref))
    for i in range(1, len(net.layers) + 1):
        assert_close(f"out_l{i}", on.acts[i], ref[f"out_l{i}"], atol=2e-6, stored=True)
    assert_close("in_diff", r["in_diff"], ref["in_diff"], atol=1e-6, rtol=1e-4, stored=True)
    assert_close("corr", on.flat_corr(), golden_arrays(ref, net), atol=2e-5, rtol=1e-4, stored=True)
    m2 = kaldi_io.read_model(d + "/out/model_out")
    assert_close("params", on.flat_params(), m2.flat_params(), atol=1e-6, stored=True)


@pytest.mark.parametrize("wl,seed", [("tiny", 1), ("small", 2), ("mid", 3)])
def test_token_error_count_matches_reference(wl, seed):
    """Ctc::ErrorRateMSeq against the restated greedy decode + edit distance, on random-weight models whose greedy
    paths contain repeats, blanks and insertions (the statistics behind the recipes' TOKEN_ACCURACY line)."""
    w, net, b = case(wl, seed, seed + 100)
    for l in net.layers:                      # larger weights -> peaky posteriors -> non-trivial greedy paths
        for k in l.params:
            l.params[k] = (l.params[k] * 8).astype(np.float32)
    with tempfile.TemporaryDirectory() as d:
        kaldi_io.write_model(d + "/model", net)
        kaldi_io.write_batch_file(d + "/batch.bin", b)
        np.save(d + "/diff.npy", np.zeros((b.feats.shape[0], w.classes), np.float32))
        with stored_runs(f"{wl}_token_errors", d, keep=("out/net_out.npy",), transform={"out/net_out.npy": onehot_argmax}):
            info = oracle.run_reference("cpu", d + "/model", d + "/batch.bin", d + "/out", 0.0, 0.0,
                                        diff_in=d + "/diff.npy")
        y = oracle.load_dump(d + "/out")["net_out"]
    err, nref = oracle.greedy_token_errors(y, b.frames, b.labels, b.S)
    assert int(info["ref_tokens"]) == nref == sum(len(l) for l in b.labels)
    assert float(info["token_err"]) == float(err)
    am = y.argmax(1)
    assert len(np.unique(am)) > 2             # the decode really saw several symbols


def _torch_ctc(logits, frames, labels, S):
    import torch
    N, K = logits.shape
    T = N // S
    lt = torch.tensor(logits.reshape(T, S, K), dtype=torch.float64, requires_grad=True)
    lp = torch.log_softmax(lt, -1)
    tg = torch.tensor(np.concatenate(labels), dtype=torch.long)
    loss = torch.nn.functional.ctc_loss(lp, tg, torch.tensor(np.asarray(frames, np.int64)),
                                        torch.tensor([len(l) for l in labels]), blank=0, reduction="none")
    loss.sum().backward()
    return -loss.detach().numpy(), lt.grad.numpy().reshape(N, K)


@pytest.mark.parametrize("seed,S,T,K,maxlab", [(0, 3, 12, 5, 4), (1, 8, 40, 12, 10), (2, 1, 9, 4, 4), (3, 5, 30, 46, 14)])
def test_oracle_ctc_matches_torch_fp64(seed, S, T, K, maxlab):
    rng = np.random.default_rng(seed)
    frames = np.sort(rng.integers(max(2 * maxlab + 1, T // 2), T + 1, size=S))[::-1].astype(np.int32)
    frames[0] = T
    labels = []
    for s in range(S):
        n = int(rng.integers(1, maxlab + 1))
        lab = rng.integers(1, K, size=n)
        if n >= 2 and s % 2 == 0:
            lab[1] = lab[0]  # force a repeated label: no skip transition across the blank
        labels.append(lab.astype(np.int32))
    logits = rng.standard_normal((T * S, K)) * 2
    y = oracle.softmax(logits, np.float64)
    pzx, diff, _, _ = oracle.ctc_eval(y, frames, labels, S, np.float64)
    tp, tg = _torch_ctc(logits, frames, labels, S)
    assert_close("pzx", pzx, tp, atol=1e-9)
    assert_close("diff", diff, tg, atol=1e-9)
    # fp32 restatement against the fp64 arbiter: the algorithm's own fp32 error
    p32, d32, _, _ = oracle.ctc_eval(y.astype(np.float32), frames, labels, S, np.float32)
    assert_close("pzx32", p32, pzx, atol=0, rtol=2e-6)
    assert_close("diff32", d32, diff, atol=2e-4)


def test_oracle_ctc_properties():
    w, net, b = case("small")
    rng = np.random.default_rng(9)
    y = oracle.softmax(rng.standard_normal((b.feats.shape[0], w.classes)), np.float64)
    pzx, diff, a, bt = oracle.ctc_eval(y, b.frames, b.labels, b.S, np.float64, want_ab=True)
    assert np.all(pzx < 0)
    T = b.T
    for s in range(b.S):
        rows = np.arange(T) * b.S + s
        valid = rows[: b.frames[s]]
        # gradient wrt logits sums to zero on every valid row; padded rows are exactly zero
        assert np.abs(diff[valid].sum(1)).max() < 1e-12
        assert np.all(diff[rows[b.frames[s]:]] == 0)
        # sum_j alpha_t(j) beta_t(j) / y_t(l_j) = p(z|x) at every valid t
        L = 2 * len(b.labels[s]) + 1
        lab = np.zeros(L, np.int64)
        lab[1::2] = b.labels[s]
        for t in (0, b.frames[s] // 2, b.frames[s] - 1):
            r = t * b.S + s
            tot = np.logaddexp.reduce(a[r, :L] + bt[r, :L] - np.log(y[r, lab]))
            assert abs(tot - pzx[s]) < 1e-9


def test_oracle_padding_independence():
    """Valid-frame outputs and all gradients do not depend on the amount of padding (SURVEY.md 7.2)."""
    w, net, b = case("tiny")
    on = oracle.OracleNet(net, np.float64)
    r1 = on.train_step(b, 1e-3, 0.0)
    # re-pack the same utterances with 3 extra all-padding frames
    S, T = b.S, b.T
    feats2 = np.zeros(((T + 3) * S, b.feats.shape[1]), np.float32)
    feats2[: T * S] = b.feats
    b2 = kaldi_io.Batch(feats2, b.frames, b.labels)
    on2 = oracle.OracleNet(net, np.float64)
    r2 = on2.train_step(b2, 1e-3, 0.0)
    assert_close("pzx", r2["pzx"], r1["pzx"], atol=1e-12)
    assert_close("corr", on2.flat_corr(), on.flat_corr(), atol=1e-12)
    for s in range(S):
        rows = np.arange(b.frames[s]) * S + s
        assert_close("net_out", r2["net_out"][rows], r1["net_out"][rows], atol=1e-12)


def test_greedy_token_errors():
    y = np.zeros((6, 3))
    # S=1, path: 1 1 0 2 2 1 -> collapse -> 1 2 1
    for t, c in enumerate([1, 1, 0, 2, 2, 1]):
        y[t, c] = 1.0
    err, ref = oracle.greedy_token_errors(y, [6], [np.array([1, 2, 2])], 1)
    assert (err, ref) == (1, 3)
