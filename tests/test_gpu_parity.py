"""GPU parity tests (run with -m gpu on the B200 box).  Everything goes through the C ABI
(include/eesen_b200.h) via eesen_b200.binding; the checker is the oracle (oracle/), the committed
golden vectors minted from the reference, and stored runs of the reference's own gpucompute build
(oracle/_ref/ref_dump_gpu, compiled from the unmodified sources for sm_100a; tests/util.py:stored_runs).

Stated tolerances (fp32 storage everywhere):
  default arithmetic "fp32x3" (3xTF32 split, fp32 accumulate): fp32-faithful
      log p(z|x)          rel 2e-5      (north_star bound: 1e-4)
      per-frame gradient  abs 1e-4 + 2e-6*|log p(z|x)|   (alpha+beta live in the log domain at magnitude
                          |log p|, where one fp32 ulp is ~1e-7*|log p|; the reference's own fp32 CTC is
                          4e-5 .. 5e-4 away from fp64 on these cases, tests/test_oracle.py)
      layer outputs       abs 2e-5
      momentum buffers    abs 2e-3 + rel 2e-3 (sums over thousands of rows, order-dependent)
  "tf32" arithmetic: log p(z|x) rel 1e-4 (still inside the north_star bound), gradients abs 5e-3.
"""
import os
import tempfile

import numpy as np
import pytest

from util import GOLDEN, assert_close, case, golden_arrays, model_file, stored_runs
from eesen_b200 import binding, kaldi_io, synth
from oracle import oracle

pytestmark = pytest.mark.gpu


def diff_atol(pzx):
    """stated per-frame gradient tolerance (see header)"""
    return 1e-4 + 2e-6 * float(np.abs(pzx).max())


def torch_():
    import torch
    return torch


# ------------------------------------------------------------------------------------ level 1
@pytest.mark.parametrize("ta,tb,M,N,K", [(0, 1, 300, 96, 40), (0, 1, 130, 46, 64), (0, 0, 257, 40, 128),
                                         (0, 0, 64, 640, 46), (1, 0, 128, 40, 700), (1, 0, 46, 64, 5000),
                                         (1, 0, 1280, 320, 9000)])
@pytest.mark.parametrize("prec,tol", [("fp32x3", 5e-6), ("tf32", 2e-3), ("bf16", 1.5e-2)])
def test_gemm(ctx, ta, tb, M, N, K, prec, tol):
    torch = torch_()
    rng = np.random.default_rng(M + N + K)
    ld = lambda c: (c + 3) // 4 * 4
    Ash = (K, M) if ta else (M, K)
    Bsh = (N, K) if tb else (K, N)
    A = np.zeros((Ash[0], ld(Ash[1])), np.float32); A[:, :Ash[1]] = rng.standard_normal(Ash)
    B = np.zeros((Bsh[0], ld(Bsh[1])), np.float32); B[:, :Bsh[1]] = rng.standard_normal(Bsh)
    A[:, Ash[1]:] = np.nan  # padding columns must never be read
    B[:, Bsh[1]:] = np.nan
    C0 = rng.standard_normal((M, ld(N))).astype(np.float32)
    dA, dB, dC = torch.from_numpy(A).cuda(), torch.from_numpy(B).cuda(), torch.from_numpy(C0).cuda()
    torch.cuda.synchronize()
    ctx.set_precision(prec, "fp32x3")
    ctx.gemm(ta, tb, M, N, K, 0.5, dA, A.shape[1], dB, B.shape[1], 0.25, dC, C0.shape[1])
    ctx.synchronize()
    ctx.set_precision("fp32x3", "fp32x3")
    a = A[:, :Ash[1]].astype(np.float64); b = B[:, :Bsh[1]].astype(np.float64)
    ref = 0.5 * ((a.T if ta else a) @ (b.T if tb else b)) + 0.25 * C0[:, :N]
    got = dC.cpu().numpy()
    scale = np.sqrt(K)
    if prec == "fp32x3" and K >= 512:
        tol = 2.5e-5   # fp32 accumulation in TMEM over long K (tensor-core accumulate rounding), ~6e-6 relative
    assert_close("gemm", got[:, :N] / scale, ref / scale, atol=tol)
    assert np.array_equal(got[:, N:], C0[:, N:])   # padding columns of C untouched
    if prec == "bf16":
        # the bf16 mode is tcgen05 kind::f16 on round-to-nearest-even bf16 copies of the operands with fp32
        # accumulation: against the exact product of the ROUNDED operands only the accumulation order is left
        r16 = lambda x: torch.from_numpy(np.ascontiguousarray(x)).to(torch.bfloat16).to(torch.float64).numpy()
        a = r16(A[:, :Ash[1]]); b = r16(B[:, :Bsh[1]])
        ref16 = 0.5 * ((a.T if ta else a) @ (b.T if tb else b)) + 0.25 * C0[:, :N]
        assert_close("gemm_bf16_rounded_operands", got[:, :N] / scale, ref16 / scale, atol=2.5e-5 if K >= 512 else 5e-6)


@pytest.mark.parametrize("N,K", [(7, 5), (1000, 46), (333, 300)])
def test_softmax_and_argmax(ctx, N, K):
    torch = torch_()
    rng = np.random.default_rng(N)
    ldp = (K + 3) // 4 * 4
    x = np.zeros((N, ldp), np.float32); x[:, :K] = rng.standard_normal((N, K)) * 3
    dx = torch.from_numpy(x).cuda()
    dy = torch.full((N, ldp), 7.0, dtype=torch.float32, device="cuda")
    da = torch.zeros(N, dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    ctx.softmax(N, K, dx, ldp, dy, ldp, da)
    ctx.synchronize()
    ref = oracle.softmax(x[:, :K], np.float64)
    got = dy.cpu().numpy()
    assert_close("softmax", got[:, :K], ref, atol=2e-7)
    assert np.all(got[:, K:] == 0)
    assert np.array_equal(da.cpu().numpy(), np.argmax(x[:, :K], 1))


def _ctc_case(seed, S, T, K, maxlab, ragged=True):
    rng = np.random.default_rng(seed)
    frames = np.full(S, T, np.int32)
    if ragged:
        frames = np.sort(rng.integers(max(2 * maxlab + 1, T // 2), T + 1, size=S))[::-1].astype(np.int32)
        frames[0] = T
    labels = []
    for s in range(S):
        n = int(rng.integers(1, maxlab + 1))
        lab = rng.integers(1, K, size=n)
        if n >= 2 and s % 2 == 0:
            lab[1] = lab[0]
        labels.append(lab.astype(np.int32))
    labels[0] = rng.integers(1, K, size=maxlab).astype(np.int32)   # one utterance at the maximum label length
    if S >= 3:
        labels[2] = np.zeros(0, np.int32)   # empty transcription: only the all-blank path (|l| = 0, L' = 1)
    logits = (rng.standard_normal((T * S, K)) * 2).astype(np.float32)
    return frames, labels, logits


@pytest.mark.parametrize("seed,S,T,K,maxlab", [(0, 3, 12, 5, 4), (1, 8, 40, 12, 10), (2, 1, 9, 4, 1), (3, 5, 64, 46, 15),
                                               (4, 64, 120, 46, 31), (5, 4, 300, 32, 60), (6, 2, 700, 32, 130),
                                               (7, 3, 1100, 8, 255)])
def test_ctc_eval_vs_oracle(ctx, seed, S, T, K, maxlab):
    torch = torch_()
    frames, labels, logits = _ctc_case(seed, S, T, K, maxlab)
    ldp = (K + 3) // 4 * 4
    y = oracle.softmax(logits, np.float32)
    yp = np.zeros((T * S, ldp), np.float32); yp[:, :K] = y
    lab = np.zeros((S, maxlab), np.int32)
    for s, l in enumerate(labels):
        lab[s, :len(l)] = l
    d_y = torch.from_numpy(yp).cuda()
    d_len = torch.from_numpy(frames).cuda()
    d_lab = torch.from_numpy(lab).cuda()
    d_ll = torch.tensor([len(l) for l in labels], dtype=torch.int32, device="cuda")
    d_pzx = torch.zeros(S, dtype=torch.float32, device="cuda")
    d_diff = torch.full((T * S, ldp), 3.0, dtype=torch.float32, device="cuda")
    torch.cuda.synchronize()
    ctx.ctc_eval(T, S, K, maxlab, d_len, d_lab, d_ll, d_y, ldp, d_pzx, d_diff, ldp)
    ctx.synchronize()
    pzx64, diff64, _, _ = oracle.ctc_eval(y.astype(np.float64), frames, labels, S, np.float64)
    got_p, got_d = d_pzx.cpu().numpy(), d_diff.cpu().numpy()
    assert_close("pzx", got_p, pzx64, atol=0, rtol=2e-5)
    assert_close("diff", got_d[:, :K], diff64, atol=diff_atol(pzx64))
    for s in range(S):   # rows past the utterance end are exactly zero
        rows = np.arange(frames[s], T) * S + s
        assert np.all(got_d[rows, :K] == 0)


@pytest.mark.parametrize("S,T,I,C", [(4, 9, 8, 16), (2, 30, 40, 128), (20, 17, 40, 64), (16, 40, 40, 320), (3, 5, 64, 24),
                                     (100, 7, 40, 320), (1, 1, 40, 64),    # 100 utts: two utterance chunks (64 + 36)
                                     (4, 11, 40, 192), (3, 9, 40, 384),    # backward tile mixes: 128 + stacked 64; 3 x 128
                                     (3, 7, 40, 512), (18, 6, 40, 448),    # wide plans (C4's 512 cells): W_lo' partly / tiles 3-4 in smem
                                     (8, 300, 40, 64), (6, 290, 40, 320),  # T >= 256: input product streamed in chunks
                                     (3, 9, 40, 256), (40, 21, 40, 256)])  # full tiles only + ragged last group (cluster exchange)
@pytest.mark.parametrize("rec", ["fp32x3", "tf32", "legacy-engine", "tcfwd-engine", "l2-exchange"])
def test_bilstm_layer_vs_oracle(ctx, S, T, I, C, rec, monkeypatch):
    """Level-1 BiLSTM forward/backward of one layer against the fp64 oracle, ragged lengths.  Shapes with
    cells % 64 == 0 run on the tcgen05 recurrent kernels (lstm_tc.cu), the others -- and every shape under
    EESEN_B200_LSTM_ENGINE=legacy -- on the warp-level kernels (lstm.cu): same tolerances for both."""
    torch = torch_()
    monkeypatch.delenv("EESEN_B200_LSTM_EXCHANGE", raising=False)
    if rec in ("legacy-engine", "tcfwd-engine"):   # default: tcgen05 for both passes (lstm.cu:engine_for_pass)
        if C % 64 != 0:
            pytest.skip("only the warp-level kernels take this shape")
        monkeypatch.setenv("EESEN_B200_LSTM_ENGINE", rec.split("-")[0])
        rec = "fp32x3"
    elif rec == "l2-exchange":   # default for cells <= 384: thread-block clusters exchanging through DSMEM (lstm_tc.cu, CL = 1)
        if C % 64 != 0 or C > 384:
            pytest.skip("the cluster exchange does not apply to this shape")
        monkeypatch.delenv("EESEN_B200_LSTM_ENGINE", raising=False)
        monkeypatch.setenv("EESEN_B200_LSTM_EXCHANGE", "l2")
        rec = "fp32x3"
    else:
        monkeypatch.delenv("EESEN_B200_LSTM_ENGINE", raising=False)
    rng = np.random.default_rng(S * 1000 + T)
    frames = np.sort(rng.integers(max(1, T // 2), T + 1, size=S))[::-1].astype(np.int32)
    frames[0] = T
    x = rng.standard_normal((T * S, I)).astype(np.float32)
    for s in range(S):
        x[np.arange(frames[s], T) * S + s] = 0
    l = kaldi_io.LayerSpec("bilstm", I, 2 * C)
    # U(-0.3, 0.3) is 3x the model's init range; over hundreds of steps a 320-cell recurrence with such weights is
    # chaotic (rounding differences grow exponentially in ANY fp32 implementation), so the long shapes use the init range
    wr = 0.3 if T <= 100 else 0.1
    params = [rng.uniform(-wr, wr, size=l.param_shapes()[n]).astype(np.float32) for n in l.param_names()]
    dout = rng.standard_normal((T * S, 2 * C)).astype(np.float32)
    for s in range(S):
        dout[np.arange(frames[s], T) * S + s] = 0   # upper layers hand back zero gradient on padded rows
    # oracle (fp64)
    L = oracle.lib(np.float64)
    p64 = [L.arr(p) for p in params]
    bf = np.zeros(((T + 2) * S, 7 * C)); bb = np.zeros_like(bf); out64 = np.zeros((T * S, 2 * C))
    L.lib.oracle_bilstm_forward(T, S, I, C, L.p(frames), L.p(L.arr(x)), L.pp(p64), L.p(bf), L.p(bb), L.p(out64))
    corr = [np.zeros_like(p) for p in p64]
    dbf = np.zeros_like(bf); dbb = np.zeros_like(bf); dx64 = np.zeros((T * S, I))
    L.lib.oracle_bilstm_backward(T, S, I, C, L.p(L.arr(x)), L.pp(p64), L.p(bf), L.p(bb), L.p(L.arr(dout)), L.p(dbf),
                                 L.p(dbb), L.p(dx64), L.pp(corr), L.real(0.0))
    # device
    dp = [torch.from_numpy(p).cuda() for p in params]
    dg = [torch.full_like(p, 9.0) for p in dp]
    d_x = torch.from_numpy(x).cuda(); d_len = torch.from_numpy(frames).cuda()
    gates = torch.empty((T * S, 8 * C), device="cuda"); cell = torch.empty((T * S, 2 * C), device="cuda")
    out = torch.empty((T * S, 2 * C), device="cuda"); dgates = torch.empty((T * S, 8 * C), device="cuda")
    d_dout = torch.from_numpy(dout).cuda(); dx = torch.empty((T * S, I), device="cuda")
    torch.cuda.synchronize()
    ctx.set_precision("fp32x3", rec)
    ctx.bilstm_forward(T, S, I, C, d_len, d_x, I, dp, gates, cell, out, 2 * C)
    ctx.bilstm_backward(T, S, I, C, d_x, I, dp, gates, cell, out, 2 * C, d_dout, 2 * C, dgates, dx, I, dg)
    ctx.synchronize()
    ctx.set_precision("fp32x3", "fp32x3")
    tol = 1.0 if rec == "fp32x3" else 500.0   # weights here are U(-0.3, 0.3): 3x the model init range
    assert_close("out", out.cpu().numpy(), out64, atol=1e-5 * tol)
    # saved state: cols of the reference's 7-block buffers (g,i,f,o | c)
    g_fw = gates.cpu().numpy()[:, :4 * C]; g_bw = gates.cpu().numpy()[:, 4 * C:]
    assert_close("gates_fw", g_fw, bf[S:(T + 1) * S, :4 * C], atol=1e-5 * tol)
    assert_close("gates_bw", g_bw, bb[S:(T + 1) * S, :4 * C], atol=1e-5 * tol)
    assert_close("cell_fw", cell.cpu().numpy()[:, :C], bf[S:(T + 1) * S, 4 * C:5 * C], atol=2e-5 * tol)
    assert_close("dgates_fw", dgates.cpu().numpy()[:, :4 * C], dbf[S:(T + 1) * S, :4 * C], atol=2e-5 * tol, rtol=1e-4)
    assert_close("dgates_bw", dgates.cpu().numpy()[:, 4 * C:], dbb[S:(T + 1) * S, :4 * C], atol=2e-5 * tol, rtol=1e-4)
    assert_close("dx", dx.cpu().numpy(), dx64, atol=5e-5 * tol, rtol=1e-4)
    for k, n in enumerate(l.param_names()):
        scale = max(1.0, np.abs(corr[k]).max())
        assert_close(f"grad_{n}", dg[k].cpu().numpy() / scale, corr[k] / scale, atol=2e-5 * tol)
    # padding semantics (bilstm-parallel-layer.h:201-204): backward cells are zero past the end, forward are not
    for s in range(S):
        rows = np.arange(frames[s], T) * S + s
        if len(rows):
            assert np.all(out.cpu().numpy()[rows, C:] == 0)
            assert np.all(dgates.cpu().numpy()[rows] == 0)


@pytest.mark.parametrize("S,T,I,C", [(16, 12, 40, 64), (5, 9, 40, 24)])
def test_bilstm_pitched_weights_bind_without_repacking(ctx, S, T, I, C):
    """The reference's CuMatrix weights are cudaMallocPitch'ed (cuda-matrix.cc:46-79): wx / wm (and their gradient
    matrices) with a row stride > cols must give the same bits as the dense layout (ldwx / ldwm of the ABI structs),
    on both recurrent engines."""
    torch = torch_()
    rng = np.random.default_rng(11)
    frames = np.sort(rng.integers(max(1, T // 2), T + 1, size=S))[::-1].astype(np.int32); frames[0] = T
    x = rng.standard_normal((T * S, I)).astype(np.float32)
    l = kaldi_io.LayerSpec("bilstm", I, 2 * C)
    params = [rng.uniform(-0.3, 0.3, size=l.param_shapes()[n]).astype(np.float32) for n in l.param_names()]
    dout = rng.standard_normal((T * S, 2 * C)).astype(np.float32)
    d_x = torch.from_numpy(x).cuda(); d_len = torch.from_numpy(frames).cuda(); d_dout = torch.from_numpy(dout).cuda()
    ldwx, ldwm = I + 4, C + 8     # 16-byte aligned pitches, as cudaMallocPitch returns

    def run(pitched):
        dp, dg, views = [], [], []
        for p, n in zip(params, l.param_names()):
            if pitched and p.ndim == 2:
                ld = ldwx if p.shape[1] == I and "wx" in n else ldwm
                big = torch.full((p.shape[0], ld), float("nan"), device="cuda")
                big[:, :p.shape[1]] = torch.from_numpy(p).cuda()
                gbig = torch.full((p.shape[0], ld), 7.0, device="cuda")
                dp.append(big); dg.append(gbig); views.append(gbig[:, :p.shape[1]])
            else:
                dp.append(torch.from_numpy(p).cuda()); g = torch.full(p.shape, 9.0, device="cuda"); dg.append(g); views.append(g)
        gates = torch.empty((T * S, 8 * C), device="cuda"); cell = torch.empty((T * S, 2 * C), device="cuda")
        out = torch.empty((T * S, 2 * C), device="cuda"); dgates = torch.empty((T * S, 8 * C), device="cuda")
        dx = torch.empty((T * S, I), device="cuda")
        torch.cuda.synchronize()
        kw = dict(ldwx=ldwx, ldwm=ldwm) if pitched else {}
        ctx.bilstm_forward(T, S, I, C, d_len, d_x, I, dp, gates, cell, out, 2 * C, **kw)
        kwb = dict(ldwx=ldwx, ldwm=ldwm, gldwx=ldwx, gldwm=ldwm) if pitched else {}
        ctx.bilstm_backward(T, S, I, C, d_x, I, dp, gates, cell, out, 2 * C, d_dout, 2 * C, dgates, dx, I, dg, **kwb)
        ctx.synchronize()
        if pitched:   # the padding columns of the gradient matrices are never written
            for gb, p in zip(dg, params):
                if p.ndim == 2:
                    assert torch.all(gb[:, p.shape[1]:] == 7.0)
        return [out.cpu().numpy(), dx.cpu().numpy()] + [v.cpu().numpy().copy() for v in views]

    dense, pitched = run(False), run(True)
    for a, b in zip(dense, pitched):
        assert_close("pitched_vs_dense", b, a, atol=2e-6)


def test_sgd_update_segments(ctx):
    torch = torch_()
    rng = np.random.default_rng(0)
    n = 1003
    w = rng.standard_normal(n).astype(np.float32); c = rng.standard_normal(n).astype(np.float32) * 3
    g = rng.standard_normal(n).astype(np.float32) * 3
    segs = [(0, 501, 0.1, 2.0), (501, 502, 0.05, 0.0)]
    dw, dc, dg = (torch.from_numpy(a.copy()).cuda() for a in (w, c, g))
    torch.cuda.synchronize()
    ctx.sgd_update(dw, dc, dg, n, 0.9, segs)
    ctx.synchronize()
    cref = g + np.float32(0.9) * c
    cref[:501] = np.clip(cref[:501], -2.0, 2.0)
    wref = w.copy(); wref[:501] -= np.float32(0.1) * cref[:501]; wref[501:] -= np.float32(0.05) * cref[501:]
    assert_close("corr", dc.cpu().numpy(), cref, atol=1e-6)
    assert_close("w", dw.cpu().numpy(), wref, atol=1e-6)


# ------------------------------------------------------------------------------------ level 2
def _gpu_steps(ctx, net, b, lr, mom, steps, want_in_diff=True):
    n = binding.Net(ctx, model_file(net))
    n.set_train_options(lr, mom)
    if want_in_diff:
        n.get(102)
    st = None
    for _ in range(steps):
        st = n.train_step(b.feats, b.frames, b.labels, True)
    return n, st


@pytest.mark.parametrize("wl", ["tiny", "small", "mid"])
def test_train_step_vs_oracle(ctx, wl):
    w, net, b = case(wl)
    lr, mom = 1e-3, 0.9
    n, st = _gpu_steps(ctx, net, b, lr, mom, 1)
    on = oracle.OracleNet(net, np.float64)
    ro = on.train_step(b, lr, mom)
    for i in range(1, len(net.layers) + 1):
        assert_close(f"out_l{i}", n.get(i), on.acts[i], atol=2e-5)
    assert_close("pzx", n.get(101).ravel(), ro["pzx"], atol=0, rtol=2e-5)
    assert abs(st["obj"] - ro["pzx"].sum()) <= 2e-5 * abs(ro["pzx"].sum())
    assert_close("obj_diff", n.get(100), ro["obj_diff"], atol=diff_atol(ro["pzx"]))
    assert_close("in_diff", n.get(102), ro["in_diff"], atol=2e-5, rtol=1e-3)
    assert_close("corr", n.corr(), on.flat_corr(), atol=2e-3, rtol=2e-3)
    assert_close("params", n.params(), on.flat_params(), atol=2e-6)
    err, ref = oracle.greedy_token_errors(ro["net_out"], b.frames, b.labels, b.S)
    assert (st["token_err"], st["ref_tokens"], st["frames"]) == (err, ref, b.valid_frames)
    # second step exercises the momentum carry
    st2 = n.train_step(b.feats, b.frames, b.labels, True)
    ro2 = on.train_step(b, lr, mom)
    assert abs(st2["obj"] - ro2["pzx"].sum()) <= 5e-5 * abs(ro2["pzx"].sum())
    assert_close("params2", n.params(), on.flat_params(), atol=5e-6)
    n.close()


@pytest.mark.parametrize("wl", ["tiny", "small", "c1"])
@pytest.mark.parametrize("kind", ["cpu", "gpu"])
def test_train_step_vs_reference_golden(ctx, wl, kind):
    """Against the committed outputs of the UNMODIFIED reference (tests/golden/make_golden.py)."""
    path = os.path.join(GOLDEN, f"{wl}_ref{kind}.npz")
    if not os.path.exists(path):
        pytest.skip(f"{path} not generated")
    g = np.load(path)
    mseed, bseed, steps = [int(v) for v in g["meta"]]
    lr, mom = [float(v) for v in g["hyper"]]
    w, net, b = case(wl, mseed, bseed)
    n, st = _gpu_steps(ctx, net, b, lr, mom, steps)
    if kind == "gpu":   # the reference's own CUDA CTC drove both steps, as ours did
        assert_close("pzx", n.get(101).ravel(), g["pzx"], atol=0, rtol=2e-5)
        assert_close("obj_diff", n.get(100), g["obj_diff"], atol=diff_atol(g["pzx"]))
        assert_close("params", n.params(), g["params_out"], atol=5e-6)
        assert_close("corr", n.corr(), golden_arrays(g, net), atol=2e-3, rtol=2e-3)
        for i in range(1, len(net.layers) + 1):
            assert_close(f"out_l{i}", n.get(i), g[f"out_l{i}"], atol=2e-5)
    else:
        # CPU reference has no CTC: its backward was driven by a stored diff, so only the forward of
        # step 1 is comparable end to end; compare the first-step forward
        n1, _ = _gpu_steps(ctx, net, b, lr, mom, 0)
        n1.train_step(b.feats, b.frames, b.labels, False)
        g1 = oracle.OracleNet(net, np.float32)
        g1.forward(b.feats, b.frames)
        for i in range(1, len(net.layers) + 1):
            assert_close(f"out_l{i}", n1.get(i), g1.acts[i], atol=2e-5)
        n1.close()
    n.close()


# what the comparisons with ref_dump_gpu read of its output directory, and the cells the stored runs keep of each
# compared tensor (spread over every utterance and every weight matrix; the momentum buffers, grad_*, count as one).
# log p(z|x) is kept whole.
REF_STEP_OUTPUTS = ("out/pzx.npy", "out/net_out.npy", "out/obj_diff.npy", "out/in_diff.npy", "out/grad_*", "out/model_out")
REF_STEP_CELLS = {"small": 1024, "mid": 2048}
REF_FULL_SIZE_OUTPUTS = ("out/pzx.npy", "out/net_out.npy", "out/obj_diff.npy", "out/model_out")
REF_FULL_SIZE_CELLS = {"out/net_out.npy": 3072, "out/obj_diff.npy": 3072, "out/model_out": 3072}


@pytest.mark.parametrize("wl,steps", [("small", 2), ("mid", 1)])
def test_train_step_vs_reference_gpucompute_live(ctx, wl, steps):
    """Same inputs through the reference's own gpucompute kernels (compiled for sm_100a) on this GPU."""
    w, net, b = case(wl, 21, 22)
    lr, mom = 1e-3, 0.9
    d = tempfile.mkdtemp()
    kaldi_io.write_model(d + "/model", net)
    kaldi_io.write_batch_file(d + "/batch.bin", b)
    with stored_runs(f"{wl}_gpucompute_{steps}steps", d, keep=REF_STEP_OUTPUTS, whole=("out/pzx.npy",),
                     cells={p: REF_STEP_CELLS[wl] for p in REF_STEP_OUTPUTS[1:]}):
        oracle.run_reference("gpu", d + "/model", d + "/batch.bin", d + "/out", lr, mom, steps=steps)
    ref = oracle.load_dump(d + "/out")
    n, st = _gpu_steps(ctx, net, b, lr, mom, steps)
    assert_close("pzx", n.get(101).ravel(), ref["pzx"], atol=0, rtol=2e-5)      # north_star: 1e-4 relative
    assert_close("net_out", n.get(len(net.layers)), ref["net_out"], atol=2e-5, stored=True)
    assert_close("obj_diff", n.get(100), ref["obj_diff"], atol=diff_atol(ref["pzx"]), stored=True)
    assert_close("in_diff", n.get(102), ref["in_diff"], atol=2e-5, rtol=1e-3, stored=True)
    assert_close("corr", n.corr(), golden_arrays(ref, net), atol=2e-3, rtol=2e-3, stored=True)
    m2 = kaldi_io.read_model(d + "/out/model_out")
    assert_close("params", n.params(), m2.flat_params(), atol=5e-6, stored=True)
    n.close()


# ------------------------------------------------------------------------------------ LstmParallel (uni-directional)
@pytest.mark.parametrize("wl", ["tiny", "small", "mid"])
def test_lstm_parallel_train_step_vs_oracle(ctx, wl):
    """<LstmParallel> stack (lstm-parallel-layer.h): the forward cells alone, nothing masked."""
    w, net, b = case(wl, bidirectional=False)
    lr, mom = 1e-3, 0.9
    n, st = _gpu_steps(ctx, net, b, lr, mom, 1)
    on = oracle.OracleNet(net, np.float64)
    ro = on.train_step(b, lr, mom)
    for i in range(1, len(net.layers) + 1):
        assert_close(f"out_l{i}", n.get(i), on.acts[i], atol=2e-5)
    assert_close("pzx", n.get(101).ravel(), ro["pzx"], atol=0, rtol=2e-5)
    assert_close("obj_diff", n.get(100), ro["obj_diff"], atol=diff_atol(ro["pzx"]))
    assert_close("in_diff", n.get(102), ro["in_diff"], atol=2e-5, rtol=1e-3)
    assert_close("corr", n.corr(), on.flat_corr(), atol=2e-3, rtol=2e-3)
    assert_close("params", n.params(), on.flat_params(), atol=2e-6)
    n.train_step(b.feats, b.frames, b.labels, True)
    on.train_step(b, lr, mom)
    assert_close("params2", n.params(), on.flat_params(), atol=5e-6)
    n.close()


@pytest.mark.parametrize("wl", ["tiny", "small"])
def test_lstm_parallel_vs_reference_golden(ctx, wl):
    path = os.path.join(GOLDEN, f"{wl}_uni_refgpu.npz")
    if not os.path.exists(path):
        pytest.skip(f"{path} not generated")
    g = np.load(path)
    mseed, bseed, steps = [int(v) for v in g["meta"]]
    lr, mom = [float(v) for v in g["hyper"]]
    w, net, b = case(wl, mseed, bseed, bidirectional=False)
    n, st = _gpu_steps(ctx, net, b, lr, mom, steps)
    assert_close("pzx", n.get(101).ravel(), g["pzx"], atol=0, rtol=2e-5)
    assert_close("obj_diff", n.get(100), g["obj_diff"], atol=diff_atol(g["pzx"]))
    assert_close("params", n.params(), g["params_out"], atol=5e-6)
    assert_close("corr", n.corr(), golden_arrays(g, net), atol=2e-3, rtol=2e-3)
    for i in range(1, len(net.layers) + 1):
        assert_close(f"out_l{i}", n.get(i), g[f"out_l{i}"], atol=2e-5)
    n.close()


def test_lstm_parallel_vs_reference_gpucompute_live_and_model_bytes(ctx):
    """Live against the reference's GPU build with Adagrad, incl. the model file.  The reference stores the
    WEIGHTS a second time under <LstmAccus> (lstm-layer.h:153-163, a bug: a reloaded model then takes
    sqrt(weight + eps)); our writer keeps the same byte layout but stores the real accumulators."""
    w, net, b = case("small", 21, 22, bidirectional=False)
    lr, mom = 1e-3, 0.9
    d = tempfile.mkdtemp()
    kaldi_io.write_model(d + "/model", net)
    kaldi_io.write_batch_file(d + "/batch.bin", b)
    with stored_runs("small_uni_gpucompute_adagrad", d, keep=("out/model_out",)):
        oracle.run_reference("gpu", d + "/model", d + "/batch.bin", d + "/out", lr, mom, steps=2, opt="Adagrad")
    m2 = kaldi_io.read_model(d + "/out/model_out")
    n = _adaptive_steps(ctx, net, b, lr, mom, "Adagrad", 2)
    assert_close("params", n.params(), m2.flat_params(), atol=_ada_atol(lr), stored=True)
    n.write(d + "/ours_out", True)
    ours = kaldi_io.read_model(d + "/ours_out")
    for lo, lt in zip(ours.layers, m2.layers):
        if lo.kind == "lstm":
            for k in lo.param_names():      # theirs: <LstmAccus> block == the weights block; ours: the accumulators
                assert np.array_equal(lt.accus[k], lt.params[k], equal_nan=True)
                assert lo.accus[k].shape == lo.params[k].shape and (lo.accus[k] >= 0).all()
            assert any(not np.array_equal(lo.accus[k], lo.params[k]) for k in lo.param_names())
    assert len(open(d + "/ours_out", "rb").read()) == len(open(d + "/out/model_out", "rb").read())
    n.close()


def test_lstm_nonparallel_marker_and_feedforward(ctx):
    w, net, b = case("tiny", bidirectional=False)
    p = model_file(net)
    n = binding.Net(ctx, p)
    n.write_nonparallel(p + ".np")
    assert open(p + ".np", "rb").read() == open(p, "rb").read().replace(b"<LstmParallel>", b"<Lstm>")
    n2 = binding.Net(ctx, p + ".np")
    y = n.feedforward(b.feats, b.frames, True)
    on = oracle.OracleNet(net, np.float64)
    ref = np.log(on.forward(b.feats, b.frames))
    s = 1
    rows = np.arange(b.frames[s]) * b.S + s
    assert_close("packed", y[rows], ref[rows], atol=2e-5, rtol=1e-5)
    u = b.feats[rows]
    assert_close("<Lstm> one sequence", n2.feedforward(u, None, True), y[rows], atol=2e-5, rtol=1e-5)
    n.close(); n2.close()


# ------------------------------------------------------------------------------------ Adagrad / RMSProp
def _adaptive_steps(ctx, net, b, lr, mom, opt, steps, model_path=None, **kw):
    n = binding.Net(ctx, model_path or model_file(net))
    n.set_train_options(lr, mom)
    n.set_optimizer(opt, **kw)
    for _ in range(steps):
        n.train_step(b.feats, b.frames, b.labels, True)
    return n


# the adaptive step lr*c/sqrt(accu+eps) has slope <= lr/sqrt(eps) = 1e3*lr in c: a momentum-buffer
# difference of 1e-6 (fp32 reduction order) may move a parameter by 1e-3*lr*... -> budget 2% of one step
def _ada_atol(lr):
    return 0.02 * lr


@pytest.mark.parametrize("opt", ["Adagrad", "RMSProp"])
@pytest.mark.parametrize("wl", ["tiny", "small"])
def test_adaptive_update_vs_oracle(ctx, wl, opt):
    """Net::SetUpdateAlgorithm(Adagrad|RMSProp): three steps against the fp64 restatement."""
    w, net, b = case(wl)
    lr, mom = 2e-3, 0.5
    n = _adaptive_steps(ctx, net, b, lr, mom, opt, 3)
    on = oracle.OracleNet(net, np.float64)
    on.set_optimizer(opt)
    for _ in range(3):
        on.train_step(b, lr, mom)
    assert_close("accu", n.accu(), on.flat_accu(), atol=1e-7, rtol=5e-3)
    assert_close("params", n.params(), on.flat_params(), atol=_ada_atol(lr))
    moved = np.abs(on.flat_params() - net.flat_params()).max()
    assert moved > 1.5 * lr          # the rule really is adaptive: ~lr per step whatever the gradient scale
    n.close()


def test_adaptive_options_and_learn_rate_coef(ctx):
    """eps / rho / one_minus_rho are honoured; learn_rate_coef is ignored by the adaptive branch
    (bilstm-layer.h:865-869 vs :885-955) while max_grad still clips."""
    w, net, b = case("tiny")
    for l in net.layers:
        if l.kind != "softmax":
            l.learn_rate_coef, l.max_grad = 0.25, 0.01
    lr, mom = 1e-3, 0.9
    n = _adaptive_steps(ctx, net, b, lr, mom, "RMSProp", 2, adagrad_epsilon=1e-4, rmsprop_rho=0.8,
                        rmsprop_one_minus_rho=0.3)
    on = oracle.OracleNet(net, np.float64)
    on.set_optimizer("RMSProp", 1e-4, 0.8, 0.3)
    for _ in range(2):
        on.train_step(b, lr, mom)
    assert_close("accu", n.accu(), on.flat_accu(), atol=1e-9, rtol=5e-3)
    assert_close("params", n.params(), on.flat_params(), atol=_ada_atol(lr))
    assert np.abs(n.corr()).max() <= 0.01 + 1e-9
    n.close()


@pytest.mark.parametrize("opt", ["adagrad", "rmsprop"])
@pytest.mark.parametrize("wl", ["tiny", "small"])
def test_adaptive_update_vs_reference_golden(ctx, wl, opt):
    """Against the committed output of the reference's GPU build run with --opt-algorithm (make_golden.py adaptive)."""
    path = os.path.join(GOLDEN, f"{wl}_refgpu_{opt}.npz")
    if not os.path.exists(path):
        pytest.skip(f"{path} not generated")
    g = np.load(path)
    mseed, bseed, steps = [int(v) for v in g["meta"]]
    lr, mom = [float(v) for v in g["hyper"]]
    w, net, b = case(wl, mseed, bseed)
    n = _adaptive_steps(ctx, net, b, lr, mom, {"adagrad": "Adagrad", "rmsprop": "RMSProp"}[opt], steps)
    assert_close("pzx", n.get(101).ravel(), g["pzx"], atol=0, rtol=5e-5)
    assert_close("accu", n.accu(), g["accus_out"], atol=1e-7, rtol=5e-3)
    assert_close("params", n.params(), g["params_out"], atol=_ada_atol(lr))
    n.close()


@pytest.mark.parametrize("opt", ["Adagrad", "RMSProp"])
def test_adaptive_update_vs_reference_gpucompute_live(ctx, opt):
    w, net, b = case("small", 21, 22)
    lr, mom = 1e-3, 0.9
    d = tempfile.mkdtemp()
    kaldi_io.write_model(d + "/model", net)
    kaldi_io.write_batch_file(d + "/batch.bin", b)
    with stored_runs(f"small_gpucompute_{opt.lower()}", d, keep=("out/model_out",)):
        oracle.run_reference("gpu", d + "/model", d + "/batch.bin", d + "/out", lr, mom, steps=3, opt=opt)
    m2 = kaldi_io.read_model(d + "/out/model_out")
    n = _adaptive_steps(ctx, net, b, lr, mom, opt, 3)
    assert_close("accu", n.accu(), m2.flat_accus(), atol=1e-7, rtol=5e-3, stored=True)
    assert_close("params", n.params(), m2.flat_params(), atol=_ada_atol(lr), stored=True)
    # the model we write carries the accumulators where the reference puts them: the reference's own
    # writer and ours agree token for token (same length, same tokens; payload compared above)
    out = d + "/ours_out"
    n.write(out, True)
    ours, theirs = open(out, "rb").read(), open(d + "/out/model_out", "rb").read()
    assert len(ours) == len(theirs) and ours.count(b"<BiLstmAccus>") == theirs.count(b"<BiLstmAccus>") == sum(
        l.kind == "bilstm" for l in net.layers) and ours.count(b"<AffineAccus>") == theirs.count(b"<AffineAccus>") == 1
    n.close()


def test_adaptive_resume_from_written_model(ctx):
    """Accumulators survive Net::Write -> Net::Read (the reference resumes Adagrad across epochs this way;
    momentum buffers are NOT stored, so the check uses momentum 0)."""
    w, net, b = case("tiny")
    lr = 1e-3
    full = _adaptive_steps(ctx, net, b, lr, 0.0, "Adagrad", 4)
    half = _adaptive_steps(ctx, net, b, lr, 0.0, "Adagrad", 2)
    p = model_file(net) + ".half"
    half.write(p, True)
    m = kaldi_io.read_model(p)
    assert_close("accus in file", m.flat_accus(), half.accu(), atol=0)
    rest = _adaptive_steps(ctx, net, b, lr, 0.0, "Adagrad", 2, model_path=p)
    assert np.array_equal(rest.params(), full.params()) and np.array_equal(rest.accu(), full.accu())
    # SGD on a model that carries accumulators keeps and re-writes them untouched (adaBuffersInitialized)
    sgd = binding.Net(ctx, p)
    sgd.set_train_options(lr, 0.0)
    sgd.train_step(b.feats, b.frames, b.labels, True)
    assert np.array_equal(sgd.accu(), half.accu())
    sgd.write(p + ".sgd", True)
    assert_close("accus kept", kaldi_io.read_model(p + ".sgd").flat_accus(), half.accu(), atol=0)
    for x in (full, half, rest, sgd):
        x.close()


def test_model_write_is_byte_compatible(ctx):
    w, net, b = case("tiny")
    p = model_file(net)
    n = binding.Net(ctx, p)
    out = p + ".out"
    n.write(out, True)
    assert open(out, "rb").read() == open(p, "rb").read()        # Net::Write(Net::Read(x)) == x
    txt = p + ".txt"
    n.write(txt, False)
    n2 = binding.Net(ctx, txt)                                     # text mode round trip
    assert_close("text", n2.params(), n.params(), atol=1e-6)
    n.close(); n2.close()


def test_tf32_mode_within_north_star_tolerance(ctx):
    w, net, b = case("mid")
    ctx.set_precision("tf32", "tf32")
    try:
        n, st = _gpu_steps(ctx, net, b, 1e-3, 0.9, 1)
    finally:
        ctx.set_precision("fp32x3", "fp32x3")
    on = oracle.OracleNet(net, np.float64)
    ro = on.train_step(b, 1e-3, 0.9)
    assert_close("pzx", n.get(101).ravel(), ro["pzx"], atol=0, rtol=1e-4)
    assert_close("obj_diff", n.get(100), ro["obj_diff"], atol=5e-3)
    n.close()


# ------------------------------------------------------------------------------------ full size (C2)
@pytest.fixture(scope="module")
def c2_run(ctx):
    w = synth.WORKLOADS["c2"]
    net = synth.make_model(w, seed=0)
    b = synth.make_batch(w, seed=1)
    n = binding.Net(ctx, model_file(net))
    n.set_train_options(w.learn_rate, w.momentum)
    st = n.train_step(b.feats, b.frames, b.labels, True)
    yield w, net, b, n, st
    n.close()


def test_c2_full_size_properties(ctx, c2_run):
    """BASELINE configs[1] at full size: size-independent properties of the result."""
    w, net, b, n, st = c2_run
    diff = n.get(100)
    y = n.get(len(net.layers))
    pzx = n.get(101).ravel()
    assert st["frames"] == b.valid_frames and np.isfinite(st["obj"]) and np.all(pzx < 0)
    T, S = b.T, b.S
    valid = np.zeros(T * S, bool)
    for s in range(S):
        valid[np.arange(b.frames[s]) * S + s] = True
    assert np.abs(y.sum(1) - 1).max() < 1e-5                      # softmax rows
    assert np.abs(diff[valid].sum(1)).max() < 2e-5                # CTC gradient rows sum to zero
    assert np.all(diff[~valid] == 0)                              # padded rows exactly zero
    # the CTC of the full-size posteriors against the fp64 oracle (CTC alone is cheap on the CPU)
    p64, d64, _, _ = oracle.ctc_eval(y.astype(np.float64), b.frames, b.labels, S, np.float64)
    assert_close("pzx", pzx, p64, atol=0, rtol=2e-5)
    assert_close("diff", diff, d64, atol=diff_atol(p64))
    # backward cells of the last BiLSTM layer are zero on padded rows; forward cells are not masked
    top = n.get(len(net.layers) - 2)
    assert np.all(top[~valid][:, w.cells:] == 0) and np.abs(top[~valid][:, :w.cells]).max() > 0
    assert np.all(np.isfinite(n.params()))


def test_c2_full_size_deterministic(ctx, c2_run):
    """Two independent runs of the same step are bit-identical (fixed reduction orders, no atomics
    on the data path)."""
    w, net, b, n, st = c2_run
    n2 = binding.Net(ctx, model_file(net))
    n2.set_train_options(w.learn_rate, w.momentum)
    st2 = n2.train_step(b.feats, b.frames, b.labels, True)
    assert st2["obj"] == st["obj"]
    assert np.array_equal(n2.params(), n.params())
    n2.close()


def test_c2_stream_knobs_give_the_same_step(ctx, c2_run, monkeypatch):
    """The stream-level schedules are pure reorderings: the streamed dX of the recurrent backward pass (opt-in,
    EESEN_B200_STREAM_DX=1: chunk pairs behind flags on the side stream, the kernel of the layer below waits per chunk),
    planes of x / m made early on the side stream (default) or behind the kernel, everything on one stream
    (EESEN_B200_OVERLAP=0) -- all give the parameters of the default schedule after one C2 step (row-chunked GEMMs
    compute every output row exactly as the whole product does; only the split-K weight-gradient sums are shared)."""
    w, net, b, n, st = c2_run
    ref = n.params()
    for env in ({"EESEN_B200_STREAM_DX": "1"}, {"EESEN_B200_STREAM_DX": "1", "EESEN_B200_DX_READY": "2", "EESEN_B200_EARLY_CONV": "0"},
                {"EESEN_B200_OVERLAP": "0"}):
        for k in ("EESEN_B200_STREAM_DX", "EESEN_B200_DX_READY", "EESEN_B200_EARLY_CONV", "EESEN_B200_OVERLAP"):
            monkeypatch.delenv(k, raising=False)
        for k, v in env.items():
            monkeypatch.setenv(k, v)
        c2 = binding.Context(0)          # the knobs are read when a context is created
        n2 = binding.Net(c2, model_file(net))
        n2.set_train_options(w.learn_rate, w.momentum)
        st2 = n2.train_step(b.feats, b.frames, b.labels, True)
        assert st2["obj"] == st["obj"], env
        assert np.abs(n2.params() - ref).max() <= 1e-7, (env, np.abs(n2.params() - ref).max())
        n2.close()
        c2.close()


def test_c2_full_size_vs_reference_gpucompute(ctx):
    """BASELINE configs[1] at full size against the reference's own gpucompute run on the same inputs:
    CTC log-prob within 1e-4 relative (north_star) and per-frame gradients within the stated tolerance."""
    w = synth.WORKLOADS["c2"]
    net = synth.make_model(w, seed=0)
    b = synth.make_batch(w, seed=1)
    d = tempfile.mkdtemp()
    kaldi_io.write_model(d + "/model", net)
    kaldi_io.write_batch_file(d + "/batch.bin", b)
    with stored_runs("c2_gpucompute", d, keep=REF_FULL_SIZE_OUTPUTS, whole=("out/pzx.npy",), cells=REF_FULL_SIZE_CELLS):
        oracle.run_reference("gpu", d + "/model", d + "/batch.bin", d + "/out", w.learn_rate, w.momentum, steps=1,
                             dump_layers=False)      # the layer outputs are not compared here
    ref = oracle.load_dump(d + "/out")
    n, st = _gpu_steps(ctx, net, b, w.learn_rate, w.momentum, 1, want_in_diff=False)
    pzx = n.get(101).ravel()
    rel = np.abs(pzx - ref["pzx"]) / np.abs(ref["pzx"])
    assert rel.max() < 2e-5, rel.max()
    assert_close("net_out", n.get(len(net.layers)), ref["net_out"], atol=5e-5, stored=True)
    assert_close("obj_diff", n.get(100), ref["obj_diff"], atol=2 * diff_atol(ref["pzx"]), stored=True)
    m2 = kaldi_io.read_model(d + "/out/model_out")
    # parameter update = lr * (momentum buffer); the buffers are sums over all T*S rows of per-frame
    # gradients that individually agree only to diff_atol (fp32 log-domain CTC at |log p| ~ 2000 in BOTH
    # implementations), so their difference random-walks to ~sqrt(T*S) * diff_atol
    rows = b.feats.shape[0]
    assert_close("params", n.params(), m2.flat_params(),
                 atol=5e-6 + w.learn_rate * np.sqrt(rows) * diff_atol(ref["pzx"]), stored=True)
    n.close()


# ------------------------------------------------------------------------------------ BASELINE config 4 (bf16 gate GEMM)
# Stated tolerances of the bf16 arithmetic mode (--gemm-precision bf16: every dense contraction is tcgen05 kind::f16 on
# round-to-nearest-even bf16 copies of both operands, fp32 accumulation; the recurrence stays fp32-faithful):
#   against the fp64 restatement fed the SAME bf16-rounded operands (oracle_set_dense_rounding): what is left is
#     accumulation order plus roundings that flip because our fp32 activations differ from fp64 in the last bits --
#     layer outputs abs 2e-3, log p(z|x) rel 1e-3, per-frame gradient abs 5e-3, parameters after the step abs 2e-5;
#   against the exact fp64 restatement (what the rounding itself costs): log p(z|x) rel 2e-2.
# The fp32x3 mode keeps the north-star tolerance (log p rel 1e-4; asserted at 2e-5 throughout this file).
BF16_OUT_ATOL, BF16_PZX_RTOL, BF16_DIFF_ATOL, BF16_PARAM_ATOL = 2e-3, 1e-3, 5e-3, 2e-5


def test_bf16_train_step_vs_oracle_fed_bf16_rounded_operands(ctx):
    w, net, b = case("mid")
    lr, mom = 1e-3, 0.9
    ctx.set_precision("bf16", "fp32x3")
    try:
        n, st = _gpu_steps(ctx, net, b, lr, mom, 1)
    finally:
        ctx.set_precision("fp32x3", "fp32x3")
    exact = oracle.OracleNet(net, np.float64)
    re_ = exact.train_step(b, lr, mom)
    oracle.set_dense_rounding(np.float64, 1)
    try:
        on = oracle.OracleNet(net, np.float64)
        ro = on.train_step(b, lr, mom)
    finally:
        oracle.set_dense_rounding(np.float64, 0)
    for i in range(1, len(net.layers) + 1):
        assert_close(f"out_l{i}", n.get(i), on.acts[i], atol=BF16_OUT_ATOL)
    assert_close("pzx", n.get(101).ravel(), ro["pzx"], atol=0, rtol=BF16_PZX_RTOL)
    assert_close("obj_diff", n.get(100), ro["obj_diff"], atol=BF16_DIFF_ATOL)
    assert_close("params", n.params(), on.flat_params(), atol=BF16_PARAM_ATOL)
    assert_close("pzx_vs_exact", n.get(101).ravel(), re_["pzx"], atol=0, rtol=2e-2)
    # the rounding is really happening: the bf16 run is measurably off the exact one, the emulation explains it
    d_exact = np.abs(n.get(1) - exact.acts[1]).max()
    d_emul = np.abs(n.get(1) - on.acts[1]).max()
    assert d_exact > 5 * d_emul and d_exact > 1e-4, (d_exact, d_emul)
    n.close()


@pytest.fixture(scope="module")
def c4_inputs():
    w = synth.WORKLOADS["c4"]
    return w, synth.make_model(w, seed=0), synth.make_batch(w, seed=4)


def test_c4_vs_reference_gpucompute_at_the_reference_row_limit(ctx):
    """BASELINE configs[3] (5x512 BiLSTM, K = 32, 64 utterances) against the reference's own gpucompute.  The
    reference CANNOT run the config at its full 2000 frames: CuVectorBase::AddColSumMat launches a grid of
    (1, rows) blocks (src/gpucompute/cuda-vector.cc:880-899, called from Ctc::EvalParallel ctc-loss.cc:162), and
    rows = T*S = 128 000 exceeds the 65 535 limit of gridDim.y ("invalid configuration argument" -- measured on the
    B200).  So the live comparison runs at the largest length it can take, T = 1000 (64 000 rows); the full length
    is covered by test_c4_full_size_bf16_vs_fp32x3 below."""
    import dataclasses
    w = dataclasses.replace(synth.WORKLOADS["c4"], t_lo=1000, t_hi=1000, lab_lo=80, lab_hi=120)
    net, b = synth.make_model(w, seed=0), synth.make_batch(w, seed=4)
    d = tempfile.mkdtemp()
    kaldi_io.write_model(d + "/model", net)
    kaldi_io.write_batch_file(d + "/batch.bin", b)
    with stored_runs("c4_t1000_gpucompute", d, keep=REF_FULL_SIZE_OUTPUTS, whole=("out/pzx.npy",),
                     cells=REF_FULL_SIZE_CELLS):
        oracle.run_reference("gpu", d + "/model", d + "/batch.bin", d + "/out", w.learn_rate, w.momentum, steps=1,
                             dump_layers=False)      # 1.3 GB of layer outputs are not needed here
    ref = {k: np.load(os.path.join(d, "out", k + ".npy")) for k in ("pzx", "net_out", "obj_diff")}
    n, st = _gpu_steps(ctx, net, b, w.learn_rate, w.momentum, 1, want_in_diff=False)
    pzx = n.get(101).ravel()
    rel = np.abs(pzx - ref["pzx"]) / np.abs(ref["pzx"])
    assert rel.max() < 1e-4, rel.max()                       # north_star: CTC log-prob within 1e-4 relative
    assert_close("net_out", n.get(len(net.layers)), ref["net_out"], atol=1e-4, stored=True)
    assert_close("obj_diff", n.get(100), ref["obj_diff"], atol=4 * diff_atol(ref["pzx"]), stored=True)
    m2 = kaldi_io.read_model(d + "/out/model_out")
    rows = b.feats.shape[0]
    assert_close("params", n.params(), m2.flat_params(), atol=5e-6 + w.learn_rate * np.sqrt(rows) * 4 * diff_atol(ref["pzx"]),
                 stored=True)
    n.close()


def test_c4_full_size_bf16_vs_fp32x3(ctx, c4_inputs):
    """BASELINE configs[3] at FULL size (5x512, 64 x 2000 frames = 128 000 rows), one train step in fp32x3 and in bf16
    arithmetic: size-independent properties of the fp32x3 result, then the bf16 run against it at the stated bf16
    tolerances (log p rel 2e-2, posteriors abs 5e-2)."""
    w, net, b = c4_inputs
    n, st = _gpu_steps(ctx, net, b, w.learn_rate, w.momentum, 1, want_in_diff=False)
    pzx32 = n.get(101).ravel().copy()
    out32 = n.get(len(net.layers)).copy()
    diff = n.get(100)
    assert st["frames"] == b.valid_frames and np.all(np.isfinite(pzx32)) and np.all(pzx32 < 0)
    assert np.abs(out32.sum(1) - 1).max() < 1e-5                 # softmax rows
    assert np.abs(diff.sum(1)).max() < 5e-5                      # CTC gradient rows sum to zero (all rows valid here)
    p64, d64, _, _ = oracle.ctc_eval(out32.astype(np.float64), b.frames, b.labels, b.S, np.float64)
    assert_close("pzx_vs_fp64_ctc", pzx32, p64, atol=0, rtol=5e-5)
    assert np.all(np.isfinite(n.params()))
    n.close()
    ctx.set_precision("bf16", "fp32x3")
    try:
        n16, _ = _gpu_steps(ctx, net, b, w.learn_rate, w.momentum, 1, want_in_diff=False)
    finally:
        ctx.set_precision("fp32x3", "fp32x3")
    p16 = n16.get(101).ravel()
    assert np.all(np.isfinite(p16)) and np.all(np.isfinite(n16.params()))
    assert (np.abs(p16 - pzx32) / np.abs(pzx32)).max() < 2e-2     # stated bf16 tolerance on log p(z|x) vs fp32-faithful
    assert np.abs(n16.get(len(net.layers)) - out32).max() < 5e-2  # posteriors
    n16.close()


def test_train_ctc_parallel_driver_matches_api(ctx, tmp_path):
    """The C++ driver (host logic of reference src/netbin/train-ctc-parallel.cc) on Kaldi archives gives
    the same model as the level-2 API fed the same minibatches, and prints the recipe-facing log lines."""
    import subprocess
    from util import ROOT
    w, net, b = case("small")
    mpath = str(tmp_path / "nnet.in")
    kaldi_io.write_model(mpath, net)
    S, T = b.S, b.T
    utts = [b.feats[np.arange(b.frames[s]) * S + s] for s in range(S)]
    keys = [f"utt{s:03d}" for s in range(S)]
    kaldi_io.write_feature_ark(str(tmp_path / "feats.ark"), keys, utts)
    kaldi_io.write_label_ark(str(tmp_path / "labels.ark"), keys, b.labels)
    out = str(tmp_path / "nnet.out")
    exe = os.path.join(ROOT, "eesen_b200", "bin", "train-ctc-parallel")
    r = subprocess.run([exe, "--learn-rate=0.001", "--momentum=0.9", "--num-sequence=4", "--frame-limit=100000",
                        "--report-step=4", "--verbose=1", f"ark:{tmp_path}/feats.ark", f"ark,t:{tmp_path}/labels.ark",
                        mpath, out], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, r.stderr[-3000:]
    assert "TOKEN_ACCURACY >>" in r.stderr and "fps" in r.stderr and "TRAINING STARTED" in r.stderr
    got = kaldi_io.read_model(out).flat_params()
    # the same two minibatches (utterances 0-3, then 4-7) through the level-2 API
    n = binding.Net(ctx, mpath)
    n.set_train_options(1e-3, 0.9)
    for lo in (0, 4):
        feats, frames = kaldi_io.pack_utterances(utts[lo:lo + 4])
        n.train_step(feats, frames, b.labels[lo:lo + 4], True)
    assert_close("driver_vs_api", got, n.params(), atol=1e-7)
    n.close()


def test_reference_driver_on_the_b200_library_matches_our_driver(ctx, tmp_path):
    """The drop-in, compiled: the reference's UNMODIFIED train-ctc-parallel.cc / Net / Layer factory / Affine /
    Softmax / Update code (GPU build of /root/reference) with BiLstmParallel::{PropagateFnc,BackpropagateFnc},
    Ctc::EvalParallel and CuMatrixBase<float>::AddMatMat re-pointed at libeesen_b200.so (oracle/shim, oracle/Makefile
    target ref_train_ctc_parallel_b200) trains the same model as this repo's own driver on the same archives.
    Reference call sites: src/netbin/train-ctc-parallel.cc:195-207, src/net/layer.h:149-155."""
    import subprocess
    from util import ROOT
    exe_ref = os.path.join(ROOT, "oracle", "_ref", "ref_train_ctc_parallel_b200")
    if not os.path.exists(exe_ref):
        pytest.skip("oracle/_ref/ref_train_ctc_parallel_b200 not built (needs /root/reference at build time)")
    w, net, b = case("small")
    mpath = str(tmp_path / "nnet.in")
    kaldi_io.write_model(mpath, net)
    S = b.S
    utts = [b.feats[np.arange(b.frames[s]) * S + s] for s in range(S)]
    keys = [f"utt{s:03d}" for s in range(S)]
    kaldi_io.write_feature_ark(str(tmp_path / "feats.ark"), keys, utts)
    kaldi_io.write_label_ark(str(tmp_path / "labels.ark"), keys, b.labels)
    args = ["--learn-rate=0.001", "--momentum=0.9", "--num-sequence=4", "--frame-limit=100000", "--report-step=4",
            "--verbose=1", f"ark:{tmp_path}/feats.ark", f"ark,t:{tmp_path}/labels.ark", mpath]
    outs = {}
    for name, exe in (("reference_on_b200", exe_ref), ("ours", os.path.join(ROOT, "eesen_b200", "bin", "train-ctc-parallel"))):
        out = str(tmp_path / f"nnet.{name}")
        r = subprocess.run([exe] + args + [out], capture_output=True, text=True, timeout=300)
        assert r.returncode == 0, (name, r.stderr[-3000:])
        assert "TOKEN_ACCURACY >>" in r.stderr, (name, r.stderr[-2000:])
        outs[name] = kaldi_io.read_model(out).flat_params()
    # same kernels for the BiLSTM layers, CTC and every AddMatMat; what differs is the reference's own softmax,
    # bias / column-sum and update kernels (fp32 rounding only)
    assert_close("reference_driver_on_b200_vs_ours", outs["reference_on_b200"], outs["ours"], atol=5e-6)
