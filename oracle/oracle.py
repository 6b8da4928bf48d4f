"""oracle/oracle.py -- TEST INFRASTRUCTURE ONLY.

ctypes front-end to the CPU restatement (oracle/cpu_ref.c -> oracle/_ref/liboracle_f{32,64}.so)
plus a runner for the UNMODIFIED reference binaries (oracle/_ref/ref_dump_{cpu,gpu}).
Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference leg may
import this module; the product (eesen_b200/) never does.

`train_step` strings the restated ops together exactly as train-ctc-parallel.cc:195-207 +
Net::Propagate/Backpropagate (net.cc:67-108) do.
"""
from __future__ import annotations

import ctypes as C
import json
import os
import subprocess
import tempfile
from typing import Dict, List, Optional

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
REFDIR = os.path.join(HERE, "_ref")


def build(quiet: bool = True) -> None:
    """Compile the restatement (always) and the reference binaries (when /root/reference exists)."""
    cmd = ["make", "-C", HERE, "-j8", "all"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("oracle build failed:\n" + r.stdout[-4000:] + r.stderr[-4000:])


class _Lib:
    def __init__(self, dtype):
        self.dtype = np.dtype(dtype)
        name = "liboracle_f32.so" if self.dtype == np.float32 else "liboracle_f64.so"
        path = os.path.join(REFDIR, name)
        if not os.path.exists(path):
            build()
        self.lib = C.CDLL(path)
        assert self.lib.oracle_real_size() == self.dtype.itemsize
        self.real = C.c_float if self.dtype == np.float32 else C.c_double

    def arr(self, a):
        a = np.ascontiguousarray(a, self.dtype)
        return a

    @staticmethod
    def p(a):
        return a.ctypes.data_as(C.c_void_p)

    def pp(self, arrs):
        t = (C.c_void_p * len(arrs))(*[a.ctypes.data for a in arrs])
        return t


_LIBS: Dict[str, _Lib] = {}


def lib(dtype=np.float32) -> _Lib:
    k = np.dtype(dtype).name
    if k not in _LIBS:
        _LIBS[k] = _Lib(dtype)
    return _LIBS[k]


def set_dense_rounding(dtype, mode: int) -> None:
    """mode 1: the restatement rounds both operands of every dense (input-side / affine) product to bf16, as the
    product's bf16 arithmetic mode does (BASELINE config 4); 0 restores exact operands."""
    lib(dtype).lib.oracle_set_dense_rounding(int(mode))


def ctc_eval(y: np.ndarray, frames, labels: List[np.ndarray], S: int, dtype=np.float32, want_ab=False):
    L = lib(dtype)
    y = L.arr(y)
    N, K = y.shape
    T = N // S
    frames = np.ascontiguousarray(frames, np.int32)
    lab_len = np.array([len(l) for l in labels], np.int32)
    flat = np.concatenate([np.asarray(l, np.int32) for l in labels]) if lab_len.sum() else np.zeros(1, np.int32)
    flat = np.ascontiguousarray(flat, np.int32)
    pzx = np.zeros(S, L.dtype)
    diff = np.zeros((N, K), L.dtype)
    Lp = 2 * int(lab_len.max()) + 1
    alpha = np.zeros((N, Lp), L.dtype) if want_ab else None
    beta = np.zeros((N, Lp), L.dtype) if want_ab else None
    L.lib.oracle_ctc_eval_parallel(T, S, K, L.p(frames), L.p(flat), L.p(lab_len), L.p(y), L.p(pzx), L.p(diff),
                                   L.p(alpha) if want_ab else None, L.p(beta) if want_ab else None)
    return pzx, diff, alpha, beta


def softmax(x: np.ndarray, dtype=np.float32) -> np.ndarray:
    L = lib(dtype)
    x = L.arr(x)
    y = np.empty_like(x)
    L.lib.oracle_softmax(x.shape[0], x.shape[1], L.p(x), L.p(y))
    return y


class OracleNet:
    """Holds parameters + momentum buffers in the oracle's precision and runs train steps."""

    def __init__(self, net, dtype=np.float32):
        self.L = lib(dtype)
        self.spec = net
        self.params = [{n: self.L.arr(l.params[n]).copy() for n in l.param_names()} for l in net.layers]
        self.corr = [{n: np.zeros_like(v) for n, v in p.items()} for p in self.params]
        # Net::SetUpdateAlgorithm (net.cc:481-496) + NetTrainOptions (train-opts.h:33-50)
        self.algorithm = "SGD"
        self.adagrad_epsilon, self.rmsprop_rho, self.rmsprop_one_minus_rho = 1e-6, 0.9, 0.1   # train-opts.h:40-42,50
        self.accu = [{n: np.zeros_like(v) for n, v in p.items()} for p in self.params]

    def set_optimizer(self, algorithm="SGD", adagrad_epsilon=1e-6, rmsprop_rho=0.9, rmsprop_one_minus_rho=0.1):
        assert algorithm in ("SGD", "Adagrad", "RMSProp")
        self.algorithm, self.adagrad_epsilon = algorithm, adagrad_epsilon
        self.rmsprop_rho, self.rmsprop_one_minus_rho = rmsprop_rho, rmsprop_one_minus_rho

    # ---- dropout (bilstm-parallel-layer.h:46-94, 209-377, 604-879).  masks: one dict per layer (or None):
    #   "fmask": scaled forward mask [T*S x 2C] applied to the layer OUTPUT and to out_diff (:409-416, :891-895)
    #   "rmask": scaled recurrent mask [T*S x 2C] (step dropout, row (t-1)*S+s) or [S x 2C] (sequence dropout),
    #            forward cells in columns [0,C), backward cells in [C,2C) (:85-88)
    # The reference draws them from a thread-local mt19937 seeded by std::random_device (kaldi-math.h:107-131):
    # not reproducible by design, so parity is "same masks -> same numbers"; the masks are always inputs here.
    def forward(self, feats, frames, masks=None):
        self.masks = masks
        L = self.L
        S = len(frames)
        frames = np.ascontiguousarray(frames, np.int32)
        x = L.arr(feats)
        N = x.shape[0]
        T = N // S
        acts = [x]
        self.bufs = []
        for li, l in enumerate(self.spec.layers):
            p = self.params[li]
            if l.kind == "bilstm":
                Cc = l.cells
                buf_fw = np.zeros(((T + 2) * S, 7 * Cc), L.dtype)
                buf_bw = np.zeros(((T + 2) * S, 7 * Cc), L.dtype)
                out = np.zeros((N, 2 * Cc), L.dtype)
                plist = [p[n] for n in l.param_names()]
                mk = masks[li] if masks else None
                drop = 0
                if mk is not None and mk.get("rmask") is not None:
                    drop = 2 if l.dropout.get("rnndrop") else 1
                    rm = L.arr(mk["rmask"])
                    rfw, rbw = np.ascontiguousarray(rm[:, :Cc]), np.ascontiguousarray(rm[:, Cc:])
                    per_step = int(rm.shape[0] == N)
                    L.lib.oracle_bilstm_forward_drop(T, S, l.in_dim, Cc, L.p(frames), L.p(acts[-1]), L.pp(plist),
                                                     L.p(buf_fw), L.p(buf_bw), L.p(out), drop, L.p(rfw), L.p(rbw), per_step)
                    self.bufs.append((buf_fw, buf_bw, drop, rfw, rbw, per_step))
                else:
                    L.lib.oracle_bilstm_forward(T, S, l.in_dim, Cc, L.p(frames), L.p(acts[-1]), L.pp(plist),
                                                L.p(buf_fw), L.p(buf_bw), L.p(out))
                    self.bufs.append((buf_fw, buf_bw, 0, None, None, 0))
                if mk is not None and mk.get("fmask") is not None:
                    out = out * L.arr(mk["fmask"])
                acts.append(out)
            elif l.kind == "lstm":
                Cc = l.cells
                buf = np.zeros(((T + 2) * S, 7 * Cc), L.dtype)
                out = np.zeros((N, Cc), L.dtype)
                plist = [p[n] for n in l.param_names()]
                L.lib.oracle_lstm_forward(T, S, l.in_dim, Cc, L.p(acts[-1]), L.pp(plist), L.p(buf), L.p(out))
                self.bufs.append((buf,))
                acts.append(out)
            elif l.kind == "affine":
                out = np.zeros((N, l.out_dim), L.dtype)
                L.lib.oracle_affine_forward(N, l.in_dim, l.out_dim, L.p(acts[-1]), L.p(p["w"]), L.p(p["b"]), L.p(out))
                self.bufs.append(None)
                acts.append(out)
            elif l.kind == "softmax":
                out = np.zeros((N, l.out_dim), L.dtype)
                L.lib.oracle_softmax(N, l.out_dim, L.p(acts[-1]), L.p(out))
                self.bufs.append(None)
                acts.append(out)
        self.acts = acts
        return acts[-1]

    def backward_update(self, obj_diff, frames, lr: float, momentum: float):
        L = self.L
        S = len(frames)
        N = obj_diff.shape[0]
        T = N // S
        d = L.arr(obj_diff)
        self.in_diffs = {}
        for li in range(len(self.spec.layers) - 1, -1, -1):
            l = self.spec.layers[li]
            p, c = self.params[li], self.corr[li]
            x = self.acts[li]
            if l.kind == "softmax":
                nd = d.copy()  # softmax-layer.h:49-57: identity
            elif l.kind == "affine":
                nd = np.zeros((N, l.in_dim), L.dtype)
                L.lib.oracle_affine_backward(N, l.in_dim, l.out_dim, L.p(d), L.p(p["w"]), L.p(nd))
                L.lib.oracle_affine_grad(N, l.in_dim, l.out_dim, L.p(x), L.p(d), L.p(c["w"]), L.p(c["b"]),
                                         L.real(momentum))
            elif l.kind == "lstm":
                Cc = l.cells
                nd = np.zeros((N, l.in_dim), L.dtype)
                dbuf = np.zeros(((T + 2) * S, 7 * Cc), L.dtype)
                plist = [p[n] for n in l.param_names()]
                clist = [c[n] for n in l.param_names()]
                L.lib.oracle_lstm_backward(T, S, l.in_dim, Cc, L.p(x), L.pp(plist), L.p(self.bufs[li][0]), L.p(d),
                                           L.p(dbuf), L.p(nd), L.pp(clist), L.real(momentum))
            else:
                Cc = l.cells
                nd = np.zeros((N, l.in_dim), L.dtype)
                dfw = np.zeros(((T + 2) * S, 7 * Cc), L.dtype)
                dbw = np.zeros(((T + 2) * S, 7 * Cc), L.dtype)
                plist = [p[n] for n in l.param_names()]
                clist = [c[n] for n in l.param_names()]
                bf, bb, drop, rfw, rbw, per_step = self.bufs[li]
                mk = self.masks[li] if getattr(self, "masks", None) else None
                if mk is not None and mk.get("fmask") is not None:
                    d = np.ascontiguousarray(d * L.arr(mk["fmask"]))
                if drop:
                    L.lib.oracle_bilstm_backward_drop(T, S, l.in_dim, Cc, L.p(x), L.pp(plist), L.p(bf), L.p(bb), L.p(d),
                                                      L.p(dfw), L.p(dbw), L.p(nd), L.pp(clist), L.real(momentum), drop,
                                                      L.p(rfw), L.p(rbw), per_step)
                else:
                    L.lib.oracle_bilstm_backward(T, S, l.in_dim, Cc, L.p(x), L.pp(plist), L.p(bf), L.p(bb), L.p(d),
                                                 L.p(dfw), L.p(dbw), L.p(nd), L.pp(clist), L.real(momentum))
                self.last_dbuf = (dfw, dbw)
            # TrainableLayer::Update right after the layer's Backpropagate (net.cc:98-105)
            for n in l.param_names():
                if self.algorithm == "SGD":
                    L.lib.oracle_sgd_update(C.c_long(p[n].size), L.p(p[n]), L.p(c[n]),
                                            L.real(lr * l.learn_rate_coef), L.real(l.max_grad))
                else:   # the adaptive branch ignores learn_rate_coef (bilstm-layer.h:885-955)
                    a = self.accu[li][n]
                    L.lib.oracle_ada_update(C.c_long(p[n].size), L.p(p[n]), L.p(c[n]), L.p(a), L.real(lr),
                                            L.real(l.max_grad), L.real(self.adagrad_epsilon),
                                            L.real(self.rmsprop_rho), L.real(self.rmsprop_one_minus_rho),
                                            1 if self.algorithm == "Adagrad" else 2)
            self.in_diffs[li] = nd
            d = nd
        return d

    def train_step(self, batch, lr: float, momentum: float, diff_override: Optional[np.ndarray] = None, masks=None):
        y = self.forward(batch.feats, batch.frames, masks)
        pzx, diff, _, _ = ctc_eval(y, batch.frames, batch.labels, batch.S, self.L.dtype)
        if diff_override is not None:
            diff = self.L.arr(diff_override)
        in_diff = self.backward_update(diff, batch.frames, lr, momentum)
        return {"net_out": y, "pzx": pzx, "obj_diff": diff, "in_diff": in_diff}

    def flat_params(self) -> np.ndarray:
        return np.concatenate([self.params[i][n].ravel() for i, l in enumerate(self.spec.layers) for n in l.param_names()])

    def flat_accu(self) -> np.ndarray:
        return np.concatenate([self.accu[i][n].ravel() for i, l in enumerate(self.spec.layers) for n in l.param_names()])

    def flat_corr(self) -> np.ndarray:
        return np.concatenate([self.corr[i][n].ravel() for i, l in enumerate(self.spec.layers) for n in l.param_names()])


def dropout_mask(rows: int, cols: int, p: float, per_col: bool, seed: int, stream: int) -> np.ndarray:
    """Replica of the product's device mask generator (eesen_b200/csrc/optim.cu:uniform01 / dropout_mask_kernel):
    splitmix64 finaliser of (seed, stream, index) -> 24 bits -> u in (0,1); mask = (u - p > 0) / (1 - p), one draw
    per element or per column.  (The reference's own generator is random_device-seeded; this only checks that OUR
    generator is the documented function of its seed.)"""
    M = np.uint64(0xFFFFFFFFFFFFFFFF)
    n = cols if per_col else rows * cols
    idx = np.arange(n, dtype=np.uint64)
    with np.errstate(over="ignore"):
        z = np.uint64(seed & 0xFFFFFFFFFFFFFFFF) + np.uint64(0x9e3779b97f4a7c15) * (idx + np.uint64(1)) \
            + np.uint64(0xbf58476d1ce4e5b9) * np.uint64((stream + 1) & 0xFFFFFFFFFFFFFFFF)
        z = (z ^ (z >> np.uint64(30))) * np.uint64(0xbf58476d1ce4e5b9)
        z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94d049bb133111eb)
        z = z ^ (z >> np.uint64(31))
    u = ((z >> np.uint64(40)).astype(np.float32) + np.float32(0.5)) * np.float32(1.0 / 16777216.0)
    m = np.where(u - np.float32(p) > 0, np.float32(1.0) / (np.float32(1.0) - np.float32(p)), np.float32(0.0)).astype(np.float32)
    return np.tile(m[None, :], (rows, 1)) if per_col else m.reshape(rows, cols)


def class_log_priors(counts, prior_cutoff=1e-10, blank_scale=1.0) -> np.ndarray:
    """ClassPrior::ClassPrior (class-prior.cc:28-76): counts below the cutoff are floored and masked with
    FLT_MAX/2, class 0 scaled by blank_scale, normalised, log in double, cast to float, mask added."""
    p = np.asarray(counts, np.float64).copy()
    cut = np.float64(np.float32(prior_cutoff))
    mask = np.zeros(p.size, np.float32)
    low = p < cut
    p[low] = cut
    mask[low] = np.finfo(np.float32).max / 2
    if blank_scale != 1.0:
        p[0] *= np.float64(np.float32(blank_scale))
    p = p * (1.0 / p.sum())
    return (np.log(p).astype(np.float32) + mask).astype(np.float32)


def net_output(on: "OracleNet", feats, frames, apply_log=False, log_priors=None, prior_scale=1.0) -> np.ndarray:
    """net-output-extract.cc:96-110 on a packed batch: Feedforward, ApplyLog, SubtractOnLogpost."""
    y = on.forward(feats, frames).astype(on.L.dtype).copy()
    if apply_log:
        with np.errstate(divide="ignore"):
            y = np.log(y)
    if log_priors is not None:
        y = y + np.asarray(-prior_scale, on.L.dtype) * np.asarray(log_priors, on.L.dtype)[None, :]
    return y


# Every call of a binary under oracle/_ref goes through RUNNER (same signature as subprocess.run with
# capture_output=True, text=True).  The tests set it to replay the runs stored under tests/golden/runs, so they do
# not need the reference's sources (tests/util.py:stored_runs).
RUNNER = None


def _run(cmd: List[str], env=None, timeout: Optional[int] = None):
    if RUNNER is not None:
        return RUNNER(cmd, env=env, timeout=timeout)
    return subprocess.run(cmd, capture_output=True, text=True, env=env, timeout=timeout)


def run_reference_tool(tool: str, args: List[str], timeout: int = 600, threads: Optional[int] = None):
    """Run one of the reference's own command-line tools built under oracle/_ref."""
    exe = os.path.join(REFDIR, tool)
    env = dict(os.environ)
    if threads is not None:
        env["OPENBLAS_NUM_THREADS"] = str(threads)
    r = _run([exe] + list(args), env=env, timeout=timeout)
    if r.returncode != 0:
        raise RuntimeError(f"{tool} failed ({r.returncode}):\n{r.stdout[-2000:]}\n{r.stderr[-4000:]}")
    return r


def greedy_token_errors(y: np.ndarray, frames, labels, S: int):
    """Ctc::ErrorRateMSeq (ctc-loss.cc:235-298): argmax path -> collapse repeats -> drop blanks ->
    Levenshtein (util/edit-distance-inl.h:28-75).  Returns (errors, ref_tokens)."""
    am = np.argmax(y, axis=1)
    err = 0
    ref = 0
    for s in range(S):
        seq = am[np.arange(int(frames[s])) * S + s]
        keep = np.concatenate([[True], seq[1:] != seq[:-1]])
        hyp = [int(v) for v in seq[keep] if v != 0]
        r = [int(v) for v in labels[s]]
        # plain DP edit distance
        prev = list(range(len(hyp) + 1))
        for i in range(1, len(r) + 1):
            cur = [i] + [0] * len(hyp)
            for j in range(1, len(hyp) + 1):
                cur[j] = min(prev[j] + 1, cur[j - 1] + 1, prev[j - 1] + (r[i - 1] != hyp[j - 1]))
            prev = cur
        err += prev[-1]
        ref += len(r)
    return err, ref


# --------------------------------------------------------------------------- the real reference
def have_reference(kind: str) -> bool:
    return os.path.exists(os.path.join(REFDIR, f"ref_dump_{kind}"))


def run_reference(kind: str, model_path: str, batch_path: str, outdir: str, lr: float, momentum: float,
                  steps: int = 1, diff_in: Optional[str] = None, time_only: bool = False,
                  threads: Optional[int] = None, timeout: int = 3600, opt: str = "SGD", dump_layers: bool = True):
    """Run oracle/_ref/ref_dump_{cpu,gpu} (the unmodified reference objects) on one batch."""
    exe = os.path.join(REFDIR, f"ref_dump_{kind}")
    os.makedirs(outdir, exist_ok=True)
    cmd = [exe, model_path, batch_path, outdir, "--lr", repr(float(lr)), "--momentum", repr(float(momentum)),
           "--steps", str(steps)]
    if opt != "SGD":
        cmd += ["--opt", opt]
    if diff_in:
        cmd += ["--diff-in", diff_in]
    if time_only:
        cmd += ["--time-only"]
    if not dump_layers:
        cmd += ["--no-dump-layers"]
    env = dict(os.environ)
    if threads is not None:
        env["OPENBLAS_NUM_THREADS"] = str(threads)
    r = _run(cmd, env=env, timeout=timeout)
    if r.returncode != 0:
        raise RuntimeError(f"reference run failed ({r.returncode}):\n{r.stdout[-2000:]}\n{r.stderr[-4000:]}")
    info = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])
    return info


def load_dump(outdir: str) -> Dict[str, np.ndarray]:
    out = {}
    for f in os.listdir(outdir):
        if f.endswith(".npy"):
            out[f[:-4]] = np.load(os.path.join(outdir, f))
    return out


# --------------------------------------------------------------------------- WFST one-best search (row N3)
_DEC = None


def decode_best_path(g, loglikes: np.ndarray, acoustic_scale: float, beam: float, max_active: int = 2147483647,
                     min_active: int = 0, max_out: int = 4096):
    """oracle/decoder_ref.c: the restated LatticeFasterDecoder search, one utterance.  g: eesen_b200.wfst.Graph (plain
    arrays); loglikes [T x K].  Returns (words | None, cost, frames_decoded, arcs_expanded)."""
    global _DEC
    if _DEC is None:
        path = os.path.join(REFDIR, "liboracle_dec.so")
        if not os.path.exists(path):
            build()
        _DEC = C.CDLL(path)
        _DEC.oracle_decode_best_path.restype = C.c_int
    ll = np.ascontiguousarray(loglikes, np.float32)
    T, K = ll.shape
    out = np.zeros(max_out, np.int32)
    cost = C.c_float(0.0); nf = C.c_int(0); na = C.c_long(0)
    P = lambda a, t: np.ascontiguousarray(a, t).ctypes.data_as(C.c_void_p)
    keep = [np.ascontiguousarray(g.row, np.int32), np.ascontiguousarray(g.eps, np.int32), np.ascontiguousarray(g.ilabel, np.int32),
            np.ascontiguousarray(g.olabel, np.int32), np.ascontiguousarray(g.weight, np.float32),
            np.ascontiguousarray(g.nextstate, np.int32), np.ascontiguousarray(g.final, np.float32)]
    p = [a.ctypes.data_as(C.c_void_p) for a in keep]
    n = _DEC.oracle_decode_best_path(g.num_states, g.start, p[0], p[1], p[2], p[3], p[4], p[5], p[6], T, K,
                                     ll.ctypes.data_as(C.c_void_p), C.c_float(acoustic_scale), C.c_float(beam),
                                     int(max_active), int(min_active), out.ctypes.data_as(C.c_void_p), max_out,
                                     C.byref(cost), C.byref(nf), C.byref(na))
    return (out[:n].tolist() if n >= 0 else None), float(cost.value), int(nf.value), int(na.value)
