"""ctypes binding of the C ABI (include/eesen_b200.h) for tests and bench.

Plumbing only: it loads ``eesen_b200/lib/libeesen_b200.so`` (built in-tree by ``make`` /
``__graft_entry__.build()``) and raises if the library or a CUDA device is missing -- there is
no CPU fallback and nothing here imports the oracle.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import List, Optional, Sequence

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "lib", "libeesen_b200.so")

PREC = {"fp32x3": 0, "tf32": 1, "bf16": 2}


class EesenB200Error(RuntimeError):
    pass


class BilstmParams(C.Structure):
    _fields_ = [(n, C.c_void_p * 2) for n in ("wx", "wm", "bias", "pi", "pf", "po")] + [("ldwx", C.c_int), ("ldwm", C.c_int)]


class SgdSegment(C.Structure):
    _fields_ = [("offset", C.c_int64), ("count", C.c_int64), ("lr", C.c_float), ("max_grad", C.c_float)]


_lib = None


def load_library() -> C.CDLL:
    global _lib
    if _lib is not None:
        return _lib
    path = os.environ.get("EESEN_B200_LIB", LIB_PATH)   # instrumented builds (make TIMING=1 LIBDIR=...) for tests/lstm_timing.py
    if not os.path.exists(path):
        raise EesenB200Error(f"{path} not built: run `make` (or __graft_entry__.build()) first")
    lib = C.CDLL(path)
    lib.eesen_b200_last_error.restype = C.c_char_p
    lib.eesen_b200_last_error.argtypes = [C.c_void_p]
    lib.eesen_b200_stream.restype = C.c_void_p
    lib.eesen_b200_stream.argtypes = [C.c_void_p]
    lib.eesen_b200_launch_count.restype = C.c_long
    lib.eesen_b200_launch_count.argtypes = [C.c_void_p]
    lib.eesen_b200_sm_count.argtypes = [C.c_void_p]
    lib.eesen_b200_destroy.argtypes = [C.c_void_p]
    lib.eesen_b200_destroy.restype = None
    lib.eesen_b200_net_free.argtypes = [C.c_void_p]
    lib.eesen_b200_net_free.restype = None
    lib.eesen_b200_net_last_loss.argtypes = [C.c_void_p]
    _lib = lib
    return lib


def _p(x) -> C.c_void_p:
    """device pointer of a torch tensor / int / None"""
    if x is None:
        return C.c_void_p(0)
    if isinstance(x, int):
        return C.c_void_p(x)
    return C.c_void_p(x.data_ptr())


class Context:
    """One per process/GPU (reference: the CuDevice singleton)."""

    def __init__(self, device: int = -1, gemm_precision: str = "fp32x3", recurrent_precision: str = "fp32x3"):
        self.lib = load_library()
        h = C.c_void_p()
        rc = self.lib.eesen_b200_create(C.byref(h), C.c_int(device))
        if rc != 0:
            raise EesenB200Error(f"eesen_b200_create failed ({rc}): {self.lib.eesen_b200_last_error(None).decode()}")
        self.h = h
        self.set_precision(gemm_precision, recurrent_precision)

    def close(self):
        if getattr(self, "h", None):
            self.lib.eesen_b200_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def check(self, rc: int, what: str):
        if rc != 0:
            raise EesenB200Error(f"{what} failed ({rc}): {self.lib.eesen_b200_last_error(self.h).decode()}")

    def set_precision(self, gemm: str, rec: str):
        self.check(self.lib.eesen_b200_set_precision(self.h, PREC[gemm], PREC[rec]), "set_precision")

    def synchronize(self):
        self.check(self.lib.eesen_b200_synchronize(self.h), "synchronize")

    @property
    def stream(self) -> int:
        return int(self.lib.eesen_b200_stream(self.h) or 0)

    @property
    def launches(self) -> int:
        return int(self.lib.eesen_b200_launch_count(self.h))

    @property
    def sm_count(self) -> int:
        return int(self.lib.eesen_b200_sm_count(self.h))

    def lstm_engine(self, num_utts: int, cells: int, ndir: int = 2, backward: bool = False) -> int:
        """1 = tcgen05 recurrent kernels, 0 = warp-level kernels, -1 = no plan (eesen_b200_lstm_engine)."""
        return int(self.lib.eesen_b200_lstm_engine(self.h, C.c_int(num_utts), C.c_int(cells), C.c_int(ndir), C.c_int(1 if backward else 0)))

    PROFILE_CATEGORIES = ("gemm", "lstm_fwd", "lstm_bwd", "softmax", "ctc", "sgd", "allreduce", "misc", "gemm_side")

    def profile(self, enable: int = -1):
        """Returns ({category: ms}, {category: launches}) since the last reset; enable=1/0 switches+resets."""
        ms = (C.c_double * 9)()
        cnt = (C.c_long * 9)()
        self.check(self.lib.eesen_b200_profile(self.h, int(enable), ms, cnt), "profile")
        return ({k: ms[i] for i, k in enumerate(self.PROFILE_CATEGORIES)},
                {k: cnt[i] for i, k in enumerate(self.PROFILE_CATEGORIES)})

    # ---- level 1 (torch CUDA tensors carry the device memory)
    def gemm(self, ta, tb, M, N, K, alpha, A, lda, B, ldb, beta, Cm, ldc):
        self.check(self.lib.eesen_b200_gemm(self.h, ta, tb, M, N, K, C.c_float(alpha), _p(A), lda, _p(B), ldb,
                                            C.c_float(beta), _p(Cm), ldc), "gemm")

    @staticmethod
    def _pack(tensors12, ldwx=0, ldwm=0) -> BilstmParams:
        """ldwx / ldwm: row strides of the wx / wm matrices in floats (0 = dense), e.g. pitched reference weights"""
        s = BilstmParams()
        names = ("wx", "wm", "bias", "pi", "pf", "po")
        for d in range(2):
            for k, n in enumerate(names):
                getattr(s, n)[d] = tensors12[d * 6 + k].data_ptr()
        s.ldwx, s.ldwm = ldwx, ldwm
        return s

    def bilstm_forward(self, T, S, I, Cc, d_len, x, ldx, params12, gates, cell, out, ldo, ldwx=0, ldwm=0):
        p = self._pack(params12, ldwx, ldwm)
        self.check(self.lib.eesen_b200_bilstm_forward(self.h, T, S, I, Cc, _p(d_len), _p(x), ldx, C.byref(p),
                                                      _p(gates), _p(cell), _p(out), ldo), "bilstm_forward")

    def bilstm_backward(self, T, S, I, Cc, x, ldx, params12, gates, cell, out, ldo, dout, ldd, dgates, dx, lddx,
                        grads12, ldwx=0, ldwm=0, gldwx=0, gldwm=0):
        p, g = self._pack(params12, ldwx, ldwm), self._pack(grads12, gldwx, gldwm)
        self.check(self.lib.eesen_b200_bilstm_backward(self.h, T, S, I, Cc, _p(x), ldx, C.byref(p), _p(gates),
                                                       _p(cell), _p(out), ldo, _p(dout), ldd, _p(dgates), _p(dx),
                                                       lddx, C.byref(g)), "bilstm_backward")

    def affine_forward(self, N, D, K, x, ldx, W, b, y, ldy):
        self.check(self.lib.eesen_b200_affine_forward(self.h, N, D, K, _p(x), ldx, _p(W), _p(b), _p(y), ldy),
                   "affine_forward")

    def affine_backward(self, N, D, K, x, ldx, diff, lddiff, W, dx, lddx, dW, db):
        self.check(self.lib.eesen_b200_affine_backward(self.h, N, D, K, _p(x), ldx, _p(diff), lddiff, _p(W), _p(dx),
                                                       lddx, _p(dW), _p(db)), "affine_backward")

    def softmax(self, N, K, logits, ld, probs, ldp, argmax=None):
        self.check(self.lib.eesen_b200_softmax(self.h, N, K, _p(logits), ld, _p(probs), ldp, _p(argmax)), "softmax")

    def ctc_eval(self, T, S, K, max_lab, d_len, d_labels, d_lab_len, probs, ldp, pzx, diff, ldd):
        self.check(self.lib.eesen_b200_ctc_eval(self.h, T, S, K, max_lab, _p(d_len), _p(d_labels), _p(d_lab_len),
                                                _p(probs), ldp, _p(pzx), _p(diff), ldd), "ctc_eval")

    def ce_eval(self, T, S, K, d_len, probs, ldp, d_targets, diff, ldd, d_stats):
        """Frame-level cross-entropy (CE::EvalParallel); d_stats: device float64[3] <- obj, correct, valid frames."""
        self.check(self.lib.eesen_b200_ce_eval(self.h, T, S, K, _p(d_len), _p(probs), ldp, _p(d_targets), _p(diff), ldd,
                                               _p(d_stats)), "ce_eval")

    def sgd_update(self, w, corr, grad, n, momentum, segments: Sequence[tuple]):
        arr = (SgdSegment * len(segments))(*[SgdSegment(*s) for s in segments])
        self.check(self.lib.eesen_b200_sgd_update(self.h, _p(w), _p(corr), _p(grad), C.c_int64(n),
                                                  C.c_float(momentum), arr, len(segments)), "sgd_update")

    # ---- NCCL
    def nccl_unique_id(self) -> bytes:
        buf = C.create_string_buffer(128)
        rc = self.lib.eesen_b200_nccl_unique_id(buf)
        if rc != 0:
            raise EesenB200Error("ncclGetUniqueId failed")
        return buf.raw

    def nccl_init(self, rank: int, nranks: int, uid: bytes):
        self.check(self.lib.eesen_b200_nccl_init(self.h, rank, nranks, C.c_char_p(uid)), "nccl_init")

    def allreduce_sum(self, buf, n):
        self.check(self.lib.eesen_b200_allreduce_sum(self.h, _p(buf), C.c_int64(n)), "allreduce_sum")


def class_log_priors(counts, prior_cutoff: float = 1e-10, blank_scale: float = 1.0) -> np.ndarray:
    """ClassPrior::ClassPrior host arithmetic (class-prior.cc:28-76) through the C ABI."""
    lib = load_library()
    c = np.ascontiguousarray(counts, np.float64)
    out = np.empty(c.size, np.float32)
    rc = lib.eesen_b200_class_log_priors(c.ctypes.data_as(C.c_void_p), int(c.size), C.c_float(prior_cutoff),
                                         C.c_float(blank_scale), out.ctypes.data_as(C.c_void_p))
    if rc:
        raise EesenB200Error(f"class_log_priors failed ({rc})")
    return out


class Net:
    """Level-2 handle: the Net + Ctc host mirror (reference train-ctc-parallel.cc call sequence)."""

    def __init__(self, ctx: Context, model_path: str):
        self.ctx = ctx
        self.lib = ctx.lib
        h = C.c_void_p()
        ctx.check(self.lib.eesen_b200_net_read(ctx.h, model_path.encode(), C.byref(h)), "net_read")
        self.h = h
        i, o, l, n = C.c_int(), C.c_int(), C.c_int(), C.c_int64()
        self.lib.eesen_b200_net_dims(self.h, C.byref(i), C.byref(o), C.byref(l), C.byref(n))
        self.in_dim, self.out_dim, self.num_layers, self.num_params = i.value, o.value, l.value, n.value

    def close(self):
        if getattr(self, "h", None):
            self.lib.eesen_b200_net_free(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_train_options(self, learn_rate: float, momentum: float):
        self.ctx.check(self.lib.eesen_b200_net_set_train_options(self.h, C.c_float(learn_rate), C.c_float(momentum)),
                       "net_set_train_options")

    def set_optimizer(self, algorithm: str = "SGD", adagrad_epsilon: float = 1e-6, rmsprop_rho: float = 0.9,
                      rmsprop_one_minus_rho: float = -1.0):
        """Net::SetUpdateAlgorithm + the adaptive NetTrainOptions (one_minus_rho < 0: the reference's fixed 0.1)."""
        self.ctx.check(self.lib.eesen_b200_net_set_optimizer(self.h, algorithm.encode(), C.c_float(adagrad_epsilon),
                                                             C.c_float(rmsprop_rho), C.c_float(rmsprop_one_minus_rho)),
                       "net_set_optimizer")

    def feedforward(self, feats: np.ndarray, frames, apply_log: bool = False, log_priors: Optional[np.ndarray] = None,
                    prior_scale: float = 1.0) -> np.ndarray:
        """Forward-only pass of one packed batch (net-output-extract): returns [T*S, K] host array."""
        feats = np.ascontiguousarray(feats, np.float32)
        if frames is None:      # the reference's call pattern: no SetSeqLengths, one sequence
            S, fptr = 1, None
        else:
            frames = np.ascontiguousarray(frames, np.int32)
            S, fptr = frames.size, frames.ctypes.data_as(C.c_void_p)
        T = feats.shape[0] // S
        out = np.empty((T * S, self.out_dim), np.float32)
        lp = None
        if log_priors is not None:
            lp = np.ascontiguousarray(log_priors, np.float32)
            assert lp.size == self.out_dim
        self.ctx.check(self.lib.eesen_b200_net_feedforward(
            self.h, feats.ctypes.data_as(C.c_void_p), T, S, fptr, int(apply_log),
            lp.ctypes.data_as(C.c_void_p) if lp is not None else None, C.c_float(prior_scale),
            out.ctypes.data_as(C.c_void_p)), "net_feedforward")
        return out

    def write_nonparallel(self, path: str, binary: bool = True):
        self.ctx.check(self.lib.eesen_b200_net_write_nonparallel(self.h, path.encode(), int(binary)), "net_write_nonparallel")

    def change_dropout(self, forward=0.0, fw_step=False, fw_seq=False, rnndrop=False, nml=False, recurrent=0.0,
                       rec_step=False, rec_seq=False, twiddle=False):
        """Net::ChangeDropoutParameters (the options net-change-model writes into the model)."""
        self.ctx.check(self.lib.eesen_b200_net_change_dropout(
            self.h, C.c_float(forward), int(fw_step), int(fw_seq), int(rnndrop), int(nml), C.c_float(recurrent),
            int(rec_step), int(rec_seq), int(twiddle)), "net_change_dropout")

    def set_dropout_seed(self, seed: int):
        self.ctx.check(self.lib.eesen_b200_net_set_dropout_seed(self.h, C.c_ulonglong(seed)), "net_set_dropout_seed")

    def set_dropout_masks(self, layer: int, fmask: Optional[np.ndarray] = None, rmask: Optional[np.ndarray] = None):
        """Inject explicit scaled masks for one BiLSTM layer (None clears); kept until replaced."""
        f = np.ascontiguousarray(fmask, np.float32) if fmask is not None else None
        r = np.ascontiguousarray(rmask, np.float32) if rmask is not None else None
        self.ctx.check(self.lib.eesen_b200_net_set_dropout_masks(
            self.h, int(layer), f.ctypes.data_as(C.c_void_p) if f is not None else None, f.shape[0] if f is not None else 0,
            r.ctypes.data_as(C.c_void_p) if r is not None else None, r.shape[0] if r is not None else 0),
            "net_set_dropout_masks")

    def write(self, path: str, binary: bool = True):
        self.ctx.check(self.lib.eesen_b200_net_write(self.h, path.encode(), int(binary)), "net_write")

    @staticmethod
    def _labels(labels: List[np.ndarray]):
        lab_len = np.array([len(l) for l in labels], np.int32)
        flat = np.concatenate([np.asarray(l, np.int32) for l in labels]) if lab_len.sum() else np.zeros(1, np.int32)
        return np.ascontiguousarray(flat, np.int32), lab_len

    def train_step(self, feats: np.ndarray, frames: np.ndarray, labels: List[np.ndarray], train: bool = True):
        """HOST inputs; H2D copy, forward, CTC, error rate, backward+update; returns stats dict."""
        feats = np.ascontiguousarray(feats, np.float32)
        frames = np.ascontiguousarray(frames, np.int32)
        S = frames.shape[0]
        T = feats.shape[0] // S
        flat, lab_len = self._labels(labels)
        st = (C.c_double * 4)()
        self.ctx.check(self.lib.eesen_b200_net_train_step(self.h, feats.ctypes.data_as(C.c_void_p), T, S,
                                                          frames.ctypes.data_as(C.c_void_p),
                                                          flat.ctypes.data_as(C.c_void_p),
                                                          lab_len.ctypes.data_as(C.c_void_p), int(train), st),
                       "net_train_step")
        return {"obj": st[0], "token_err": st[1], "ref_tokens": st[2], "frames": st[3]}

    def train_step_device(self, d_feats, T: int, S: int, frames: np.ndarray, flat_labels: np.ndarray,
                          lab_len: np.ndarray, train: bool = True):
        self.ctx.check(self.lib.eesen_b200_net_train_step_device(self.h, _p(d_feats), T, S,
                                                                 frames.ctypes.data_as(C.c_void_p),
                                                                 flat_labels.ctypes.data_as(C.c_void_p),
                                                                 lab_len.ctypes.data_as(C.c_void_p), int(train)),
                       "net_train_step_device")

    def train_step_ce(self, feats: np.ndarray, frames: np.ndarray, targets: List[np.ndarray], train: bool = True):
        """Frame-level cross-entropy step, HOST inputs: targets[s] holds frames[s] class ids.  Returns
        {obj: sum of -log y[target], correct, frames: valid frames, padded: T*S rows}."""
        feats = np.ascontiguousarray(feats, np.float32)
        frames = np.ascontiguousarray(frames, np.int32)
        S = frames.shape[0]
        T = feats.shape[0] // S
        assert all(len(t) == f for t, f in zip(targets, frames)), "one target per frame"
        flat = np.ascontiguousarray(np.concatenate([np.asarray(t, np.int32) for t in targets]), np.int32)
        st = (C.c_double * 4)()
        self.ctx.check(self.lib.eesen_b200_net_train_step_ce(self.h, feats.ctypes.data_as(C.c_void_p), T, S,
                                                             frames.ctypes.data_as(C.c_void_p),
                                                             flat.ctypes.data_as(C.c_void_p), int(train), st),
                       "net_train_step_ce")
        return self._ce_stats(st)

    def train_step_ce_device(self, d_feats, T: int, S: int, frames: np.ndarray, d_targets, train: bool = True):
        """Device-resident CE step: d_targets int32 [T*S] packed like the rows; statistics via read_stats(ce=True)."""
        frames = np.ascontiguousarray(frames, np.int32)
        self.ctx.check(self.lib.eesen_b200_net_train_step_ce_device(self.h, _p(d_feats), T, S,
                                                                    frames.ctypes.data_as(C.c_void_p), _p(d_targets),
                                                                    int(train)), "net_train_step_ce_device")

    @staticmethod
    def _ce_stats(st):
        return {"obj": st[0], "correct": st[1], "frames": st[2], "padded": st[3]}

    def read_stats(self, ce: Optional[bool] = None):
        """Statistics of the last step, named after the loss that step used (eesen_b200_net_last_loss); passing ce
        states the expected loss and raises if the last step used the other one."""
        st = (C.c_double * 4)()
        self.ctx.check(self.lib.eesen_b200_net_read_stats(self.h, st), "net_read_stats")
        last_ce = bool(self.lib.eesen_b200_net_last_loss(self.h))
        if ce is not None and bool(ce) != last_ce:
            raise EesenB200Error(f"read_stats(ce={ce}): the last step used {'CE' if last_ce else 'CTC'}")
        if last_ce:
            return self._ce_stats(st)
        return {"obj": st[0], "token_err": st[1], "ref_tokens": st[2], "frames": st[3]}

    def get(self, which: int) -> np.ndarray:
        r, c = C.c_int(), C.c_int()
        self.ctx.check(self.lib.eesen_b200_net_get(self.h, which, None, C.c_int64(0), C.byref(r), C.byref(c)), "net_get")
        out = np.zeros((r.value, c.value), np.float32)
        if out.size:
            self.ctx.check(self.lib.eesen_b200_net_get(self.h, which, out.ctypes.data_as(C.c_void_p),
                                                       C.c_int64(out.size), C.byref(r), C.byref(c)), "net_get")
        return out

    def params(self) -> np.ndarray:
        return self.get(200).ravel()

    def corr(self) -> np.ndarray:
        return self.get(201).ravel()

    def accu(self) -> np.ndarray:
        return self.get(203).ravel()

    def grads(self) -> np.ndarray:
        return self.get(202).ravel()

    def set_params(self, flat: np.ndarray):
        flat = np.ascontiguousarray(flat, np.float32)
        self.ctx.check(self.lib.eesen_b200_net_set_params(self.h, flat.ctypes.data_as(C.c_void_p),
                                                          C.c_int64(flat.size)), "net_set_params")
