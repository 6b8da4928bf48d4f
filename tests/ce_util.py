"""Restatement of the reference's frame-level cross-entropy (src/net/ce-loss.cc:94-169) for the CE tests.

CE::EvalParallel, on softmax posteriors y packed as [T*S x K] with row r = t*S + s, valid iff t < frames[s]:
  diff     = (y - onehot(target)) * mask          (AddMat(-1, onehot) then MulRowsVec(mask))
  correct  = #valid rows with FindRowMaxId(y) == target   (first index of the row maximum)
  obj      = -sum over valid rows of log y[r, target[r]]
The reference takes log of the whole matrix and multiplies by the one-hot matrix, so a posterior that underflows to
0 anywhere makes its objective NaN (log 0 * 0); this restatement reads the target column only, as the library does.
"""
import numpy as np


def pack_targets(targets, frames, T):
    """per-utterance targets (frames[s] each) -> [T*S] packed like the rows; padded rows hold 0"""
    S = len(frames)
    out = np.zeros(T * S, np.int32)
    for s in range(S):
        out[np.arange(int(frames[s])) * S + s] = np.asarray(targets[s][:frames[s]], np.int32)
    return out


def valid_rows(frames, T):
    S = len(frames)
    r = np.arange(T * S)
    return (r // S) < np.asarray(frames)[r % S]


def ce_eval(y, frames, packed, dtype=np.float32):
    """returns diff [T*S x K] in dtype, obj (float64), correct (int), valid rows (int)"""
    y = np.asarray(y, dtype)
    N, K = y.shape
    S = len(frames)
    mask = valid_rows(frames, N // S)
    onehot = np.zeros_like(y)
    onehot[np.nonzero(mask)[0], packed[mask]] = 1
    diff = (y - onehot) * mask[:, None].astype(dtype)
    diff[~mask] = 0          # +0 in padded rows ((y - 1) * 0 is -0 in the reference, equal under ==)
    rows = np.nonzero(mask)[0]
    with np.errstate(divide="ignore"):       # a target posterior of 0 gives +inf, as in the library
        obj = -np.log(y[rows, packed[rows]]).astype(np.float64).sum()
    correct = int((np.argmax(y[rows], axis=1) == packed[rows]).sum())
    return diff, float(obj), correct, int(mask.sum())


def random_targets(frames, K, seed):
    """one target per frame, including 0 and K-1"""
    rng = np.random.default_rng(seed)
    out = [rng.integers(0, K, size=int(f)).astype(np.int32) for f in frames]
    out[0][0] = 0
    out[0][-1] = K - 1
    return out


def reference_case(seed, S, T, K):
    """seeded posteriors (softmax of N(0, 9) logits, fp32), ragged frames (one utterance without frames when S >= 3)
    and packed targets including 0 and K-1, for the comparisons with the reference's own CE::EvalParallel"""
    rng = np.random.default_rng(seed)
    frames = np.sort(rng.integers(max(1, T // 3), T + 1, size=S))[::-1].astype(np.int32)
    frames[0] = T
    if S >= 3:
        frames[-1] = 0
    x = rng.standard_normal((T * S, K)) * 3
    y = np.exp(x - x.max(1, keepdims=True))
    y = (y / y.sum(1, keepdims=True)).astype(np.float32)
    packed = pack_targets(random_targets(frames, K, seed + 1), frames, T)
    return frames, packed, y


def run_reference_ce(work, y, packed, frames):
    """oracle/_ref/ref_ce_cpu: the reference's CE::EvalParallel on the CPU (call inside tests/util.py:stored_runs).
    Returns (diff [T*S x K], {obj, correct, frames (padded rows), sequences})."""
    import json
    import os
    from oracle import oracle
    np.save(os.path.join(work, "y.npy"), np.ascontiguousarray(y, np.float32))
    np.save(os.path.join(work, "targets.npy"), np.ascontiguousarray(packed, np.int32))
    np.save(os.path.join(work, "frames.npy"), np.ascontiguousarray(frames, np.int32))
    os.makedirs(os.path.join(work, "out"), exist_ok=True)
    r = oracle.run_reference_tool("ref_ce_cpu", [os.path.join(work, f) for f in ("y.npy", "targets.npy", "frames.npy", "out")])
    info = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])
    return np.load(os.path.join(work, "out", "ce_diff.npy")), info
