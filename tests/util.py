"""Shared helpers for the parity tests."""
import contextlib
import fnmatch
import hashlib
import json
import os
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from eesen_b200 import kaldi_io, synth  # noqa: E402

GOLDEN = os.path.join(ROOT, "tests", "golden")
RUNS = os.path.join(GOLDEN, "runs")


def assert_close(name, got, ref, atol, rtol=0.0, stored=False):
    """stored=True: ref was restored by stored_runs and holds NaN in the cells the fixture did not keep; only the
    kept cells are compared (there must be some), and every cell of got must still be finite."""
    got = np.asarray(got, np.float64)
    ref = np.asarray(ref, np.float64)
    assert got.shape == ref.shape, f"{name}: shape {got.shape} vs {ref.shape}"
    if stored:
        assert np.isfinite(got).all(), f"{name}: non-finite values"
        keep = ~np.isnan(ref)
        assert keep.any() or not keep.size, f"{name}: no stored cell to compare"
        got, ref = got[keep], ref[keep]
    err = np.abs(got - ref)
    bound = atol + rtol * np.abs(ref)
    worst = (err - bound).max() if err.size else 0.0
    assert worst <= 0, (f"{name}: max abs err {err.max():.3e} (|ref| max {np.abs(ref).max():.3e}) exceeds "
                        f"atol={atol:g} rtol={rtol:g}")


def model_file(net):
    d = tempfile.mkdtemp(prefix="eesen_b200_test_")
    p = os.path.join(d, "model")
    kaldi_io.write_model(p, net)
    return p


def case(wl, mseed=3, bseed=5, bidirectional=True):
    w = synth.WORKLOADS[wl]
    return w, synth.make_model(w, seed=mseed, bidirectional=bidirectional), synth.make_batch(w, seed=bseed)


def golden_arrays(dump, net):
    """Flatten the reference's grad_<layer>_<name> dumps into model-file (arena) order."""
    names = {"wx": "wx", "wm": "wm", "b": "b", "pi": "pi", "pf": "pf", "po": "po"}
    out = []
    for li, l in enumerate(net.layers):
        for n in l.param_names():
            out.append(np.asarray(dump[f"grad_{li}_{n}"]).ravel())
    return np.concatenate(out)


# ------------------------------------------------------------------------------------ stored runs of the reference
# The reference binaries (oracle/_ref, built from the reference's sources) are not available wherever the suite runs.
# A test that compares with them wraps its calls in `with stored_runs(name, work):`; every call of a binary is then
# replayed from tests/golden/runs/<name>.npz: the stored return code, stdout / stderr and the files the call wrote
# under `work` are restored in place.  The files under `work` the call read must hash to what the reference was
# given, and the command line must be the recorded one, so a fixture only ever answers the question it was made for.
# EESEN_B200_RECORD_RUNS=1 (with the reference built) runs the binaries instead and writes the fixtures.
#
# Size: the outputs of a call fall into groups, one per pattern of `cells` (the first that matches) plus one for the
# rest.  A group keeps about cells[pattern] float cells (BUDGET for the rest) in all: every float array, and every
# matrix / vector of a binary Kaldi file, in it keeps a share in proportion to its size, at least FLOOR cells (or all
# of them), at the fixed positions sample_index(n, k).  The other cells come back as NaN; assert_close(stored=True)
# compares the kept ones.  Outputs matching `whole` are stored complete, and a Kaldi payload equal to that of one of
# the call's input files as a pointer to it.
RECORD = os.environ.get("EESEN_B200_RECORD_RUNS") == "1"
BUDGET = 384
FLOOR = 8


def sample_index(n, k):
    """k fixed, evenly spread flat indices into an n-element array (multiplicative hash; all of them if k >= n)."""
    if k >= n:
        return np.arange(n)
    return np.unique((np.arange(k, dtype=np.int64) * 2654435761 + 97) % n)


def _float_blocks(raw, cut=False):
    """(offset, count) of the float32 payload of every binary Kaldi matrix ("FM ") and vector ("FV ") in raw
    (cut: raw holds the headers only, the payloads cut out)."""
    out, i = [], 0
    while True:
        m, v = raw.find(b"FM \x04", i), raw.find(b"FV \x04", i)
        j = min(x for x in (m, v, len(raw)) if x >= 0)
        if j == len(raw):
            return out
        if j == m:
            rows, cols = int(np.frombuffer(raw, np.int32, 1, j + 4)[0]), int(np.frombuffer(raw, np.int32, 1, j + 9)[0])
            off, cnt = j + 13, rows * cols
        else:
            off, cnt = j + 8, int(np.frombuffer(raw, np.int32, 1, j + 4)[0])
        out.append((off, cnt))
        i = off if cut else off + 4 * cnt


def _payload(raw):
    blocks = _float_blocks(raw)
    if not blocks:
        return blocks, np.zeros(0, np.float32)
    return blocks, np.concatenate([np.frombuffer(raw, np.float32, c, o) for o, c in blocks])


def _share(n, budget, total):
    return min(n, max(FLOOR, -(-budget * n // max(total, 1))))


def _unsampled(vals, n, k, dtype=np.float32):
    if k >= n:
        return np.asarray(vals, dtype)
    full = np.full(n, np.nan, dtype)
    full[sample_index(n, k)] = vals
    return full


def _files(work):
    out = {}
    for dp, _, fs in os.walk(work):
        for f in fs:
            p = os.path.join(dp, f)
            out[os.path.relpath(p, work)] = hashlib.sha256(open(p, "rb").read()).hexdigest()
    return out


def _save_runs(path, calls, arrays):
    """one pool per dtype and a JSON index: a fixture is a handful of npz members, not one per array"""
    pools, index = {}, {}
    for k, a in arrays.items():
        pool = pools.setdefault(a.dtype.str, [])
        index[k] = [a.dtype.str, sum(x.size for x in pool), int(a.size)]
        pool.append(a.ravel())
    np.savez_compressed(path, calls=np.frombuffer(json.dumps({"calls": calls, "index": index}).encode(), np.uint8),
                        **{"pool" + dt.replace("<", "_").replace("|", "_"): np.concatenate(v) for dt, v in pools.items()})


def _load_runs(path):
    g = np.load(path)
    d = json.loads(g["calls"].tobytes())
    pools = {k: g[k] for k in g.files if k.startswith("pool")}
    arrays = {k: pools["pool" + dt.replace("<", "_").replace("|", "_")][off:off + n] for k, (dt, off, n) in d["index"].items()}
    return d["calls"], arrays


@contextlib.contextmanager
def stored_runs(name, work, keep=("*",), whole=(), cells=None, transform=None, sample=True):
    """Replay (or, when recording, run and store) every oracle/_ref binary called inside the block.
    keep: patterns of the output files to store (relative to work); whole: patterns of outputs stored complete;
    cells: {pattern: cells kept of the outputs it matches}; transform: {pattern: f} applied to a .npy output before
    it is stored (whole), for a test that needs less than the array; sample=False stores every output complete
    (small outputs a test needs whole)."""
    cells = dict(cells or {})
    from oracle import oracle
    path = os.path.join(RUNS, name + ".npz")
    work = os.path.abspath(work)
    ref_dir = os.path.abspath(oracle.REFDIR)
    calls, arrays, produced = [], {}, set()
    if not RECORD:
        calls, arrays = _load_runs(path)

    def norm(cmd):
        return [str(c).replace(ref_dir, "<ref>").replace(work, "<work>") for c in cmd]

    def runner(cmd, env=None, timeout=None):
        inputs = {k: v for k, v in _files(work).items() if k not in produced}
        if RECORD:
            r = subprocess.run(cmd, capture_output=True, text=True, env=env, timeout=timeout)
            after = _files(work)
            c = {"cmd": norm(cmd), "inputs": inputs, "rc": r.returncode, "stdout": r.stdout, "stderr": r.stderr,
                 "outputs": []}
            pays = {}
            outs = [rel for rel in sorted(after) if not (rel in inputs and inputs[rel] == after[rel])
                    and any(fnmatch.fnmatch(rel, k) for k in keep)]
            size = {rel: _payload(open(os.path.join(work, rel), "rb").read())[1].size if not rel.endswith(".npy")
                    else np.load(os.path.join(work, rel)).size for rel in outs}
            group = {rel: next((pat for pat in cells if fnmatch.fnmatch(rel, pat)), None) for rel in outs}
            total = {g: sum(size[rel] for rel in outs if group[rel] == g) for g in set(group.values())}

            def share(rel, n):
                return _share(n, cells.get(group[rel], BUDGET), total[group[rel]])

            for rel in outs:
                full = not sample or any(fnmatch.fnmatch(rel, k) for k in whole)
                key = f"c{len(calls)}_{len(c['outputs'])}"
                o = {"path": rel, "key": key}
                p = os.path.join(work, rel)
                fn = next((f for pat, f in (transform or {}).items() if fnmatch.fnmatch(rel, pat)), None)
                if rel.endswith(".npy"):
                    a = np.load(p)
                    a = fn(a) if fn else a
                    o.update(kind="npy", shape=list(a.shape), dtype=a.dtype.str, n=int(a.size))
                    o["whole"] = bool(fn) or full
                    o["k"] = int(a.size) if o["whole"] else share(rel, a.size)
                    arrays[key] = a.ravel()[sample_index(a.size, o["k"])]
                else:
                    raw = open(p, "rb").read()
                    blocks, pay = _payload(raw)
                    if not blocks:
                        o["kind"] = "bytes"
                        arrays[key] = np.frombuffer(raw, np.uint8)
                    else:
                        skel, i = [], 0
                        for off, cnt in blocks:
                            skel.append(raw[i:off])
                            i = off + 4 * cnt
                        o.update(kind="kaldi", n=int(pay.size))
                        arrays[key + "_skeleton"] = np.frombuffer(b"".join(skel) + raw[i:], np.uint8)
                        for src in inputs:
                            if src not in pays:
                                pays[src] = _payload(open(os.path.join(work, src), "rb").read())[1]
                            if pays[src].size == pay.size and np.array_equal(pays[src].view(np.uint32), pay.view(np.uint32)):
                                o["payload_of"] = src
                                break
                        else:
                            o["ks"] = [cnt if full else share(rel, cnt) for _, cnt in blocks]
                            parts, i = [], 0
                            for (_, cnt), k in zip(blocks, o["ks"]):
                                parts.append(pay[i:i + cnt][sample_index(cnt, k)])
                                i += cnt
                            arrays[key] = np.concatenate(parts)
                c["outputs"].append(o)
            calls.append(c)
            produced.update(rel for rel in after if inputs.get(rel) != after[rel])
            return r
        assert calls, f"{name}: more reference calls than stored"
        c = calls.pop(0)
        assert c["cmd"] == norm(cmd), f"{name}: command differs from the stored run:\n{c['cmd']}\n{norm(cmd)}"
        assert c["inputs"] == inputs, f"{name}: the inputs differ from those of the stored run"
        for o in c["outputs"]:
            p = os.path.join(work, o["path"])
            os.makedirs(os.path.dirname(p), exist_ok=True)
            if o["kind"] == "npy":
                a = _unsampled(arrays[o["key"]], o["n"], o["k"], np.dtype(o["dtype"]))
                np.save(p, a.reshape(o["shape"]))
            elif o["kind"] == "bytes":
                open(p, "wb").write(arrays[o["key"]].tobytes())
            else:
                skel = arrays[o["key"] + "_skeleton"].tobytes()
                blocks = _float_blocks(skel, cut=True)
                if "payload_of" in o:
                    pay = _payload(open(os.path.join(work, o["payload_of"]), "rb").read())[1]
                else:
                    vals, parts, i = arrays[o["key"]], [], 0
                    for (_, cnt), k in zip(blocks, o["ks"]):
                        n = sample_index(cnt, k).size
                        parts.append(_unsampled(vals[i:i + n], cnt, k))
                        i += n
                    pay = np.concatenate(parts) if parts else vals
                parts, i, j = [], 0, 0
                for off, cnt in blocks:
                    parts += [skel[j:off], pay[i:i + cnt].astype("<f4").tobytes()]
                    i, j = i + cnt, off
                open(p, "wb").write(b"".join(parts) + skel[j:])
            produced.add(o["path"])
        return subprocess.CompletedProcess(cmd, c["rc"], c["stdout"], c["stderr"])

    oracle.RUNNER = runner
    try:
        yield
    finally:
        oracle.RUNNER = None
    if RECORD:
        os.makedirs(RUNS, exist_ok=True)
        _save_runs(path, calls, arrays)
    else:
        assert not calls, f"{name}: {len(calls)} stored reference call(s) not made"
