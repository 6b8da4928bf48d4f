"""CPU pins of the dropout variants of BiLstmParallel (SURVEY.md 8f N1): the restatement against the reference's
CPU build with the masks the reference itself drew (they come from a std::random_device-seeded generator, so the
comparison is always "same masks -> same numbers"; tests/golden/*_drop_*.npz store masks + outputs)."""
import os
import tempfile

import numpy as np
import pytest

from util import GOLDEN, assert_close, case, golden_arrays, stored_runs
from eesen_b200 import kaldi_io
from oracle import oracle

# name -> dropout options of every BiLSTM layer
VARIANTS = {
    "fwdstep": dict(forward=0.2, fw_step=True),
    "fwdseq": dict(forward=0.3, fw_seq=True),
    "nmlstep": dict(recurrent=0.25, rec_step=True, nml=True),
    "nmlseq": dict(recurrent=0.25, rec_seq=True, nml=True),
    "rnndropstep": dict(recurrent=0.2, rec_step=True, rnndrop=True),
    "rnndropseq": dict(recurrent=0.3, rec_seq=True, rnndrop=True),
    "fwd+nml": dict(forward=0.2, fw_step=True, recurrent=0.25, rec_seq=True, nml=True),
}


def drop_case(wl, variant, mseed=3, bseed=5):
    w, net, b = case(wl, mseed, bseed)
    for l in net.layers:
        if l.kind == "bilstm":
            l.dropout = dict(VARIANTS[variant])
    return w, net, b


def masks_from_dump(dump, net, b):
    """Reference layouts -> ours: forward [T*S x 2C] as is; recurrent fw|bw concatenated, step masks lose the two
    boundary slots ((T+2)*S rows -> T*S rows), sequence masks stay [S x 2C]."""
    out = []
    for li, l in enumerate(net.layers):
        if l.kind != "bilstm":
            out.append(None)
            continue
        m = {}
        if f"mask_{li}_fwd" in dump:
            m["fmask"] = dump[f"mask_{li}_fwd"]
        if f"mask_{li}_rec_fw" in dump:
            r = np.concatenate([dump[f"mask_{li}_rec_fw"], dump[f"mask_{li}_rec_bw"]], axis=1)
            if r.shape[0] != b.S:
                r = r[b.S:b.S + b.T * b.S]
            m["rmask"] = np.ascontiguousarray(r)
        out.append(m or None)
    return out


def check_mask_statistics(masks, net):
    for l, m in zip(net.layers, masks):
        if m is None:
            continue
        for key, p in (("fmask", l.dropout.get("forward", 0.0)), ("rmask", l.dropout.get("recurrent", 0.0))):
            if key in m:
                vals = np.unique(m[key])
                assert np.allclose(vals, [0.0, 1.0 / (1.0 - p)]) or np.allclose(vals, [1.0 / (1.0 - p)])
                seq_key = l.dropout.get("fw_seq") if key == "fmask" else l.dropout.get("rec_seq")
                n = m[key].shape[1] if seq_key else m[key].size        # independent draws
                assert abs((m[key] == 0).mean() - p) < 5.0 * np.sqrt(p * (1 - p) / n) + 0.01
        seq = l.dropout.get("fw_seq") and "fmask" in m
        if seq:   # SetRandUniformCol: one value per column, identical in every row (cpucompute/matrix.cc:952-965)
            assert np.all(m["fmask"] == m["fmask"][0])
        if l.dropout.get("rec_seq") and "rmask" in m:
            assert np.all(m["rmask"] == m["rmask"][0])


@pytest.mark.parametrize("variant", sorted(VARIANTS))
def test_oracle_dropout_matches_reference_cpu_live(variant):
    w, net, b = drop_case("tiny", variant)
    lr, mom = 1e-3, 0.9
    with tempfile.TemporaryDirectory() as d:
        kaldi_io.write_model(d + "/model", net)
        kaldi_io.write_batch_file(d + "/batch.bin", b)
        diff = (np.random.default_rng(1).standard_normal((b.feats.shape[0], w.classes)) * 0.1).astype(np.float32)
        rows_pad = np.concatenate([np.arange(b.frames[s], b.T) * b.S + s for s in range(b.S)])
        diff[rows_pad.astype(np.int64)] = 0.0          # CTC never produces gradient on padding frames
        np.save(d + "/diff.npy", diff)
        with stored_runs(f"tiny_drop_{variant.replace('+', '_')}_cpu", d, whole=("out/mask_*",),
                         keep=("out/out_l[1-9].npy", "out/in_diff.npy", "out/grad_*", "out/mask_*", "out/model_out")):
            oracle.run_reference("cpu", d + "/model", d + "/batch.bin", d + "/out", lr, mom, steps=1,
                                 diff_in=d + "/diff.npy")
        dump = oracle.load_dump(d + "/out")
        m2 = kaldi_io.read_model(d + "/out/model_out")
    masks = masks_from_dump(dump, net, b)
    assert any(m is not None for m in masks)
    check_mask_statistics(masks, net)
    on = oracle.OracleNet(net, np.float32)
    r = on.train_step(b, lr, mom, diff_override=diff, masks=masks)
    for i in range(1, len(net.layers) + 1):
        assert_close(f"out_l{i}", on.acts[i], dump[f"out_l{i}"], atol=2e-6, stored=True)
    assert_close("in_diff", r["in_diff"], dump["in_diff"], atol=1e-6, rtol=1e-4, stored=True)
    assert_close("corr", on.flat_corr(), golden_arrays(dump, net), atol=2e-5, rtol=1e-4, stored=True)
    assert_close("params", on.flat_params(), m2.flat_params(), atol=1e-6, stored=True)
    assert m2.layers[0].dropout == net.layers[0].dropout or all(
        abs(float(m2.layers[0].dropout.get(k, 0)) - float(v)) < 1e-7 for k, v in net.layers[0].dropout.items())


def golden_drop_case(wl, variant):
    """(net, batch, masks, fixture) of a committed dropout fixture (make_golden.py dropcpu)."""
    path = os.path.join(GOLDEN, f"{wl}_drop_{variant.replace('+', '_')}_refcpu.npz")
    g = np.load(path)
    w, net, b = drop_case(wl, variant)
    masks = []
    for li, l in enumerate(net.layers):
        m = {}
        if l.kind == "bilstm":
            if f"fmask_{li}" in g:
                m["fmask"] = g[f"fmask_{li}"].astype(np.float32) / np.float32(1.0 - l.dropout["forward"])
            if f"rmask_{li}" in g:
                m["rmask"] = g[f"rmask_{li}"].astype(np.float32) / np.float32(1.0 - l.dropout["recurrent"])
        masks.append(m or None)
    return w, net, b, masks, g


GOLDEN_CASES = [("tiny", v) for v in sorted(VARIANTS)] + [("small", "fwd+nml"), ("small", "rnndropstep")]


@pytest.mark.parametrize("wl,variant", GOLDEN_CASES)
def test_oracle_dropout_matches_reference_cpu_golden(wl, variant):
    w, net, b, masks, g = golden_drop_case(wl, variant)
    lr, mom = [float(v) for v in g["hyper"]]
    on = oracle.OracleNet(net, np.float32)
    r = on.train_step(b, lr, mom, diff_override=g["diff_in"], masks=masks)
    assert_close("last bilstm out", on.acts[w.layers], g[f"out_l{w.layers}"], atol=2e-6)
    assert_close("in_diff", r["in_diff"], g["in_diff"], atol=1e-6, rtol=1e-4)
    assert_close("corr", on.flat_corr(), golden_arrays(g, net), atol=2e-5, rtol=1e-4)
    assert_close("params", on.flat_params(), g["params_out"], atol=1e-6)
