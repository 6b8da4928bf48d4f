"""GPU tests: the fused CE kernel and the CE train step against the reference's own code, replayed from stored runs
of the reference's CPU build (tests/util.py:stored_runs):
  * ce_eval against CE::EvalParallel (oracle/_ref/ref_ce_cpu): diff bit-equal, objective rel 1e-6, correct exact;
  * one train_step_ce against the reference's CPU Net: Propagate (ref_dump_cpu), CE::EvalParallel on its posteriors
    (ref_ce_cpu), Backpropagate + explicit SGD driven by that gradient (ref_dump_cpu --diff-in), at the bounds of
    tests/test_gpu_parity.py (layer outputs and obj_diff abs 2e-5, parameters abs 2e-6)."""
import os
import tempfile

import numpy as np
import pytest

import ce_util
from test_ce_reference import CASES, reference
from util import assert_close, case, model_file, stored_runs
from eesen_b200 import binding, kaldi_io
from oracle import oracle

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("name", sorted(CASES))
def test_ce_eval_vs_reference(ctx, name):
    import torch
    (frames, packed, y, T, S), rdiff, info = reference(name)
    K = y.shape[1]
    ld = (K + 3) // 4 * 4
    yp = np.zeros((T * S, ld), np.float32); yp[:, :K] = y
    d_y = torch.from_numpy(yp).cuda()
    d_len = torch.from_numpy(frames).cuda()
    d_tgt = torch.from_numpy(packed).cuda()
    d_diff = torch.zeros((T * S, ld), dtype=torch.float32, device="cuda")
    d_st = torch.zeros(3, dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()
    ctx.ce_eval(T, S, K, d_len, d_y, ld, d_tgt, d_diff, ld, d_st)
    ctx.synchronize()
    st = d_st.cpu().numpy()
    assert_close("diff", d_diff.cpu().numpy()[:, :K], rdiff, atol=0, stored=True)
    assert abs(st[0] - info["obj"]) <= 1e-6 * abs(info["obj"])
    assert (st[1], st[2]) == (info["correct"], frames.sum())


STEP_KEEP = ("out1/net_out.npy", "ce/*", "out2/obj_diff.npy", "out2/model_out", "out2/out_l*")


def reference_step():
    """the reference's CPU CE step on the `small` case (records or replays small_ce_cpu_step)"""
    w, net, b = case("small", 21, 22)
    lr, mom = 1e-3, 0.9
    targets = ce_util.random_targets(b.frames, w.classes, 23)
    packed = ce_util.pack_targets(targets, b.frames, b.T)
    d = tempfile.mkdtemp(prefix="eesen_b200_ce_step_")
    kaldi_io.write_model(d + "/model", net)
    kaldi_io.write_batch_file(d + "/batch.bin", b)
    np.save(d + "/zero.npy", np.zeros((b.T * b.S, w.classes), np.float32))
    os.makedirs(d + "/ce")
    with stored_runs("small_ce_cpu_step", d, keep=STEP_KEEP, whole=("out1/net_out.npy", "ce/*"),
                     cells={"out2/*": 1024}):
        # the reference's forward (the zero gradient of this first run is discarded with its model)
        oracle.run_reference("cpu", d + "/model", d + "/batch.bin", d + "/out1", lr, mom, diff_in=d + "/zero.npy")
        y = np.load(d + "/out1/net_out.npy")
        rdiff, info = ce_util.run_reference_ce(d + "/ce", y, packed, b.frames)
        oracle.run_reference("cpu", d + "/model", d + "/batch.bin", d + "/out2", lr, mom,
                             diff_in=d + "/ce/out/ce_diff.npy")
    return (w, net, b, lr, mom, targets), d, y, rdiff, info


def test_train_step_ce_vs_reference_cpu_step(ctx):
    (w, net, b, lr, mom, targets), d, y, rdiff, info = reference_step()
    ref = oracle.load_dump(d + "/out2")
    n = binding.Net(ctx, model_file(net))
    n.set_train_options(lr, mom)
    st = n.train_step_ce(b.feats, b.frames, targets, True)
    L = len(net.layers)
    assert_close("net_out", n.get(L), y, atol=2e-5)
    for i in range(1, L + 1):
        assert_close(f"out_l{i}", n.get(i), ref[f"out_l{i}"], atol=2e-5, stored=True)
    assert_close("obj_diff", n.get(100), rdiff, atol=2e-5)
    assert abs(st["obj"] - info["obj"]) <= 2e-5 * abs(info["obj"])
    assert st["padded"] == info["frames"] and st["frames"] == b.valid_frames
    m2 = kaldi_io.read_model(d + "/out2/model_out")
    assert_close("params", n.params(), m2.flat_params(), atol=2e-6, stored=True)
    assert not np.array_equal(m2.flat_params()[np.isfinite(m2.flat_params())],
                              net.flat_params()[np.isfinite(m2.flat_params())]), "the reference step did not train"
    n.close()
