"""CPU tests: the restatement of frame-level cross-entropy (tests/ce_util.py) that the GPU tests use, held to the
reference's own CE::EvalParallel (src/net/ce-loss.cc:94-169) run through oracle/_ref/ref_ce_cpu, replayed from
tests/golden/runs where the reference is absent (tests/util.py:stored_runs)."""
import tempfile

import numpy as np
import pytest

import ce_util
from util import assert_close, stored_runs

# name: (seed, S, T, K); the small case is stored whole, the K = 4000 one keeps a sample of the gradient
CASES = {"small": (0, 8, 40, 12), "k4000": (1, 4, 12, 4000)}


def reference(name):
    seed, S, T, K = CASES[name]
    frames, packed, y = ce_util.reference_case(seed, S, T, K)
    d = tempfile.mkdtemp(prefix="eesen_b200_ce_ref_")
    with stored_runs(f"ce_eval_{name}", d, keep=("out/*",), cells={"out/ce_diff.npy": 4096},
                     sample=name != "small"):
        diff, info = ce_util.run_reference_ce(d, y, packed, frames)
    return (frames, packed, y, T, S), diff, info


@pytest.mark.parametrize("name", sorted(CASES))
@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_restatement_matches_reference_ce_evalparallel(name, dtype):
    (frames, packed, y, T, S), rdiff, info = reference(name)
    diff, obj, correct, valid = ce_util.ce_eval(y, frames, packed, dtype)
    if dtype == np.float32:
        assert_close("diff", diff, rdiff, atol=0, stored=True)      # bit-equal where stored
    else:
        assert_close("diff", diff, rdiff, atol=1e-7, stored=True)
    assert abs(obj - info["obj"]) <= 1e-6 * abs(info["obj"])
    assert correct == info["correct"]
    assert info["frames"] == T * S and info["sequences"] == S      # the reference counts padded rows
    assert valid == int(frames.sum())
