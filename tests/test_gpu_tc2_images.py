"""The second-generation tcgen05 pass (k <= 16, kl_tiled_tc2.cu) reproduces, bit for bit, the factors, iteration counts, stop
reasons and objectives that the pass computed before its V operand images moved into a producer kernel and its X tiles into
the step-contiguous swizzled layout (tests/golden/tc2_pass.npz, written by tests/golden/make_tc2_golden.py: small outputs whole,
the factors as the SHA-256 of their bytes plus 64 sampled entries).  Neither change touches the arithmetic: the same MMA
sequence, the same per-unit FP32 drains in the same order, the same per-element quotient."""
import importlib.util
import os

import numpy as np
import pytest

import nmfk_b200 as nb

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))


def _golden_module():
    spec = importlib.util.spec_from_file_location("make_tc2_golden", os.path.join(HERE, "golden", "make_tc2_golden.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


G = _golden_module()


@pytest.fixture(scope="module")
def ctx():
    c = nb.Context()
    yield c
    c.close()


@pytest.fixture(scope="module")
def golden():
    return dict(np.load(G.GOLDEN))


def test_golden_cases_cover_the_tc2_range():
    ks = {case[3] for case in G.CASES}
    assert {1, 5, 8, 9, 16} <= ks
    assert any(case[4] % 2 for case in G.CASES)  # shadow units
    assert any(case[1] % 128 and case[2] % 64 for case in G.CASES)
    assert any(case[6] for case in G.CASES) and any("Hfixed" in case[5] for case in G.CASES) and any("Wfixed" in case[5] for case in G.CASES)


@pytest.mark.parametrize("case", G.CASES, ids=[c[0] for c in G.CASES])
def test_tc2_pass_bit_identical_to_golden(ctx, golden, case):
    rec = G.compact(G.run_case(ctx, case))
    assert sorted(rec) == sorted(k for k in golden if k.startswith(case[0] + "_"))
    # samples and small arrays first: a mismatch there reports by how much the run differs
    for key in sorted(rec, key=lambda k: k.endswith("_sha256")):
        val, ref = rec[key], golden[key]
        assert val.shape == ref.shape and val.dtype == ref.dtype, key
        assert np.array_equal(val, ref), (key, float(np.max(np.abs(val.astype(np.float64) - ref.astype(np.float64)))))


def test_golden_has_restarts_stopping_at_different_iterations(golden):
    its = golden["k5_r5_stops_iters"]
    assert len(set(its.tolist())) > 1, its
