"""CPU: the a-contrario RANSAC oracle (oracle/acransac_oracle.cpp, SURVEY §8f N4) against the committed golden outputs
of the reference's own ACRANSAC + ACKernelAdaptor<SevenPointSolver, EpipolarDistanceError, UnnormalizerT>
(tests/golden/reference_outputs.json "geom_F", reference_oracle_cases.npz)."""
import json
import os
import sys

import numpy as np
import pytest

import checkers as ck
from openmvg_b200 import synth

sys.path.insert(0, os.path.join(os.path.dirname(__file__), "golden"))
_ALL = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "reference_outputs.json")))
GOLD = _ALL.get("geom_F", [])
GOLD_H = _ALL.get("geom_H", [])
REF = np.load(os.path.join(os.path.dirname(__file__), "golden", "reference_oracle_cases.npz"))


def case_inputs(c):
    wh = tuple(c.get("wh", (1000, 1000)))
    xI, xJ, _ = synth.two_view_matches(c["n"], c["outlier_frac"], seed=c["seed"], wh=wh)
    return xI, xJ, (wh[0], wh[1], wh[0], wh[1])


def case_inputs_h(c):
    wh = tuple(c.get("wh", (1000, 1000)))
    xI, xJ, _ = synth.two_view_matches(c["n"], c["outlier_frac"], seed=c["seed"], wh=wh, planar=True)
    return xI, xJ, (wh[0], wh[1], wh[0], wh[1])


def inlier_hash(inliers):
    a = np.ascontiguousarray(np.stack([inliers, inliers], 1).astype(np.uint32))
    return str(int(ck.oracle().oracle_fnv1a_ij(ck._P(a), ck.ctypes.c_int64(len(a)))))


def check_against_gold(r, c):
    assert len(r["inliers"]) == c["n_inliers"] and inlier_hash(r["inliers"]) == c["inliers_fnv1a"], c["name"]
    em, nfa = float(c["error_max"]), float(c["min_nfa"])
    if np.isfinite(em):
        assert abs(r["error_max"] - em) <= 1e-9 * max(1.0, abs(em)) and abs(r["min_nfa"] - nfa) <= 1e-9 * max(1.0, abs(nfa))
    else:
        assert r["error_max"] == em and r["min_nfa"] == nfa
    if c["n_inliers"]:
        F = r["F"] / np.linalg.norm(r["F"]); G = np.array(c["F_unit"]).reshape(3, 3)
        assert min(np.abs(F - G).max(), np.abs(F + G).max()) <= 1e-7


@pytest.mark.parametrize("c", GOLD, ids=lambda c: c["name"])
def test_oracle_against_reference_golden(c):
    xI, xJ, wh = case_inputs(c)
    check_against_gold(ck.oracle_acransac_fundamental(xI, xJ, wh, 4.0, 2048), c)


def test_some_cases_exercise_every_branch():
    """The golden set covers: early exit without a model, too few matches, a model found in max-consensus mode at
    iteration 0 and later, the focused-sampling phase."""
    names = {c["name"]: c for c in GOLD}
    assert names["p200_no_model"]["n_inliers"] == 0 and names["p7"]["n_inliers"] == 0 and names["p8"]["n_inliers"] == 0
    assert names["p1500_half_outliers"]["n_inliers"] > 600 and names["p18"]["n_inliers"] >= 0


def reference_case(prefix):
    """The reference's ACRANSAC result for one seed (tests/golden/reference_oracle_cases.npz)."""
    return {k: REF[f"{prefix}.{k}"] for k in ("inliers", "error_max", "min_nfa") if f"{prefix}.{k}" in REF.files}


@pytest.mark.parametrize("seed", range(20, 32))
def test_oracle_against_compiled_reference(seed):
    rng = np.random.default_rng(seed)
    n = int(rng.integers(9, 900)); of = float(rng.uniform(0.0, 0.7)); it = int(rng.choice([64, 256, 2048]))
    xI, xJ, _ = synth.two_view_matches(n, of, seed=seed, wh=(1600, 1200))
    wh = (1600, 1200, 1600, 1200)
    r = reference_case(f"geom_F.{seed}"); o = ck.oracle_acransac_fundamental(xI, xJ, wh, 4.0, it)
    assert np.array_equal(r["inliers"], o["inliers"]), (n, of, it)
    assert r["error_max"] == o["error_max"] or abs(r["error_max"] - o["error_max"]) <= 1e-9 * abs(r["error_max"])
    assert r["min_nfa"] == o["min_nfa"] or abs(r["min_nfa"] - o["min_nfa"]) <= 1e-9 * abs(r["min_nfa"])


@pytest.mark.parametrize("c", GOLD_H, ids=lambda c: c["name"])
def test_homography_oracle_against_reference_golden(c):
    """The homography model (GeometricFilter_HMatrix_AC: 4-point DLT, asymmetric transfer error, point-to-point NFA)."""
    xI, xJ, wh = case_inputs_h(c)
    check_against_gold(ck.oracle_acransac_homography(xI, xJ, wh, 4.0, 2048), c)


@pytest.mark.parametrize("seed", range(40, 48))
def test_homography_oracle_against_compiled_reference(seed):
    rng = np.random.default_rng(seed)
    n = int(rng.integers(5, 900)); of = float(rng.uniform(0.0, 0.7)); it = int(rng.choice([64, 2048]))
    xI, xJ, _ = synth.two_view_matches(n, of, seed=seed, wh=(1600, 1200), planar=True)
    wh = (1600, 1200, 1600, 1200)
    r = reference_case(f"geom_H.{seed}"); o = ck.oracle_acransac_homography(xI, xJ, wh, 4.0, it)
    assert np.array_equal(r["inliers"], o["inliers"]), (n, of, it)
    assert r["min_nfa"] == o["min_nfa"] or abs(r["min_nfa"] - o["min_nfa"]) <= 1e-9 * abs(r["min_nfa"])
