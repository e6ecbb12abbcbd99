"""CPU: the BA oracle against the committed golden outputs of the reference's own
Bundle_Adjustment_Ceres::Adjust (tests/golden/reference_outputs.json, reference_oracle_cases.npz)."""
import json
import os
import sys

import numpy as np
import pytest

import checkers as ck

sys.path.insert(0, os.path.join(os.path.dirname(__file__), "golden"))
from make_golden import ORACLE_BA_EXT_KW, ORACLE_BA_KW, kw_key
from openmvg_b200 import synth

G = os.path.join(os.path.dirname(__file__), "golden")
GOLD = json.load(open(os.path.join(G, "reference_outputs.json")))
REF = np.load(os.path.join(G, "reference_oracle_cases.npz"))
SMALL = [c for c in GOLD["ba"] if c["scene"]["n_cams"] <= 100]


@pytest.mark.parametrize("case", SMALL, ids=lambda c: c["name"])
def test_golden_final_cost(case):
    s = synth.ba_scene(**case["scene"])
    o = ck.oracle_ba_solve(s, **case["opts"])
    assert o["usable"] == case["ok"]
    assert abs(o["initial_cost"] - case["initial_cost"]) <= 1e-12 * case["initial_cost"]
    # the golden cost is recomputed from the scene Adjust RETURNS (write-back rules included)
    returned = ck.oracle_ba_cost(s, o["poses"], o["intrinsics"], o["points"], use_loss=case["opts"].get("use_loss", 1))
    assert abs(returned - case["final_cost"]) <= 1e-9 * case["final_cost"]        # observed: ~1e-15
    if case["opts"].get("extrinsics_opt", 6) != 2:
        assert abs(o["final_cost"] - case["final_cost"]) <= 1e-9 * case["final_cost"]
    assert o["iterations"] == case["iterations"] and o["successful"] == case["successful"] and o["unsuccessful"] == case["unsuccessful"]
    assert ("Function tolerance" in case["termination"]) == (o["termination"] == 0)


def test_cost_matches_reference_formula():
    """1/2 sum rho(|r|^2), Huber a=16 (sfm_data_BA_ceres.cpp:249; loss_function.cc:47-61)."""
    s = synth.ba_scene(6, 100, 4, seed=1, outlier_frac=0.3)
    _, r, *_ = ck.oracle_ba_eval(s, use_loss=0)
    sq = (r ** 2).sum(1)
    want = 0.5 * np.where(sq <= 256.0, sq, 32.0 * np.sqrt(sq) - 256.0).sum()
    assert abs(ck.oracle_ba_cost(s) - want) <= 1e-12 * want
    assert (sq > 256).any() and (sq <= 256).any()


def test_jacobian_against_finite_differences():
    s = synth.ba_scene(4, 30, 4, seed=9, model=4)
    s["intrinsics"][:, 3:] = s["gt_dist"][3:]
    _, r0, Ji, Jc, Jp = ck.oracle_ba_eval(s, use_loss=0)
    h = 1e-6
    for name, J, arr, width in (("poses", Jc, "poses", 6), ("points", Jp, "points", 3), ("intrinsics", Ji, "intrinsics", 8)):
        for k in range(width):
            s2 = dict(s); a = s[arr].copy(); a[:, k] += h; s2[arr] = a
            _, r1, *_ = ck.oracle_ba_eval(s2, use_loss=0)
            fd = (r1 - r0) / h
            assert np.abs(fd - J[:, :, k]).max() <= 2e-4 * max(1.0, np.abs(J[:, :, k]).max()), (name, k)


def reference_case(prefix):
    """The reference's results for one case of tests/golden/reference_oracle_cases.npz (make_golden.py oracle_cases)."""
    return {k[len(prefix) + 1:]: REF[k] for k in REF.files if k.startswith(prefix + ".") and "." not in k[len(prefix) + 1:]}


def registered_scene(s, r):
    """The scene after the reference's pre-solve registration of the priors (ck.ref_ba_register_priors)."""
    t = dict(s)
    if r["reg_fit"] >= 0:
        t.update(poses=r["reg_poses"].copy(), points=r["reg_points"].copy(), prior_center=r["reg_prior_center"].copy(),
                 prior_huber_a=float(r["reg_fit"]) ** 2)
    return t


@pytest.mark.parametrize("kw", ORACLE_BA_KW)
def test_against_compiled_reference(kw):
    s = synth.ba_scene(12, 400, 5, seed=13, outlier_frac=0.01)
    r = reference_case("ba." + kw_key(kw))
    o = ck.oracle_ba_solve(s, **kw)
    assert r["ok"] and o["usable"]
    assert abs(o["final_cost"] - r["final_cost"]) <= 1e-9 * r["final_cost"]
    assert o["iterations"] == r["iterations"]
    assert np.abs(o["points"] - r["points"]).max() < 1e-7 and np.abs(o["poses"][:, 3:] - r["poses"][:, 3:]).max() < 1e-7
    from scipy.spatial.transform import Rotation   # angle-axis is ambiguous at theta ~ pi: compare the rotations
    Ro = Rotation.from_rotvec(o["poses"][:, :3]).as_matrix(); Rr = Rotation.from_rotvec(r["poses"][:, :3]).as_matrix()
    assert np.abs(Ro - Rr).max() < 1e-7


# ---- ground control points and pose-centre priors (SURVEY §8a B17)
@pytest.mark.parametrize("case", GOLD.get("ba_ext", []), ids=lambda c: c["name"])
def test_golden_gcp_and_priors(case):
    """Oracle vs the reference Adjust with control points / motion priors (golden = cost of the scene
    the reference returned, GCP and prior terms included)."""
    s = ck.golden_ext_scene(case)
    o = ck.oracle_ba_solve(s, **case["opts"])
    assert o["usable"] and case["ok"]
    assert abs(o["final_cost"] - case["final_cost"]) <= 1e-9 * case["final_cost"], (o["final_cost"], case["final_cost"])
    assert o["iterations"] == case["iterations"]
    if s.get("point_fixed") is not None:                      # GCP landmarks are constant
        f = s["point_fixed"].astype(bool)
        assert np.array_equal(o["points"][f], s["points"][f])
    ret = dict(s); ret.update(poses=o["poses"], intrinsics=o["intrinsics"], points=o["points"])
    assert abs(ck.oracle_ba_cost(ret, use_loss=case["opts"].get("use_loss", 1)) - o["final_cost"]) <= 1e-12 * o["final_cost"]


def test_gcp_and_priors_against_compiled_reference():
    s = synth.add_priors(synth.add_gcp(synth.ba_scene(12, 300, 5, seed=3), 6, weight=15.0), sigma=0.02)   # GCPs live in the priors' frame
    r = reference_case("ba_ext")
    t, fit, cen = registered_scene(s, r), r["reg_fit"], r["reg_centroid"]
    assert fit == r["prior_fit"] and fit > 0
    o = ck.oracle_ba_solve(t)
    assert abs(o["final_cost"] - r["final_cost"]) <= 1e-9 * r["final_cost"]
    assert o["iterations"] == r["iterations"]
    # the reference undoes only the centring (sfm_data_BA_ceres.cpp:572): same for the oracle's result
    assert np.abs((o["points"] + cen) - r["points"]).max() <= 1e-7


def test_zero_weight_removes_observation_exactly():
    """Weight 0 must equal deleting the observation (the rejection loop relies on it)."""
    s = synth.ba_scene(10, 300, 5, seed=4, outlier_frac=0.05)
    rng = np.random.default_rng(0)
    keep = rng.random(len(s["obs_view"])) > 0.1
    w = dict(s); w["obs_weight"] = keep.astype(np.float64)
    d = dict(s); d["obs_view"] = np.ascontiguousarray(s["obs_view"][keep]); d["obs_point"] = np.ascontiguousarray(s["obs_point"][keep]); d["obs_xy"] = np.ascontiguousarray(s["obs_xy"][keep])
    a = ck.oracle_ba_solve(w); b = ck.oracle_ba_solve(d)
    assert abs(a["final_cost"] - b["final_cost"]) <= 1e-9 * b["final_cost"] and a["iterations"] == b["iterations"]   # (OpenMP atomics reorder sums)


@pytest.mark.parametrize("kw", ORACLE_BA_EXT_KW, ids=kw_key)
def test_gcp_priors_option_mixes_against_compiled_reference(kw):
    """Control points + motion priors under the option mixes of Optimize_Options and another camera model."""
    r = reference_case("ba_ext." + kw_key(kw))
    kw = dict(kw); model = kw.pop("model", 1)
    s = synth.add_priors(synth.add_gcp(synth.ba_scene(14, 400, 5, seed=6, model=model), 5, weight=12.0), sigma=0.015)
    t = registered_scene(s, r)
    o = ck.oracle_ba_solve(t, **kw)
    assert r["ok"] and o["usable"]
    assert abs(o["final_cost"] - r["final_cost"]) <= 1e-8 * r["final_cost"], (o["final_cost"], r["final_cost"])
    assert o["iterations"] == r["iterations"]
