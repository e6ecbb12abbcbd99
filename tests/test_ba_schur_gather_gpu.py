"""The reduced camera matrix Scc is gathered per block from pair lists built at context creation
(schur_gather_kernel), and landmarks outside those lists still add to it with atomics afterwards (schur_kernel).
These scenes hit the corners of that split: wide rows of Scc on the PCG path, landmarks on both sides of the
32-observation limit, landmarks seen through two intrinsic groups, control points, and landmarks removed from a
context whose lists were built before.  Each is checked against the oracle with the tolerances of test_ba_gpu.py."""
import numpy as np
import pytest

import checkers as ck
from openmvg_b200 import synth

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ba():
    from openmvg_b200 import ba as m
    return m


def _concat(a, b):
    """Scene a with the landmarks and observations of scene b (same cameras) appended."""
    s = dict(a)
    n0 = len(a["points"])
    s["points"] = np.ascontiguousarray(np.concatenate([a["points"], b["points"]]))
    s["obs_view"] = np.ascontiguousarray(np.concatenate([a["obs_view"], b["obs_view"]]))
    s["obs_point"] = np.ascontiguousarray(np.concatenate([a["obs_point"], b["obs_point"] + n0]).astype(np.int32))
    s["obs_xy"] = np.ascontiguousarray(np.concatenate([a["obs_xy"], b["obs_xy"]]))
    return s


def _check(g, o, initial=True):
    assert g["ok"] and o["usable"]
    if initial:
        assert abs(g["initial_cost"] - o["initial_cost"]) <= 1e-12 * o["initial_cost"]
    assert abs(g["final_cost"] - o["final_cost"]) <= 1e-6 * o["final_cost"], (g["final_cost"], o["final_cost"])
    assert g["iterations"] == o["iterations"]


def test_dense_camera_graph_on_the_pcg_path(ba, monkeypatch):
    """31 consecutive cameras per landmark on a ring of 64: every row of Scc has 61 blocks, and each diagonal block
    sums ~240 landmark terms against ~8 per off-diagonal block."""
    monkeypatch.setenv("OMVG_BA_DENSE_MAX", "0"); monkeypatch.setenv("OMVG_BA_DENSE2_MAX", "0")
    s = synth.ba_scene(64, 500, 31, seed=11)
    g = ba.solve(s)
    assert g["pcg_iterations"] > 0
    _check(g, ck.oracle_ba_solve(s))


def test_landmarks_with_32_and_33_observations(ba):
    """32 observations: the last landmark size in the pair lists; 33: left to the atomic kernel, which then adds to
    blocks the gather already wrote (both triangles)."""
    s = _concat(_concat(synth.ba_scene(40, 60, 32, seed=2), synth.ba_scene(40, 60, 33, seed=3)), synth.ba_scene(40, 400, 5, seed=4))
    assert set(np.bincount(s["obs_point"])) == {32, 33, 5}
    _check(ba.solve(s), ck.oracle_ba_solve(s))


def test_two_intrinsic_groups(ba, monkeypatch):
    """Even and odd cameras in different intrinsic groups: stride-2 landmarks stay in one group (pair lists), the
    others see both (atomic kernel).  On the direct solve and on the PCG path."""
    s = synth.ba_scene(48, 1500, 6, seed=6, n_intrinsics=2)
    o = ck.oracle_ba_solve(s)
    _check(ba.solve(s), o)
    monkeypatch.setenv("OMVG_BA_DENSE_MAX", "0"); monkeypatch.setenv("OMVG_BA_DENSE2_MAX", "0")
    _check(ba.solve(s), o)


def test_control_points(ba):
    """Fixed, weighted, loss-free control-point landmarks are in the pair lists like any other landmark."""
    s = synth.add_gcp(synth.ba_scene(30, 900, 6, seed=8), 6, weight=12.0)
    _check(ba.solve(s), ck.oracle_ba_solve(s))


def test_remove_points_after_a_solve(ba, monkeypatch):
    """Lists built at creation stay valid when landmarks are removed after a first solve: the removed tracks then
    contribute nothing, as in a scene built without them."""
    monkeypatch.setenv("OMVG_BA_DENSE_MAX", "0"); monkeypatch.setenv("OMVG_BA_DENSE2_MAX", "0")
    s = synth.ba_scene(50, 2000, 6, seed=9)
    ctx = ba.BAContext(s)
    ctx.run()
    mask = np.zeros(len(s["points"]), np.uint8); mask[::5] = 1
    removed, nt = ctx.remove_points(mask)
    assert nt == int(mask.sum())
    ctx.reset()
    b = ctx.run(); ctx.close()
    keep = ~removed; remap = np.cumsum(mask == 0) - 1
    d = dict(s); d.update(points=np.ascontiguousarray(s["points"][mask == 0]), obs_view=np.ascontiguousarray(s["obs_view"][keep]),
                          obs_point=np.ascontiguousarray(remap[s["obs_point"][keep]].astype(np.int32)), obs_xy=np.ascontiguousarray(s["obs_xy"][keep]))
    o = ck.oracle_ba_solve(d)
    assert abs(b["final_cost"] - o["final_cost"]) <= 1e-7 * o["final_cost"] and b["iterations"] == o["iterations"]
