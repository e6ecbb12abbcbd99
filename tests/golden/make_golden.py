"""Generate tests/golden/*.json|npz by running THE REFERENCE ITSELF (oracle/_ref, built by
oracle/Makefile from /root/reference sources in place) on seeded inputs from openmvg_b200.synth.
Run in the build container:  python tests/golden/make_golden.py
The inputs are regenerated from their seeds at test time; only the reference's outputs are stored."""
import hashlib
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
import checkers as ck          # noqa: E402
from openmvg_b200 import synth  # noqa: E402

MATCH_CASES = [
    dict(name="ragged5", counts=[300, 129, 2, 257, 1000], seed=11, ratio=0.8),
    dict(name="tiles3", counts=[128, 256, 384], seed=11, ratio=0.8),
    dict(name="ratio06", counts=[400, 500, 300], seed=4, ratio=0.6),
    dict(name="pair5000", counts=[5000, 5000], seed=11, ratio=0.8),
]
BA_CASES = [
    dict(name="c1", scene=dict(n_cams=10, n_points=500, obs_per_point=4), opts={}),
    dict(name="c30", scene=dict(n_cams=30, n_points=1500, obs_per_point=8), opts={}),
    dict(name="c100", scene=dict(n_cams=100, n_points=5000, obs_per_point=10), opts={}),
    dict(name="outliers", scene=dict(n_cams=16, n_points=800, obs_per_point=6, seed=5, outlier_frac=0.02), opts={}),
    dict(name="intr_none", scene=dict(n_cams=16, n_points=800, obs_per_point=6, seed=5, outlier_frac=0.02), opts=dict(intrinsics_opt=1)),
    dict(name="translation_only", scene=dict(n_cams=16, n_points=800, obs_per_point=6, seed=5, outlier_frac=0.02), opts=dict(extrinsics_opt=4)),
    dict(name="focal_rotation", scene=dict(n_cams=16, n_points=800, obs_per_point=6, seed=5, outlier_frac=0.02), opts=dict(intrinsics_opt=2, extrinsics_opt=2)),
    dict(name="structure_fixed", scene=dict(n_cams=16, n_points=800, obs_per_point=6, seed=5, outlier_frac=0.02), opts=dict(structure_opt=0)),
    dict(name="points_only", scene=dict(n_cams=16, n_points=800, obs_per_point=6, seed=5, outlier_frac=0.02), opts=dict(intrinsics_opt=1, extrinsics_opt=1)),
    dict(name="no_loss", scene=dict(n_cams=16, n_points=800, obs_per_point=6, seed=5, outlier_frac=0.02), opts=dict(use_loss=0)),
    dict(name="radial1", scene=dict(n_cams=14, n_points=700, obs_per_point=6, seed=8, model=2), opts={}),
    dict(name="radial3", scene=dict(n_cams=14, n_points=700, obs_per_point=6, seed=8, model=3), opts={}),
    dict(name="brown", scene=dict(n_cams=14, n_points=700, obs_per_point=6, seed=8, model=4), opts={}),
    dict(name="fisheye", scene=dict(n_cams=14, n_points=700, obs_per_point=6, seed=8, model=5), opts={}),
    dict(name="config2_1000_100k_1M", scene=dict(n_cams=1000, n_points=100000, obs_per_point=10), opts={}),
]

# Ground control points / pose-centre priors (sfm_data_BA_ceres.cpp:183-236, 398-472).  For prior cases the
# reference's own pre-solve registration (LMedS similarity + centring) is stored too, so the tests can hand
# the LM core the scene the reference's LM saw without the reference being present.
BA_EXT_CASES = [
    dict(name="gcp", scene=dict(n_cams=16, n_points=800, obs_per_point=6, seed=5), gcp=dict(n_gcp=8, weight=20.0), opts={}),
    dict(name="gcp_radial3", scene=dict(n_cams=14, n_points=700, obs_per_point=6, seed=8, model=3), gcp=dict(n_gcp=6, weight=10.0), opts={}),
    dict(name="priors", scene=dict(n_cams=16, n_points=800, obs_per_point=6, seed=5), priors=dict(sigma=0.01, offset=(5.0, -3.0, 2.0), scale=2.0), opts={}),
    dict(name="priors_weighted", scene=dict(n_cams=20, n_points=600, obs_per_point=5, seed=9), priors=dict(sigma=0.02, weight=(4.0, 4.0, 0.5)), opts=dict(intrinsics_opt=1)),
    dict(name="gcp_priors", scene=dict(n_cams=16, n_points=800, obs_per_point=6, seed=5), gcp=dict(n_gcp=8, weight=20.0), priors=dict(sigma=0.02), opts={}),
]


def ext_scene(c):
    s = synth.ba_scene(**c["scene"])
    if "gcp" in c:
        s = synth.add_gcp(s, **c["gcp"])
    if "priors" in c:
        s = synth.add_priors(s, **c["priors"])
    return s


def main_ext():
    path = os.path.join(HERE, "reference_outputs.json")
    out = json.load(open(path))
    out["ba_ext"] = []
    arrays = {}
    for c in BA_EXT_CASES:
        s = ext_scene(c)
        ref_opts = {k: v for k, v in c["opts"].items() if k in ("intrinsics_opt", "extrinsics_opt", "structure_opt", "use_loss")}
        r = ck.ref_ba_adjust_ex(s, threads=8, **ref_opts)
        e = dict(name=c["name"], scene=c["scene"], gcp=c.get("gcp"), priors=c.get("priors"), opts=c["opts"], ok=r["ok"],
                 initial_cost=r["initial_cost"], final_cost=r["final_cost"], iterations=r["iterations"], prior_fit=r["prior_fit"])
        if "priors" in c:
            t, fit, cen = ck.ref_ba_register_priors(s)
            assert fit == r["prior_fit"]
            e["centroid"] = [float(x) for x in cen]
            arrays[c["name"] + "_poses"] = t["poses"]; arrays[c["name"] + "_points"] = t["points"]; arrays[c["name"] + "_prior_center"] = t["prior_center"]
        out["ba_ext"].append(e)
        print("ba_ext", c["name"], r["initial_cost"], r["final_cost"], r["iterations"], r["prior_fit"])
    json.dump(out, open(path, "w"), indent=1)
    np.savez_compressed(os.path.join(HERE, "reference_ba_ext.npz"), **arrays)


CASCADE_CASES = [
    dict(name="ragged5", counts=[300, 129, 2, 257, 1000], seed=11, ratio=0.8),
    dict(name="three2k", counts=[2000, 1800, 1500], seed=4, ratio=0.8),
    dict(name="ratio06", counts=[1500, 1200, 0, 900], seed=11, ratio=0.6),
]


def main_cascade():
    """Cascade_Hashing_Matcher_Regions::Match (the reference's default matcher) on seeded collections, and the
    projections CascadeHasher::Init draws (std::mt19937 + std::normal_distribution, via the reference driver)."""
    path = os.path.join(HERE, "reference_outputs.json")
    out = json.load(open(path))
    out["cascade"] = []
    P, S = ck.ref_cascade_projections()
    np.savez_compressed(os.path.join(HERE, "cascade_projections.npz"), primary=P, secondary=S)
    arrays = {}
    for c in CASCADE_CASES:
        descs = synth.descriptors(len(c["counts"]), c["counts"], seed=c["seed"])
        pi, pj = synth.exhaustive_pairs(len(c["counts"]))
        off, ij = ck.ref_cascade_collection(descs, pi, pj, c["ratio"])
        fnv = int(ck.oracle().oracle_fnv1a_ij(ij.ctypes.data_as(ck.ctypes.c_void_p), ck.ctypes.c_int64(len(ij))))
        out["cascade"].append(dict(name=c["name"], counts=c["counts"], seed=c["seed"], ratio=c["ratio"], n_matches=int(len(ij)), fnv1a=str(fnv),
                                   offsets=[int(x) for x in off]))
        arrays["cascade_" + c["name"]] = ij
        print("cascade", c["name"], len(ij), fnv)
    json.dump(out, open(path, "w"), indent=1)
    np.savez_compressed(os.path.join(HERE, "reference_cascade_matches.npz"), **arrays)


def main_io():
    """File-format fixtures written by the reference's own writers (matching::Save, saveDescsToBinFile)."""
    pI = np.array([7, 2, 2, 9, 4], np.uint32); pJ = np.array([9, 5, 3, 11, 6], np.uint32)
    off = np.concatenate([[0], np.cumsum([3, 2, 4, 0, 1])]).astype(np.uint64)
    ij = np.random.default_rng(0).integers(0, 5000, (int(off[-1]), 2)).astype(np.uint32)
    for ext in ("txt", "bin"):
        ck.ref_save_matches(os.path.join(HERE, f"matches_fixture.{ext}"), pI, pJ, off, ij)
    ck.ref_save_descs(os.path.join(HERE, "desc_fixture.desc"), synth.descriptors(1, [37], seed=3)[0])


# Added after the first golden run (round 2): the sixth camera model and scenes with many intrinsic groups.  `more`
# appends / replaces these in reference_outputs.json without touching the rest.
BA_MORE_CASES = [
    dict(name="spherical", scene=dict(n_cams=14, n_points=700, obs_per_point=6, seed=8, model=7), opts={}),
    dict(name="spherical_rotation_only", scene=dict(n_cams=14, n_points=700, obs_per_point=6, seed=8, model=7), opts=dict(extrinsics_opt=2)),
    dict(name="intr40", scene=dict(n_cams=40, n_points=2000, obs_per_point=6, seed=3, n_intrinsics=40), opts={}),
    dict(name="intr200_radial3", scene=dict(n_cams=200, n_points=6000, obs_per_point=8, seed=3, n_intrinsics=200, model=3), opts={}),
    dict(name="intr5_brown", scene=dict(n_cams=30, n_points=1500, obs_per_point=8, seed=3, n_intrinsics=5, model=4), opts={}),
]


def main_more():
    path = os.path.join(HERE, "reference_outputs.json")
    out = json.load(open(path))
    names = {c["name"] for c in BA_MORE_CASES}
    out["ba"] = [c for c in out["ba"] if c["name"] not in names]
    for c in BA_MORE_CASES:
        s = synth.ba_scene(**c["scene"])
        ref_opts = {k: v for k, v in c["opts"].items() if k in ("intrinsics_opt", "extrinsics_opt", "structure_opt", "use_loss")}
        r = ck.ref_ba_adjust(s, threads=8, **ref_opts)
        out["ba"].append(dict(name=c["name"], scene=c["scene"], opts=c["opts"], ok=r["ok"], initial_cost=r["initial_cost"], final_cost=r["final_cost"],
                              iterations=r["iterations"], successful=r["successful"], unsuccessful=r["unsuccessful"], termination=r["termination"]))
        print("ba", c["name"], r["initial_cost"], r["final_cost"], r["iterations"], r["termination"])
    json.dump(out, open(path, "w"), indent=1)


# Geometric filter (SURVEY §8f N4): the reference's ACRANSAC with the fundamental-matrix kernel on seeded putative
# matches of one pair (synth.two_view_matches).  `geom` appends the section without touching the rest.
GEOM_CASES = [
    dict(name="p300", n=300, outlier_frac=0.3, seed=3), dict(name="p1500_half_outliers", n=1500, outlier_frac=0.5, seed=4),
    dict(name="p60", n=60, outlier_frac=0.2, seed=5), dict(name="p200_no_model", n=200, outlier_frac=0.9, seed=6),
    dict(name="p8", n=8, outlier_frac=0.0, seed=7), dict(name="p7", n=7, outlier_frac=0.0, seed=8),
    dict(name="p500", n=500, outlier_frac=0.3, seed=9), dict(name="p2500_wide", n=2500, outlier_frac=0.4, seed=10, wh=(4000, 3000)),
    dict(name="p30_clean", n=30, outlier_frac=0.0, seed=11), dict(name="p18", n=18, outlier_frac=0.1, seed=12),
]


def geom_case_inputs(c):
    wh = tuple(c.get("wh", (1000, 1000)))
    xI, xJ, _ = synth.two_view_matches(c["n"], c["outlier_frac"], seed=c["seed"], wh=wh)
    return xI, xJ, (wh[0], wh[1], wh[0], wh[1])


GEOM_H_CASES = [
    dict(name="h300", n=300, outlier_frac=0.3, seed=3), dict(name="h1500_half_outliers", n=1500, outlier_frac=0.5, seed=4),
    dict(name="h60", n=60, outlier_frac=0.2, seed=5), dict(name="h200_no_model", n=200, outlier_frac=0.9, seed=6),
    dict(name="h5", n=5, outlier_frac=0.0, seed=7), dict(name="h4", n=4, outlier_frac=0.0, seed=8),
    dict(name="h2500_wide", n=2500, outlier_frac=0.4, seed=10, wh=(4000, 3000)), dict(name="h12", n=12, outlier_frac=0.1, seed=10),
]


def main_geom():
    path = os.path.join(HERE, "reference_outputs.json")
    out = json.load(open(path))
    out["geom_F"] = []; out["geom_H"] = []
    for c in GEOM_H_CASES:
        wh = tuple(c.get("wh", (1000, 1000)))
        xI, xJ, _ = synth.two_view_matches(c["n"], c["outlier_frac"], seed=c["seed"], wh=wh, planar=True)
        r = ck.ref_acransac_homography(xI, xJ, (wh[0], wh[1], wh[0], wh[1]), 4.0, 2048)
        inl = np.ascontiguousarray(np.stack([r["inliers"], r["inliers"]], 1).astype(np.uint32))
        fnv = int(ck.oracle().oracle_fnv1a_ij(inl.ctypes.data_as(ck.ctypes.c_void_p), ck.ctypes.c_int64(len(inl))))
        Hn = r["F"] / np.linalg.norm(r["F"]) if len(r["inliers"]) else r["F"]
        out["geom_H"].append(dict(c, n_inliers=int(len(r["inliers"])), inliers_fnv1a=str(fnv), error_max=repr(r["error_max"]), min_nfa=repr(r["min_nfa"]),
                                  F_unit=[float(v) for v in Hn.reshape(-1)]))
        print("geom H", c["name"], len(r["inliers"]), r["error_max"], r["min_nfa"])
    for c in GEOM_CASES:
        xI, xJ, wh = geom_case_inputs(c)
        r = ck.ref_acransac_fundamental(xI, xJ, wh, 4.0, 2048)
        inl = np.ascontiguousarray(np.stack([r["inliers"], r["inliers"]], 1).astype(np.uint32))
        fnv = int(ck.oracle().oracle_fnv1a_ij(inl.ctypes.data_as(ck.ctypes.c_void_p), ck.ctypes.c_int64(len(inl))))
        Fn = r["F"] / np.linalg.norm(r["F"]) if len(r["inliers"]) else r["F"]
        out["geom_F"].append(dict(c, n_inliers=int(len(r["inliers"])), inliers_fnv1a=str(fnv), error_max=repr(r["error_max"]), min_nfa=repr(r["min_nfa"]),
                                  F_unit=[float(v) for v in Fn.reshape(-1)]))
        print("geom", c["name"], len(r["inliers"]), r["error_max"], r["min_nfa"])
    json.dump(out, open(path, "w"), indent=1)


# What the oracle tests (tests/test_oracle_{ba,match,geom}.py) compare against when they check the oracle case by
# case: the reference's own results on the same seeded inputs, so those comparisons run without the reference.
ORACLE_BA_KW = [dict(), dict(intrinsics_opt=1), dict(extrinsics_opt=4), dict(structure_opt=0)]
ORACLE_BA_EXT_KW = [dict(intrinsics_opt=1), dict(extrinsics_opt=4), dict(structure_opt=0), dict(use_loss=0), dict(model=3)]


def kw_key(kw):
    return "_".join(f"{a}{b}" for a, b in kw.items()) or "default"


def main_oracle_cases():
    out = {}

    def put(prefix, **arrays):
        for k, v in arrays.items():
            out[f"{prefix}.{k}"] = np.asarray(v)

    def registered(prefix, s, **ref_kw):
        r = ck.ref_ba_adjust_ex(s, **ref_kw)
        t, fit, cen = ck.ref_ba_register_priors(s)
        put(prefix, ok=r["ok"], final_cost=r["final_cost"], iterations=r["iterations"], points=r["points"], prior_fit=r["prior_fit"],
            reg_poses=t["poses"], reg_points=t["points"], reg_prior_center=t["prior_center"], reg_fit=fit, reg_centroid=cen)

    for kw in ORACLE_BA_KW:
        r = ck.ref_ba_adjust(synth.ba_scene(12, 400, 5, seed=13, outlier_frac=0.01), threads=2, **kw)
        put("ba." + kw_key(kw), ok=r["ok"], final_cost=r["final_cost"], iterations=r["iterations"], poses=r["poses"], points=r["points"])
    registered("ba_ext", synth.add_priors(synth.add_gcp(synth.ba_scene(12, 300, 5, seed=3), 6, weight=15.0), sigma=0.02))
    for kw in ORACLE_BA_EXT_KW:
        kw = dict(kw); model = kw.pop("model", 1)
        s = synth.add_priors(synth.add_gcp(synth.ba_scene(14, 400, 5, seed=6, model=model), 5, weight=12.0), sigma=0.015)
        registered("ba_ext." + kw_key(kw or dict(model=model)), s, **kw)

    descs = synth.descriptors(4, [257, 300, 64, 129], seed=77)
    pi, pj = np.meshgrid(np.arange(4), np.arange(4), indexing="ij")
    keep = pi != pj
    pi = pi[keep].astype(np.uint32); pj = pj[keep].astype(np.uint32)
    order = np.lexsort((pj, pi)); pi, pj = pi[order], pj[order]
    for ratio in (0.8, 0.95, 0.5):
        roff, rij = ck.ref_match_collection(descs, pi, pj, ratio)
        put(f"match.{ratio}", offsets=roff, ij=rij)
    put("match", pair01=ck.ref_match_pair(descs[0], descs[1]))

    descs = synth.descriptors(3, [1200, 1000, 700], seed=21)
    P, S = ck.ref_cascade_projections()
    put("cascade", projections_sha256=np.frombuffer(hashlib.sha256(P.tobytes() + S.tobytes()).digest(), np.uint8),
        zero_mean=ck.ref_cascade_zero_mean(descs, [0, 1, 2]))
    for k, d in enumerate(descs):
        codes, bids = ck.ref_cascade_hash(d, out["cascade.zero_mean"])
        put(f"cascade.{k}", codes=codes, bids=bids)
    roff, rij = ck.ref_cascade_collection(descs, *synth.exhaustive_pairs(3), 0.8)
    put("cascade", offsets=roff, ij=rij)

    for seed in range(20, 32):
        rng = np.random.default_rng(seed)
        n = int(rng.integers(9, 900)); of = float(rng.uniform(0.0, 0.7)); it = int(rng.choice([64, 256, 2048]))
        xI, xJ, _ = synth.two_view_matches(n, of, seed=seed, wh=(1600, 1200))
        r = ck.ref_acransac_fundamental(xI, xJ, (1600, 1200, 1600, 1200), 4.0, it)
        put(f"geom_F.{seed}", inliers=r["inliers"], error_max=r["error_max"], min_nfa=r["min_nfa"])
    for seed in range(40, 48):
        rng = np.random.default_rng(seed)
        n = int(rng.integers(5, 900)); of = float(rng.uniform(0.0, 0.7)); it = int(rng.choice([64, 2048]))
        xI, xJ, _ = synth.two_view_matches(n, of, seed=seed, wh=(1600, 1200), planar=True)
        r = ck.ref_acransac_homography(xI, xJ, (1600, 1200, 1600, 1200), 4.0, it)
        put(f"geom_H.{seed}", inliers=r["inliers"], min_nfa=r["min_nfa"])
    np.savez_compressed(os.path.join(HERE, "reference_oracle_cases.npz"), **out)
    print("oracle cases", len(out), "arrays")


def main():
    out = {"match": [], "ba": []}
    arrays = {}
    for c in MATCH_CASES:
        descs = synth.descriptors(len(c["counts"]), c["counts"], seed=c["seed"])
        pi, pj = synth.exhaustive_pairs(len(c["counts"]))
        off, ij = ck.ref_match_collection(descs, pi, pj, c["ratio"])
        fnv = int(ck.oracle().oracle_fnv1a_ij(ij.ctypes.data_as(ck.ctypes.c_void_p), ck.ctypes.c_int64(len(ij))))
        out["match"].append(dict(name=c["name"], counts=c["counts"], seed=c["seed"], ratio=c["ratio"], n_matches=int(len(ij)), fnv1a=str(fnv),
                                 offsets=[int(x) for x in off]))
        if len(ij) < 4000:
            arrays["match_" + c["name"]] = ij
        print("match", c["name"], len(ij), fnv)
    for c in BA_CASES:
        s = synth.ba_scene(**c["scene"])
        ref_opts = {k: v for k, v in c["opts"].items() if k in ("intrinsics_opt", "extrinsics_opt", "structure_opt", "use_loss")}
        r = ck.ref_ba_adjust(s, threads=8, **ref_opts)
        out["ba"].append(dict(name=c["name"], scene=c["scene"], opts=c["opts"], ok=r["ok"], initial_cost=r["initial_cost"], final_cost=r["final_cost"],
                              iterations=r["iterations"], successful=r["successful"], unsuccessful=r["unsuccessful"], termination=r["termination"]))
        print("ba", c["name"], r["initial_cost"], r["final_cost"], r["iterations"], r["termination"])
    json.dump(out, open(os.path.join(HERE, "reference_outputs.json"), "w"), indent=1)
    np.savez_compressed(os.path.join(HERE, "reference_matches.npz"), **arrays)


if __name__ == "__main__":
    if len(sys.argv) > 1 and sys.argv[1] == "ext":      # only the GCP / prior section (keeps the rest untouched)
        main_ext()
    elif len(sys.argv) > 1 and sys.argv[1] == "cascade":
        main_cascade()
    elif len(sys.argv) > 1 and sys.argv[1] == "io":
        main_io()
    elif len(sys.argv) > 1 and sys.argv[1] == "more":
        main_more()
    elif len(sys.argv) > 1 and sys.argv[1] == "geom":
        main_geom()
    elif len(sys.argv) > 1 and sys.argv[1] == "oracle_cases":
        main_oracle_cases()
    else:
        main()
        main_ext()
        main_cascade()
        main_io()
