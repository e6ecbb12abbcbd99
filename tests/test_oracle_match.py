"""CPU: the MATCH oracle against the reference's known answers and the committed golden vectors
(generated from the compiled reference)."""
import hashlib
import json
import os

import numpy as np
import pytest

import checkers as ck
from openmvg_b200 import synth

G = os.path.join(os.path.dirname(__file__), "golden")
GOLD = json.load(open(os.path.join(G, "reference_outputs.json")))
GOLD_IJ = np.load(os.path.join(G, "reference_matches.npz"))
REF = np.load(os.path.join(G, "reference_oracle_cases.npz"))


def test_l2_known_answer():
    """matching/metric_test.cpp:25-39 — L2 of (0..7) and (7..0) is 168."""
    a = np.arange(8, dtype=np.uint8); b = a[::-1].copy()
    assert ck.oracle().oracle_l2_u8(ck._P(a), ck._P(b), 8) == 168


def test_l2_dim128_equals_squared_norm():
    """matching/metric_test.cpp:132-147 — L2<uint8_t> on random 128-D vectors equals (a-b).squaredNorm()."""
    rng = np.random.default_rng(0)
    for _ in range(20):
        a = rng.integers(0, 256, 128, dtype=np.int64).astype(np.uint8); b = rng.integers(0, 256, 128, dtype=np.int64).astype(np.uint8)
        assert ck.oracle().oracle_l2_u8(ck._P(a), ck._P(b), 128) == int(((a.astype(int) - b.astype(int)) ** 2).sum())
    full = np.full(128, 255, np.uint8); zero = np.zeros(128, np.uint8)
    assert ck.oracle().oracle_l2_u8(ck._P(full), ck._P(zero), 128) == 128 * 255 * 255     # the int32 maximum of the path


def test_search_neighbours_guards():
    """matcher_brute_force.hpp:108-113 — NN(=2) > rows or no query => false; Build(nullptr,0,..) false
    (matching_test.cpp:155-163)."""
    d = synth.descriptors(1, 4, seed=1)[0]
    assert ck.oracle_top2(d[:1], d)[0] == -1
    assert ck.oracle_top2(d, d[:0])[0] == -1
    assert len(ck.oracle_match_pair(d[:1], d)) == 0 and len(ck.oracle_match_pair(d[:0], d)) == 0 and len(ck.oracle_match_pair(d, d[:0])) == 0


def test_top2_toy():
    """Dim-4 toy of matching_test.cpp:74-87 lifted to 128-D: the query equal to row 1 finds index 1 at distance 0;
    with multiplicity the second distance of a duplicated minimum equals the first."""
    db = np.zeros((3, 128), np.uint8); db[0, :4] = [0, 1, 2, 3]; db[1, :4] = [4, 5, 6, 7]; db[2, :4] = [8, 9, 10, 11]
    q = db[1:2].copy()
    rc, d1, i1, d2 = ck.oracle_top2(db, q)
    assert rc == 0 and d1[0] == 0 and i1[0] == 1 and d2[0] == 64
    rc, d1, i1, d2 = ck.oracle_top2(np.concatenate([db, db[1:2]]), q)
    assert d1[0] == 0 and d2[0] == 0 and i1[0] == 1


def test_ratio_is_float_arithmetic():
    """matching_filters.hpp:57: (float)d1 < fratio*(float)d2 with fratio = 0.8f*0.8f."""
    fr = np.float32(0.8) * np.float32(0.8)
    for d1, d2 in [(64, 100), (63, 100), (640000, 1000000), (640001, 1000000), (0, 0), (5, 5), (8323200, 8323200)]:
        want = bool(np.float32(d1) < fr * np.float32(d2))
        assert bool(ck.oracle().oracle_ratio_keep(d1, d2, ck.ctypes.c_float(fr))) == want


@pytest.mark.parametrize("case", GOLD["match"], ids=lambda c: c["name"])
def test_golden_collections(case):
    descs = synth.descriptors(len(case["counts"]), case["counts"], seed=case["seed"])
    pi, pj = synth.exhaustive_pairs(len(case["counts"]))
    off, ij = ck.oracle_match_collection(descs, pi, pj, case["ratio"])
    assert [int(x) for x in off] == case["offsets"]
    assert len(ij) == case["n_matches"]
    fnv = int(ck.oracle().oracle_fnv1a_ij(ck._P(np.ascontiguousarray(ij)), ck.ctypes.c_int64(len(ij))))
    assert str(fnv) == case["fnv1a"]
    key = "match_" + case["name"]
    if key in GOLD_IJ:
        assert np.array_equal(ij, GOLD_IJ[key])


def test_against_compiled_reference():
    """Against the reference's Matcher_Regions on the same collection (tests/golden/reference_oracle_cases.npz)."""
    descs = synth.descriptors(4, [257, 300, 64, 129], seed=77)
    pi, pj = np.meshgrid(np.arange(4), np.arange(4), indexing="ij")
    keep = pi != pj
    pi = pi[keep].astype(np.uint32); pj = pj[keep].astype(np.uint32)
    # Pair_Set is an ordered set: present pairs in sorted order to both
    order = np.lexsort((pj, pi)); pi, pj = pi[order], pj[order]
    for ratio in (0.8, 0.95, 0.5):
        roff, rij = REF[f"match.{ratio}.offsets"], REF[f"match.{ratio}.ij"]
        ooff, oij = ck.oracle_match_collection(descs, pi, pj, ratio)
        assert np.array_equal(roff, ooff) and np.array_equal(rij, oij)
    a = REF["match.pair01"]; b = ck.oracle_match_pair(descs[0], descs[1])
    assert np.array_equal(a, b)


# ---- cascade hashing (SURVEY M9 / N2): oracle vs the reference's Cascade_Hashing_Matcher_Regions
def _sorted_rows(off, ij, p):
    m = ij[int(off[p]):int(off[p + 1])]
    return m[np.lexsort((m[:, 1], m[:, 0]))]


@pytest.mark.parametrize("case", GOLD.get("cascade", []), ids=lambda c: c["name"])
def test_cascade_golden(case):
    """Whole pipeline (zero-mean, hashing, buckets, Hamming top-10, exact L2 top-2, ratio) against the committed
    output of the reference's Cascade_Hashing_Matcher_Regions::Match.  The reference sorts each pair's matches by
    (i, j); the oracle emits them in query order, so rows are compared after that sort.  The hashing is a float
    mat-vec whose summation order differs (Eigen GEMV vs k-ascending here): a projection within rounding of zero
    could flip a bit, so the bar is statistical (>= 99.9 % of the matches identical); on these cases it is exact."""
    descs = synth.descriptors(len(case["counts"]), case["counts"], seed=case["seed"])
    pi, pj = synth.exhaustive_pairs(len(case["counts"]))
    off, ij, _, _ = ck.oracle_cascade_collection(descs, pi, pj, case["ratio"])
    gold = np.load(os.path.join(os.path.dirname(__file__), "golden", "reference_cascade_matches.npz"))["cascade_" + case["name"]]
    goff = case["offsets"]
    same = tot = 0
    for p in range(len(pi)):
        a = set(map(tuple, _sorted_rows(off, ij, p))); b = set(map(tuple, gold[goff[p]:goff[p + 1]]))
        same += len(a & b); tot += len(a | b)
    assert tot == 0 or same >= 0.999 * tot, (same, tot)
    assert tot > 0 or case["n_matches"] == 0


def test_cascade_stages_against_compiled_reference():
    """Stage by stage against the reference's CascadeHasher (tests/golden/reference_oracle_cases.npz)."""
    descs = synth.descriptors(3, [1200, 1000, 700], seed=21)
    P, S = ck.cascade_projections()
    digest = np.frombuffer(hashlib.sha256(P.tobytes() + S.tobytes()).digest(), np.uint8)
    assert np.array_equal(digest, REF["cascade.projections_sha256"])   # the committed fixture is the reference's draw
    used = [0, 1, 2]
    zo = ck.oracle_cascade_zero_mean(descs, used); zr = REF["cascade.zero_mean"]
    assert np.array_equal(zo, zr)
    bits = diff = 0
    for k, d in enumerate(descs):
        co, bo = ck.oracle_cascade_hash(d, zr, P, S); cr, br = REF[f"cascade.{k}.codes"], REF[f"cascade.{k}.bids"]
        diff += sum(bin(int(x)).count("1") for x in (co ^ cr).ravel()) + sum(bin(int(x)).count("1") for x in (bo ^ br).ravel())
        bits += co.size * 32 + bo.size * 10
    assert diff <= 1e-5 * bits, (diff, bits)
    pi, pj = synth.exhaustive_pairs(3)
    off, ij, _, _ = ck.oracle_cascade_collection(descs, pi, pj, 0.8, P, S)
    roff, rij = REF["cascade.offsets"], REF["cascade.ij"]
    same = tot = 0
    for p in range(len(pi)):
        a = set(map(tuple, _sorted_rows(off, ij, p))); b = set(map(tuple, rij[int(roff[p]):int(roff[p + 1])]))
        same += len(a & b); tot += len(a | b)
    assert tot > 50 and same >= 0.999 * tot, (same, tot)


def test_cascade_recall_against_brute_force():
    """What main_benchANN scores: the approximate matcher against the exhaustive one (same ratio test)."""
    descs = synth.descriptors(3, [1500, 1500, 1500], seed=8)
    pi, pj = synth.exhaustive_pairs(3)
    off, ij, _, _ = ck.oracle_cascade_collection(descs, pi, pj, 0.8)
    boff, bij = ck.oracle_match_collection(descs, pi, pj, 0.8)
    a = set(); b = set()
    for p in range(len(pi)):
        a |= {(p,) + tuple(r) for r in ij[int(off[p]):int(off[p + 1])]}; b |= {(p,) + tuple(r) for r in bij[int(boff[p]):int(boff[p + 1])]}
    assert len(b) > 100 and len(a & b) >= 0.9 * len(b), (len(a), len(b), len(a & b))
