"""MATCH parity on the GPU: the CUDA path (through the C-ABI) against the oracle, bit-exact."""
import numpy as np
import pytest

import checkers as ck
from openmvg_b200 import synth

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def matching():
    from openmvg_b200 import matching as m
    return m


def _csr_equal(off_a, ij_a, off_b, ij_b):
    assert np.array_equal(np.asarray(off_a, np.uint64), np.asarray(off_b, np.uint64))
    assert np.array_equal(ij_a, ij_b)


def test_tc_top2_against_simt_and_oracle(matching):
    """Raw tensor-core result: exact d1, the group of i1, and an upper bound of d2."""
    descs = synth.descriptors(2, [700, 1000], seed=3)
    ctx = matching.MatchContext(0)
    ctx.load(descs)
    sd1, si1, sd2 = ctx.debug_top2_simt(0, 1)
    rc, od1, oi1, od2 = ck.oracle_top2(descs[0], descs[1])
    assert rc == 0
    assert np.array_equal(sd1, od1) and np.array_equal(sd2, od2)
    uniq = od1 < od2
    assert np.array_equal(si1[uniq], oi1[uniq])
    td1, tg1, tub2 = ctx.debug_top2_tc(0, 1)
    assert np.array_equal(td1, od1)
    assert np.array_equal(tg1[uniq], (oi1 // 32)[uniq])
    assert np.all(tub2 >= od2)
    ctx.close()


@pytest.mark.parametrize("counts", [[5000, 5000], [300, 129, 2, 257, 1000], [128, 256, 384]])
def test_collection_bit_exact(matching, counts):
    descs = synth.descriptors(len(counts), counts, seed=11)
    pi, pj = synth.exhaustive_pairs(len(counts))
    ctx = matching.MatchContext(0)
    ctx.load(descs)
    ctx.run(pi, pj, 0.8)
    off, ij = ctx.fetch()
    ooff, oij = ck.oracle_match_collection(descs, pi, pj, 0.8)
    _csr_equal(off, ij, ooff, oij)
    assert len(ij) > 0
    ctx.close()


def test_edge_cases(matching):
    """Empty images, a 1-row database (NN=2 > rows => nothing), duplicates (d1 == d2), ratio 1.0 / 0.0."""
    rng = np.random.default_rng(5)
    base = synth.descriptors(1, 64, seed=9)[0]
    dup = np.concatenate([base, base])                  # every row twice: d1 == d2 == 0 for queries = base
    descs = [base, np.zeros((0, 128), np.uint8), base[:1].copy(), dup,
             rng.integers(0, 256, (40, 128), dtype=np.int64).astype(np.uint8), np.full((33, 128), 255, np.uint8)]
    n = len(descs)
    pi, pj = np.meshgrid(np.arange(n), np.arange(n), indexing="ij")
    pi = pi.reshape(-1).astype(np.uint32); pj = pj.reshape(-1).astype(np.uint32)     # incl. I == J and I > J
    ctx = matching.MatchContext(0)
    ctx.load(descs)
    for ratio in (0.8, 1.0, 0.0, 0.6):
        ctx.run(pi, pj, ratio)
        off, ij = ctx.fetch()
        ooff, oij = ck.oracle_match_collection(descs, pi, pj, ratio)
        _csr_equal(off, ij, ooff, oij)
    ctx.close()


def test_large_database_groups(matching):
    """> 8192 rows in the database: group size 64 (re-scan spans two 32-row chunks)."""
    descs = synth.descriptors(2, [9000, 600], seed=21)
    ctx = matching.MatchContext(0)
    ctx.load(descs)
    pi = np.array([0, 1], np.uint32); pj = np.array([1, 0], np.uint32)
    ctx.run(pi, pj, 0.8)
    off, ij = ctx.fetch()
    ooff, oij = ck.oracle_match_collection(descs, pi, pj, 0.8)
    _csr_equal(off, ij, ooff, oij)
    ctx.close()


def test_batched_runs_match_single(matching, monkeypatch):
    """Small k12 budget forces several batches; result must not change."""
    import os
    descs = synth.descriptors(6, [400, 500, 300, 450, 380, 410], seed=4)
    pi, pj = synth.exhaustive_pairs(6)
    ctx = matching.MatchContext(0)
    ctx.load(descs); ctx.run(pi, pj, 0.8); off1, ij1 = ctx.fetch(); ctx.close()
    monkeypatch.setenv("OMVG_MATCH_K12_MB", "0")        # 0 MB => one pair per batch
    ctx = matching.MatchContext(0)
    ctx.load(descs); ctx.run(pi, pj, 0.8); off2, ij2 = ctx.fetch(); ctx.close()
    _csr_equal(off1, ij1, off2, ij2)


def test_matcher_interface(matching):
    """The Matcher::Match mirror: non-dense image ids, only non-empty pairs inserted."""
    d = synth.descriptors(3, [300, 300, 0], seed=2)
    provider = {10: d[0], 42: d[1], 7: d[2]}
    pairs = {(10, 42), (7, 10), (7, 42)}
    out = matching.Matcher_Regions_B200(0.8).Match(provider, pairs)
    assert set(out.keys()) == {(10, 42)}
    assert np.array_equal(out[(10, 42)], ck.oracle_match_pair(d[0], d[1], 0.8))


def test_reference_golden_hashes(matching):
    """Golden outputs of the compiled reference (tests/golden): counts, CSR offsets and FNV-1a of the (i,j) list,
    including the 5000 x 5000 pair of the survey probe shape."""
    import json, os
    gold = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "reference_outputs.json")))
    for case in gold["match"]:
        descs = synth.descriptors(len(case["counts"]), case["counts"], seed=case["seed"])
        pi, pj = synth.exhaustive_pairs(len(case["counts"]))
        ctx = matching.MatchContext(0)
        ctx.load(descs); ctx.run(pi, pj, case["ratio"]); off, ij = ctx.fetch(); ctx.close()
        assert [int(x) for x in off] == case["offsets"]
        ij = np.ascontiguousarray(ij)
        fnv = int(ck.oracle().oracle_fnv1a_ij(ck._P(ij), ck.ctypes.c_int64(len(ij))))
        assert str(fnv) == case["fnv1a"], case["name"]


def test_full_size_properties(matching):
    """BASELINE-size slice (40 images x 5000): size-independent properties — every kept match passes the ratio
    test when re-evaluated exactly for its own query, rows are sorted by query index, and the self-pair (I,I)
    matches nothing (d1 = 0 needs 0 < fratio*d2: true only if d2 > 0, then i == j)."""
    descs = synth.descriptors(40, 5000, seed=1000)
    pi, pj = synth.exhaustive_pairs(40)
    ctx = matching.MatchContext(0)
    ctx.load(descs); ctx.run(pi, pj, 0.8); off, ij = ctx.fetch()
    assert len(ij) > 10000
    rng = np.random.default_rng(0)
    for p in rng.choice(len(pi), 12, replace=False):
        rows = ij[int(off[p]):int(off[p + 1])]
        assert np.all(np.diff(rows[:, 1].astype(np.int64)) > 0)              # ascending query index
        if len(rows) == 0:
            continue
        I, J = descs[int(pi[p])].astype(np.int64), descs[int(pj[p])].astype(np.int64)
        for i, j in rows[rng.choice(len(rows), min(5, len(rows)), replace=False)]:
            d = ((I - J[int(j)]) ** 2).sum(1)
            o = np.argsort(d, kind="stable")
            assert o[0] == i and np.float32(d[o[0]]) < np.float32(0.8) * np.float32(0.8) * np.float32(d[o[1]])
    # a pair sample bit-exact against the oracle
    for p in (0, len(pi) // 2, len(pi) - 1):
        want = ck.oracle_match_pair(descs[int(pi[p])], descs[int(pj[p])], 0.8)
        assert np.array_equal(ij[int(off[p]):int(off[p + 1])], want)
    ctx.run(np.array([3], np.uint32), np.array([3], np.uint32), 0.8); o2, ij2 = ctx.fetch()
    assert np.array_equal(ij2[:, 0], ij2[:, 1])                                   # self pair: only i == j can survive
    ctx.close()


# ---- whole-collection goldens of the compiled reference (tests/golden/make_golden_m1m2.py)
def _m1m2_gold():
    import os
    path = os.path.join(os.path.dirname(__file__), "golden", "reference_m1_m2.npz")
    if not os.path.exists(path):
        pytest.skip("tests/golden/reference_m1_m2.npz not generated")
    return np.load(path)


def test_whole_m1_against_reference_golden(matching):
    """BASELINE configs[2] IN FULL: 200 images x 5000, all 19 900 pairs, per-pair match count and FNV-1a of the (i, j)
    list identical to what the reference's Matcher_Regions(0.8, BRUTE_FORCE_L2)::Match produced for every pair."""
    g = _m1m2_gold()
    descs = synth.descriptor_collection(200, 5000, seed=1000)
    pi, pj = synth.exhaustive_pairs(200)
    ctx = matching.MatchContext(0)
    ctx.load(descs); ctx.run(pi, pj, 0.8); off, ij = ctx.fetch(); ctx.close()
    counts, fnv = ck.per_pair_digest(off, ij)
    assert int(counts.sum()) == int(g["m1_counts"].sum()) > 100000
    assert np.array_equal(counts, g["m1_counts"])
    bad = np.flatnonzero(fnv != g["m1_fnv"])
    assert len(bad) == 0, f"{len(bad)} of 19900 pairs differ, first {bad[:5]}"


def test_sampled_m2_multibatch_against_reference_golden(matching, monkeypatch):
    """BASELINE configs[3] sample: 256 seeded pairs of the 1000-image collection, run through the MULTI-BATCH path
    (result-buffer budget cut so the pass takes several launches), bit-exact against the reference golden.
    Only the images the sample names are uploaded (the others stay zero rows: they are never read)."""
    g = _m1m2_gold()
    spi, spj = g["m2_pair_i"], g["m2_pair_j"]
    wpi, wpj = synth.sampled_pairs(1000, 256, seed=5)
    assert np.array_equal(spi, wpi) and np.array_equal(spj, wpj)
    used = sorted(set(spi.tolist()) | set(spj.tolist()))
    monkeypatch.setenv("OMVG_MATCH_K12_MB", "4")        # ~100 pairs of 5000 queries per batch => 3 batches
    ctx = matching.MatchContext(0)
    ctx.set_images([5000] * 1000)
    blocks = {}
    for v in used:
        b = v // 25
        if b not in blocks:
            blocks[b] = synth.descriptor_collection(1000, 5000, seed=1000, lo=25 * b, hi=25 * b + 25)
        ctx.upload_host(v, blocks[b][v - 25 * b])
    ctx.prepare(); ctx.run(spi, spj, 0.8); off, ij = ctx.fetch()
    counts, fnv = ck.per_pair_digest(off, ij)
    assert np.array_equal(counts, g["m2_counts"]) and np.array_equal(fnv, g["m2_fnv"])
    ctx.close()


# ---- cascade hashing on the GPU (SURVEY M9 / N2)
def _cascade_gpu(descs, pi, pj, ratio):
    from openmvg_b200 import matching
    P, S = ck.cascade_projections()
    used = np.zeros(len(descs), np.uint8)
    used[np.asarray(pi, np.int64)] = 1; used[np.asarray(pj, np.int64)] = 1
    ctx = matching.MatchContext()
    ctx.load(descs)
    ctx.cascade_prepare(P, S, used)
    hashes = [ctx.cascade_debug_hash(k) for k in range(len(descs))]
    ctx.cascade_run(pi, pj, ratio)
    off, ij = ctx.fetch()
    off = off.copy(); ij = ij.copy()
    ctx.close()
    return off, ij, hashes


@pytest.mark.parametrize("counts,seed,ratio", [([300, 129, 2, 257, 1000], 11, 0.8), ([2000, 1800, 1500], 4, 0.8), ([1500, 1200, 0, 900], 11, 0.6),
                                               ([1, 40, 3], 5, 0.8)])
def test_cascade_matches_oracle_bit_exact(counts, seed, ratio):
    """Zero-mean vector, hash codes, bucket ids and the final (i, j) rows of every pair, bit for bit."""
    descs = synth.descriptors(len(counts), counts, seed=seed)
    pi, pj = synth.exhaustive_pairs(len(counts))
    off, ij, hashes = _cascade_gpu(descs, pi, pj, ratio)
    ooff, oij, zm, oh = ck.oracle_cascade_collection(descs, pi, pj, ratio)
    for k in range(len(counts)):
        codes, bids, gzm = hashes[k]
        assert np.array_equal(gzm, zm)
        if k in oh:
            assert np.array_equal(codes, oh[k][0]) and np.array_equal(bids, oh[k][1]), k
    assert np.array_equal(off, ooff)
    assert np.array_equal(ij, oij)


@pytest.mark.parametrize("name", ["ragged5", "three2k", "ratio06"])
def test_cascade_against_reference_golden(name):
    """Against the committed output of the reference's Cascade_Hashing_Matcher_Regions::Match (rows sorted by
    (i, j) as the reference leaves them); statistical bar 99.9 %, see tests/test_oracle_match.py."""
    import json, os
    gold = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "reference_outputs.json")))
    case = [c for c in gold["cascade"] if c["name"] == name][0]
    ref = np.load(os.path.join(os.path.dirname(__file__), "golden", "reference_cascade_matches.npz"))["cascade_" + name]
    descs = synth.descriptors(len(case["counts"]), case["counts"], seed=case["seed"])
    pi, pj = synth.exhaustive_pairs(len(case["counts"]))
    off, ij, _ = _cascade_gpu(descs, pi, pj, case["ratio"])
    same = tot = 0
    for p in range(len(pi)):
        a = set(map(tuple, ij[int(off[p]):int(off[p + 1])])); b = set(map(tuple, ref[case["offsets"][p]:case["offsets"][p + 1]]))
        same += len(a & b); tot += len(a | b)
    assert tot > 0 and same >= 0.999 * tot, (same, tot)


def test_cascade_full_size_pairs_properties():
    """5000 x 5000 descriptors per image (BASELINE size): every emitted match is a true ratio-test survivor of the
    candidates' exact distances and most brute-force matches are found (recall as main_benchANN scores it)."""
    from openmvg_b200 import matching
    descs = synth.descriptors(4, [5000] * 4, seed=3)
    pi, pj = synth.exhaustive_pairs(4)
    off, ij, _ = _cascade_gpu(descs, pi, pj, 0.8)
    ctx = matching.MatchContext(); ctx.load(descs); ctx.run(pi, pj, 0.8); boff, bij = ctx.fetch(); boff = boff.copy(); bij = bij.copy(); ctx.close()
    a = set(); b = set()
    for p in range(len(pi)):
        a |= {(p,) + tuple(r) for r in ij[int(off[p]):int(off[p + 1])]}; b |= {(p,) + tuple(r) for r in bij[int(boff[p]):int(boff[p + 1])]}
    assert len(b) > 1000 and len(a & b) >= 0.9 * len(b), (len(a), len(b), len(a & b))
    for p in range(len(pi)):                                    # ascending query order inside a pair
        m = ij[int(off[p]):int(off[p + 1])]
        assert np.all(np.diff(m[:, 1].astype(np.int64)) > 0)


def test_cascade_large_buckets_take_the_streaming_path():
    """More than 128 candidates per query (many near-identical descriptors share buckets): the streaming selection
    rounds, duplicate suppression across groups and the (Hamming, insertion order) tie-breaks, bit for bit."""
    rng = np.random.default_rng(5)
    descs = synth.descriptors(3, [900, 800, 700], seed=9)
    for d in descs:                                            # 300 rows of each image collapse onto 3 prototypes +-1
        for k in range(3):
            rows = slice(100 * k, 100 * k + 100)
            d[rows] = np.clip(d[100 * k].astype(np.int16) + rng.integers(-1, 2, (100, 128)), 0, 255).astype(np.uint8)
    descs[1][:300] = descs[0][:300]                            # and the same prototypes across images
    pi, pj = synth.exhaustive_pairs(3)
    off, ij, hashes = _cascade_gpu(descs, pi, pj, 0.8)
    ooff, oij, zm, oh = ck.oracle_cascade_collection(descs, pi, pj, 0.8)
    assert np.array_equal(off, ooff) and np.array_equal(ij, oij)
    # the case really exercises more than 128 candidates per query (query 0 of image 1 against image 0)
    tot = sum(int((oh[0][1][:, g] == oh[1][1][0, g]).sum()) for g in range(6))
    assert tot > 128, tot


def test_load_desc_files_equals_in_memory_upload(tmp_path):
    """N3: '.desc' files read by the library's thread pool into pinned memory give the same matches as uploading the
    arrays, and the result written by omvg_matches_save reads back identically (text format parsed here)."""
    from openmvg_b200 import matching
    counts = [700, 0, 650, 300]
    descs = synth.descriptors(len(counts), counts, seed=1)
    paths = []
    for k, d in enumerate(descs):
        p = tmp_path / f"img{k}.desc"; matching.write_desc_file(str(p), d); paths.append(str(p))
    pi, pj = synth.exhaustive_pairs(len(counts))
    a = matching.MatchContext(); got = a.load_desc_files(paths); a.run(pi, pj, 0.8); aoff, aij = a.fetch(); aoff = aoff.copy(); aij = aij.copy(); a.close()
    assert list(got) == counts
    b = matching.MatchContext(); b.load(descs); b.run(pi, pj, 0.8); boff, bij = b.fetch()
    assert np.array_equal(aoff, boff) and np.array_equal(aij, bij)
    b.close()
    out = tmp_path / "matches.putative.txt"
    matching.save_matches(str(out), pi * 10 + 1, pj * 10 + 1, aoff, aij)        # arbitrary view ids
    tok = out.read_text().split()
    t = 0; seen = {}
    while t < len(tok):
        I, J, n = int(tok[t]), int(tok[t + 1]), int(tok[t + 2]); t += 3
        seen[(I, J)] = np.array(tok[t:t + 2 * n], np.uint32).reshape(-1, 2); t += 2 * n
    for p in range(len(pi)):
        m = aij[int(aoff[p]):int(aoff[p + 1])]
        key = (int(pi[p]) * 10 + 1, int(pj[p]) * 10 + 1)
        assert (key in seen) == (len(m) > 0)
        if len(m):
            assert np.array_equal(seen[key], m)


# ---- the fifth-K-slice kernel (match_dig2_kernel) against the key-arithmetic kernel and the oracle
def _near_tie_collection(seed):
    """Rows that differ from each other by +-1 in a few elements: distances of 0, 1, 2, ... with both parities of |b|^2,
    so the chunk maxima tie to within the parity and the exact-scan fallbacks of the finalize pass run."""
    rng = np.random.default_rng(seed)
    base = synth.descriptors(1, 40, seed=seed + 1)[0].astype(np.int64)
    rows = []
    for b in base:
        for _ in range(12):
            v = b.copy()
            k = rng.integers(0, 4)
            idx = rng.choice(128, size=k, replace=False)
            v[idx] += rng.choice([-1, 1], size=k)
            rows.append(np.clip(v, 0, 255))
    rows = np.array(rows, np.uint8)
    a = rows[rng.permutation(len(rows))]
    b = rows[rng.permutation(len(rows))][:300]
    c = np.clip(rows.astype(np.int64) + rng.integers(-1, 2, rows.shape), 0, 255).astype(np.uint8)
    return [a, b, c]


@pytest.mark.parametrize("seed", [1, 2])
def test_fifth_slice_near_ties(matching, seed):
    descs = _near_tie_collection(seed)
    n = len(descs)
    pi, pj = np.meshgrid(np.arange(n), np.arange(n), indexing="ij")
    pi = pi.reshape(-1).astype(np.uint32); pj = pj.reshape(-1).astype(np.uint32)
    ctx = matching.MatchContext(0)
    ctx.load(descs)
    assert ctx.kernel_variant() == 5
    for ratio in (0.8, 0.95, 0.999, 1.0):
        ctx.run(pi, pj, ratio)
        off, ij = ctx.fetch()
        ooff, oij = ck.oracle_match_collection(descs, pi, pj, ratio)
        _csr_equal(off, ij, ooff, oij)
    ctx.close()


def test_kernel_variants_agree(matching, monkeypatch):
    """Default (fifth slice, two query tiles per database tile) = the key-arithmetic kernel (OMVG_MATCH_TC4) = the oracle."""
    rng = np.random.default_rng(8)
    descs = synth.descriptors(5, [1500, 700, 2300, 33, 900], seed=31)
    descs.append(rng.integers(0, 256, (800, 128), dtype=np.int64).astype(np.uint8))       # |b|^2 ~ 2.8e6: c0 > 0
    descs.append(rng.integers(0, 256, (600, 128), dtype=np.int64).astype(np.uint8))
    pi, pj = synth.exhaustive_pairs(len(descs))
    pi = np.concatenate([pi, pj]); pj = np.concatenate([pj, pi[:len(pj)]])
    ooff, oij = ck.oracle_match_collection(descs, pi, pj, 0.8)
    results = []
    for env in ({}, {"OMVG_MATCH_TC4": "1"}):
        monkeypatch.delenv("OMVG_MATCH_TC4", raising=False)
        for k, v in env.items(): monkeypatch.setenv(k, v)
        ctx = matching.MatchContext(0)
        ctx.load(descs)
        assert ctx.kernel_variant() == (4 if "OMVG_MATCH_TC4" in env else 5)
        ctx.run(pi, pj, 0.8)
        off, ij = ctx.fetch()
        _csr_equal(off, ij, ooff, oij)
        ctx.close()


def test_wide_norm_spread_takes_the_key_arithmetic_kernel(matching):
    """All-zero and all-255 descriptors in ONE image: |b|^2 spans 8.3e6, more than 32 signed digits can carry."""
    rng = np.random.default_rng(3)
    mixed = np.concatenate([np.zeros((40, 128), np.uint8), np.full((40, 128), 255, np.uint8),
                            rng.integers(0, 256, (300, 128), dtype=np.int64).astype(np.uint8)])
    descs = [mixed, synth.descriptors(1, 500, seed=77)[0], mixed[::-1].copy()]
    pi, pj = synth.exhaustive_pairs(3)
    pi = np.concatenate([pi, pj]); pj = np.concatenate([pj, pi[:len(pj)]])
    ctx = matching.MatchContext(0)
    ctx.load(descs)
    assert ctx.kernel_variant() == 4
    ctx.run(pi, pj, 0.8)
    off, ij = ctx.fetch()
    ooff, oij = ck.oracle_match_collection(descs, pi, pj, 0.8)
    _csr_equal(off, ij, ooff, oij)
    ctx.close()
