"""Python binding of the MATCH C-ABI (tests / bench plumbing; the drop-in host shim is the C++
class in openmvg_b200/host/Matcher_Regions_B200.hpp).

Mirrors openMVG::matching_image_collection::Matcher_Regions(ratio, BRUTE_FORCE_L2)::Match
(reference: matching_image_collection/Matcher_Regions.cpp:32-107): same argument meaning — a
regions provider (image id -> [n,128] uint8 descriptors), a set of pairs, an output map keyed by
(I, J) that only receives non-empty results.
"""
from __future__ import annotations

import ctypes
import os

import numpy as np

from ._lib import check, lib

_vp = ctypes.c_void_p


def _p(a):
    return a.ctypes.data_as(_vp)


class MatchContext:
    """Thin RAII wrapper over omvg_match_ctx."""

    def __init__(self, device: int = 0):
        self._h = _vp()
        check(lib().omvg_match_create(ctypes.byref(self._h), int(device)))
        self.counts = None

    def close(self):
        if self._h:
            lib().omvg_match_destroy(self._h)
            self._h = _vp()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- collection
    def set_images(self, counts):
        self.counts = np.ascontiguousarray(counts, np.uint32)
        check(lib().omvg_match_set_images(self._h, len(self.counts), _p(self.counts)))

    def upload_host(self, image: int, desc: np.ndarray):
        desc = np.ascontiguousarray(desc, np.uint8)
        assert desc.size == int(self.counts[image]) * 128
        check(lib().omvg_match_upload_host(self._h, int(image), _p(desc)))

    def upload_device_packed(self, dev_ptr: int):
        check(lib().omvg_match_upload_device_packed(self._h, _vp(dev_ptr)))

    def prepare(self):
        check(lib().omvg_match_prepare(self._h))

    def load(self, descs):
        """set_images + upload every image from host arrays + prepare."""
        self.set_images([len(d) for d in descs])
        for k, d in enumerate(descs):
            self.upload_host(k, d)
        self.prepare()

    def load_desc_files(self, paths):
        """set_images + parallel read of openMVG '.desc' files into pinned memory + upload + prepare (N3)."""
        arr = (ctypes.c_char_p * len(paths))(*[os.fsencode(p) for p in paths])
        counts = np.zeros(len(paths), np.uint32)
        check(lib().omvg_match_load_desc_files(self._h, len(paths), arr, _p(counts)))
        self.counts = counts
        return counts

    # ---- matching
    def run(self, pair_i, pair_j, dist_ratio: float = 0.8):
        self._pi = np.ascontiguousarray(pair_i, np.uint32)
        self._pj = np.ascontiguousarray(pair_j, np.uint32)
        check(lib().omvg_match_run(self._h, _p(self._pi), _p(self._pj), ctypes.c_uint64(len(self._pi)),
                                   ctypes.c_float(dist_ratio)))

    def sync(self):
        check(lib().omvg_match_sync(self._h))

    def fetch(self):
        """-> (offsets[n_pairs+1] uint64, ij[n_matches,2] uint32) copied out of the context."""
        off = ctypes.POINTER(ctypes.c_uint64)()
        ij = ctypes.POINTER(ctypes.c_uint32)()
        n = ctypes.c_uint64()
        check(lib().omvg_match_fetch(self._h, ctypes.byref(off), ctypes.byref(ij), ctypes.byref(n)))
        npairs = len(self._pi)
        offsets = np.ctypeslib.as_array(off, (npairs + 1,)).copy()
        m = (np.ctypeslib.as_array(ij, (n.value * 2,)).reshape(-1, 2).copy() if n.value else np.zeros((0, 2), np.uint32))
        return offsets, m

    def launch_count(self) -> int:
        return int(lib().omvg_match_launch_count(self._h))

    def kernel_variant(self) -> int:
        """5 = fifth-K-slice kernel, 4 = key-arithmetic kernel (see omvg_match_kernel_variant)."""
        return int(lib().omvg_match_kernel_variant(self._h))

    def kernel_time(self, reset: bool = True):
        ms = ctypes.c_double(); n = ctypes.c_uint64()
        check(lib().omvg_match_kernel_time(self._h, ctypes.byref(ms), ctypes.byref(n), int(reset)))
        return ms.value, n.value

    # ---- validation aids
    # ---- cascade hashing (FASTCASCADEHASHINGL2; Cascade_Hashing_Matcher_Regions.cpp)
    def cascade_prepare(self, primary, secondary, used=None):
        P = np.ascontiguousarray(primary, np.float32).reshape(128, 128)
        S = np.ascontiguousarray(secondary, np.float32).reshape(6, 10, 128)
        u = None if used is None else np.ascontiguousarray(used, np.uint8)
        check(lib().omvg_match_cascade_prepare(self._h, _p(P), _p(S), None if u is None else _p(u)))

    def cascade_run(self, pair_i, pair_j, dist_ratio: float = 0.8):
        self._pi = np.ascontiguousarray(pair_i, np.uint32)
        self._pj = np.ascontiguousarray(pair_j, np.uint32)
        check(lib().omvg_match_cascade_run(self._h, _p(self._pi), _p(self._pj), ctypes.c_uint64(len(self._pi)),
                                           ctypes.c_float(dist_ratio)))

    def cascade_debug_hash(self, image: int):
        n = int(self.counts[image])
        codes = np.zeros((n, 4), np.uint32); bids = np.zeros((n, 6), np.uint16); zm = np.zeros(128, np.float32)
        check(lib().omvg_match_cascade_debug_hash(self._h, image, _p(codes), _p(bids), _p(zm)))
        return codes, bids, zm

    def debug_top2_simt(self, db_image: int, q_image: int):
        n = int(self.counts[q_image])
        d1 = np.zeros(n, np.int32); i1 = np.zeros(n, np.uint32); d2 = np.zeros(n, np.int32)
        check(lib().omvg_match_debug_top2_simt(self._h, db_image, q_image, _p(d1), _p(i1), _p(d2)))
        return d1, i1, d2

    def debug_top2_tc(self, db_image: int, q_image: int):
        n = int(self.counts[q_image])
        d1 = np.zeros(n, np.int32); g1 = np.zeros(n, np.uint32); ub2 = np.zeros(n, np.int32)
        check(lib().omvg_match_debug_top2_tc(self._h, db_image, q_image, _p(d1), _p(g1), _p(ub2)))
        return d1, g1, ub2


class Matcher_Regions_B200:
    """Drop-in for Matcher_Regions(distRatio, BRUTE_FORCE_L2) (Matcher_Regions.hpp / Matcher.hpp:34-48)."""

    def __init__(self, dist_ratio: float = 0.8, device: int = 0):
        self.f_dist_ratio_ = float(dist_ratio)
        self.device = device

    def Match(self, regions_provider, pairs, map_PutativeMatches=None, progress=None):
        """regions_provider: mapping image id -> [n,128] uint8; pairs: iterable of (I, J).
        Fills/returns map_PutativeMatches[(I,J)] = [n,2] uint32 (i_, j_) for non-empty pairs only."""
        out = {} if map_PutativeMatches is None else map_PutativeMatches
        pairs = sorted(set((int(a), int(b)) for a, b in pairs))      # Pair_Set is an ordered std::set
        ids = sorted(regions_provider.keys())
        dense = {v: k for k, v in enumerate(ids)}
        ctx = MatchContext(self.device)
        try:
            ctx.load([np.ascontiguousarray(regions_provider[v], np.uint8).reshape(-1, 128) for v in ids])
            pi = np.array([dense[a] for a, _ in pairs], np.uint32)
            pj = np.array([dense[b] for _, b in pairs], np.uint32)
            ctx.run(pi, pj, self.f_dist_ratio_)
            offsets, ij = ctx.fetch()
        finally:
            ctx.close()
        for k, pr in enumerate(pairs):
            a, b = int(offsets[k]), int(offsets[k + 1])
            if b > a:                                                  # Matcher_Regions.cpp:99-102
                out[pr] = ij[a:b].copy()
            if progress is not None:
                progress(1)
        return out


class Cascade_Hashing_Matcher_Regions_B200:
    """Drop-in for Cascade_Hashing_Matcher_Regions(distRatio) on {image id: [n,128] uint8}: same pairs, same
    per-pair content as the reference up to its two host-side clean-ups — rows are sorted by (i, j) here as
    IndMatch::getDeduplicated does; the equal-coordinates filter needs feature positions and lives in the C++ shim."""

    def __init__(self, dist_ratio: float = 0.8, primary=None, secondary=None, device: int = 0):
        self.f_dist_ratio_ = float(dist_ratio)
        self.primary, self.secondary, self.device = primary, secondary, device

    def Match(self, regions_provider, pairs, map_PutativeMatches=None, progress=None):
        out = {} if map_PutativeMatches is None else map_PutativeMatches
        pairs = sorted(set((int(a), int(b)) for a, b in pairs))
        ids = sorted(regions_provider.keys())
        dense = {v: k for k, v in enumerate(ids)}
        used = np.zeros(len(ids), np.uint8)
        for a, b in pairs:
            used[dense[a]] = 1; used[dense[b]] = 1
        ctx = MatchContext(self.device)
        try:
            ctx.load([np.ascontiguousarray(regions_provider[v], np.uint8).reshape(-1, 128) for v in ids])
            ctx.cascade_prepare(self.primary, self.secondary, used)
            pi = np.array([dense[a] for a, _ in pairs], np.uint32)
            pj = np.array([dense[b] for _, b in pairs], np.uint32)
            ctx.cascade_run(pi, pj, self.f_dist_ratio_)
            offsets, ij = ctx.fetch()
        finally:
            ctx.close()
        for k, pr in enumerate(pairs):
            a, b = int(offsets[k]), int(offsets[k + 1])
            if b > a:
                m = ij[a:b]
                out[pr] = m[np.lexsort((m[:, 1], m[:, 0]))].copy()
            if progress is not None:
                progress(1)
        return out


def save_matches(path: str, pair_I, pair_J, offsets, ij) -> None:
    """Write a CSR result as openMVG's matches.*.txt / matches.*.bin (matching::Save; extension picks the format)."""
    pI = np.ascontiguousarray(pair_I, np.uint32); pJ = np.ascontiguousarray(pair_J, np.uint32)
    off = np.ascontiguousarray(offsets, np.uint64); m = np.ascontiguousarray(ij, np.uint32).reshape(-1)
    check(lib().omvg_matches_save(os.fsencode(path), ctypes.c_uint64(len(pI)), _p(pI), _p(pJ), _p(off), _p(m)))


def write_desc_file(path: str, desc: np.ndarray) -> None:
    """openMVG '.desc' layout (features/descriptor.hpp:206-228): size_t count, then count x 128 bytes."""
    d = np.ascontiguousarray(desc, np.uint8).reshape(-1, 128)
    with open(path, "wb") as f:
        f.write(np.uint64(len(d)).tobytes()); f.write(d.tobytes())
