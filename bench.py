#!/usr/bin/env python
"""bench.py — the two hot paths on N B200s (one process per GPU) or, with --impl reference, the
reference's own CPU implementation of the same paths on the host cores.

Headline (`metric`/`value`): BA LM-iterations/s on BASELINE.json configs[1]
(1000 cams / 100k pts / 1M obs, shared pinhole intrinsic, Huber(16), refine all).  One "step" = one
complete Adjust (LM until Ceres' own termination test fires) on the device-resident scene;
`value` = sum(Ceres-style iteration count) / sum(device time, CUDA events).  `e2e` = the same solve
through omvg_ba_solve with HOST buffers (packing, H2D, structure build, solve, D2H inside the
timed region).  BA does not shard (SURVEY §8e): with --gpus N every rank runs a replica of the SAME
scene ("weak").

The `match` object carries the second hot path with the same keys (and `match_value`, `match_e2e`,
`match_roofline_frac` repeat its numbers at the top level): exhaustive BRUTE_FORCE_L2 + ratio
matching, 200 images x 5000 descriptors (BASELINE.json configs[2]); image pairs are sharded over the
ranks.  At N > 1 the e2e leg is the whole sharded path: every rank copies only ITS 1/N of the images from
pinned host memory, one NCCL all-gather of the per-rank descriptor tiles gives every rank the collection,
then arena fill, prepare, match, fetch — all inside the timer; `allgather_ms` is reported beside it.
At N = 8 (or with --m2) the `m2` object runs BASELINE.json configs[3]: 1000 images x 5000 the same way.
`ba_sweep` (N = 1) is configs[4]: the 50 -> 2000 camera LM-iteration latency curve.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

BA_CFG = (1000, 100_000, 10)          # cams, points, obs/point  -> 1M observations
BA_SEED = 42                          # the same scene on every rank (replicas)
BA_BYTES_PER_OBS = 232                # SURVEY §8d: 24 B in (view/point index + xy) + 16 B r + 192 B J (2x(3+6+3) doubles)
# One LM iteration with the Jacobian materialised once (DESIGN.md §5): evaluation 232 B/obs (above) + one read of
# r and J for the normal equations / Schur complement (208 + 12 B of indices) + one read for back-substitution and
# the model cost change (208 + 12) + the cost-only evaluation of the candidate (40 B/obs)  = 712 B/obs.
BA_STEP_BYTES_PER_OBS = 232 + 220 + 220 + 40
BA_WORKLOAD = "BA 1000 cams / 100k pts / 1M obs, 1 shared pinhole intrinsic, Huber(16), refine all (BASELINE configs[1]); replica per GPU"
BA_L2 = "inputs larger than L2 (J+r = 224 MB per evaluation)"
MATCH_IMAGES, MATCH_DESC, MATCH_SEED = 200, 5000, 1000
M2_IMAGES = 1000
OPS_PER_DESC_PAIR = 256               # 128 MAC
SWEEP_CAMS = (50, 100, 200, 500, 2000)
CPU_MATCH_IMAGES = 26                 # 325 pairs of 5000 x 5000: ~3 s of the reference on a 128-thread host
GEOM_PAIRS, GEOM_MATCHES = 2000, 800  # geometric-filter leg: pairs x putative matches per pair
DUMP_BYTES = 60 << 20                 # --dump-outputs budget (array data), under 64 MB with the .npy headers


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm_gbs=d["hbm_gbs"], bf16_tflops=d["bf16_tflops"], bf16_sustained=d.get("bf16_tflops_sustained", d["bf16_tflops"]), src="measured")
    return dict(hbm_gbs=6650.0, bf16_tflops=1590.0, bf16_sustained=1400.0, src="fallback")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region (B200_PROFILING.md)."""
    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.index, self.samples, self.stop, self.t = index, [], threading.Event(), None

    def _run(self):
        while not self.stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i", str(self.index)],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.samples.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            self.stop.wait(0.2)

    def __enter__(self):
        self.t = threading.Thread(target=self._run, daemon=True); self.t.start(); return self

    def __exit__(self, *a):
        self.stop.set(); self.t.join(timeout=6)

    def summary(self):
        sm = [float(s[0]) for s in self.samples if s and s[0].replace(".", "").isdigit()]
        mx = [float(s[1]) for s in self.samples if len(s) > 1 and s[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for s in self.samples for n, v in zip(names, s[2:6]) if v.lower().startswith("active")})
        return dict(sm_mhz=float(np.median(sm)) if sm else None, sm_max_mhz=max(mx) if mx else None, reasons=reasons, samples=len(sm))


def dist_env():
    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1")); local = int(os.environ.get("LOCAL_RANK", "0"))
    return rank, world, local


def image_shard(n_img, rank, world):
    """Contiguous slice of the images rank `rank` owns (host side of the NCCL all-gather) and the padded per-rank count."""
    per = (n_img + world - 1) // world
    return min(rank * per, n_img), min((rank + 1) * per, n_img), per


def pair_shard(pi, pj, rank, world):
    """Round-robin deal of the (equal-cost) pair list: rank r takes pairs r, r + world, ..."""
    sl = slice(rank, None, world)
    return np.ascontiguousarray(pi[sl]), np.ascontiguousarray(pj[sl])


def dump_outputs(path, arrays):
    """Write each array as <path>/<name>.npy.  Smallest first; an array larger than what is left of DUMP_BYTES is
    replaced by a fixed, seeded sample of its rows (the same rows for the same shape), so two builds compare row for row."""
    os.makedirs(path, exist_ok=True)
    left = DUMP_BYTES
    for name, a in sorted(arrays.items(), key=lambda kv: kv[1].nbytes):
        if a.nbytes > left:
            keep = left // (a.nbytes // len(a))
            a = a[np.sort(np.random.default_rng(0).choice(len(a), keep, replace=False))]
        np.save(os.path.join(path, name + ".npy"), a)
        left -= a.nbytes


# ===================================================================================== ours (GPU)
def run_ours(args):
    import torch
    import torch.distributed as dist
    from openmvg_b200 import ba, matching, synth
    rank, world, local = dist_env()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — openmvg_b200 has no CPU path (use --impl reference for the CPU baseline)")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def allmax(x):
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def allsum(x):
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t.item())

    pk = peaks()
    K, W = args.steps, args.warmup
    launches = 0
    outputs = {}                                      # what the last timed step of each leg returned (--dump-outputs)
    # ------------------------------------------------------------------ BA (replica per rank, same scene)
    scene = synth.ba_scene(*BA_CFG, seed=BA_SEED)
    n_obs = len(scene["obs_view"])
    ctx = ba.BAContext(scene, device=local)
    for _ in range(W):
        ctx.reset(); ctx.run()
    barrier()
    iters = 0; lm_steps = 0; dev_ms = 0.0; jac_ms = 0.0; jac_n = 0; last = None
    clk = ClockSampler(local); clk.__enter__()        # sampled over the BA and the MATCH timed regions
    t0 = time.perf_counter()
    for _ in range(K):
        ctx.reset(); r = ctx.run()
        iters += r["iterations"]; lm_steps += r["lm_steps"]; dev_ms += r["device_ms"]; jac_ms += r["jacobian_ms"]; jac_n += r["jacobian_launches"]; launches += r["kernel_launches"]; last = r
    barrier()
    wall = time.perf_counter() - t0
    ba_time = allmax(max(dev_ms / 1e3, 0.0))
    ba_wall = allmax(wall)
    ba_iters_all = allsum(iters)
    if args.dump_outputs:
        poses, intr, pts = ctx.download()
        outputs.update(ba_poses=poses, ba_intrinsics=intr, ba_points=pts, ba_cost=np.array([last["initial_cost"], last["final_cost"]]))
    ctx.close()
    # e2e: host buffers in, host buffers out, everything inside the timed region
    barrier()
    e_iters = 0; e_steps = max(1, min(K, 3))
    # inputs start in PINNED host memory (page-locked copies of the scene arrays), results land in host arrays
    scene_pinned = {k: (torch.from_numpy(np.ascontiguousarray(v)).pin_memory().numpy() if isinstance(v, np.ndarray) and k not in ("gt_R", "gt_C", "gt_dist") else v)
                    for k, v in scene.items()}
    t0 = time.perf_counter()
    for _ in range(e_steps):
        g = ba.solve(scene_pinned, device=local); e_iters += g["iterations"]; launches += g["kernel_launches"]
    barrier()
    e_wall = allmax(time.perf_counter() - t0); e_iters_all = allsum(e_iters)
    h2d = sum(scene[k].nbytes for k in ("poses", "intrinsics", "points", "intr_model", "view_pose", "view_intr", "obs_view", "obs_point", "obs_xy"))
    d2h = sum(scene[k].nbytes for k in ("poses", "intrinsics", "points"))
    jac_s = jac_ms / 1e3 / max(jac_n, 1)
    ba_roof = dict(bound="hbm", achieved=BA_BYTES_PER_OBS * n_obs / jac_s / 1e9, peak=pk["hbm_gbs"], unit="GB/s",
                   # dram__bytes_read.sum + dram__bytes_write.sum of one launch on this scene (ncu --set full capture,
                   # profiles/r01_ba_eval_kernel_full.md: 33.06 MB read + 150.79 MB written; less than the 232 MB of
                   # algorithmic bytes because the tail of the write stream is still in the 126 MB L2 when the kernel ends)
                   traffic=183.85e6 if n_obs == 1000000 else None, traffic_unit="bytes/launch",
                   kernel="eval_kernel<true> (residual+Jacobian+Huber+scaling)", launches=jac_n, avg_ms=jac_s * 1e3, peak_source=pk["src"])
    ba_roof["frac"] = ba_roof["achieved"] / ba_roof["peak"]
    # the whole LM iteration against the same bandwidth: algorithmic bytes of one iteration / device time per iteration
    step_s = dev_ms / 1e3 / max(iters, 1)
    ba_roof["step"] = dict(bytes_per_lm_iter=BA_STEP_BYTES_PER_OBS * n_obs, ms_per_lm_iter=step_s * 1e3,
                           achieved=BA_STEP_BYTES_PER_OBS * n_obs / step_s / 1e9, unit="GB/s",
                           what="712 B/obs: J+r written once (232), read once for the Schur complement (220), once for back-substitution + model change (220), cost-only candidate evaluation (40)")
    ba_roof["step"]["frac"] = ba_roof["step"]["achieved"] / pk["hbm_gbs"]

    # ------------------------------------------------------------------ BA sweep (configs[4]), rank 0 at N = 1
    sweep = None
    if world == 1 and not args.no_sweep:
        sweep = []
        for C in SWEEP_CAMS:
            s = synth.ba_scene(C, 50 * C, 10)
            c2 = ba.BAContext(s, device=local); c2.run(); c2.reset(); c2.run(); c2.reset()
            best = None
            for _ in range(3):
                c2.reset(); g = c2.run(); launches += g["kernel_launches"]
                if best is None or g["device_ms"] < best["device_ms"]:
                    best = g
            c2.close()
            sweep.append(dict(cams=C, points=50 * C, obs=500 * C, iterations=best["iterations"], device_ms=best["device_ms"],
                              ms_per_lm_iter=best["device_ms"] / best["iterations"], pcg_iterations=int(best["pcg_iterations"]),
                              kernel_launches=int(best["kernel_launches"]), final_cost=best["final_cost"]))

    # ------------------------------------------------------------------ geometric filter (SURVEY §8f N4), rank 0 at N = 1
    geom = None
    if world == 1 and not args.no_sweep:
        from openmvg_b200 import geometry
        pairs = [synth.two_view_matches(GEOM_MATCHES, 0.35, seed=500 + k, wh=(1600, 1200))[:2] for k in range(GEOM_PAIRS)]
        goff = np.concatenate([[0], np.cumsum([len(p_[0]) for p_ in pairs])]).astype(np.uint64)
        gI = np.concatenate([p_[0] for p_ in pairs]); gJ = np.concatenate([p_[1] for p_ in pairs])
        gsz = np.tile(np.array([1600, 1200, 1600, 1200], np.int32), (GEOM_PAIRS, 1))
        geometry.fundamental_acransac(goff, gI, gJ, gsz, 4.0, 2048, device=local)
        t0 = time.perf_counter(); gres = geometry.fundamental_acransac(goff, gI, gJ, gsz, 4.0, 2048, device=local); g_wall = time.perf_counter() - t0
        geom = {"metric": "pairs/sec", "value": GEOM_PAIRS / g_wall, "unit": "pairs/s", "ms_per_step": g_wall * 1e3,
                "config": {"workload": f"AC-RANSAC fundamental-matrix filter (GeometricFilter_FMatrix_AC(4.0, 2048)), {GEOM_PAIRS} pairs x {GEOM_MATCHES} putative matches, 35 % outliers"},
                "pairs_kept": int(sum(len(r_["inliers"]) > 17 for r_ in gres)), "inliers": int(sum(len(r_["inliers"]) for r_ in gres)),
                "note": "host arrays in, host arrays out (one omvg_geom_fundamental_acransac call: H2D, one CTA per pair, D2H)"}
        launches += 1

    # ------------------------------------------------------------------ MATCH (pairs sharded over ranks)
    def match_leg(n_img, steps, warm, e2e_steps, with_cascade, keep_outputs=False):
        nonlocal launches
        lo, hi, per = image_shard(n_img, rank, world)
        mine = synth.descriptor_collection(n_img, MATCH_DESC, seed=MATCH_SEED, lo=lo, hi=hi)
        host_mine = torch.zeros((per * MATCH_DESC, 128), dtype=torch.uint8).pin_memory()      # this rank's images, pinned host
        if mine:
            host_mine[: (hi - lo) * MATCH_DESC] = torch.from_numpy(np.concatenate(mine))
        dev_mine = torch.empty((per * MATCH_DESC, 128), dtype=torch.uint8, device="cuda")
        gathered = torch.empty((world * per * MATCH_DESC, 128), dtype=torch.uint8, device="cuda") if world > 1 else dev_mine
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        mctx = matching.MatchContext(local)
        mctx.set_images([MATCH_DESC] * n_img)
        pi, pj = synth.exhaustive_pairs(n_img)
        mpi, mpj = pair_shard(pi, pj, rank, world)
        desc_pairs_rank = float(len(mpi)) * MATCH_DESC * MATCH_DESC
        ag_ms = []

        def load_collection():
            """host (pinned, 1/N of the images) -> device -> all-gather -> arena + norms/keys.  Returns nothing; times the gather."""
            dev_mine.copy_(host_mine, non_blocking=True)
            if world > 1:
                ev[0].record()
                dist.all_gather_into_tensor(gathered, dev_mine)
                ev[1].record()
            torch.cuda.current_stream().synchronize()                 # the arena fill runs on the context's own stream
            if world > 1:
                ag_ms.append(ev[0].elapsed_time(ev[1]))
            mctx.upload_device_packed(gathered.data_ptr()); mctx.prepare()

        load_collection(); mctx.sync()
        for _ in range(warm):
            mctx.run(mpi, mpj, 0.8); mctx.sync()
        mctx.kernel_time(reset=True); l0 = mctx.launch_count()
        barrier()
        t0 = time.perf_counter()
        for _ in range(steps):
            mctx.run(mpi, mpj, 0.8)
        mctx.sync(); barrier()
        m_wall = allmax(time.perf_counter() - t0)
        tc_ms, tc_n = mctx.kernel_time(reset=True)
        off, ij = mctx.fetch()
        n_matches = len(ij)
        if keep_outputs:                              # indices below 2^24 (float32) and offsets below 2^53 (float64) stay exact
            outputs.update(match_offsets=off.astype(np.float64), match_ij=ij.astype(np.float32))
        # e2e: descriptors start in pinned host memory (this rank's 1/N); copy + all-gather + arena + prepare + run + fetch timed
        ag_ms.clear()
        barrier(); t0 = time.perf_counter()
        for _ in range(e2e_steps):
            load_collection(); mctx.run(mpi, mpj, 0.8); off, ij = mctx.fetch()
        barrier()
        me_wall = allmax(time.perf_counter() - t0)
        launches += mctx.launch_count() - l0
        total_pairs = allsum(desc_pairs_rank)
        all_matches = allsum(float(n_matches))
        ag = allmax(float(np.mean(ag_ms))) if ag_ms else 0.0
        tc_s = tc_ms / 1e3 / max(tc_n, 1)
        int8_peak = 2.0 * pk["bf16_sustained"]                          # dense INT8 = 2x bf16 rate; bf16 is the measured figure
        # one pass may take several launches (pair batches sized by the result-buffer budget): rate over all of them
        roof = dict(bound="tensor", achieved=OPS_PER_DESC_PAIR * desc_pairs_rank * steps / max(tc_ms / 1e3, 1e-12) / 1e12, peak=int8_peak, unit="TOP/s", traffic=None,
                    kernel="match_dig2_kernel (tcgen05 kind::i8, 4 descriptor K-slices + 1 digit slice, fused top-2; 256 algorithmic op per descriptor pair, the fifth slice is not counted)", launches=tc_n, avg_ms=tc_s * 1e3,
                    peak_source=f"2 x {pk['src']} bf16 sustained (INT8 dense rate = 2 x bf16)")
        roof["frac"] = roof["achieved"] / roof["peak"]
        gather_bytes = (world - 1) * per * MATCH_DESC * 128 if world > 1 else 0
        res = {"metric": "desc-pairs/sec", "value": total_pairs * steps / m_wall, "unit": "desc-pairs/s", "ms_per_step": m_wall * 1e3 / steps, "steps": steps, "dtype": "u8",
               "config": {"workload": f"exhaustive BRUTE_FORCE_L2 + ratio 0.8, {n_img} images x {MATCH_DESC} x 128-D uint8, {len(pi)} pairs sharded round-robin over {world} GPU(s)",
                          "l2": f"descriptor arena {n_img * MATCH_DESC * 128 / 1e6:.0f} MB + per-pair result buffers: larger than L2"},
               "matches": int(all_matches),
               "e2e": {"value": total_pairs * e2e_steps / me_wall, "unit": "desc-pairs/s", "h2d_bytes_per_step": (hi - lo) * MATCH_DESC * 128 + 8 * len(mpi),
                       "d2h_bytes_per_step": int(8 * (len(mpi) + 1) + 8 * n_matches), "ms_per_step": me_wall * 1e3 / e2e_steps, "steps": e2e_steps,
                       "allgather_ms": ag, "allgather_recv_bytes_per_rank": gather_bytes,
                       "allgather_gbs_per_rank": (gather_bytes / 1e9) / (ag / 1e3) if ag > 0 else None,
                       "path": "per rank: 1/N of the images pinned host -> device, NCCL all_gather_into_tensor, arena fill, prepare, match, fetch" if world > 1 else
                               "pinned host -> device, arena fill, prepare, match, fetch"},
               "roofline": roof}
        if with_cascade:
            # cascade hashing (openMVG's default matcher, SURVEY M9/N2) on the same pair shard: reported next to the
            # exhaustive matcher, not part of the headline (its parity against the reference is statistical: the hash
            # mat-vec order is fixed k-ascending, Eigen's GEMV order differs — 1 of 82 832 matches on 780 pairs)
            try:
                z_ = np.load(os.path.join(ROOT, "tests", "golden", "cascade_projections.npz"))      # CascadeHasher::Init's draw (fixture)
                mctx.cascade_prepare(z_["primary"], z_["secondary"], None); mctx.cascade_run(mpi, mpj, 0.8); mctx.sync()
                barrier(); t0 = time.perf_counter()
                for _ in range(steps):
                    mctx.cascade_run(mpi, mpj, 0.8)
                mctx.sync(); barrier()
                c_wall = allmax(time.perf_counter() - t0)
                res["cascade_hashing"] = {"ms_per_step": c_wall * 1e3 / steps, "pairs_per_s": allsum(float(len(mpi))) * steps / c_wall,
                                          "matches_rank0": int(len(mctx.fetch()[1])), "exhaustive_matches_rank0": int(n_matches),
                                          "parity": "bit-exact vs oracle/cascade_oracle.c; statistical vs the reference (float hashing order), >= 99.9 % identical",
                                          "note": "same pairs through omvg_match_cascade_run (hash tables resident); reference = Cascade_Hashing_Matcher_Regions"}
            except Exception as e:                                     # the fixture with the reference's projections is test data
                res["cascade_hashing"] = {"unavailable": str(e)[:120]}
        mctx.close()
        del gathered, dev_mine, host_mine
        torch.cuda.empty_cache()
        return res

    n_img = MATCH_IMAGES if args.match_images is None else args.match_images
    match = match_leg(n_img, K, W, max(1, min(K, 3)), True, keep_outputs=bool(args.dump_outputs))
    clk.__exit__()
    m2 = None
    if args.m2 or (world == 8 and not args.no_m2):
        m2 = match_leg(M2_IMAGES, 2, 1, 1, False)

    if rank == 0:
        line = {
            "metric": "BA LM-iters/sec", "value": ba_iters_all / ba_time, "unit": "LM-iter/s", "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": ba_time * 1e3 / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": BA_WORKLOAD, "l2": BA_L2},
            "detail": {"iterations_per_solve": last["iterations"], "lm_steps_per_solve": last["lm_steps"], "pcg_iterations_per_solve": last["pcg_iterations"],
                       "final_cost": last["final_cost"], "wall_ms_per_step": ba_wall * 1e3 / K, "kernel_launches_per_solve": int(last["kernel_launches"])},
            "e2e": {"value": e_iters_all / e_wall, "unit": "LM-iter/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "ms_per_step": e_wall * 1e3 / e_steps},
            "gpu_launches": int(launches), "roofline": ba_roof, "clocks": clk.summary(),
            "match": match, "match_value": match["value"], "match_unit": "desc-pairs/s", "match_e2e": match["e2e"]["value"],
            "match_roofline_frac": match["roofline"]["frac"],
        }
        if m2 is not None:
            line["m2"] = m2; line["m2_value"] = m2["value"]; line["m2_e2e"] = m2["e2e"]["value"]
        if sweep is not None:
            line["ba_sweep"] = sweep
        if geom is not None:
            line["geom"] = geom
        if not args.no_cpu and world == 1:
            cb, mb, _ = cpu_baselines(scene, full=False)
            line["cpu_baseline"], line["match"]["cpu_baseline"] = cb, mb
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, outputs)
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


# ===================================================================================== reference (CPU)
def cpu_baselines(scene, full, quick=False):
    """The reference itself (oracle/_ref) when it was built, else the oracle port; bounded samples.
    full=False (our arm's cpu_baseline): BA at {8, 32, N} threads, MATCH sample.  full=True (--impl reference):
    BA at {1, 8, 32, N/2, N} threads, MATCH sample, cascade-hashing sample, the configs[4] sweep."""
    import checkers as ck
    from openmvg_b200 import synth
    cores = os.cpu_count() or 1
    runs = []
    if ck.have_ref_ba():
        ths = sorted({min(cores, t) for t in ((1, 8, 32, max(1, cores // 2), cores) if full else (8, 32, cores))})
        if quick:
            ths = [min(cores, 8)]
        best = None
        for th in ths:
            r = ck.ref_ba_adjust(scene, threads=th)
            v = r["iterations"] / r["minimizer_s"]
            runs.append(dict(threads=th, adjust_wall_s=r["wall_s"], minimizer_s=r["minimizer_s"], lm_iter_per_s=v))
            if best is None or v > best["value"]:
                best = dict(value=v, unit="LM-iter/s", cores=th, kind="reference",
                            sample="one full Bundle_Adjustment_Ceres::Adjust on the same 1000/100k/1M scene per thread count; iterations / Ceres 'Minimizer' seconds; best thread count reported",
                            adjust_wall_s=r["wall_s"], minimizer_s=r["minimizer_s"], preprocessor_s=r["preprocessor_s"], iterations=r["iterations"],
                            final_cost=r["final_cost"], linear_solver_s=r["linear_solver_s"], jacobian_s=r["jacobian_s"])
        best["thread_sweep"] = runs; best["host_threads"] = cores
        ba_cpu = best
    else:
        small = synth.ba_scene(200, 10_000, 10)
        t0 = time.perf_counter(); o = ck.oracle_ba_solve(small); dt = time.perf_counter() - t0
        runs.append(dict(threads=cores, adjust_wall_s=dt))
        ba_cpu = dict(value=o["iterations"] / dt, unit="LM-iter/s", cores=cores, kind="port", sample="oracle port on 200 cams/10k pts/100k obs (1/10 of the workload)")
    n_img = 6 if quick else CPU_MATCH_IMAGES
    descs = synth.descriptor_collection(n_img, MATCH_DESC, seed=MATCH_SEED)
    pi, pj = synth.exhaustive_pairs(n_img)
    if ck.have_ref_match():
        ck.ref_match_collection(descs[:3], pi[:1], pj[:1])          # warm the thread pool
        t0 = time.perf_counter(); ck.ref_match_collection(descs, pi, pj); dt = time.perf_counter() - t0
        kind = "reference"
    else:
        t0 = time.perf_counter(); ck.oracle_match_collection(descs[:6], *synth.exhaustive_pairs(6)); dt = (time.perf_counter() - t0) * len(pi) / 15
        kind = "port"
    m_cpu = dict(value=len(pi) * MATCH_DESC * MATCH_DESC / dt, unit="desc-pairs/s", cores=cores, kind=kind,
                 sample=f"Matcher_Regions(BRUTE_FORCE_L2)::Match on the first {n_img} images of the collection = {len(pi)} image pairs of 5000x5000 descriptors (all host threads, AVX2 build)", seconds=dt,
                 extrapolated_m1_s=19900 * MATCH_DESC * MATCH_DESC * dt / (len(pi) * MATCH_DESC * MATCH_DESC))
    extra = {}
    if full and not quick:
        if ck.have_ref_match():
            t0 = time.perf_counter(); ck.ref_cascade_collection(descs, pi, pj, 0.8); dtc = time.perf_counter() - t0
            extra["cascade_hashing"] = dict(cpu_baseline=dict(value=len(pi) / dtc, unit="pairs/s", cores=cores, kind="reference", seconds=dtc,
                                                              sample=f"Cascade_Hashing_Matcher_Regions::Match on the same {len(pi)} pairs (hashing included)"))
        if ck.have_ref_geom():
            gp = [synth.two_view_matches(GEOM_MATCHES, 0.35, seed=500 + k, wh=(1600, 1200))[:2] for k in range(200)]
            t0 = time.perf_counter()
            for a_, b_ in gp:
                ck.ref_acransac_fundamental(a_, b_, (1600, 1200, 1600, 1200), 4.0, 2048)
            dtg = time.perf_counter() - t0
            extra["geom"] = dict(cpu_baseline=dict(value=200 / dtg, unit="pairs/s", cores=1, kind="reference", seconds=dtg,
                                                   sample="ACRANSAC + ACKernelAdaptor<SevenPointSolver, EpipolarDistanceError> on the first 200 pairs, ONE host thread (the reference runs one pair per OpenMP thread: multiply by the cores for its collection rate)"))
        if ck.have_ref_ba():
            sw = []
            for C in SWEEP_CAMS:
                s = synth.ba_scene(C, 50 * C, 10)
                b = None
                for th in sorted({min(cores, 8), min(cores, 32)}):
                    r = ck.ref_ba_adjust(s, threads=th)
                    if b is None or r["minimizer_s"] < b["minimizer_s"]:
                        b = dict(r, threads=th)
                sw.append(dict(cams=C, iterations=b["iterations"], minimizer_s=b["minimizer_s"], adjust_wall_s=b["wall_s"], threads=b["threads"],
                               ms_per_lm_iter=1e3 * b["minimizer_s"] / b["iterations"], final_cost=b["final_cost"]))
            extra["ba_sweep"] = sw
    return ba_cpu, m_cpu, extra


def run_reference(args):
    rank, world, _ = dist_env()
    if rank != 0:
        return
    from openmvg_b200 import synth
    scene = synth.ba_scene(*BA_CFG, seed=BA_SEED)
    ba_cpu, m_cpu, extra = cpu_baselines(scene, full=True, quick=args.quick)
    sweep = ba_cpu.get("thread_sweep", [])
    n_steps = max(1, len(sweep))                                  # one bounded sample (one Adjust) per thread count
    mean_wall_ms = 1e3 * float(np.mean([r["adjust_wall_s"] for r in sweep])) if sweep else 0.0
    line = {"impl": "reference", "metric": "BA LM-iters/sec", "value": ba_cpu["value"], "unit": "LM-iter/s", "n_gpus": world,
            "steps": n_steps, "steps_requested": args.steps, "warmup": 0, "warmup_requested": args.warmup,
            "ms_per_step": mean_wall_ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": BA_WORKLOAD, "l2": BA_L2},
            "cpu_baseline": ba_cpu, "e2e": {"value": ba_cpu["value"], "unit": "LM-iter/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0,
            "match": {"metric": "desc-pairs/sec", "value": m_cpu["value"], "unit": "desc-pairs/s", "cpu_baseline": m_cpu,
                      "e2e": {"value": m_cpu["value"], "unit": "desc-pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}},
            "match_value": m_cpu["value"], "match_unit": "desc-pairs/s", "match_e2e": m_cpu["value"]}
    if "cascade_hashing" in extra:
        line["match"]["cascade_hashing"] = extra["cascade_hashing"]
    if "ba_sweep" in extra:
        line["ba_sweep"] = extra["ba_sweep"]
    if "geom" in extra:
        line["geom"] = extra["geom"]
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg (profiling runs)")
    ap.add_argument("--no-sweep", action="store_true", help="skip the configs[4] BA sweep (profiling runs)")
    ap.add_argument("--m2", action="store_true", help="also run configs[3] (1000 images) at this N (default: only at N = 8)")
    ap.add_argument("--no-m2", action="store_true")
    ap.add_argument("--match-images", type=int, default=None)
    ap.add_argument("--quick", action="store_true", help="--impl reference only: one thread count, 15-pair MATCH sample, no sweep (the CPU test-suite uses it)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last BA solve and the last MATCH pass returned as DIR/<name>.npy "
                         "(float64 / float32, at most 64 MB; with --gpus N > 1, rank 0's pair shard of MATCH)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    if args.warmup < 3 and args.impl == "ours" and not args.no_cpu:
        args.warmup = 3
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
