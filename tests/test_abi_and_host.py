"""CPU: the C-ABI library loads and exports every symbol include/omvg_b200.h declares (no compute
without a GPU), fails loudly without a device, and the host-side sharding logic works over gloo."""
import ctypes
import os
import re
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    from openmvg_b200.build import build
    build()
    from openmvg_b200._lib import lib as L
    return L()


def test_every_declared_symbol_is_exported(lib):
    hdr = open(os.path.join(ROOT, "include", "omvg_b200.h")).read()
    names = set(re.findall(r"\b(omvg_[a-z0-9_]+)\s*\(", hdr))
    assert len(names) >= 25
    for n in sorted(names):
        assert hasattr(lib, n), f"{n} declared in omvg_b200.h but not exported"


def test_struct_layouts_match_header(lib):
    from openmvg_b200 import ba
    assert ctypes.sizeof(ba.Options) == 128 and ctypes.sizeof(ba.Summary) == 80 and ctypes.sizeof(ba.Problem) == 160
    o = ba.default_options()
    assert (o.intrinsics_opt, o.extrinsics_opt, o.structure_opt, o.use_loss) == (14, 6, 1, 1)
    assert o.huber_a == 16.0 and o.max_num_iterations == 50 and o.function_tolerance == 1e-6
    assert o.gradient_tolerance == 1e-10 and o.parameter_tolerance == 1e-8 and o.initial_radius == 1e4


def test_fails_loudly_without_gpu(lib):
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from openmvg_b200 import ba, matching, synth
    from openmvg_b200._lib import OmvgError
    with pytest.raises(OmvgError):
        matching.MatchContext(0)
    with pytest.raises(OmvgError):
        ba.solve(synth.ba_scene(4, 20, 3))
    assert lib.omvg_device_count() == 0


def test_product_never_imports_oracle():
    """The product path must not route through oracle/ (no CPU fallback)."""
    pkg = os.path.join(ROOT, "openmvg_b200")
    for dp, _, fs in os.walk(pkg):
        for f in fs:
            if f.endswith((".py", ".cu", ".cuh", ".hpp", ".h", ".cpp")):
                txt = open(os.path.join(dp, f), errors="replace").read()
                assert "oracle/" not in txt.replace("oracle/_ref", "").replace("oracle/)", "") or f in ("synth.py",), f
                assert "checkers" not in txt, f


WORKER = r'''
import os, sys
import numpy as np, torch, torch.distributed as dist
sys.path.insert(0, sys.argv[1])
from openmvg_b200 import synth
import bench
dist.init_process_group("gloo", init_method="tcp://127.0.0.1:%s" % sys.argv[2], rank=int(sys.argv[3]), world_size=2)
rank, world = dist.get_rank(), 2
n_img, nd = 7, 40                                   # odd on purpose: the last rank's tile is short and padded
lo, hi, per = bench.image_shard(n_img, rank, world)
mine = synth.descriptor_collection(n_img, nd, seed=1000, block=3, lo=lo, hi=hi)      # each rank draws only ITS images
assert len(mine) == hi - lo
pad = torch.zeros((per * nd, 128), dtype=torch.uint8); pad[: (hi - lo) * nd] = torch.from_numpy(np.concatenate(mine))
out = [torch.zeros_like(pad) for _ in range(world)]
dist.all_gather(out, pad)
allrows = torch.cat(out)[: n_img * nd]
# every rank must hold the whole collection, image k at rows [k*nd, (k+1)*nd) — what upload_device_packed expects
ref = np.concatenate(synth.descriptor_collection(n_img, nd, seed=1000, block=3))
assert np.array_equal(allrows.numpy(), ref)
pi, pj = synth.exhaustive_pairs(n_img)
mpi, mpj = bench.pair_shard(pi, pj, rank, world)
mine_pairs = set(zip(mpi.tolist(), mpj.tolist()))
cnt = torch.tensor([len(mine_pairs)]); dist.all_reduce(cnt)
assert int(cnt) == len(pi)                      # the shards partition the pair list
gathered = [None, None]; dist.all_gather_object(gathered, sorted(mine_pairs))
assert sorted(gathered[0] + gathered[1]) == sorted(zip(pi.tolist(), pj.tolist()))
assert not (set(map(tuple, gathered[0])) & set(map(tuple, gathered[1])))
assert abs(len(gathered[0]) - len(gathered[1])) <= 1
dist.destroy_process_group()
print("ok", rank)
'''


def test_pair_sharding_world2_gloo(tmp_path):
    """bench.py's multi-GPU plumbing on CPU: all-gather of per-rank descriptor tiles + round-robin pair
    shards partition the exhaustive pair list (world_size 2, gloo)."""
    w = tmp_path / "worker.py"; w.write_text(WORKER)
    import socket
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    procs = [subprocess.Popen([sys.executable, str(w), ROOT, str(port), str(r)], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True) for r in range(2)]
    outs = [p.communicate(timeout=240)[0] for p in procs]
    for p, o in zip(procs, outs):
        assert p.returncode == 0, o


def test_bench_dump_outputs_budget_and_sample(tmp_path):
    """bench.py --dump-outputs: one .npy per array, at most 64 MB in all; an array over the budget becomes a seeded
    sample of its rows, the same rows on every run."""
    import bench
    small = np.linspace(0.0, 1.0, 7)
    big = np.arange(3 * bench.DUMP_BYTES // 8, dtype=np.float32).reshape(-1, 2)        # 1.5 x the budget
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), {"small": small, "big": big})
    assert sorted(os.listdir(tmp_path / "a")) == ["big.npy", "small.npy"]
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in os.listdir(tmp_path / "a")) <= 64_000_000
    assert np.array_equal(np.load(tmp_path / "a" / "small.npy"), small)
    s = np.load(tmp_path / "a" / "big.npy")
    assert s.dtype == np.float32 and 0 < len(s) < len(big) and np.all(np.diff(s[:, 0]) > 0) and np.array_equal(s, big[(s[:, 0] // 2).astype(np.int64)])
    assert np.array_equal(s, np.load(tmp_path / "b" / "big.npy"))


# ---- file formats (SURVEY §8f N3): host-side, no GPU needed
def _sample_csr():
    pI = np.array([7, 2, 2, 9, 4], np.uint32); pJ = np.array([9, 5, 3, 11, 6], np.uint32)      # unsorted, one empty pair
    counts = [3, 2, 4, 0, 1]
    off = np.concatenate([[0], np.cumsum(counts)]).astype(np.uint64)
    rng = np.random.default_rng(0)
    ij = rng.integers(0, 5000, (int(off[-1]), 2)).astype(np.uint32)
    return pI, pJ, off, ij


@pytest.mark.parametrize("ext", ["txt", "bin"])
def test_matches_file_matches_reference_fixture(tmp_path, ext):
    """omvg_matches_save writes byte for byte what matching::Save writes (fixtures generated by the reference,
    tests/golden/make_golden.py): std::map order, empty pairs dropped."""
    from openmvg_b200 import matching
    pI, pJ, off, ij = _sample_csr()
    out = tmp_path / f"matches.putative.{ext}"
    matching.save_matches(str(out), pI, pJ, off, ij)
    want = open(os.path.join(ROOT, "tests", "golden", f"matches_fixture.{ext}"), "rb").read()
    assert out.read_bytes() == want


def test_matches_save_rejects_bad_arguments(tmp_path):
    from openmvg_b200 import matching
    from openmvg_b200._lib import OmvgError
    pI, pJ, off, ij = _sample_csr()
    with pytest.raises(OmvgError):
        matching.save_matches(str(tmp_path / "m.json"), pI, pJ, off, ij)
    with pytest.raises(OmvgError):
        matching.save_matches(str(tmp_path / "m.txt"), np.array([1, 1], np.uint32), np.array([2, 2], np.uint32), np.array([0, 1, 2], np.uint64), ij[:2])


def test_desc_file_layout_is_the_reference_one(tmp_path):
    """The '.desc' writer the GPU loader test uses produces the reference's bytes (fixture from saveDescsToBinFile)."""
    from openmvg_b200 import matching, synth
    d = synth.descriptors(1, [37], seed=3)[0]
    p = tmp_path / "a.desc"
    matching.write_desc_file(str(p), d)
    assert p.read_bytes() == open(os.path.join(ROOT, "tests", "golden", "desc_fixture.desc"), "rb").read()


def _build_c_example(tmp_path):
    exe = str(tmp_path / "minimal_c_abi")
    lib_dir = os.path.join(ROOT, "openmvg_b200")
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-Wextra", "-pedantic", "-Werror", os.path.join(ROOT, "examples", "minimal_c_abi.c"),
                           "-I" + os.path.join(ROOT, "include"), "-L" + lib_dir, "-lomvg_b200", "-Wl,-rpath," + lib_dir, "-lm", "-o", exe])
    return exe


def test_header_is_plain_c_and_example_fails_loudly_without_gpu(tmp_path):
    """include/omvg_b200.h compiles as strict C99; without a B200 the first call reports OMVG_E_CUDA."""
    from openmvg_b200 import build
    build.build()
    exe = _build_c_example(tmp_path)
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present: covered by the gpu-marked variant")
    r = subprocess.run([exe], capture_output=True, text=True)
    assert r.returncode == 0 and "no B200" in r.stdout


@pytest.mark.gpu
def test_c_example_runs_on_gpu(tmp_path):
    exe = _build_c_example(tmp_path)
    r = subprocess.run([exe], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "MATCH: 50 matches" in r.stdout and "BA: rc 0" in r.stdout


@pytest.mark.skipif(not os.path.exists(os.path.join(ROOT, "oracle", "_ref", "libref_ba.so")), reason="oracle/_ref not built")
def test_reference_arm_prints_the_contract_line():
    """`bench.py --impl reference` (the CPU arm the driver runs next to ours): one JSON line with the same metric,
    unit and workload string as our arm, impl == "reference", a cpu_baseline of kind "reference" and zero-copy e2e."""
    import json
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "1", "--steps", "1", "--warmup", "0", "--quick"],
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])
    assert line["impl"] == "reference" and line["metric"] == "BA LM-iters/sec" and line["unit"] == "LM-iter/s" and line["higher_is_better"] is True
    assert line["value"] > 0 and line["cpu_baseline"]["kind"] == "reference" and line["cpu_baseline"]["cores"] >= 1
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["e2e"]["d2h_bytes_per_step"] == 0 and line["e2e"]["value"] == line["value"]
    ours = open(os.path.join(ROOT, "bench.py")).read()
    assert ours.count(line["config"]["workload"]) == 1 and ours.count("BA_WORKLOAD") == 3   # one string, used by both arms
    assert line["steps"] == len(line["cpu_baseline"]["thread_sweep"]) and line["ms_per_step"] > 0    # the steps it actually ran
    assert set(line["config"]) == {"workload", "l2"}
    assert line["match"]["cpu_baseline"]["kind"] == "reference" and line["match"]["value"] > 0
