"""A/B of BA kernel variants on config 2 (and the 2000-camera sweep point): one subprocess per environment
setting (the switches are read once per process).  python tools/ba_ab.py [cams points obs_per_point]"""
import json, os, subprocess, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CHILD = r'''
import sys, json
sys.path.insert(0, %r)
from openmvg_b200 import ba, synth
C, Pn, K = %d, %d, %d
s = synth.ba_scene(C, Pn, K)
ctx = ba.BAContext(s)
for _ in range(3): ctx.reset(); ctx.run()
best = None
for _ in range(5):
    ctx.reset(); r = ctx.run()
    if best is None or r["device_ms"] < best["device_ms"]: best = r
print(json.dumps(dict(device_ms=best["device_ms"], iters=best["iterations"], pcg=best["pcg_iterations"], cost=best["final_cost"], launches=best["kernel_launches"])))
'''
cfg = [int(x) for x in sys.argv[1:4]] if len(sys.argv) >= 4 else [1000, 100000, 10]
variants = [("default (pcg5)", {}), ("pcg5 timing", {"OMVG_BA_PCG_TIMING": "1"}), ("coarse every step", {"OMVG_BA_COARSE_EVERY": "1"}), ("coarse every 4", {"OMVG_BA_COARSE_EVERY": "4"}),
            ("gj timing", {"OMVG_BA_GJ_TIMING": "1"})]
for name, env in variants:
    e = dict(os.environ); e.update(env)
    p = subprocess.run([sys.executable, "-c", CHILD % (ROOT, *cfg)], capture_output=True, text=True, env=e, timeout=600)
    tail = [l for l in p.stderr.splitlines() if "timing" in l][-3:]
    print(f"{name:22s} {p.stdout.strip()[-300:]} {' | '.join(tail)}", flush=True)
    if p.returncode:
        print(p.stderr[-1500:])
