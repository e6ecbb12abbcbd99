"""Ad-hoc probe (not a test): time the MATCH path on n images x 5000 descriptors."""
import sys, time, os
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
from openmvg_b200 import matching, synth
n = int(sys.argv[1]) if len(sys.argv) > 1 else 40
reps = int(sys.argv[2]) if len(sys.argv) > 2 else 3
descs = synth.descriptors(n, 5000, seed=1000)
pi, pj = synth.exhaustive_pairs(n)
ctx = matching.MatchContext(0)
ctx.load(descs)
print('kernel variant', ctx.kernel_variant())
for r in range(reps):
    t = time.time(); ctx.run(pi, pj, 0.8); ctx.sync(); dt = time.time() - t
    ms, k = ctx.kernel_time()
    print("run", r, "pairs", len(pi), "wall %.2f ms" % (dt * 1e3), "tc kernel %.2f ms" % ms, "desc-pairs/s %.3e" % (len(pi) * 25e6 / dt), "TOP/s(tc) %.0f" % (len(pi) * 25e6 * 256 / (ms / 1e3) / 1e12))
off, ij = ctx.fetch(); print("matches", len(ij))
