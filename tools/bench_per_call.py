import os, sys, time; sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, strkit_b200
rng = np.random.default_rng(1)
def rs(n): return "".join(rng.choice(list("ACGT"), size=n))
p = strkit_b200.RepeatCountParams("repalign", 50, 3, 1)
fl, fr, motif = rs(70), rs(70), "CAG"
tr = motif * 30
strkit_b200.get_repeat_count(30, tr, fl, fr, motif, p)
t = time.perf_counter()
for i in range(500):
    # distinct tuples (no lru_cache hits), HiFi-sized: one flank base changes per call
    f2 = fl[:i % 70] + "ACGT"[(i // 70) % 4] + fl[i % 70 + 1:]
    strkit_b200.get_repeat_count(30, tr, f2, fr, motif, p)
dt = (time.perf_counter() - t) / 500
print("get_repeat_count per call: %.1f us" % (dt * 1e6))
rp = strkit_b200.get_reference_rc_params("repalign", 30, 250)
strkit_b200.get_ref_repeat_count(30, tr, fl, fr, motif, len(tr), 5, rp)
t = time.perf_counter()
for i in range(200):
    strkit_b200.get_ref_repeat_count(30, tr + "A" * (i % 3), fl, fr, motif, len(tr) + i % 3, 5, rp)
dt = (time.perf_counter() - t) / 200
print("get_ref_repeat_count per call: %.1f us" % (dt * 1e6))
