import os, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, abo_b200 as abo
from oracle import abo_oracle as orc
c = orc.make_config("C5")
gp0 = abo.StandardGP(abo.SqExponentialKernel(), c["noise"])
for _ in range(3): v, g, i = abo.nlml_batch(gp0, c["theta"], c["X"], c["y"])
ts = []
for _ in range(10):
    t0 = time.perf_counter(); v, g, i = abo.nlml_batch(gp0, c["theta"], c["X"], c["y"]); ts.append(time.perf_counter() - t0)
print("ms", 1e3 * min(ts), 1e3 * np.median(ts), "sum", float(np.sum(v[np.isfinite(v)])), "gsum", float(np.sum(g[np.isfinite(g)])))
