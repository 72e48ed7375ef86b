"""Exercises the HBM-bound kernels of the path once each (for `ncu --set full` captures, profiles/ncu_hbm_kernels_r02_summary.json):
K build at n = 8192 (kmat_p1_kernel), O(n^2) row append (kvec / trmv_lower / trmvT_lower_partial / reduce_rows / append_commit),
copy-on-write un-share (copy_lower_tiles), the device top-k selection over 2 M scores (sel_*), the small-n fused sweep (n = 64,
HBM side: 8 (d + 1) B per candidate) and the three-kernel GradientGP sweep (ks_build_kernel<.., true>, gemm_tma_kernel<EPI_COLSUMSQ>,
acq_epilogue_kernel)."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
import abo_b200 as abo
from oracle import abo_oracle as orc

c = orc.make_config("C4", n=8192, m=8, d=20)
k = c["scale"] * abo.with_lengthscale(abo.SqExponentialKernel(), 1.0 / c["inv_ls"])
gp = abo.update(abo.StandardGP(k, c["noise"]), c["X"][:-1], c["y"][:-1])          # kmat_p1 + factorisation
snap = abo.copy(gp)
gp2 = abo.update(gp, c["X"], c["y"])                                              # un-share + append
acq = abo.ExpectedImprovement(0.01, float(c["y"].min()))
m = 1 << 21
Xc = torch.rand((m, 20), dtype=torch.float64, device="cuda", generator=torch.Generator(device="cuda").manual_seed(1))
S = torch.empty(m, dtype=torch.float64, device="cuda")
c64 = orc.make_config("C4", n=64, m=8, d=20)
g64 = abo.update(abo.StandardGP(k, c64["noise"]), c64["X"], c64["y"])
g64.gpx.acq_eval_dev(acq.acq_id, acq.params(), Xc.data_ptr(), m, S.data_ptr(), k=100)     # fused sweep at n = 64 + sel_* over 2 M scores
c3 = orc.make_config("C3", n=128, m=16384)
kg = c3["scale"] * abo.with_lengthscale(abo.ApproxMatern52Kernel(), 1.0 / c3["inv_ls"])
gg = abo.update(abo.GradientGP(kg, 11, c3["noise"]), c3["X"], c3["Y"])
abo.ExpectedImprovement(*c3["acq_params"])(gg, c3["Xc"])                                   # ks_build<GRAD> + gemm_tma<EPI_COLSUMSQ> + acq_epilogue
torch.cuda.synchronize()
print("hbm_kernels_probe done")
