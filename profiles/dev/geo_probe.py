"""Development probe: where does the CUDA geometric projection differ from the float64 host pipeline (40x40)?"""
import sys
sys.path.insert(0, ".")
import numpy as np
import torch
from ao_marl_b200 import tables
from ao_marl_b200.config import load_config_from_file
from ao_marl_b200.init import geo
from ao_marl_b200.lib import Simulator, pad_rows

t = tables.build_static(load_config_from_file("production_sh_40x40_8m_3layers.py"))
P, sifn = geo.build_geo(t)
IF = geo.influence_rows(t)
n = t.n
m = (t.mpupil != 0).ravel()
sim = Simulator(t, 2, rl=None)
sim.reset(np.array([301, 302], dtype=np.int64))
sim.move_atmos()
phase = sim.raytrace_wfs(atmos=True, dms=False).cpu().numpy().astype(np.float64)
com = sim.do_control_geo().cpu().numpy().astype(np.float64)
bdev = sim.rows("GEO_PROJ", t.nactu).cpu().numpy().astype(np.float64)
for e in range(2):
    phi = phase[e].ravel()
    mean = phi[m].mean()
    b = IF @ (m * (phi - mean))
    c = P.astype(np.float64) @ b
    print("env", e, "phase rms", phi[m].std(), "mean", mean)
    d = np.abs(bdev[e] - b)
    print("  b: max|b|", np.abs(b).max(), "max diff", d.max(), "at", d.argmax(), "tt diff", d[-2:], "median diff", np.median(d))
    print("  com: max", np.abs(c).max(), "max diff dev-host", np.abs(com[e] - c).max())
    cg = sim.gemm_tn(torch.as_tensor(pad_rows(b[None, :].astype(np.float32)), device="cuda"),
                     torch.as_tensor(pad_rows(P), device="cuda"))[0, :t.nactu].cpu().numpy()
    print("  device gemm on host b: max diff", np.abs(cg - c).max())
    for nm, cc in (("host", c), ("dev", com[e]), ("devgemm(host b)", cg), ("host P @ dev b", P.astype(np.float64) @ bdev[e])):
        r = (phi - mean) * m + IF.T @ cc
        print("  resid var", nm, r[m].var())
    worst = np.argsort(d)[-8:]
    print("  worst b rows", worst, d[worst], b[worst])
sim.close()
