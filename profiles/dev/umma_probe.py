"""Development probe: wfs_frame_umma_kernel against the float32 FFT kernel (10x10 and 40x40), for both readings of
the MN-major descriptor (AOM_UMMA_SWAP=0/1), each in its own process (an expired wait traps the context)."""
import os, subprocess, sys
sys.path.insert(0, ".")

CHILD = r'''
import sys, numpy as np, torch
sys.path.insert(0, ".")
from ao_marl_b200 import tables
from ao_marl_b200.config import load_config_from_file
from ao_marl_b200.lib import Simulator
par, E = sys.argv[1], int(sys.argv[2])
t = tables.build_static(load_config_from_file(par))
sim = Simulator(t, E, rl=None)
sim.reset(np.arange(E, dtype=np.int64) + 31)
r = np.random.default_rng(10)
volts = (r.standard_normal((E, t.nactu)) * (10 if t.nactu < 200 else 0.3)).astype(np.float32)
sim.set_dm_volts(torch.as_tensor(volts, device="cuda"))
for it in range(3):
    for _ in range(3):
        sim.move_atmos()
    res = {}
    for path in ("simt", "tensor", "umma", "umma_fast"):
        sim.set_wfs_path(path)
        name = sim.wfs_kernel()
        sim.comp_wfs_image(keep_image=(it % 2 == 0), noise=-1.0)
        sim.do_centroids()
        torch.cuda.synchronize()
        res[path] = (sim.rows("SLOPES", t.nslopes).cpu().numpy().copy(), name)
    ref = res["simt"][0]
    for path in ("tensor", "umma", "umma_fast"):
        err = np.abs(res[path][0] - ref).max() / np.abs(ref).max()
        print("it %d %-10s %-24s rel err vs simt %.3e" % (it, path, res[path][1], err), flush=True)
sim.check_device()
print("OK")
'''
for par, E in (("production_sh_10x10_2m.py", 4), ("production_sh_40x40_8m_3layers.py", 3)):
    for swap in ("0",):
        env = dict(os.environ, AOM_UMMA_SWAP=swap)
        print("=== %s E=%d AOM_UMMA_SWAP=%s" % (par, E, swap), flush=True)
        try:
            r = subprocess.run([sys.executable, "-c", CHILD, par, str(E)], env=env, capture_output=True, text=True, timeout=300)
            print(r.stdout[-3000:])
            if r.returncode != 0:
                print("rc", r.returncode, r.stderr[-1500:])
        except subprocess.TimeoutExpired:
            print("TIMEOUT")
