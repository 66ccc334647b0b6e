"""Development probe: device time of the geometric controller at the bench size (E = 4096, 40x40, 3 layers)."""
import sys
sys.path.insert(0, ".")
import numpy as np
import torch
from ao_marl_b200 import tables
from ao_marl_b200.config import load_config_from_file
from ao_marl_b200.init import geo
from ao_marl_b200.lib import Simulator

E = int(sys.argv[1]) if len(sys.argv) > 1 else 4096
t = tables.build_static(load_config_from_file("production_sh_40x40_8m_3layers.py"))
geo.build_geo(t)
sim = Simulator(t, E, rl=None)
sim.reset(1234 + np.arange(E, dtype=np.int64))
sim.move_atmos()
for _ in range(2):
    sim.do_control_geo()
torch.cuda.synchronize()
ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
ev[0].record()
for _ in range(5):
    sim.do_control_geo()
ev[1].record()
torch.cuda.synchronize()
print("do_control_geo ms", ev[0].elapsed_time(ev[1]) / 5)
ev[0].record()
for _ in range(5):
    sim.comp_strehl(1.65, geo=True)
ev[1].record()
torch.cuda.synchronize()
print("comp_strehl ms", ev[0].elapsed_time(ev[1]) / 5)
sim.close()
