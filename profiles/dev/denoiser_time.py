"""Development probe: device time of the denoiser (row a-6) per 40x40 frame: fused kernel vs cuDNN through torch."""
import sys
sys.path.insert(0, ".")
import numpy as np
import torch
from ao_marl_b200 import tables
from ao_marl_b200.config import load_config_from_file
from ao_marl_b200.denoiser import Autoencoder
from ao_marl_b200.lib import Simulator

nv = 1200
t = tables.build_static(load_config_from_file("production_sh_10x10_2m.py"))
sim = Simulator(t, 1, rl=None, atmosphere=False)
ae = Autoencoder(dict(type="cnn_single_subaperture", path="autoencoder_M9_rms_3"), device="cuda", sim=sim)
lib = Autoencoder(dict(type="cnn_single_subaperture", path="autoencoder_M9_rms_3"), device="cuda")


def timed(fn, x, reps=3):
    for _ in range(2):
        fn(x)
    torch.cuda.synchronize()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    ev[0].record()
    for _ in range(reps):
        fn(x)
    ev[1].record()
    torch.cuda.synchronize()
    return ev[0].elapsed_time(ev[1]) / reps


for E in (64, 1024):
    x = torch.rand((E * nv, 16, 16), device="cuda") * 20
    ms = timed(ae.predict, x)
    print("fused kernel  E=%d: %.2f ms per frame, %.1f us per env, %.1f TFLOP/s" % (E, ms, ms / E * 1e3, 3.42e6 * E * nv / ms / 1e9))
for E, tf32 in ((64, False), (64, True)):
    torch.backends.cudnn.allow_tf32 = tf32
    x = torch.rand((E * nv, 16, 16), device="cuda") * 20
    ms = timed(lib.predict, x)
    print("cuDNN tf32=%s E=%d: %.2f ms per frame, %.1f us per env, %.1f TFLOP/s" % (tf32, E, ms, ms / E * 1e3, 3.42e6 * E * nv / ms / 1e9))
sim.close()
