"""Tile list of the per-environment actor kernel (ctrl_tiles_host.h, what aom_set_controller_env builds), checked on the
CPU through a host build of that header: every environment on a policy slot appears exactly once, in a tile of its own slot; tiles
hold one slot and at most 128 environments, grouped by slot; integrator environments are absent and listed apart."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
TILE = 128


@pytest.fixture(scope="module")
def harness(tmp_path_factory):
    src = os.path.join(HERE, "cpu_kernels", "ctrl_tiles_harness.cpp")
    out = str(tmp_path_factory.mktemp("ctrl_tiles") / "libctrl_tiles.so")
    subprocess.run(["g++", "-O2", "-shared", "-fPIC", "-o", out, src], check=True)
    return ctypes.CDLL(out)


def P(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def build(h, ctrl):
    ctrl = np.ascontiguousarray(ctrl, np.int32)
    E = ctrl.size
    tmax = h.h_ctrl_tiles_max(E)
    slot = np.full(tmax, -7, np.int32)
    env = np.full((tmax, TILE), -7, np.int32)
    integ = np.full(E, -7, np.int32)
    ni = ctypes.c_int(-1)
    n = h.h_ctrl_tiles(P(ctrl), E, P(slot), P(env), P(integ), ctypes.byref(ni))
    assert 0 <= n <= tmax
    return slot[:n], env[:n], integ[:ni.value]


def check(h, ctrl):
    ctrl = np.asarray(ctrl, np.int32)
    slot, env, integ = build(h, ctrl)
    listed = env[env >= 0]
    on_slot = np.flatnonzero(ctrl >= 0)
    assert np.array_equal(np.sort(listed), on_slot)                      # every slot environment exactly once
    assert np.unique(listed).size == listed.size
    for t in range(slot.size):
        rows = env[t][env[t] >= 0]
        assert 0 < rows.size <= TILE
        assert (env[t][rows.size:] == -1).all()                          # padding only at the end
        assert (ctrl[rows] == slot[t]).all()                             # one slot per tile
        assert (np.diff(rows) > 0).all()
    assert (np.diff(slot) >= 0).all()                                    # tiles of a slot next to each other
    for s in np.unique(slot):
        n = int((ctrl == s).sum())
        assert int((slot == s).sum()) == (n + TILE - 1) // TILE          # the fewest tiles per slot
    assert np.array_equal(integ, np.flatnonzero(ctrl == -1))             # integrator environments apart, not in tiles
    return slot, env, integ


def test_interleaved_slots_and_integrator(harness):
    r = np.random.default_rng(1)
    for E in (1, 127, 128, 129, 300, 4096, 4099):
        check(harness, r.integers(-1, 8, E))
        check(harness, np.arange(E) % 3 - 1)


def test_single_environment(harness):
    for c in range(-1, 8):
        slot, env, integ = check(harness, [c])
        assert slot.size == (0 if c < 0 else 1)


def test_all_integrator(harness):
    slot, env, integ = check(harness, np.full(300, -1))
    assert slot.size == 0 and integ.size == 300


def test_one_slot_is_the_uniform_tiling(harness):
    """Every environment on one slot: the tiles of the uniform kernel, 128 consecutive environments each."""
    E = 300
    slot, env, _ = check(harness, np.full(E, 5))
    assert (slot == 5).all() and slot.size == 3
    ref = np.full(3 * TILE, -1)
    ref[:E] = np.arange(E)
    assert np.array_equal(env.ravel(), ref)


def test_roket_refuses_per_environment_controllers():
    """ROKET's breakdown has one controller: it raises while per-environment controllers are in force, and not otherwise."""
    import types
    from ao_marl_b200.guardians.roket import Roket
    stub = types.SimpleNamespace(sim=types.SimpleNamespace(gain_env=None, controller_env=np.array([0, -1], np.int32)))
    stub._common_gain = lambda: Roket._common_gain(stub)
    stub._one_controller = lambda: Roket._one_controller(stub)
    with pytest.raises(NotImplementedError, match="one controller"):
        Roket.do_error_breakdown(stub)
    stub.sim.controller_env = None
    Roket._one_controller(stub)
