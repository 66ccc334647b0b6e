"""Routing of aom_actor_forward between the fused actor kernel (actor_tc.cuh: hidden and head layers of at most two
128-column tiles) and the gather + three gemm_tc_kernel + sampling sequence that serves wider actors.  The sequence is
checked against the float64 reference and error bound of test_actor_forward at a hidden size outside the fused kernel's
envelope; the launch count shows which path ran."""
import pytest

from test_actor_forward import Case


@pytest.fixture(scope="module")
def torch():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch


def launches_of_one_forward(c):
    before = c.sim.launches()
    c.forward("tcgen05", True)
    return c.sim.launches() - before


@pytest.mark.gpu
@pytest.mark.parametrize("hidden,E", [(512, 300), (512, 129)])
def test_wide_actor_falls_back_inside_bound(static10, torch, hidden, E):
    """hidden_size_actor = 512 is outside the fused kernel: gather, three GEMMs and sampling (five launches), every
    action inside its bound on both GEMM paths."""
    c = Case(static10, "10x10", hidden, E, E + hidden, torch)
    try:
        assert launches_of_one_forward(c) == 5
        c.steps += 1
        c.run_modes()
    finally:
        c.close()


@pytest.mark.gpu
def test_envelope_runs_fused(static10, torch):
    """hidden_size_actor = 256 with 160 head columns (two head tiles) is served by the single fused launch."""
    c = Case(static10, "10x10", 256, 129, 7, torch)
    try:
        assert launches_of_one_forward(c) == 1
    finally:
        c.close()
