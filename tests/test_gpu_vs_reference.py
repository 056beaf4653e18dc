"""Kernel-by-kernel parity against the UNMODIFIED reference's Numba-CUDA kernels.

The reference cannot be committed to this repository, so what its kernels computed on a GPU is stored in
tests/golden/ref_numba_cuda.npz (written by oracle/make_golden_numba_cuda.py, which replays the same kernel
sequence on the same seeded scenarios).  What is asserted (same inputs on both sides: seed, PMFs, masks, params):
  * host preprocessing of the PMF grid, control noise, sampled traction maps: bit-identical (whole-array
    SHA-256, plus the stored sample of values so that a mismatch says how many differ)
  * deterministic-mode rollout costs: bit-identical
  * stochastic CVaR costs: within 1e-4 relative (only the summation order of the CVaR mean differs),
    including M > 1024 against the reference's oversized kernel at cvar_alpha = 1
  * updated control sequence given the reference's costs: within 1e-4
"""
import io
import contextlib
import os

import numpy as np
import pytest

from oracle.make_golden_numba_cuda import CASES, case_key, case_scenario, digest

pytestmark = pytest.mark.gpu


def _quiet(fn, *a, **k):
    with contextlib.redirect_stdout(io.StringIO()):
        return fn(*a, **k)


@pytest.fixture(scope="module")
def ref(golden_dir):
    return np.load(os.path.join(golden_dir, "ref_numba_cuda.npz"), allow_pickle=False)


def _assert_same_as_reference(g, name, got):
    """`got` bit-identical to the reference's array `name` of this case."""
    got = np.ascontiguousarray(got)
    assert got.shape == tuple(g(name + "_shape")) and got.dtype.str == str(g(name + "_dtype")), \
        (name, got.shape, got.dtype.str, tuple(g(name + "_shape")), str(g(name + "_dtype")))
    idx = g(name + "_idx")
    bad = int((got.reshape(-1)[idx] != g(name + "_val")).sum())
    assert bad == 0, "%s: %d of %d sampled values differ from the reference" % (name, bad, idx.size)
    assert digest(got) == str(g(name + "_sha256")), "%s differs from the reference outside the sampled values" % name


@pytest.mark.parametrize("mode,N,M,T,H,res,B,det_alpha", CASES)
def test_kernels_vs_reference_numba_cuda(ref, mode, N, M, T, H, res, B, det_alpha):
    key = case_key(mode, N, M, T, H, res, B, det_alpha)

    def g(name):
        return ref[key + "__" + name]
    import __graft_entry__
    __graft_entry__.build()
    import mppi_numba_b200 as E
    sc = case_scenario(mode, N, M, T, H, res, B, det_alpha)
    p = sc["params"]
    cfg = _quiet(E.Config, **sc["cfg"])
    el, ea = _quiet(E.TDM_Numba, cfg), _quiet(E.TDM_Numba, cfg)
    _quiet(el.set_TDM_from_PMF_grid, sc["pmf_lin"], sc["tdm_dict"], sc["obstacle"], sc["unknown"])
    _quiet(ea.set_TDM_from_PMF_grid, sc["pmf_ang"], sc["tdm_dict"], sc["obstacle"], sc["unknown"])
    ep = _quiet(E.MPPI_Numba, cfg)
    ep.setup(p, el, ea)
    ep.u_cur_d.copy_to_device(sc["u0"])
    ep.move_mppi_task_vars_to_device()
    L = E._lib
    Hp, Wp = el.pmf_grid_d.shape[1:]
    # host preprocessing of the setter
    _assert_same_as_reference(g, "pmf", el.pmf_grid_d.copy_to_host())
    # the body of solve_* kernel by kernel (same seed -> same streams as the reference's)
    alpha_dyn = 0.9 if mode == "tdm" else 1.0
    eg_l, eg_a = el.sample_grids(alpha_dyn).copy_to_host(), ea.sample_grids(alpha_dyn).copy_to_host()
    _assert_same_as_reference(g, "lin", eg_l[:, :Hp, :Wp])
    _assert_same_as_reference(g, "ang", eg_a[:, :Hp, :Wp])
    L.check(L.lib.b200mppi_planner_sample_noise(ep._handle))
    _assert_same_as_reference(g, "noise", ep.noise_samples_d.copy_to_host())
    ref_costs = g("costs")
    L.check(L.lib.b200mppi_planner_rollout(ep._handle))
    got = ep.costs_d.copy_to_host()
    assert got.shape == ref_costs.shape
    rel = np.abs(got - ref_costs) / np.maximum(np.abs(ref_costs), 1e-6)
    print("\n[%s] costs bit-identical %.4f, max rel %.2e" % (mode, float((got == ref_costs).mean()), float(rel.max())))
    if mode == "det":
        assert (got == ref_costs).all()
    else:
        assert rel.max() < 1e-4
    ref_u = g("u")
    c = np.ascontiguousarray(ref_costs)
    L.check(L.lib.b200mppi_planner_update(ep._handle, L.ptr(c)))
    eu = ep.u_cur_d.copy_to_host()
    np.testing.assert_allclose(eu, ref_u, rtol=1e-4, atol=1e-5)
