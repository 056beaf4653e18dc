"""The CUDA engine at planner parameters away from the defaults (run with ``-m gpu`` on a B200): per-(n,m) costs of the
windowed and the generic rollout kernels, CVaR, the deterministic and speed-map kernels and the update, through the
C-ABI, against the reference's own kernels at the two points of tests/golden/ref_params.npz; a whole solve() sequence
through the public API at P1; the windowed kernel against the generic one at scale; and reach-box sampling when the
traction exceeds 1 and speeds go negative.  Costs cross zero at these points, so relative errors are taken against
max(|ref|, 1)."""
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

from oracle import mppi_ref as MR                          # noqa: E402
from tests.scenarios import make_scenario                  # noqa: E402
from tests.test_gpu_parity import RawPlanner              # noqa: E402

POINTS = ("p1", "p2")


@pytest.fixture(scope="module")
def eng():
    import __graft_entry__
    __graft_entry__.build()
    import mppi_numba_b200 as E
    assert E.device_count() >= 1, "GPU tests need a CUDA device"
    return E


def load_all(golden_dir):
    return np.load(os.path.join(golden_dir, "ref_params.npz"), allow_pickle=False)


def point(golden_dir, name):
    g = load_all(golden_dir)
    return {k[len(name) + 1:]: g[k] for k in g.files if k.startswith(name + "_")}


def rel1(a, ref):
    return np.abs(np.asarray(a, np.float64) - ref) / np.maximum(np.abs(np.asarray(ref, np.float64)), 1.0)


def _planner(eng, d, mode, M):
    """RawPlanner on the point's maps: the sampled grids, masks and risk map of the golden data, the point's traction
    bounds (the PMF is a placeholder: the grids are set directly)."""
    R, Cc = d["lin"].shape[1:]
    Hp, Wp = d["obs"].shape
    N, T = d["noise"].shape[:2]
    rp = RawPlanner(eng, mode, N, M, T, R, Cc)
    dummy = np.zeros((2, Hp, Wp), dtype=np.int8)
    dummy[1] = 100
    for which in ("lin", "ang"):
        rp.set_map(which, dummy, d[which + "_bounds"], d[which + "_bounds"], d["res"], d["xlim"], d["ylim"],
                   d["obs"], d["unk"], d["risk"][0] if mode == 2 else None)
    rp.set_grids("lin", d["lin"][:rp.M])
    rp.set_grids("ang", d["ang"][:rp.M])
    rp.copy_in(eng._lib.BUF_NOISE, d["noise"])
    rp.copy_in(eng._lib.BUF_U_CUR, d["u_cur"])
    return rp


def _point_params(d, gname, **kw):
    return dict(x0=list(d["x0"]), xgoal=list(d["xgoal_" + gname]), dt=float(d["dt"]), goal_tolerance=float(d["goal_tol"]),
                v_post_rollout=float(d["v_post"]), lambda_weight=float(d["lam"]), u_std=list(d["u_std"]),
                vrange=list(d["vrange"]), wrange=list(d["wrange"]), obs_penalty=float(d["obs_cost"]),
                unknown_penalty=float(d["unk_cost"]), dist_weight=float(d["dist_weight"]), **kw)


# ----------------------------------------------------------------------------- kernels through the C-ABI
@pytest.mark.parametrize("name", POINTS)
@pytest.mark.parametrize("gname", ["near", "far"])
@pytest.mark.parametrize("no_window", [False, True])
def test_stochastic_rollout_and_cvar_vs_reference_at_param_point(eng, golden_dir, monkeypatch, name, gname, no_window):
    """Per-(n,m) costs of the windowed kernel (no_window False) or the generic kernel (B200MPPI_NO_WINDOW=1), and the
    CVaR at alpha 0.5 / 0.9, every element within 1e-4."""
    if no_window:
        monkeypatch.setenv("B200MPPI_NO_WINDOW", "1")            # read when the planner handle is created
    d = point(golden_dir, name)
    M = d["lin"].shape[0]
    N = d["noise"].shape[0]
    for alpha in (0.5, 0.9):
        rp = _planner(eng, d, 0, M)
        try:
            rp.set_params(**_point_params(d, gname, cvar_alpha=alpha))
            rp.call("rollout")
            cnm = rp.copy_out(eng._lib.BUF_COSTS_NM, (N, M))
            r = rel1(cnm, d["sto_cnm_" + gname])
            assert r.max() < 1e-4, (np.unravel_index(r.argmax(), r.shape), r.max())
            cv = rp.copy_out(eng._lib.BUF_COSTS, (N,))
            assert rel1(cv, d["sto_cvar%02d_%s" % (int(alpha * 10), gname)]).max() < 1e-4
        finally:
            rp.close()


@pytest.mark.parametrize("name", POINTS)
@pytest.mark.parametrize("gname", ["near", "far"])
def test_det_and_speed_map_rollouts_vs_reference_at_param_point(eng, golden_dir, name, gname):
    d = point(golden_dir, name)
    N = d["noise"].shape[0]
    for mode, key in ((1, "det_"), (2, "spd_")):
        rp = _planner(eng, d, mode, 1)
        try:
            rp.set_params(**_point_params(d, gname))
            rp.call("rollout")
            c = rp.copy_out(eng._lib.BUF_COSTS, (N,))
            assert rel1(c, d[key + gname]).max() < 1e-4, key
        finally:
            rp.close()


@pytest.mark.parametrize("name", POINTS)
def test_update_vs_reference_at_param_point(eng, golden_dir, name):
    """The point's lambda and clip ranges; slabs of penalty-sized costs whose weights underflow."""
    d = point(golden_dir, name)
    N, T = d["upd_noise"].shape[:2]
    rp = RawPlanner(eng, 1, N, 1, T, 8, 8)
    try:
        rp.set_params(lambda_weight=float(d["lam"]), vrange=list(d["vrange"]), wrange=list(d["wrange"]))
        rp.copy_in(eng._lib.BUF_NOISE, d["upd_noise"])
        rp.copy_in(eng._lib.BUF_U_CUR, d["upd_u0"])
        c = np.ascontiguousarray(d["upd_costs"])
        rp.call("update", eng._lib.ptr(c))
        u = rp.copy_out(eng._lib.BUF_U_CUR, (T, 2))
        w = rp.copy_out(eng._lib.BUF_WEIGHTS, (N,))
        assert rel1(u, d["upd_u"]).max() < 1e-4
        assert rel1(w, d["upd_w"]).max() < 1e-4
        np.testing.assert_allclose(w, d["upd_w"], rtol=1e-4, atol=1e-9)
        assert (w[64:160] == 0).all()
    finally:
        rp.close()


# ----------------------------------------------------------------------------- whole solve through the public API
@pytest.mark.parametrize("mode", ["tdm", "det", "spd"])
def test_solve_sequence_vs_reference_at_p1(eng, golden_dir, mode):
    """Config -> TDM setters -> setup -> solve -> get_state_rollout -> shift_and_update -> solve at P1's lambda, dt,
    u_std, ranges, dist_weight, penalties, goal tolerance, v_post, cvar_alpha and alpha_dyn != 1, all passed through
    the params dict, against the reference's run of the same sequence."""
    g = load_all(golden_dir)
    d = point(golden_dir, "p1")
    S = {k[6:]: g[k] for k in g.files if k.startswith("solve_")}
    flags = dict(tdm=dict(use_tdm=True), det=dict(use_det_dynamics=True),
                 spd=dict(use_nom_dynamics_with_speed_map=True))[mode]
    cfg = eng.Config(T=float(S["T_s"]), dt=float(d["dt"]), num_grid_samples=int(S["M"]), num_control_rollouts=int(S["N"]),
                     seed=int(S["seed"]), max_map_dim=tuple(int(v) for v in S["max_map_dim"]),
                     tdm_sample_thread_dim=tuple(int(v) for v in S["thread_dim"]),
                     max_speed_padding=float(S["max_speed_padding"]), num_vis_state_rollouts=5, **flags)
    H, W = S["obstacle"].shape
    res = float(S["res"])
    lin, ang = eng.TDM_Numba(cfg), eng.TDM_Numba(cfg)
    for t_, which in ((lin, "lin"), (ang, "ang")):
        dd = dict(res=res, xlimits=np.array([0.0, W * res]), ylimits=np.array([0.0, H * res]),
                  bin_values=S[which + "_bin_values"], bin_values_bounds=S[which + "_bounds"],
                  det_dynamics_cvar_alpha=float(S["det_alpha"]))
        t_.set_TDM_from_PMF_grid(S["pmf_" + which], dd, S["obstacle"], S["unknown"])
    pl = eng.MPPI_Numba(cfg)
    p = dict(dt=float(d["dt"]), x0=np.array(S["x0"], float), xgoal=np.array(S["xgoal"], float),
             goal_tolerance=float(d["goal_tol"]), v_post_rollout=float(d["v_post"]), cvar_alpha=float(S["cvar_alpha"]),
             alpha_dyn=float(S["alpha_dyn"]), dist_weight=float(d["dist_weight"]), lambda_weight=float(d["lam"]),
             num_opt=1, u_std=np.array(d["u_std"]), vrange=np.array(d["vrange"]), wrange=np.array(d["wrange"]),
             obs_penalty=float(d["obs_cost"]), unknown_penalty=float(d["unk_cost"]))
    pl.setup(p, lin, ang)
    u1 = pl.solve()
    assert (lin.sample_grid_batch_d.copy_to_host() == S[mode + "_lin_grid1"]).all()
    assert (ang.sample_grid_batch_d.copy_to_host() == S[mode + "_ang_grid1"]).all()
    np.testing.assert_allclose(pl.noise_samples_d.copy_to_host(), S[mode + "_noise1"], rtol=3e-6, atol=2e-6)
    np.testing.assert_allclose(u1, S[mode + "_u1"], rtol=1e-3, atol=2e-4)
    st = pl.get_state_rollout()
    assert st.shape == S[mode + "_states1"].shape
    np.testing.assert_allclose(st, S[mode + "_states1"], rtol=2e-3, atol=2e-3)
    pl.shift_and_update(np.array(S["x0_next"], float), S[mode + "_u1"], num_shifts=1)
    u2 = pl.solve()
    np.testing.assert_allclose(u2, S[mode + "_u2"], rtol=2e-3, atol=5e-4)
    w = pl.weights_d.copy_to_host()
    assert abs(float(w.sum()) - 1.0) < 1e-5


# ----------------------------------------------------------------------------- windowed vs generic at scale
def _scale_params(d):
    return dict(lambda_weight=float(d["lam"]), u_std=np.array(d["u_std"]), vrange=np.array(d["vrange"]),
                wrange=np.array(d["wrange"]), dist_weight=float(d["dist_weight"]), goal_tolerance=float(d["goal_tol"]),
                v_post_rollout=float(d["v_post"]), obs_penalty=float(d["obs_cost"]), unknown_penalty=float(d["unk_cost"]))


def _set_pmf_any_bounds(tdm, pmf_grid, tdm_dict, obstacle, unknown):
    """set_TDM_from_PMF_grid for the sampled-map mode without its lo == 0 assertion (kept from the reference's setter):
    the engine itself decodes any traction bounds."""
    tdm.num_pmf_bins = pmf_grid.shape[0]
    tdm.res = tdm_dict["res"]
    tdm.cell_dimensions = (tdm.res, tdm.res)
    tdm.xlimits, tdm.ylimits = tdm_dict["xlimits"], tdm_dict["ylimits"]
    tdm.bin_values = np.asarray(tdm_dict["bin_values"]).astype(np.float32)
    tdm.bin_values_bounds = np.asarray(tdm_dict["bin_values_bounds"]).astype(np.float32)
    tdm.pmf_grid = np.asarray(pmf_grid).astype(np.int8)
    tdm._upload(tdm.res, tdm.xlimits, tdm.ylimits, obstacle, unknown, None)
    tdm.pmf_grid_initialized = True


@pytest.mark.parametrize("name", POINTS)
@pytest.mark.parametrize("maskmax", [1, 3])
def test_window_kernel_equals_generic_kernel_at_param_point(eng, golden_dir, monkeypatch, name, maskmax):
    """test_window_kernel_equals_generic_kernel's scenario (res 0.05 m, T = 128, rollouts leave the staged window) at
    the point's traction bounds (lo != 0) and planner parameters: MASK01 (maskmax 1) and the general penalty variant."""
    d = point(golden_dir, name)
    lb = [float(v) for v in d["lin_bounds"]]
    sc = make_scenario("tdm", N=512, M=16, T=128, H=900, W=900, res=0.05, B=12, seed=8, warm_start=True,
                       bin_bounds=lb, dt=float(d["dt"]), params=_scale_params(d))
    if maskmax > 1:
        rng = np.random.default_rng(3)
        sc["obstacle"] = (sc["obstacle"].astype(np.int64) * rng.integers(1, maskmax + 1, sc["obstacle"].shape)).astype(np.int8)
        assert sc["obstacle"].max() > 1
    L = eng._lib
    outs = []
    for no_win in (False, True):
        if no_win:
            monkeypatch.setenv("B200MPPI_NO_WINDOW", "1")
        cfg = eng.Config(**sc["cfg"])
        lin, ang = eng.TDM_Numba(cfg), eng.TDM_Numba(cfg)
        _set_pmf_any_bounds(lin, sc["pmf_lin"], sc["tdm_dict"], sc["obstacle"], sc["unknown"])
        _set_pmf_any_bounds(ang, sc["pmf_ang"], sc["tdm_dict"], sc["obstacle"], sc["unknown"])
        pl = eng.MPPI_Numba(cfg)
        pl.setup(sc["params"], lin, ang)
        pl.u_cur_d.copy_to_device(sc["u0"])
        pl.move_mppi_task_vars_to_device()
        lin.sample_grids(1.0)
        ang.sample_grids(1.0)
        assert lin.sample_grid_batch_d.copy_to_host().min() == 0           # the lowest bin decodes to lo != 0
        L.check(L.lib.b200mppi_planner_sample_noise(pl._handle))
        L.check(L.lib.b200mppi_planner_rollout(pl._handle))
        outs.append(pl.costs_nm_d.copy_to_host())
    monkeypatch.delenv("B200MPPI_NO_WINDOW")
    r = rel1(outs[0], outs[1])
    assert r.max() < 2e-6, r.max()


# ----------------------------------------------------------------------------- reach box: traction > 1, negative speeds
def _reach_scenario(vrange, v_warm, seed):
    """tdm scenario with traction bins over [-0.3, 1.8] (mostly high traction) and a warm start whose speeds hold
    negative values; small heading noise, so that rollouts travel far."""
    B = 8
    sc = make_scenario("tdm", N=512, M=32, T=32, H=420, W=420, res=0.1, B=B, seed=seed, warm_start=True,
                       thread_dim=(7, 5), bin_bounds=(-0.3, 1.8),
                       params=dict(vrange=np.array(vrange), wrange=np.array([-0.5, 0.8]), u_std=np.array([1.0, 0.3]),
                                   lambda_weight=0.6))
    rng = np.random.default_rng(seed + 10)
    pmf = np.zeros_like(sc["pmf_lin"])
    pmf[0] = 10                                                           # traction -0.3: some rollouts move backwards
    pmf[B - 2] = rng.integers(0, 40, pmf.shape[1:])
    pmf[B - 1] = 90 - pmf[B - 2]
    sc["pmf_lin"] = pmf.astype(np.int8)
    sc["u0"][:, 0] = v_warm
    sc["u0"][5:9, 0] = vrange[0] * 0.8                                    # negative speeds in the warm start
    sc["u0"][:, 1] *= 0.3
    return sc


def _reach_planner(eng, sc, monkeypatch, box):
    monkeypatch.setenv("B200MPPI_SAMPLE_BOX", box)
    cfg = eng.Config(**sc["cfg"])
    lin, ang = eng.TDM_Numba(cfg), eng.TDM_Numba(cfg)
    _set_pmf_any_bounds(lin, sc["pmf_lin"], sc["tdm_dict"], sc["obstacle"], sc["unknown"])
    _set_pmf_any_bounds(ang, sc["pmf_ang"], sc["tdm_dict"], sc["obstacle"], sc["unknown"])
    pl = eng.MPPI_Numba(cfg)
    pl.setup(sc["params"], lin, ang)
    pl.u_cur_d.copy_to_device(sc["u0"])
    return lin, ang, pl


def _closed_loop(eng, sc, monkeypatch, boxes):
    runs = {}
    for box in boxes:
        lin, ang, pl = _reach_planner(eng, sc, monkeypatch, box)
        x0 = sc["params"]["x0"].copy()
        hist, modes, first = [], [], None
        for k in range(4):
            u = pl.solve()
            modes.append(pl.sample_box())
            hist.append((u.copy(), pl.costs_d.copy_to_host(), pl.costs_nm_d.copy_to_host()))
            if k == 0:
                first = (pl.noise_samples_d.copy_to_host(), lin.sample_grid_batch_d.copy_to_host(),
                         ang.sample_grid_batch_d.copy_to_host(), lin, pl)
            x0 = x0 + np.array([0.37, -0.21, 0.05])
            pl.shift_and_update(x0, u, 1)
        runs[box] = dict(hist=hist, modes=modes, first=first, lin_rng=lin.rng_states_d.copy_to_host(),
                         ang_rng=ang.rng_states_d.copy_to_host(), rng=pl.rng_states_d.copy_to_host(),
                         noise=pl.noise_samples_d.copy_to_host(), lin_grid=lin.sample_grid_batch_d.copy_to_host(),
                         ang_grid=ang.sample_grid_batch_d.copy_to_host())
    ref = runs[boxes[0]]
    for box in boxes[1:]:
        r = runs[box]
        for k, ((u, c, cnm), (u0, c0, cnm0)) in enumerate(zip(r["hist"], ref["hist"])):
            assert (cnm == cnm0).all(), (box, k)
            assert (c == c0).all(), (box, k)
            assert (u == u0).all(), (box, k)
        for key in ("lin_rng", "ang_rng", "rng", "noise", "lin_grid", "ang_grid"):
            assert (r[key] == ref[key]).all(), (box, key)
    return runs


def _first_solve_states(sc, first):
    """The oracle's trajectories of the first solve (its noise, its whole sampled maps, the warm start)."""
    noise, gl, ga, lin, _ = first
    p = sc["params"]
    _, st = MR.rollout_costs(MR.MODE_STOCHASTIC, gl, ga, lin.bin_values_bounds, lin.bin_values_bounds,
                             lin.obstacle_map_d.copy_to_host(), lin.unknown_map_d.copy_to_host(), np.float32(lin.res),
                             lin.padded_xlimits.astype(np.float32), lin.padded_ylimits.astype(np.float32), p["vrange"],
                             p["wrange"], p["xgoal"], p["v_post_rollout"], 1e5, 1e2, p["goal_tolerance"],
                             p["lambda_weight"], p["u_std"], p["x0"], p["dt"], p["dist_weight"], noise, sc["u0"],
                             return_states=True)
    v = np.clip((sc["u0"][None, :, 0] + noise[:, :, 0]).astype(np.float32), np.float32(p["vrange"][0]),
                np.float32(p["vrange"][1]))
    return st, np.abs(v.astype(np.float64)).sum(1)


def test_boxed_solve_identical_to_whole_map_solve_with_traction_above_one(eng, monkeypatch):
    """Traction bins over [-0.3, 1.8], vrange [-1.5, 2.5], a warm start with negative speeds: off / static / dynamic
    box give bit-identical closed loops.  Not vacuous: some rollout of the first solve ends farther from x0 than
    dt * 1.0 * S (S = the largest sum_t |v| over the drawn controls), so a box that ignored the traction bound would be
    too small; and some rollout moves backwards."""
    sc = _reach_scenario([-1.5, 2.5], 2.2, seed=11)
    runs = _closed_loop(eng, sc, monkeypatch, ("off", "static", "dynamic"))
    assert all(m[0] == 0 for m in runs["off"]["modes"])
    assert runs["static"]["modes"][0][0] == 1, runs["static"]["modes"]
    assert all(m[0] == 2 for m in runs["dynamic"]["modes"]), runs["dynamic"]["modes"]
    st, vsum = _first_solve_states(sc, runs["off"]["first"])
    p = sc["params"]
    x0 = np.asarray(p["x0"][:2], np.float64)
    dist = np.sqrt(((st[:, :, -1, :2].astype(np.float64) - x0) ** 2).sum(-1))
    assert dist.max() > p["dt"] * 1.0 * vsum.max(), (dist.max(), p["dt"] * vsum.max())
    step = np.diff(st[..., :2].astype(np.float64), axis=2)
    heading = st[:, :, :-1, 2].astype(np.float64)
    along = step[..., 0] * np.cos(heading) + step[..., 1] * np.sin(heading)
    assert (along < -1e-3).any()


def test_static_box_uses_the_larger_speed_bound(eng, monkeypatch):
    """|vrange[0]| > vrange[1], speeds mostly negative: the static box must be sized by max(|vrange[0]|, |vrange[1]|)
    and the dynamic one by sum_t |v|; off / static / dynamic give bit-identical closed loops.  Some rollout ends
    farther from x0 than dt * max|traction| * T * vrange[1], so a box sized by vrange[1] would be too small."""
    sc = _reach_scenario([-2.5, 0.6], -2.0, seed=12)
    runs = _closed_loop(eng, sc, monkeypatch, ("off", "static", "dynamic"))
    assert runs["static"]["modes"][0][0] == 1, runs["static"]["modes"]
    assert all(m[0] == 2 for m in runs["dynamic"]["modes"]), runs["dynamic"]["modes"]     # sum_t |v| of backward runs
    st, _ = _first_solve_states(sc, runs["off"]["first"])
    p = sc["params"]
    x0 = np.asarray(p["x0"][:2], np.float64)
    dist = np.sqrt(((st[:, :, -1, :2].astype(np.float64) - x0) ** 2).sum(-1))
    assert dist.max() > p["dt"] * 1.8 * sc["T"] * p["vrange"][1]
