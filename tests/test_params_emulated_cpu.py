"""Rollout, control-cost, CVaR and update arithmetic at planner parameters away from the defaults
(tests/golden/ref_params.npz, produced by the reference's own kernels under Numba's simulator, oracle/make_golden.py
--only-params).  At the default parameters (lambda 1, traction bounds [0, 1], vrange [0, 3], a symmetric wrange,
dist_weight 1, the default penalties) several wrong formulas give the right numbers; the two points here break those
ties: the oracle and the real kernel source (executed on the host by the tests/emu_*.py harnesses) must follow the
reference there too.  A sensitivity check keeps the points meaningful: with any one parameter set back to its
degenerate value the oracle misses the golden data by far more than the tolerance.

Costs cross zero at these points: the control cost is negative for some rollouts and can cancel most of the running
and terminal cost.  Relative errors are therefore taken against max(|ref|, 1) and, for rollout costs, against the size
of the two terms that were added (``scale``): a float32 sum of two terms of size 100 that nearly cancel carries their
rounding error, 100 * 2^-24, whatever its own size."""
import ctypes as C
import os

import numpy as np
import pytest

from oracle import mppi_ref as MR
from oracle import xoroshiro as X
from tests.emu_cvar import build as build_cvar
from tests.emu_rollout import build as build_generic
from tests.emu_rollout_win import build as build_win
from tests.emu_update import build as build_update
from tests.test_rollout_emulated_cpu import _c, _fparams, _p, _ratios

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
F32 = np.float32
POINTS = ("p1", "p2")
GOALS = ("near", "far")


def point(name):
    """The inputs and reference outputs of one parameter point, keyed like ref_rollout.npz."""
    g = np.load(os.path.join(GOLDEN, "ref_params.npz"))
    return {k[len(name) + 1:]: g[k] for k in g.files if k.startswith(name + "_")}


def rel1(a, ref):
    return np.abs(np.asarray(a, np.float64) - ref) / np.maximum(np.abs(np.asarray(ref, np.float64)), 1.0)


def oracle_rollout(d, mode, goal, **over):
    """Oracle costs at the point ``d`` with entries of ``d`` replaced by ``over``; per-(n,m) for the stochastic mode,
    per-n otherwise."""
    q = dict(d, **over)
    maps = slice(None) if mode == MR.MODE_STOCHASTIC else slice(0, 1)
    c = MR.rollout_costs(mode, q["lin"][maps], q["ang"][maps], q["lin_bounds"], q["ang_bounds"], q["obs"], q["unk"],
                         q["res"], q["xlim"], q["ylim"], q["vrange"], q["wrange"], q["xgoal_" + goal], q["v_post"],
                         q["obs_cost"], q["unk_cost"], q["goal_tol"], q["lam"], q["u_std"], q["x0"], q["dt"],
                         q["dist_weight"], q["noise"], q["u_cur"], risk_map=q["risk"])
    return c if mode == MR.MODE_STOCHASTIC else c[:, 0]


def scale(d, mode, gname, ref):
    """max(|ref|, |cost without the control cost|, 1), elementwise."""
    return np.maximum(np.maximum(np.abs(np.asarray(ref, np.float64)), 1.0),
                      np.abs(oracle_rollout(d, mode, gname, lam=0.0).astype(np.float64)))


def rel_terms(a, ref, d, mode, gname):
    return np.abs(np.asarray(a, np.float64) - ref) / scale(d, mode, gname, ref)


def oracle_update(d, **over):
    q = dict(d, **over)
    return MR.update_useq(q["lam"], q["upd_costs"], q["upd_noise"], q["vrange"], q["wrange"], q["upd_u0"])


def rel_cvar(a, ref, cnm):
    """CVaR: a mean of terms of both signs, its error bounded relative to the mean of their magnitudes."""
    return np.abs(np.asarray(a, np.float64) - ref) / np.maximum(MR.cvar_reduce(np.abs(cnm), 1.0), 1.0)


def reach_exact(d):
    """max_n sum_t |clip(u_v + e_v)|: the bound the prepare kernels' reach statistic must not fall below."""
    v = np.clip((d["u_cur"][None, :, 0] + d["noise"][:, :, 0]).astype(F32), F32(d["vrange"][0]), F32(d["vrange"][1]))
    return np.abs(v.astype(np.float64)).sum(1).max()


# ----------------------------------------------------------------------------- the points are what they claim to be
@pytest.mark.parametrize("name", POINTS)
def test_points_break_the_default_ties(name):
    d = point(name)
    assert d["lam"] != 1 and d["dist_weight"] != 1 and d["lin_bounds"][0] != 0 and d["ang_bounds"][0] != 0
    assert d["lin_bounds"][1] - d["lin_bounds"][0] != 1 and d["wrange"][0] != -d["wrange"][1]
    assert (d["obs_cost"], d["unk_cost"]) != (1e5, 1e2)
    assert (d["sto_cnm_near"] < 0).any() and (d["sto_cnm_near"] > 1).any()                 # costs cross zero
    reached = rel1(d["sto_cnm_near"], d["sto_cnm_far"]) > 0.5
    assert reached.any()                                                                    # early exits
    pen = oracle_rollout(d, MR.MODE_STOCHASTIC, "far", obs=0 * d["obs"], unk=0 * d["unk"])
    assert (pen != d["sto_cnm_far"]).any()                                                  # mask cells are visited
    assert (d["upd_costs"] > d["upd_costs"].min() + 1e3).sum() >= 64                        # penalty-sized outliers
    if name == "p1":
        assert d["vrange"][0] < 0 < d["vrange"][1] and abs(d["vrange"][0]) != d["vrange"][1]
        assert d["obs"].max() > 1 and d["unk"].max() > 1                                    # general penalty variant
        assert d["lin"].min() < 0 and d["lin"].max() > 100 and d["ang"].min() < 0           # bytes outside 0..100
        assert ((d["u_cur"][None, :, 0] + d["noise"][:, :, 0]) < 0).any()                  # backwards commands
    else:
        assert d["vrange"][0] > 0 and d["obs_cost"] == 0


# ----------------------------------------------------------------------------- oracle vs reference
@pytest.mark.parametrize("name", POINTS)
@pytest.mark.parametrize("gname", GOALS)
def test_oracle_matches_reference_at_param_point(name, gname):
    d = point(name)
    cnm = oracle_rollout(d, MR.MODE_STOCHASTIC, gname)
    ref_cnm = d["sto_cnm_" + gname]
    assert rel_terms(cnm, ref_cnm, d, MR.MODE_STOCHASTIC, gname).max() < 2e-6
    for alpha in (0.5, 0.9):
        ref = d["sto_cvar%02d_%s" % (int(alpha * 10), gname)]
        assert rel1(MR.cvar_reduce(ref_cnm, alpha), ref).max() < 2e-6          # the reduction on the same inputs
        assert rel_cvar(MR.cvar_reduce(cnm, alpha), ref, ref_cnm).max() < 2e-6
    assert rel_terms(oracle_rollout(d, MR.MODE_DET_DYN, gname), d["det_" + gname], d, MR.MODE_DET_DYN, gname).max() < 2e-6
    assert rel_terms(oracle_rollout(d, MR.MODE_SPEED_MAP, gname), d["spd_" + gname], d, MR.MODE_SPEED_MAP,
                     gname).max() < 2e-6


@pytest.mark.parametrize("name", POINTS)
def test_oracle_update_matches_reference_at_param_point(name):
    d = point(name)
    u, w = oracle_update(d)
    np.testing.assert_allclose(w, d["upd_w"], rtol=2e-5, atol=1e-9)
    np.testing.assert_allclose(u, d["upd_u"], rtol=1e-5, atol=2e-6)
    assert (d["upd_w"][64:160] == 0).all()                       # the outliers' weights underflow


# ----------------------------------------------------------------------------- sensitivity of the points
def _mirror(r):
    return np.array([-r[1], r[1]])


SENSITIVITY = {
    "lambda = 1": dict(lam=1.0),
    "lin lo = 0": lambda d: dict(lin_bounds=d["lin_bounds"] - d["lin_bounds"][0]),
    "ang lo = 0": lambda d: dict(ang_bounds=d["ang_bounds"] - d["ang_bounds"][0]),
    "lin range = 1": lambda d: dict(lin_bounds=np.array([d["lin_bounds"][0], d["lin_bounds"][0] + 1])),
    "dist_weight = 1": dict(dist_weight=1.0),
    "wrange mirrored": lambda d: dict(wrange=_mirror(d["wrange"])),
    "wrange swapped": lambda d: dict(wrange=d["wrange"][::-1].copy()),
    "vrange from 0": lambda d: dict(vrange=np.array([0.0, d["vrange"][1]])),
    "u_std swapped": lambda d: dict(u_std=d["u_std"][::-1].copy()),
    "goal_tolerance 0.5": dict(goal_tol=0.5),
    "v_post 0.01": dict(v_post=0.01),
    "default penalties": dict(obs_cost=1e5, unk_cost=1e2),
    "obs_penalty ignored": dict(obs_cost=1e5),
    "unknown_penalty ignored": dict(unk_cost=1e2),
    "masks read as 0 / 1": lambda d: dict(obs=np.minimum(d["obs"], 1), unk=np.minimum(d["unk"], 1)),
    "bytes read unsigned": lambda d: dict(lin=d["lin"].view(np.uint8), ang=d["ang"].view(np.uint8)),
}


@pytest.mark.parametrize("variant", sorted(SENSITIVITY))
def test_degenerate_parameter_misses_the_golden(variant):
    """Each parameter set back to the value that hides it: the oracle's outputs (per-(n,m), deterministic and
    speed-map costs, the updated controls) then miss the golden by at least 100 times the 2e-6 tolerance."""
    worst = 0.0
    for name in POINTS:
        d = point(name)
        over = SENSITIVITY[variant]
        over = over(d) if callable(over) else over
        for gname in GOALS:
            for mode, key in ((MR.MODE_STOCHASTIC, "sto_cnm_"), (MR.MODE_DET_DYN, "det_"), (MR.MODE_SPEED_MAP, "spd_")):
                worst = max(worst, float(rel1(oracle_rollout(d, mode, gname, **over), d[key + gname]).max()))
        u, _ = oracle_update(d, **over)
        worst = max(worst, float(rel1(u, d["upd_u"]).max()))
    assert worst > 100 * 2e-6, (variant, worst)


def test_reach_statistic_needs_the_absolute_value():
    """At P1 the speed commands go negative: a reach statistic without |v| (max_n sum_t v) is far below the true
    bound max_n sum_t |v|."""
    d = point("p1")
    v = np.clip((d["u_cur"][None, :, 0] + d["noise"][:, :, 0]).astype(F32), F32(d["vrange"][0]), F32(d["vrange"][1]))
    signed = np.abs(v.astype(np.float64).sum(1)).max()
    assert reach_exact(d) > signed * (1 + 100 * 1e-5)


# ----------------------------------------------------------------------------- kernel source (host emulation)
@pytest.fixture(scope="module")
def emu(tmp_path_factory):
    d = str(tmp_path_factory.mktemp("emu_params"))
    return dict(win=build_win(d), gen=build_generic(d), cvar=build_cvar(d), upd=build_update(d))


def _kernel_inputs(d, gname):
    lin, ang = _c(d["lin"], np.int8), _c(d["ang"], np.int8)
    obs, unk, risk = _c(d["obs"], np.int8), _c(d["unk"], np.int8), _c(d["risk"][0], np.int8)
    noise, u_cur = _c(d["noise"], F32), _c(d["u_cur"], F32)
    f = _fparams(d["res"], d["xlim"][0], d["ylim"][0], d["dt"], d["x0"], d["xgoal_" + gname], d["goal_tol"], d["v_post"],
                 d["lam"], d["u_std"], d["vrange"], d["wrange"], d["obs_cost"], d["unk_cost"], d["dist_weight"],
                 d["lin_bounds"][0], d["ang_bounds"][0])
    return lin, ang, obs, unk, risk, noise, u_cur, f, _ratios(d["lin_bounds"], d["ang_bounds"])


@pytest.mark.parametrize("name", POINTS)
@pytest.mark.parametrize("gname", GOALS)
def test_generic_kernels_match_reference_at_param_point(emu, name, gname):
    d = point(name)
    lin, ang, obs, unk, risk, noise, u_cur, f, ratios = _kernel_inputs(d, gname)
    M, R, Cc = lin.shape
    Hp, Wp = obs.shape
    N, T = noise.shape[:2]

    def launch(mode, Mk):
        geo = _c([Hp, Wp, R, Cc, Cc, Wp, T, N, Mk], np.int32)
        cnm, costs = np.zeros((N, Mk), F32), np.zeros(N, F32)
        emu["gen"].emu_rollout(mode, _p(f), _p(geo), _p(ratios), _p(lin), _p(ang), _p(obs), _p(unk), _p(risk), _p(noise),
                               _p(u_cur), _p(cnm), _p(costs), None, 0)
        return cnm, costs
    cnm, _ = launch(0, M)
    assert rel_terms(cnm, d["sto_cnm_" + gname], d, MR.MODE_STOCHASTIC, gname).max() < 3e-6
    _, det = launch(1, 1)
    assert rel_terms(det, d["det_" + gname], d, MR.MODE_DET_DYN, gname).max() < 3e-6
    _, spd = launch(2, 1)
    assert rel_terms(spd, d["spd_" + gname], d, MR.MODE_SPEED_MAP, gname).max() < 3e-6


@pytest.mark.parametrize("name", POINTS)
@pytest.mark.parametrize("gname", GOALS)
def test_windowed_kernel_matches_reference_at_param_point(emu, name, gname):
    """prepare_rollout_kernel + the windowed kernel (the penalty variant the launcher picks for the point's masks),
    window around the robot and pushed away, against the reference and the generic kernel; the reach statistic."""
    d = point(name)
    lin, ang, obs, unk, risk, noise, u_cur, f, ratios = _kernel_inputs(d, gname)
    M, R, Cc = lin.shape
    Hp, Wp = obs.shape
    N, T = noise.shape[:2]
    geo = _c([Hp, Wp, R, Cc, Cc, Wp, T, N, M], np.int32)
    m01 = int(((obs & ~1) == 0).all() and ((unk & ~1) == 0).all())
    assert m01 == (0 if name == "p1" else 1)

    def run_win(sx, sy):
        out, origin, reach = np.zeros((N, M), F32), np.zeros(2, np.int32), np.zeros(1, F32)
        assert emu["win"].emu_rollout_win(_p(f), _p(geo), _p(ratios), _p(lin), _p(ang), _p(obs), _p(unk), _p(noise),
                                          _p(u_cur), _p(out), sx, sy, _p(origin), _p(reach), 0, 1, 0, 0, m01) == 0
        return out, reach[0]
    inside, reach = run_win(0, 0)
    ref = d["sto_cnm_" + gname]
    assert rel_terms(inside, ref, d, MR.MODE_STOCHASTIC, gname).max() < 5e-6
    shifted, _ = run_win(4000, -4000)
    assert (shifted == inside).all()
    cnm, costs = np.zeros((N, M), F32), np.zeros(N, F32)
    emu["gen"].emu_rollout(0, _p(f), _p(geo), _p(ratios), _p(lin), _p(ang), _p(obs), _p(unk), None, _p(noise), _p(u_cur),
                           _p(cnm), _p(costs), None, 0)
    assert rel_terms(inside, cnm, d, MR.MODE_STOCHASTIC, gname).max() < 2e-6
    vsum = reach_exact(d)
    assert vsum <= float(reach) <= vsum * (1 + 1e-5)


@pytest.mark.parametrize("name", POINTS)
def test_windowed_kernel_equals_generic_kernel_bit_for_bit_without_control_cost(emu, name):
    """With u_cur = 0 the control cost is exactly 0 in both kernels, and the two walk the same float sequence: the
    traction tables of the windowed kernel (lo + ratio * byte, times dt, in float64) and the generic kernel's per-step
    decode must agree to the last bit, for every byte the maps hold."""
    d = point(name)
    lin, ang, obs, unk, risk, noise, _, f, ratios = _kernel_inputs(d, "near")
    u_cur = np.zeros_like(d["u_cur"])
    M, R, Cc = lin.shape
    Hp, Wp = obs.shape
    N, T = noise.shape[:2]
    geo = _c([Hp, Wp, R, Cc, Cc, Wp, T, N, M], np.int32)
    m01 = int(((obs & ~1) == 0).all() and ((unk & ~1) == 0).all())
    out = np.zeros((N, M), F32)
    assert emu["win"].emu_rollout_win(_p(f), _p(geo), _p(ratios), _p(lin), _p(ang), _p(obs), _p(unk), _p(noise),
                                      _p(u_cur), _p(out), 0, 0, None, None, 0, 1, 0, 0, m01) == 0
    cnm, costs = np.zeros((N, M), F32), np.zeros(N, F32)
    emu["gen"].emu_rollout(0, _p(f), _p(geo), _p(ratios), _p(lin), _p(ang), _p(obs), _p(unk), None, _p(noise), _p(u_cur),
                           _p(cnm), _p(costs), None, 0)
    assert (out == cnm).all(), np.abs(out - cnm).max()
    want = oracle_rollout(d, MR.MODE_STOCHASTIC, "near", u_cur=u_cur)
    assert rel1(out, want).max() < 5e-6


@pytest.mark.parametrize("name", POINTS)
def test_noise_prepare_kernel_at_param_point(emu, name):
    """noise_prepare_kernel (what solve() launches; the harness also checks it against sample_noise + prepare_rollout
    bit for bit) at the point's u_std, lambda, vrange and wrange: clipped float64 controls, control costs
    sum_t lambda * (u_v/sv2 * e_v + u_w/sw2 * e_w) in the reference's order, and the reach statistic."""
    d = point(name)
    N, T = 37, 12
    rng = np.random.default_rng(7)
    u_cur = np.stack([rng.uniform(d["vrange"][0] - 0.5, d["vrange"][1], T),
                      rng.uniform(d["wrange"][0] - 0.5, d["wrange"][1] + 0.5, T)], 1).astype(F32)
    states = np.ascontiguousarray(X.create_states(N * T, 9))
    us, vr, wr = d["u_std"].astype(F32), _c(d["vrange"], F32), _c(d["wrange"], F32)
    npad = (N + 31) // 32 * 32
    st_out = np.zeros_like(states)
    noise, noiseT = np.zeros((N, T, 2), F32), np.zeros((T, npad, 2), np.float64)
    ctrl, reach = np.zeros(npad, F32), np.zeros(1, F32)
    rc = emu["win"].emu_noise_prepare(_p(states), _p(u_cur), N, T, us[0], us[1], F32(d["lam"]), _p(vr), _p(wr), _p(st_out),
                                      _p(noise), _p(noiseT), _p(ctrl), _p(reach))
    assert rc == 0, rc
    np.testing.assert_allclose(noise, MR.sample_noise(states.copy(), us, N, T), rtol=3e-6, atol=2e-6)
    v = np.clip((u_cur[None, :, 0] + noise[:, :, 0]).astype(F32), vr[0], vr[1])
    w = np.clip((u_cur[None, :, 1] + noise[:, :, 1]).astype(F32), wr[0], wr[1])
    assert (noiseT[:, :N, 0] == v.T.astype(np.float64)).all()
    assert (noiseT[:, :N, 1] == w.T.astype(np.float64)).all()
    assert (v < 0).any() == (name == "p1") and (w == wr[0]).any() and (w == wr[1]).any()     # both clip ends active
    # control cost: the oracle's epilogue on a zero running cost
    want = MR.rollout_costs(MR.MODE_DET_DYN, np.zeros((1, 4, 4), np.int8), np.zeros((1, 4, 4), np.int8), [0, 1], [0, 1],
                            np.zeros((4, 4), np.int8), np.zeros((4, 4), np.int8), 1.0, [0, 4], [0, 4], [0, 0], [0, 0],
                            [1, 1], 1e30, 0, 0, 0, d["lam"], us, [2, 2, 0], 0.0, 0.0, noise, u_cur)[:, 0]
    assert rel1(ctrl[:N], want).max() < 2e-6
    vs = np.abs(v.astype(np.float64)).sum(1).max()
    assert vs <= float(reach[0]) <= vs * (1 + 1e-5)


@pytest.mark.parametrize("name", POINTS)
@pytest.mark.parametrize("gname", GOALS)
def test_cvar_kernel_matches_reference_at_param_point(emu, name, gname):
    d = point(name)
    cnm = _c(d["sto_cnm_" + gname], F32)
    N, M = cnm.shape
    for alpha in (0.5, 0.9):
        out = np.zeros(N, F32)
        assert emu["cvar"].emu_cvar(_p(cnm), _p(out), N, M, N, F32(alpha)) == 0
        assert rel_cvar(out, d["sto_cvar%02d_%s" % (int(alpha * 10), gname)], cnm).max() < 2e-6


@pytest.mark.parametrize("name", POINTS)
def test_update_kernels_match_reference_at_param_point(emu, name):
    """The one-launch update (what solve() runs) and the partial + finish path at the point's lambda and clip ranges,
    with slabs of penalty-sized costs whose CTA scale exp(-(beta_cta - beta) / lambda) underflows to 0."""
    d = point(name)
    E = emu["upd"]
    costs, noise, u0 = (_c(d[k], F32) for k in ("upd_costs", "upd_noise", "upd_u0"))
    vr, wr = _c(d["vrange"], F32), _c(d["wrange"], F32)
    N, T = noise.shape[:2]
    lam = F32(d["lam"])
    ctas = E.emu_update_num_ctas(N)
    w_raw, parts, rank = np.zeros(N, F32), np.zeros((ctas, 2 * T + 2), F32), np.zeros(2 * T + 2, F32)
    u1, w1 = u0.copy(), np.zeros(N, F32)
    assert E.emu_update_one_rank(_p(costs), _p(noise), _p(w_raw), _p(parts), _p(rank), _p(u1), _p(w1), N, T, lam,
                                 _p(vr), _p(wr)) == 0
    np.testing.assert_allclose(u1, d["upd_u"], rtol=1e-5, atol=2e-6)
    np.testing.assert_allclose(w1, d["upd_w"], rtol=1e-4, atol=1e-12)
    scale = np.exp(-(parts[:, 0].astype(np.float64) - float(parts[:, 0].min())) / float(lam)).astype(F32)
    assert (scale == 0).sum() >= 2                                    # several CTAs contribute nothing
    u2, w2 = u0.copy(), np.zeros(N, F32)
    E.emu_update_partial(_p(costs), _p(noise), _p(w_raw), _p(parts), _p(rank), N, T, lam)
    E.emu_update_finish(_p(_c(rank[None, :], F32)), 1, _p(w_raw), _p(parts), _p(u2), _p(w2), N, T, lam, _p(vr), _p(wr))
    assert (u2 == u1).all() and (w2 == w1).all()
    assert (u1[:, 0] == vr[0]).any() or (u1[:, 0] == vr[1]).any() or (u1[:, 1] == wr[0]).any() or (u1[:, 1] == wr[1]).any()
