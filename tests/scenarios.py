"""Seeded synthetic scenarios shared by the GPU parity tests, smoke() and bench.py
(SURVEY.md 8(d): random PMFs summing to 100, Bernoulli(0.01) masks, goal out of reach unless
``near_goal``)."""
import numpy as np


def random_pmf(rng, B, H, W):
    if B == 2:                                   # "nominal" 2-bin grid: all mass on traction 1.0
        pmf = np.zeros((2, H, W), dtype=np.int8)
        pmf[1] = 100
        return pmf
    cuts = np.sort(rng.integers(0, 101, (B - 1, H, W)), axis=0)
    pmf = np.empty((B, H, W), dtype=np.int64)
    pmf[0] = cuts[0]
    pmf[1:B - 1] = cuts[1:] - cuts[:-1]
    pmf[B - 1] = 100 - cuts[B - 2]
    return pmf.astype(np.int8)


def make_scenario(mode, N, M, T, H, W, res, B, seed=1, near_goal=False, warm_start=False,
                  det_alpha=1.0, cvar_alpha=0.5, pad_speed=5.0, thread_dim=(16, 16), bin_values=None,
                  mask_p=0.01, bin_bounds=(0.0, 1.0), dt=0.1, params=None):
    """``bin_values`` / ``bin_bounds``: the traction bins and bounds of both maps (default: B values evenly over
    [0, 1]); ``params``: entries that replace or extend the planner's params dict (``dt`` is set here, because the
    horizon and the map padding depend on it)."""
    overrides = dict(params or {})
    pad = int(np.ceil(pad_speed * dt / res))
    flags = dict(tdm=dict(use_tdm=True), det=dict(use_det_dynamics=True),
                 spd=dict(use_nom_dynamics_with_speed_map=True))[mode]
    cfg = dict(T=T * dt + dt / 2, dt=dt, num_grid_samples=M, num_control_rollouts=N, seed=seed,
               max_map_dim=(H + 2 * pad, W + 2 * pad), tdm_sample_thread_dim=thread_dim,
               max_speed_padding=pad_speed, num_vis_state_rollouts=min(8, M if mode == "tdm" else N), **flags)
    rng_l, rng_a = np.random.default_rng(seed), np.random.default_rng(seed + 1)
    pmf_lin, pmf_ang = random_pmf(rng_l, B, H, W), random_pmf(rng_a, B, H, W)
    obstacle = (np.random.default_rng(seed + 2).random((H, W)) < mask_p).astype(np.int8)
    unknown = (np.random.default_rng(seed + 3).random((H, W)) < mask_p).astype(np.int8)
    L = H * res
    r5 = np.random.default_rng(seed + 4)
    x0 = np.array([L / 2 + r5.uniform(-2, 2) * min(1.0, L / 20), L / 2 + r5.uniform(-2, 2) * min(1.0, L / 20),
                   r5.uniform(-np.pi, np.pi)])
    obstacle[int(x0[1] / res), int(x0[0] / res)] = 0
    xgoal = x0[:2] + (np.array([1.2, 1.2]) * min(1.0, L / 20) if near_goal else 0.42 * L * np.ones(2))
    if bin_values is None:
        bin_values = np.linspace(bin_bounds[0], bin_bounds[1], B)
    tdm_dict = dict(res=res, xlimits=np.array([0.0, W * res]), ylimits=np.array([0.0, H * res]),
                    bin_values=np.asarray(bin_values), bin_values_bounds=np.array(bin_bounds, dtype=float),
                    det_dynamics_cvar_alpha=det_alpha)
    params = dict(dt=dt, x0=x0, xgoal=xgoal, goal_tolerance=0.5, v_post_rollout=0.01, cvar_alpha=cvar_alpha,
                  alpha_dyn=1.0, dist_weight=1.0, lambda_weight=1.0, num_opt=1, u_std=np.array([2.0, 3.0]),
                  vrange=np.array([0.0, 3.0]), wrange=np.array([-np.pi, np.pi]))
    params.update(overrides)
    sc = dict(mode=mode, cfg=cfg, pmf_lin=pmf_lin, pmf_ang=pmf_ang, obstacle=obstacle, unknown=unknown,
              tdm_dict=tdm_dict, params=params, N=N, M=M, T=T)
    if warm_start:
        r6 = np.random.default_rng(seed + 5)
        sc["u0"] = np.stack([r6.uniform(0, 2, T), r6.uniform(-1, 1, T)], 1).astype(np.float32)
    return sc


def oracle_rollout_costs(sc, lin, ang, noise, u_cur, grids=None):
    """Oracle per-(n,m) costs for a scenario given the engine's TDM objects (for geometry / padded masks)."""
    from oracle import mppi_ref as MR
    p = sc["params"]
    mode = dict(tdm=MR.MODE_STOCHASTIC, det=MR.MODE_DET_DYN, spd=MR.MODE_SPEED_MAP)[sc["mode"]]
    gl = lin.sample_grid_batch_d.copy_to_host() if grids is None else grids[0]
    ga = ang.sample_grid_batch_d.copy_to_host() if grids is None else grids[1]
    risk = lin.risk_traction_map_d.copy_to_host() if sc["mode"] == "spd" else None
    return MR.rollout_costs(
        mode, gl, ga, lin.bin_values_bounds, ang.bin_values_bounds, lin.obstacle_map_d.copy_to_host(),
        lin.unknown_map_d.copy_to_host(), np.float32(lin.res), lin.padded_xlimits.astype(np.float32),
        lin.padded_ylimits.astype(np.float32), p["vrange"], p["wrange"], p["xgoal"], p["v_post_rollout"],
        p.get("obs_penalty", 1e5), p.get("unknown_penalty", 1e2), p["goal_tolerance"], p["lambda_weight"],
        p["u_std"], p["x0"], p["dt"], p.get("dist_weight", 1.0), noise, u_cur, risk_map=risk)
