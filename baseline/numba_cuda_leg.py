#!/usr/bin/env python
"""The reference's own GPU path (mit-acl/mppi_numba, Numba-CUDA) timed on this box's GPU -- the
`numba_cuda_baseline` leg of bench.py (BASELINE.md section 3, row 1; north_star: "next to the reference's
Numba-CUDA path on 1 GPU ... in the same run").

Runs in its OWN process (bench.py spawns it before it touches CUDA itself) so that numba's CUDA context, its JIT
cache and the reference's import-time GPU query never share a process with the engine.  The reference is used
UNMODIFIED through its public API, imported from a checkout placed at baseline/_ref/ (git-ignored); nothing of it
is part of the repository.  One shim: ``np.float = float`` (mppi_numba/mppi.py:32-33 uses the alias numpy removed).

    python baseline/numba_cuda_leg.py c5 [c3 c2 c4]      ->  ONE JSON line on stdout

Per workload (bench.py WORKLOADS, same seeded scenario as the engine's arm):
  ms_per_solve : median wall time of the stock MPPI_Numba.solve() (it ends in a blocking D2H), >= 10 calls after
                 the JIT warm-up calls;  value = N*M*T / that
  kernels      : the body of solve_stochastic / solve_det_dyn (mppi.py:378-451, 308-375) replayed kernel by kernel
                 with cuda.synchronize() brackets: sample_grids x2, sample_noise, rollout, update (median of 5)
If the reference (or numba, or a GPU) is missing the line is {"unavailable": "<why>"} and the exit code 0.
"""
import contextlib
import json
import os
import sys
import time

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)


def locate():
    cand = os.path.join(HERE, "_ref")
    return cand if os.path.isdir(os.path.join(cand, "mppi_numba")) else None


def main():
    real_stdout = os.dup(1)
    os.dup2(2, 1)                                   # the reference prints; keep stdout for the one JSON line

    def emit(obj):
        os.write(real_stdout, (json.dumps(obj) + "\n").encode())
    ref_root = locate()
    if ref_root is None:
        return emit({"unavailable": "reference package not found (baseline/_ref)"})
    try:
        import numpy as np
        np.float = float
        sys.path.insert(0, ref_root)
        sys.path.insert(0, ROOT)
        from numba import cuda
        if not cuda.is_available():
            return emit({"unavailable": "numba finds no CUDA device"})
        from mppi_numba.config import Config as RConfig
        from mppi_numba.terrain import TDM_Numba as RTDM
        from mppi_numba.mppi import MPPI_Numba as RMPPI
    except Exception as e:                          # noqa: BLE001
        return emit({"unavailable": "reference import failed: %r" % (e,)})
    from bench import WORKLOADS, build_scenario
    names = [a for a in sys.argv[1:] if a in WORKLOADS] or ["c5"]
    out = {"impl": "reference Numba-CUDA (unmodified, %s)" % ref_root,
           "numba_compute_capability": list(cuda.get_current_device().compute_capability), "workloads": {}}
    med = lambda xs: float(np.median(xs))
    for name in names:
        sc = build_scenario(name)
        p = sc["params"]
        with contextlib.redirect_stdout(sys.stderr):
            rcfg = RConfig(**sc["cfg"])
            rl, ra = RTDM(rcfg), RTDM(rcfg)
            rl.set_TDM_from_PMF_grid(sc["pmf_lin"], sc["tdm_dict"], sc["obstacle"], sc["unknown"])
            ra.set_TDM_from_PMF_grid(sc["pmf_ang"], sc["tdm_dict"], sc["obstacle"], sc["unknown"])
            rp = RMPPI(rcfg)
            rp.setup(p, rl, ra)
            N, M, T = sc["N"], (sc["M"] if sc["mode"] == "tdm" else 1), sc["T"]
            t0 = time.perf_counter()
            for _ in range(3):
                rp.solve()                          # JIT + warm-up
            jit_s = time.perf_counter() - t0
            ts = []
            for _ in range(12):
                cuda.synchronize()
                t0 = time.perf_counter()
                rp.solve()
                ts.append(time.perf_counter() - t0)
            # kernel by kernel (the reference's own launch configurations)
            (res_d, xl_d, yl_d, vr_d, wr_d, xg_d, vpost_d, tol_d, lam_d, ustd_d, cvar_d, x0_d, dt_d, obs_c, unk_c) = \
                rp.move_mppi_task_vars_to_device()
            k = {"sample_grids_x2": [], "sample_noise": [], "rollout": [], "update": []}

            def timed(key, fn):
                cuda.synchronize()
                t0 = time.perf_counter()
                r = fn()
                cuda.synchronize()
                k[key].append(1e3 * (time.perf_counter() - t0))
                return r
            for _ in range(5):
                lin_g, ang_g = timed("sample_grids_x2", lambda: (rl.sample_grids(1.0), ra.sample_grids(1.0)))
                timed("sample_noise", lambda: RMPPI.sample_noise_numba[N, T](rp.rng_states_d, ustd_d, rp.noise_samples_d))
                if sc["mode"] == "tdm":
                    timed("rollout", lambda: RMPPI.rollout_numba[N, M, 0, 4 * M](
                        lin_g, ang_g, rl.bin_values_bounds_d, ra.bin_values_bounds_d, rl.obstacle_map_d,
                        rl.unknown_map_d, res_d, xl_d, yl_d, vr_d, wr_d, xg_d, vpost_d, obs_c, unk_c, tol_d, lam_d,
                        ustd_d, cvar_d, x0_d, dt_d, 1.0, rp.noise_samples_d, rp.u_cur_d, rp.costs_d))
                else:
                    timed("rollout", lambda: RMPPI.rollout_det_dyn_numba[N, 1](
                        lin_g, ang_g, rl.bin_values_bounds_d, ra.bin_values_bounds_d, rl.obstacle_map_d,
                        rl.unknown_map_d, res_d, xl_d, yl_d, vr_d, wr_d, xg_d, vpost_d, obs_c, unk_c, tol_d, lam_d,
                        ustd_d, x0_d, dt_d, 1.0, rp.noise_samples_d, rp.u_cur_d, rp.costs_d))
                timed("update", lambda: RMPPI.update_useq_numba[1, 32](
                    lam_d, rp.costs_d, rp.noise_samples_d, rp.weights_d, vr_d, wr_d, rp.u_cur_d))
        out["workloads"][name] = {"N": N, "M": M, "T": T, "ms_per_solve": 1e3 * med(ts), "solves_timed": len(ts),
                                  "value": N * M * T / med(ts), "unit": "state-steps/s",
                                  "jit_and_warmup_s": jit_s, "kernels_ms": {kk: med(v) for kk, v in k.items()}}
        del rp, rl, ra
    emit(out)


if __name__ == "__main__":
    main()
