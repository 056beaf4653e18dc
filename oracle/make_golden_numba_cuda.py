"""Generate tests/golden/ref_numba_cuda.npz by running the reference's own Numba-CUDA kernels (unmodified)
on a GPU.  TEST INFRASTRUCTURE: the fixture of tests/test_gpu_vs_reference.py.

    python -m oracle.make_golden_numba_cuda --reference DIR [--out FILE]

DIR is a checkout of the reference (the directory holding its ``mppi_numba`` package); it needs a CUDA GPU and
numba.  For every case of the test the body of the reference's solve_* is replayed kernel by kernel on the test's
seeded scenario (sample both traction maps, sample the control noise, roll out, update), exactly as the test
replays it on the engine, and the file keeps per case:
  costs, u                the rollout costs and the control sequence the update makes of them, in full;
  pmf, lin, ang, noise    the host-preprocessed PMF grid, both sampled traction maps and the control noise:
                          shape, dtype and SHA-256 of the whole array, plus the values at a seeded sample of
                          positions -- the test's bit-identity checks stay whole while the file stays small.
"""
import argparse
import contextlib
import hashlib
import io
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
OUT = os.path.join(ROOT, "tests", "golden", "ref_numba_cuda.npz")

#        mode   N     M     T    H     res  B   det_alpha
CASES = [("tdm", 1024, 64, 64, 512, 0.1, 12, 1.0),        # BASELINE config 3
         ("det", 4096, 1, 128, 512, 0.2, 32, 0.3),        # BASELINE config 4
         ("tdm", 8192, 256, 128, 1024, 0.1, 12, 1.0),     # BASELINE config 5, the headline workload, full size
         ("tdm", 128, 1100, 32, 128, 0.1, 12, 1.0)]       # M > 1024: rollout_oversized_numba, cvar_alpha = 1
SAMPLES = 2048


def case_key(mode, N, M, T, H, res, B, det_alpha):
    return "%s_N%d_M%d_T%d_H%d_res%g_B%d_da%g" % (mode, N, M, T, H, res, B, det_alpha)


def case_scenario(mode, N, M, T, H, res, B, det_alpha):
    """The seeded scenario of one case, with the warm start and CVaR level the test uses."""
    from tests.scenarios import make_scenario
    return make_scenario(mode, N=N, M=M, T=T, H=H, W=H, res=res, B=B, seed=1, det_alpha=det_alpha, warm_start=True,
                         cvar_alpha=1.0 if M > 1024 else 0.5)


def digest(a):
    """SHA-256 of a C-contiguous array's bytes (shape and dtype are stored and compared on their own)."""
    return hashlib.sha256(np.ascontiguousarray(a).data).hexdigest()


def _quiet(fn, *a, **k):
    with contextlib.redirect_stdout(io.StringIO()):
        return fn(*a, **k)


def run_case(ref, case, rng):
    RConfig, RTDM, RMPPI, cuda = ref
    mode, N, M, T = case[:4]
    sc = case_scenario(*case)
    p = sc["params"]
    rcfg = _quiet(RConfig, **sc["cfg"])
    rl, ra = _quiet(RTDM, rcfg), _quiet(RTDM, rcfg)
    _quiet(rl.set_TDM_from_PMF_grid, sc["pmf_lin"], sc["tdm_dict"], sc["obstacle"], sc["unknown"])
    _quiet(ra.set_TDM_from_PMF_grid, sc["pmf_ang"], sc["tdm_dict"], sc["obstacle"], sc["unknown"])
    rp = _quiet(RMPPI, rcfg)
    _quiet(rp.setup, p, rl, ra)
    rp.u_cur_d = cuda.to_device(sc["u0"])
    pmf = rl.pmf_grid_d.copy_to_host()
    Hp, Wp = pmf.shape[1:]
    (res_d, xl_d, yl_d, vr_d, wr_d, xg_d, vpost_d, tol_d, lam_d, ustd_d, cvar_d, x0_d, dt_d, obs_c, unk_c) = \
        rp.move_mppi_task_vars_to_device()
    alpha_dyn = 0.9 if mode == "tdm" else 1.0
    lin_g, ang_g = rl.sample_grids(alpha_dyn), ra.sample_grids(alpha_dyn)
    RMPPI.sample_noise_numba[N, T](rp.rng_states_d, ustd_d, rp.noise_samples_d)
    if mode == "tdm":
        kern = RMPPI.rollout_numba[N, M, 0, 4 * M] if M <= 1024 else RMPPI.rollout_oversized_numba[N, 1024, 0, 4 * M]
        kern(
            lin_g, ang_g, rl.bin_values_bounds_d, ra.bin_values_bounds_d, rl.obstacle_map_d, rl.unknown_map_d, res_d,
            xl_d, yl_d, vr_d, wr_d, xg_d, vpost_d, obs_c, unk_c, tol_d, lam_d, ustd_d, cvar_d, x0_d, dt_d, 1.0,
            rp.noise_samples_d, rp.u_cur_d, rp.costs_d)
    else:
        RMPPI.rollout_det_dyn_numba[N, 1](
            lin_g, ang_g, rl.bin_values_bounds_d, ra.bin_values_bounds_d, rl.obstacle_map_d, rl.unknown_map_d, res_d,
            xl_d, yl_d, vr_d, wr_d, xg_d, vpost_d, obs_c, unk_c, tol_d, lam_d, ustd_d, x0_d, dt_d, 1.0,
            rp.noise_samples_d, rp.u_cur_d, rp.costs_d)
    cuda.synchronize()
    costs = rp.costs_d.copy_to_host().copy()       # before the update, which reuses costs_d as scratch
    RMPPI.update_useq_numba[1, 32](lam_d, rp.costs_d, rp.noise_samples_d, rp.weights_d, vr_d, wr_d, rp.u_cur_d)
    cuda.synchronize()
    out = {"costs": costs, "u": rp.u_cur_d.copy_to_host()}
    arrays = {"pmf": pmf, "lin": lin_g.copy_to_host()[:, :Hp, :Wp], "ang": ang_g.copy_to_host()[:, :Hp, :Wp],
              "noise": rp.noise_samples_d.copy_to_host()}
    for name, a in arrays.items():
        a = np.ascontiguousarray(a)
        idx = np.unique(rng.integers(0, a.size, SAMPLES)).astype(np.int64)
        out.update({name + "_shape": np.array(a.shape, np.int64), name + "_dtype": np.array(a.dtype.str),
                    name + "_sha256": np.array(digest(a)), name + "_idx": idx, name + "_val": a.reshape(-1)[idx]})
    del rp, rl, ra
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--reference", required=True, help="directory holding the reference's mppi_numba package")
    ap.add_argument("--out", default=OUT)
    args = ap.parse_args()
    if not os.path.isdir(os.path.join(args.reference, "mppi_numba")):
        raise SystemExit("no mppi_numba package under %s" % args.reference)
    np.float = float                      # the reference's mppi.py uses the alias numpy removed
    sys.path.insert(0, os.path.abspath(args.reference))
    if ROOT not in sys.path:
        sys.path.insert(0, ROOT)
    from numba import cuda
    if not cuda.is_available():
        raise SystemExit("numba finds no CUDA device")
    from mppi_numba.config import Config
    from mppi_numba.terrain import TDM_Numba
    from mppi_numba.mppi import MPPI_Numba
    ref = (Config, TDM_Numba, MPPI_Numba, cuda)
    rng = np.random.default_rng(2024)
    dev = cuda.get_current_device()
    name = dev.name.decode() if isinstance(dev.name, bytes) else str(dev.name)
    blob = {"device": np.array("%s, compute capability %d.%d" % ((name,) + tuple(dev.compute_capability)))}
    for case in CASES:
        key = case_key(*case)
        for name, v in run_case(ref, case, rng).items():
            blob[key + "__" + name] = v
        print("%s: done" % key, file=sys.stderr)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    np.savez_compressed(args.out, **blob)
    print("wrote %s (%d bytes)" % (args.out, os.path.getsize(args.out)))


if __name__ == "__main__":
    main()
