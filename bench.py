#!/usr/bin/env python
"""bench.py -- rollouts/s (N*M*T state-steps per solve / time) of the MPPI hot path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--workload c5|c3|c2|c4]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A "step" is one MPPI_Numba.solve() (num_opt = 1): control noise, both traction-distribution maps sampled (M maps
each), N x M x T rollouts with cost accumulation, CVaR over M, softmax update, D2H of the T x 2 control sequence.
Workload (BASELINE.json configs[4], the one the metric and the north-star target are quoted on; it fits one GPU):
CVaR-cost MPPI, N=8192, M=256, T=128, 1024x1024 PMF grid (12 bins, res 0.1 m) -- at N GPUs the 256 sampled maps
are sharded over the ranks ("strong" scaling): every rank rolls all 8192 control sequences out on its M/N maps,
the per-(n,m) costs are exchanged all-to-all and the 2T+2-float softmax partials all-gathered, by the library's
own peer-memory kernels over NVLink (B200MPPI_EXCHANGE=nccl: by two NCCL collectives).

`value`  : device-timed (CUDA events on the planner's stream), inputs resident in HBM.
`e2e`    : the same metric through the public Python API from HOST buffers -- every step does
           shift_and_update(x0, u) (H2D of the T x 2 warm start + the params POD) and solve()
           (D2H of the T x 2 result), wall-clock, max over ranks.
`roofline`: the dominant kernel's algorithmic bytes / its CUDA-event time vs the measured HBM peak, and -- because
           ncu shows both dominant kernels bound by instruction issue, not by HBM -- its warp instructions
           (ncu, profiles/) / its time vs the SM issue peak (148 SMs x 4 schedulers x the SM clock sampled here).
`parity_check` (N > 1): before the timed region the sharded solve is checked on the real GPUs against a 1-rank
           solve of the same scenario and seed run by rank 0: u identical on all ranks, u vs 1-rank within 1e-5,
           every rank's CVaR-cost slice bit-identical to the 1-rank costs.  A failure exits non-zero.
`numba_cuda_baseline` (N = 1): the UNMODIFIED reference (Numba-CUDA) timed on the same GPU in the same run, in a
           subprocess (baseline/numba_cuda_leg.py): its stock solve() and its kernels one by one.
`others` (N = 1): the remaining BASELINE configs (c2, c3, c4) through the same engine, device-timed and end to end.
`cpu_baseline`: the numpy oracle (oracle/mppi_ref.py) on a bounded N-slice, on this box's host cores.
--impl reference: times that CPU path alone (the reference has no CPU implementation of its own; its GPU path is
the numba_cuda_baseline leg above).
--dump-outputs DIR: after the device-timed steps, what the last of them returned is written as DIR/u.npy (the T x 2
           control sequence) and DIR/costs.npy (the N CVaR costs, all ranks' slices in order), float32.  The steps
           before the timed ones are fixed by the arguments (see run_b200), so two builds can be compared output for
           output.
The benchmark runs from the tree build() left and writes nothing into it (it may be read-only).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

sys.dont_write_bytecode = True          # no __pycache__ in the tree
ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

WORKLOADS = {
    #       mode   N     M    T    H     res  B   det_alpha
    "c5": ("tdm", 8192, 256, 128, 1024, 0.1, 12, 1.0),
    "c3": ("tdm", 1024, 64, 64, 512, 0.1, 12, 1.0),
    "c2": ("det", 1024, 1, 64, 256, 0.2, 2, 1.0),
    "c4": ("det", 4096, 1, 128, 512, 0.2, 32, 0.3),
}


def build_scenario(name):
    from tests.scenarios import make_scenario
    mode, N, M, T, H, res, B, da = WORKLOADS[name]
    return make_scenario(mode, N=N, M=M, T=T, H=H, W=H, res=res, B=B, seed=1, det_alpha=da)


# ----------------------------------------------------------------------------- CPU baseline (oracle port)
_CPU_SHARED = {}


def _cpu_chunk(args):
    n0, n1, seed = args
    sc, maps = _CPU_SHARED["sc"], _CPU_SHARED["maps"]       # inherited through fork, not pickled
    from oracle import mppi_ref as MR
    from oracle import xoroshiro as X
    p = sc["params"]
    T = sc["T"]
    rng = np.random.default_rng(seed + n0)
    noise = (rng.standard_normal((n1 - n0, T, 2)) * p["u_std"]).astype(np.float32)
    mode = dict(tdm=MR.MODE_STOCHASTIC, det=MR.MODE_DET_DYN, spd=MR.MODE_SPEED_MAP)[sc["mode"]]
    cnm = MR.rollout_costs(mode, maps["lin"], maps["ang"], [0, 1], [0, 1], maps["obs"], maps["unk"],
                           np.float32(maps["res"]), maps["pxl"], maps["pyl"], p["vrange"], p["wrange"], p["xgoal"],
                           p["v_post_rollout"], 1e5, 1e2, p["goal_tolerance"], p["lambda_weight"], p["u_std"],
                           p["x0"], p["dt"], 1.0, noise, np.zeros((T, 2), np.float32))
    cn = MR.cvar_reduce(cnm, p["cvar_alpha"]) if sc["mode"] == "tdm" else cnm[:, 0]
    return cn, noise


def cpu_baseline_maps(sc, m_cpu):
    """Sampled maps for the CPU baseline's rollouts: m_cpu iid maps drawn with numpy from the same PMF
    (statistically the workload's maps; drawing them is set-up, outside the timed region -- the GPU arm's timed
    region does include its map sampling, so the CPU arm does less work per state-step, not more)."""
    from oracle import terrain_ref as TR
    cfgd = sc["cfg"]
    d = sc["tdm_dict"]
    pl, pxl, pyl, pad = TR.set_padding(sc["pmf_lin"], cfgd["max_speed_padding"], cfgd["dt"], d["res"],
                                       d["xlimits"], d["ylimits"], cfgd["max_map_dim"])
    pa, _, _, _ = TR.set_padding(sc["pmf_ang"], cfgd["max_speed_padding"], cfgd["dt"], d["res"],
                                 d["xlimits"], d["ylimits"], cfgd["max_map_dim"])
    q = TR.quantise_bin_values(d["bin_values"], [0, 1])
    rng = np.random.default_rng(0)

    def draw(pmf):
        cum = np.cumsum(pmf.astype(np.int64), axis=0)
        out = np.empty((m_cpu,) + pmf.shape[1:], dtype=np.int8)
        for m in range(m_cpu):
            u = rng.integers(1, 101, pmf.shape[1:])
            out[m] = q[np.argmax(cum >= u[None], axis=0)]
        return out
    mmd = cfgd["max_map_dim"]
    obs = TR.set_padding_2d(sc["obstacle"], cfgd["max_speed_padding"], cfgd["dt"], d["res"], mmd)
    unk = TR.set_padding_2d(sc["unknown"], cfgd["max_speed_padding"], cfgd["dt"], d["res"], mmd)
    return dict(lin=draw(pl), ang=draw(pa), obs=obs, unk=unk, res=d["res"], pxl=pxl.astype(np.float32),
                pyl=pyl.astype(np.float32))


class CpuBaseline:
    """numpy oracle: rollouts + CVaR + update on an (n_sample x m_sample x T) slice of the workload, N-sharded over
    all host cores.  ONE pool of worker processes is forked (before CUDA is touched) and warmed with an untimed
    pass -- first-touch imports of `oracle`, page faults on the fork-shared maps -- then every timed pass runs on
    the same warm workers."""

    def __init__(self, sc, n_sample, m_sample):
        import multiprocessing as mp
        self.sc = sc
        cores = os.cpu_count() or 1
        sc2 = dict(sc)
        sc2["M"] = m_sample if sc["mode"] == "tdm" else 1
        self.m = sc2["M"]
        self.n = n_sample
        maps = cpu_baseline_maps(sc, sc2["M"])
        self.chunks = max(1, min(cores, n_sample // 8))
        b = [n_sample * i // self.chunks for i in range(self.chunks + 1)]
        self.jobs = [(b[i], b[i + 1], 99) for i in range(self.chunks)]
        _CPU_SHARED["sc"], _CPU_SHARED["maps"] = sc2, maps
        self.pool = mp.get_context("fork").Pool(self.chunks)
        self.steps = n_sample * sc2["M"] * sc["T"]
        self.desc = "numpy oracle, N-slice %d of %d x M-slice %d of %d x T %d (%d state-steps), %d warmed processes" % (
            n_sample, sc["N"], sc2["M"], sc["M"], sc["T"], self.steps, self.chunks)
        self.one_pass()                                  # warm-up, untimed

    def one_pass(self):
        from oracle import mppi_ref as MR
        t0 = time.perf_counter()
        res = self.pool.map(_cpu_chunk, self.jobs)
        cn = np.concatenate([r[0] for r in res])
        noise = np.concatenate([r[1] for r in res])
        p = self.sc["params"]
        MR.update_useq(p["lambda_weight"], cn, noise, p["vrange"], p["wrange"], np.zeros((self.sc["T"], 2), np.float32))
        return time.perf_counter() - t0

    def measure(self, passes):
        ts = [self.one_pass() for _ in range(max(1, passes))]
        return ts

    def close(self):
        self.pool.close()
        self.pool.join()


def cpu_sample_size(sc):
    return (min(sc["N"], 4096), min(sc["M"], 64)) if sc["mode"] == "tdm" else (min(sc["N"], 4096), 1)


# ----------------------------------------------------------------------------- clocks
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.lines, self.proc = [], None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._pump, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for nm, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def measured_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


# ----------------------------------------------------------------------------- algorithmic bytes (DESIGN.md)
def algorithmic_bytes(sc, cfg, n_local, m_local, box=None):
    """HBM bytes per solve and per kernel on ONE rank, each operand once.
    `total` follows SURVEY.md 8(d) / BASELINE.md 4 literally -- the bytes the REFERENCE's algorithm has to move
    (whole maps sampled every solve, a reach window of +-vmax*T*dt read by the rollouts): the denominator of the
    north-star "fraction of the HBM roofline".  The per-kernel entries are what THIS engine's kernels have to move:
    the rollout kernel stages a 240 x 232-cell window per map (csrc/rollout_win.cu), the sampler writes only the
    reach box of this solve when it is boxed (`box` = rows x cols of it; include/b200mppi.h)."""
    N, M, T = n_local, m_local, sc["T"]
    B = sc["pmf_lin"].shape[0]
    Hp, Wp = cfg.max_map_dim
    p = sc["params"]
    reach = int(np.ceil(p["vrange"][1] * T * p["dt"] / sc["tdm_dict"]["res"]))
    Hw = min(Hp, 2 * reach + 3)
    noise = 32 * N * T + 8 * N * T                             # RNG state R+W, noise W
    cvar = 4 * N * M + 4 * N
    update = 4 * N + 8 * N * T + 16 * T
    ref_sample = 2 * (B * Hp * Wp + M * Hp * Wp)              # PMF read + sampled maps written, both TDMs
    ref_rollout = 2 * M * Hw * Hw + 2 * Hw * Hw + 8 * N * T + 4 * N * M
    if sc["mode"] == "tdm":
        win = min(Hp, 232) * min(Wp, 240)                      # the staged window (WIN_WW x WH)
        rollout = 2 * M * win + 2 * win + 16 * N * T + 4 * N * M   # windows + masks + f64 controls + costs
    else:
        rollout = ref_rollout
    bh, bw = box if box else (Hp, Wp)
    sample = 2 * (B * bh * bw + M * bh * bw)
    return dict(sample_grids=sample, rollout=rollout, noise=noise, cvar=cvar, update=update,
                total=ref_sample + ref_rollout + noise + cvar + update,
                engine_total=sample + rollout + noise + cvar + update)


def kernel_metrics(workload):
    """ncu figures of the dominant kernels (per launch: DRAM bytes, warp instructions) from the committed capture
    summary profiles/kernel_metrics.json -- written from an `ncu --set full` capture of tools/ncu_target.py; the
    live part of the roofline (kernel time, SM clock) is measured here."""
    try:
        with open(os.path.join(ROOT, "profiles", "kernel_metrics.json")) as f:
            j = json.load(f)
        return j if j.get("workload") == workload else None
    except Exception:
        return None


def numba_cuda_leg(names, timeout_s=900):
    """The reference's Numba-CUDA path on this GPU, in a subprocess (its own CUDA context): baseline/numba_cuda_leg.py."""
    cmd = [sys.executable, os.path.join(ROOT, "baseline", "numba_cuda_leg.py")] + list(names)
    try:
        r = subprocess.run(cmd, capture_output=True, text=True, timeout=timeout_s, cwd=ROOT,
                           env=dict(os.environ, PYTHONDONTWRITEBYTECODE="1"))
        lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
        if not lines:
            return {"unavailable": "no output (rc %d): %s" % (r.returncode, r.stderr[-300:])}
        return json.loads(lines[-1])
    except subprocess.TimeoutExpired:
        return {"unavailable": "timed out after %d s" % timeout_s}
    except Exception as e:                               # noqa: BLE001
        return {"unavailable": repr(e)}


# ----------------------------------------------------------------------------- main arms
def run_reference(args, sc):
    """--impl reference: the CPU restatement of the path (oracle port), all host cores, bounded sample; one warmed
    pool, each step = one pass over the sample, median over the timed steps."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    n_s, m_s = cpu_sample_size(sc)
    cb = CpuBaseline(sc, n_s, m_s)
    for _ in range(max(0, args.warmup - 1)):             # the constructor ran one warm-up pass already
        cb.one_pass()
    times = cb.measure(args.steps)
    cb.close()
    t = float(np.median(times))
    v = cb.steps / t
    out = {"impl": "reference", "metric": "rollouts/sec (N*M*T state-steps/s)", "value": v,
           "unit": "state-steps/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
           "ms_per_step": 1e3 * t, "higher_is_better": True, "scaling": "strong",
           "vs_baseline": None, "dtype": "f32", "data": "synthetic",
           "config": {"workload": workload_name(args, sc)},
           "cpu_baseline": {"value": v, "unit": "state-steps/s", "cores": cb.chunks, "kind": "port", "sample": cb.desc,
                            "statistic": "median of %d passes" % len(times),
                            "pass_ms_min_max": [1e3 * min(times), 1e3 * max(times)]},
           "e2e": {"value": v, "unit": "state-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
           "gpu_launches": 0}
    _emit(json.dumps(out))


def workload_name(args, sc):
    return workload_name_of(args.workload)


def workload_name_of(name):
    mode, N, M, T, H, res, B, da = WORKLOADS[name]
    return "%s: %s MPPI N=%d M=%d T=%d, %dx%d PMF grid (%d bins, res %.1f m), num_opt=1" % (
        name, {"tdm": "CVaR-cost", "det": "CVaR-dynamics"}[mode], N, M, T, H, H, B, res)


def _quiet():
    import contextlib
    import io
    return contextlib.redirect_stdout(io.StringIO())


def make_planner(E, sc, device, rank=0, world=1, pg=None):
    with _quiet():
        cfg = E.Config(**sc["cfg"])
        lin = E.TDM_Numba(cfg, device=device, rank=rank, world_size=world)
        ang = E.TDM_Numba(cfg, device=device, rank=rank, world_size=world)
        lin.set_TDM_from_PMF_grid(sc["pmf_lin"], sc["tdm_dict"], sc["obstacle"], sc["unknown"])
        ang.set_TDM_from_PMF_grid(sc["pmf_ang"], sc["tdm_dict"], sc["obstacle"], sc["unknown"])
        pl = E.MPPI_Numba(cfg, device=device, rank=rank, world_size=world, process_group=pg)
        pl.setup(sc["params"], lin, ang)
    return cfg, lin, ang, pl


def parity_check(E, torch, sc, pl, local, rank, world, solves=2):
    """The sharded solve on the real GPUs against a 1-rank solve of the same scenario and seed (run by rank 0 on
    its own GPU), solve by solve: (a) u bit-identical on every rank, (b) u vs the 1-rank u within rtol 1e-5 (the
    softmax partials are merged in a different order), (c) every rank's slice of the CVaR costs bit-identical to the
    same slice of the 1-rank costs.  After each solve every planner's warm start is set to the 1-rank u, so that the
    next solve starts from identical inputs and its costs compare bitwise again.  `pl` must be fresh (no solve yet)."""
    import torch.distributed as dist
    dev = torch.device("cuda", local)
    p1 = None
    if rank == 0:
        _, l1, a1, p1 = make_planner(E, sc, local)
    ranks_agree, u_ok, cvar_bitwise, rel = True, True, True, 0.0
    detail = []
    T = sc["T"]
    for _ in range(solves):
        u = pl.solve()
        c = pl.costs_d.copy_to_host()
        u_t = torch.from_numpy(u.copy()).to(dev)
        c_t = torch.from_numpy(c).to(dev)
        u_all = [torch.empty_like(u_t) for _ in range(world)]
        c_all = [torch.empty_like(c_t) for _ in range(world)]
        dist.all_gather(u_all, u_t)
        dist.all_gather(c_all, c_t)
        u1_t = torch.empty((T, 2), dtype=torch.float32, device=dev)
        if rank == 0:
            u1 = p1.solve()
            c1 = p1.costs_d.copy_to_host()
            u0 = u_all[0].cpu().numpy()
            ranks_agree &= all(bool((u_all[r] == u_all[0]).all().item()) for r in range(world))
            rel = max(rel, float((np.abs(u0 - u1) / np.maximum(np.abs(u1), 1e-3)).max()))
            u_ok &= bool(np.allclose(u0, u1, rtol=1e-5, atol=1e-6))
            call = np.concatenate([x.cpu().numpy() for x in c_all])              # rank slices in rank order = n order
            same = call.shape == c1.shape and bool((call == c1).all())
            cvar_bitwise &= same
            detail.append({"cvar_bitwise": same,
                           "cvar_mismatch_frac": float((call != c1).mean()) if call.shape == c1.shape else 1.0,
                           "cvar_max_rel": float((np.abs(call - c1) / np.maximum(np.abs(c1), 1e-6)).max()) if call.shape == c1.shape else None})
            u1_t.copy_(torch.from_numpy(u1))
        dist.broadcast(u1_t, 0)
        u1h = u1_t.cpu().numpy()
        pl.u_cur_d.copy_to_device(u1h)                 # identical warm start everywhere for the next solve
        if rank == 0:
            p1.u_cur_d.copy_to_device(u1h)
    res = torch.tensor([float(ranks_agree), float(u_ok), float(cvar_bitwise), rel], dtype=torch.float64, device=dev)
    dist.broadcast(res, 0)
    r = res.cpu().numpy()
    out = {"ranks_agree": bool(r[0]), "u_within_1e-5": bool(r[1]), "cvar_bitwise": bool(r[2]), "u_max_rel": float(r[3]),
           "solves": solves, "against": "1-rank solve of the same scenario and seed on rank 0's GPU, solve by solve"}
    out["passed"] = out["ranks_agree"] and out["u_within_1e-5"] and out["cvar_bitwise"]
    if rank == 0:
        out["per_solve"] = detail
    return out


def time_small_workload(E, torch, name, local, steps, warmup):
    """One of the other BASELINE configs on this GPU: device-timed solves and the end-to-end loop, as the main arm."""
    import ctypes as C
    from mppi_numba_b200._lib import lib, check
    sc = build_scenario(name)
    dev = torch.device("cuda", local)
    cfg, lin, ang, pl = make_planner(E, sc, local)
    stream = torch.cuda.Stream(device=dev)
    check(lib.b200mppi_planner_set_stream(pl._handle, C.c_void_p(stream.cuda_stream)))   # solve() samples on this stream too
    N, M, T = sc["N"], (sc["M"] if sc["mode"] == "tdm" else 1), sc["T"]
    t_w = time.perf_counter()                                    # small solves (~0.1 ms): keep the GPU loaded for 0.4 s so
    n_w = 0                                                      # that the clocks have ramped up before anything is timed
    while n_w < max(warmup, 3) or time.perf_counter() - t_w < 0.4:
        u = pl.solve()
        n_w += 1
    torch.cuda.synchronize(dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    l0 = pl.launch_count()
    with torch.cuda.stream(stream):
        e0.record(stream)
        for _ in range(steps):
            u = pl.solve()
        e1.record(stream)
    torch.cuda.synchronize(dev)
    ms = e0.elapsed_time(e1) / steps
    launches = (pl.launch_count() - l0) / steps
    x0 = sc["params"]["x0"].copy()
    t0 = time.perf_counter()
    for _ in range(steps):
        pl.shift_and_update(x0, u, 1)
        u = pl.solve()
    torch.cuda.synchronize(dev)
    wall = (time.perf_counter() - t0) / steps
    pl.set_profiling(True)
    acc = {}
    for _ in range(5):
        pl.solve()
        for k, v in pl.last_timings().items():
            acc.setdefault(k, []).append(v)
    out = {"workload": workload_name_of(name), "ms_per_step": ms, "value": N * M * T / (ms * 1e-3),
           "e2e_ms_per_step": wall * 1e3, "e2e_value": N * M * T / wall, "unit": "state-steps/s",
           "launches_per_step": launches, "stage_ms": {k: float(np.mean(v)) for k, v in acc.items()},
           "map_sampling": ["whole maps", "reach box (speed limit)", "reach box (this solve's controls)"][pl.sample_box()[0]]}
    del pl, lin, ang
    return out


def run_b200(args, sc):
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    cpu_base = None
    if rank == 0 and world == 1 and not args.no_cpu:
        # CPU baseline FIRST: it forks worker processes, which must happen before CUDA is initialised
        n_s, m_s = cpu_sample_size(sc)
        cb = CpuBaseline(sc, n_s, m_s)
        times = cb.measure(3)
        cb.close()
        t = float(np.median(times))
        cpu_base = {"value": cb.steps / t, "unit": "state-steps/s", "cores": cb.chunks, "kind": "port",
                    "sample": cb.desc, "statistic": "median of %d passes after one warm-up pass" % len(times)}
    others = [w for w in ("c2", "c3", "c4", "c5") if w != args.workload] if (world == 1 and not args.no_others) else []
    numba = None
    if rank == 0 and world == 1 and not args.no_numba:
        # the reference's Numba-CUDA path, same GPU, same run, its own process (before this one creates a context)
        numba = numba_cuda_leg([args.workload] + [w for w in others if w != "c5"])
    import torch
    if world != args.gpus:
        raise SystemExit("--gpus %d but WORLD_SIZE=%d: launch with torch.distributed.run" % (args.gpus, world))
    import mppi_numba_b200 as E           # the library build() compiled (importing fails loudly without it)
    torch.cuda.set_device(local)
    pg = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local)

    cfg, lin, ang, pl = make_planner(E, sc, local, rank, world, pg)
    N, M, T = sc["N"], (sc["M"] if sc["mode"] == "tdm" else 1), sc["T"]
    units = N * M * T

    # all work on one torch stream so that torch.cuda.Event brackets exactly the engine's kernels
    import ctypes as C
    from mppi_numba_b200._lib import lib, check
    stream = torch.cuda.Stream(device=dev)
    if world == 1:
        check(lib.b200mppi_planner_set_stream(pl._handle, C.c_void_p(stream.cuda_stream)))   # solve() samples on this stream too
    else:
        pl._ensure_exchange()
        stream = pl._stream

    def barrier():
        if world > 1:
            import torch.distributed as dist
            dist.barrier()
        torch.cuda.synchronize(dev)

    def max_over_ranks(x):
        if world == 1:
            return x
        import torch.distributed as dist
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- N > 1: correctness of the sharded solve on these GPUs, before anything is timed
    parity = None
    if world > 1:
        parity = parity_check(E, torch, sc, pl, local, rank, world)
        if not parity["passed"]:
            if rank == 0:
                sys.stderr.write("bench.py: PARITY CHECK FAILED at %d GPUs: %s\n" % (world, json.dumps(parity)))
                _emit(json.dumps({"metric": "rollouts/sec (N*M*T state-steps/s)", "n_gpus": world,
                                  "error": "parity_check failed", "parity_check": parity}))
            import torch.distributed as dist
            dist.destroy_process_group()
            raise SystemExit(3)

    # ---- device-timed region: K solves, inputs resident
    clocks = ClockSampler(local)          # started before the warm-up: nvidia-smi needs ~0.3 s to produce a sample
    t_w = time.perf_counter()
    for _ in range(args.warmup):
        pl.solve()
    per_solve = max((time.perf_counter() - t_w) / args.warmup, 1e-5) if args.warmup > 0 else 2e-3
    # keep the GPU under the benchmark load for ~0.5 s while the clock sampler starts.  Every solve() of a
    # multi-rank run contains exchanges, so the NUMBER of extra solves must be the same on every rank:
    # agree on it (max over ranks) instead of looping on each rank's own wall clock.
    n_settle = int(max_over_ranks(float(min(5000, int(0.5 / per_solve) + 1))))
    # that number depends on the wall clock: the settle solves start from a checkpoint (warm start + RNG streams)
    # that is restored after them, so the timed steps are always solves warmup+1 .. warmup+K of the seeded planner
    checkpoint = pl.get_state()
    for _ in range(n_settle):
        pl.solve()
    barrier()
    pl.set_state(checkpoint)
    barrier()
    clocks.lines.clear()
    l0 = pl.launch_count()          # includes the TDM kernels launched inside solve()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with torch.cuda.stream(stream):
        e0.record(stream)
        for _ in range(args.steps):
            u = pl.solve()
        e1.record(stream)
    barrier()
    ms = max_over_ranks(e0.elapsed_time(e1)) / args.steps
    launches = pl.launch_count() - l0      # kernels launched in the timed region
    if args.dump_outputs:
        costs = pl.costs_d.copy_to_host()
        if world > 1:
            import torch.distributed as dist
            parts = [None] * world
            dist.all_gather_object(parts, costs)
            costs = np.concatenate(parts)
        dump = {"u": u, "costs": costs}
    # very short timed region: extend the load for the clock sampler only (same count on every rank)
    if max_over_ranks(1.0 if len(clocks.lines) < 3 else 0.0) > 0.0:
        for _ in range(int(min(5000, int(0.4 / (ms * 1e-3)) + 1))):
            pl.solve()
    clk = clocks.stop()
    value = units / (ms * 1e-3)

    # ---- end to end through the public API from host buffers (wall clock, H2D + D2H inside)
    x0 = sc["params"]["x0"].copy()
    for _ in range(2):
        pl.shift_and_update(x0, u, 1)
        u = pl.solve()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        pl.shift_and_update(x0, u, 1)          # H2D: T x 2 warm start (+ params POD by value)
        u = pl.solve()                         # D2H: T x 2 result, synchronous
    torch.cuda.synchronize(dev)
    wall = max_over_ranks(time.perf_counter() - t0) / args.steps
    barrier()
    e2e = units / wall

    # ---- per-kernel times (CUDA events inside the library) for the roofline of the dominant kernel
    pl.set_profiling(True)
    acc = {}
    reps = max(3, min(10, args.steps))
    for _ in range(reps):
        pl.solve()
        for k, v in pl.last_timings().items():
            acc.setdefault(k, []).append(v)
    pl.set_profiling(False)
    stage_ms = {k: float(np.mean(v)) for k, v in acc.items()}
    box = pl.sample_box()
    box_dims = (box[2] - box[1], box[4] - box[3]) if box[0] else None
    ab = algorithmic_bytes(sc, cfg, pl.n_local, pl.m_local, box_dims)
    peak, peak_src = measured_peaks()
    dom = max(("sample_grids", "rollout", "noise", "cvar", "update"), key=lambda k: stage_ms.get(k, 0.0))
    dom_ms = stage_ms[dom]            # sample_grids: ONE fused launch samples the linear and the angular maps
    dom_bytes = ab[dom]
    achieved = dom_bytes / (dom_ms * 1e-3) / 1e9
    km = kernel_metrics(args.workload) if world == 1 else None
    kd = (km or {}).get("kernels", {}).get(dom)
    if dom == "sample_grids" and not box[0]:
        kd = None                         # the committed capture is of the boxed launch
    traffic = kd.get("dram_bytes") if kd else None
    sm_hz = (clk.get("sm_mhz") or 1965.0) * 1e6
    issue_peak = 148 * 4 * sm_hz
    issue = None
    if kd and kd.get("warp_inst"):
        rate = kd["warp_inst"] / (dom_ms * 1e-3)
        issue = {"warp_inst": kd["warp_inst"], "peak_warp_inst_per_s": issue_peak, "achieved_warp_inst_per_s": rate,
                 "frac": rate / issue_peak, "sm_mhz": sm_hz / 1e6,
                 "source": "smsp__inst_executed.sum of %s (%s), live kernel time and SM clock" % (kd.get("kernel", dom), km.get("capture"))}
    roofline = {"bound": (kd or {}).get("bound", "issue" if sc["mode"] == "tdm" else "latency"),
                "kernel": dom, "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src,
                "algorithmic_bytes_per_launch": dom_bytes, "kernel_ms": dom_ms,
                "note": "achieved/peak/frac are the HBM figures of the contract; `bound` is the resource ncu shows "
                        "saturated for this kernel (profiles/), `issue` its instruction-issue roofline",
                "issue": issue,
                "solve_algorithmic_bytes": ab["total"],
                "solve_frac_of_hbm_roofline": (ab["total"] / (ms * 1e-3) / 1e9) / peak,
                "solve_engine_bytes": ab["engine_total"],
                "stage_ms": stage_ms}

    out = None
    if rank == 0:
        smode = ["whole maps every solve", "reach box from the speed limit", "reach box from this solve's own controls"][box[0]]
        out = {"metric": "rollouts/sec (N*M*T state-steps/s)", "value": value, "unit": "state-steps/s",
               "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms,
               "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32",
               "data": "synthetic",
               "config": {"workload": workload_name(args, sc), "global_rollouts": N, "maps": M, "horizon": T,
                          "parallelism": "single GPU" if world == 1 else ("maps sharded x%d (M/G maps per rank, all N rollouts), all-to-all of N*M/G costs + all-gather of %d floats per solve" if sc["mode"] == "tdm" else "N-sharded x%d, 1 all-gather of %d floats per solve") % (world, 2 * T + 2),
                          "exchange": ("none (1 rank)" if world == 1 else
                                       "peer-memory kernels over NVLink (csrc/p2p.cu)" if getattr(pl, "_p2p", False)
                                       else "NCCL all_to_all_single + all_gather"),
                          "map_sampling": smode + (" (%d x %d of %d x %d cells; identical costs / u / RNG states, "
                                                   "tests/test_gpu_parity.py::test_boxed_solve_identical_to_whole_map_solve)"
                                                   % (box_dims + tuple(cfg.max_map_dim)) if box_dims else ""),
                          "l2": "no explicit flush: every solve rewrites its sampled maps (2 x %d MB per rank) and re-reads them through TMA"
                                % (M // world * (box_dims[0] * box_dims[1] if box_dims else cfg.max_map_dim[0] * cfg.max_map_dim[1]) // 2 ** 20)},
               "clocks": clk,
               "e2e": {"value": e2e, "unit": "state-steps/s", "ms_per_step": wall * 1e3,
                       "h2d_bytes_per_step": 8 * T + 88, "d2h_bytes_per_step": 8 * T + (4 if box[0] == 2 else 0)},
               "gpu_launches": int(launches),
               "roofline": roofline}
        if parity is not None:
            out["parity_check"] = parity
        if cpu_base is not None:
            out["cpu_baseline"] = cpu_base
        if numba is not None:
            nb = dict(numba)
            w = nb.get("workloads", {}).get(args.workload)
            if w:
                nb.update({"ms_per_solve": w["ms_per_solve"], "value": w["value"], "unit": "state-steps/s",
                           "kernels": w["kernels_ms"], "engine_speedup_device_timed": value / w["value"],
                           "engine_speedup_e2e": e2e / w["value"]})
            out["numba_cuda_baseline"] = nb
    if others:
        del pl, lin, ang
        res = {}
        for name in others:
            try:
                res[name] = time_small_workload(E, torch, name, local, args.steps, args.warmup)
                w = (numba or {}).get("workloads", {}).get(name)
                if w:
                    res[name]["numba_cuda_ms_per_solve"] = w["ms_per_solve"]
                    res[name]["speedup_vs_numba_cuda_e2e"] = w["ms_per_solve"] / res[name]["e2e_ms_per_step"]
            except Exception as e:                       # noqa: BLE001
                res[name] = {"error": repr(e)}
        out["others"] = res
    if rank == 0:
        if args.dump_outputs:
            os.makedirs(args.dump_outputs, exist_ok=True)
            for name, a in dump.items():
                np.save(os.path.join(args.dump_outputs, name + ".npy"), np.ascontiguousarray(a, dtype=np.float32))
        _emit(json.dumps(out))
    if world > 1:
        import torch.distributed as dist
        dist.destroy_process_group()


_emit = print


def main():
    # The contract is ONE JSON line on stdout.  Libraries (NCCL's version banner, the engine's allocation
    # notices) also write to fd 1, so everything is routed to stderr and only the final line goes to the
    # real stdout.
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    sys.stdout = os.fdopen(os.dup(2), "w", buffering=1)
    global _emit

    def _emit(line):
        os.write(real_stdout, (line + "\n").encode())
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="c5", choices=sorted(WORKLOADS))
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-numba", action="store_true", help="skip the reference's Numba-CUDA leg (N = 1)")
    ap.add_argument("--no-others", action="store_true", help="skip the other BASELINE configs (N = 1)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write u and the CVaR costs of the last timed solve to DIR/<name>.npy (--impl b200)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs needs --impl b200")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    sc = build_scenario(args.workload)
    if args.impl == "reference":
        run_reference(args, sc)
    else:
        run_b200(args, sc)


if __name__ == "__main__":
    main()
