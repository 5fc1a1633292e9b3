#!/usr/bin/env python3
"""bench.py -- headline benchmark of the batched Hunter NMPC + WBC control step (BASELINE.json metric).

  python bench.py --gpus N --steps K --warmup W              this repo's CUDA path (N>1: launched by torch.distributed.run)
  python bench.py --impl reference --gpus N --steps K ...    the reference arm: the CPU restatement of the reference's
                                                             algorithm (oracle/, "port": the upstream OCS2+qpOASES binaries
                                                             cannot be built offline) on all host threads, rank 0 only
  python bench.py --config {1,2,3,4}                         BASELINE.json configs[1..4]; the default (and what the driver runs) is 1

One "step" = one pass of the hot path over one batch: for every instance one SQP iteration of the N=100, dt=10 ms centroidal
NMPC from the initializer's cold start (LQ approximation, projection, Riccati, forward pass, filter line search), policy
evaluation at t0 + 2 ms, and one WeightedWbc QP.

  configs[1]  1024 instances per GPU, trot gait, randomised initial base pose (seed 20240901 + instance index)         [default]
  configs[2]  8192 instances on one GPU, walking mode (WBC non-stance tasks), trot schedule, cmd_vel grid
              v_x in linspace(-0.5, 0.5, 32) x w_z in linspace(-0.5, 0.5, 32) x 8 initial-pose seeds
  configs[3]  8192 instances per GPU (65 536 on 8 GPUs), schedule of instance i = i mod 4 in {stance, trot, standing_trot,
              flying_trot} with a random phase, instances sorted by schedule inside a GPU, outputs un-permuted and gathered with NCCL
  configs[4]  WBC-only raw QP sweep, B = 2^10 ... 2^20 WeightedWbc problems (38 variables, 56-60 rows) in the qpOASES layout

N>1 keeps the per-GPU instance count (weak scaling), sharded by contiguous blocks with no data-path collective; the per-instance
torques are gathered to rank 0 with NCCL every step on a side stream.

  --dump-outputs DIR   configs[1..3]: after the timed device-resident steps, rank 0 writes what the last step returned for its instances
                       (xt, ut, info, sol, tau, status; info as columns alpha, merit0, merit1, viol0, viol1, armijo, status, n_trials)
                       as DIR/<name>.npy in float64, rows in instance order, plus instance.npy (the global instance index of every row).
                       Inputs depend only on the arguments, so two builds can be compared file by file.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

sys.dont_write_bytecode = True      # the source tree may be read-only: nothing is written into it
ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "MPC+WBC control-step solves/sec (Hunter N=100)"
UNIT = "solves/s"
PER_GPU_BATCH = {1: 1024, 2: 8192, 3: 8192}
HORIZON_N, DT = 100, 0.01
T_POLICY = 0.002
SEED = 20240901
# SURVEY.md 8(d) / BASELINE.md 4: algorithmic HBM bytes and flops of one control-step solve
BYTES_PER_MPC_SOLVE = 0.48e6
BYTES_PER_WBC_SOLVE = 616 + 304
BYTES_PER_RAW_QP = 8 * (38 * 38 + 58 * 38 + 38 + 2 * 58) + 304     # SURVEY 8(d): 30.4 KB in + 304 B out
FLOPS_PER_SOLVE = 3.6e7 + 2.0e6
FP64_NOMINAL_TFLOPS = 37.0   # B200 FP64 CUDA-core peak (not in MEASURED_PEAKS.json; nominal)
GAIT_NAMES = ["stance", "trot", "standing_trot", "flying_trot"]
GAIT_PERIOD = {"stance": 0.5, "trot": 0.6, "standing_trot": 0.6, "flying_trot": 0.4}
KERNEL_OF = {"mpc_lq_project": "lq_kernel", "mpc_linearise": "lin_kernel", "mpc_riccati": "riccati_kernel", "mpc_forward_linesearch": "forward_linesearch2_kernel"}
DUMP_LIMIT_BYTES = 64 * 2 ** 20


def dump_outputs(path, outputs, instance):
    """Write every [rows, ...] array of `outputs` and the row -> instance index as path/<name>.npy in float64. Above DUMP_LIMIT_BYTES in all,
    every array keeps the same fixed, seeded sample of rows (configs[1] at its default size is written whole)."""
    arrays = {k: np.asarray(v, dtype=np.float64) for k, v in dict(outputs, instance=instance).items()}
    rows = len(instance)
    row_bytes = sum(a[:1].nbytes for a in arrays.values())
    keep = min(rows, (DUMP_LIMIT_BYTES - 1024 * len(arrays)) // row_bytes)     # 1 KB per file covers the .npy header
    if keep < rows:
        sel = np.sort(np.random.default_rng(SEED).choice(rows, keep, replace=False))
        arrays = {k: a[sel] for k, a in arrays.items()}
    os.makedirs(path, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(path, k + ".npy"), a)


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return json.load(open(p)), "measured"
    return {"hbm_gbs": 6650.0}, "fallback"


def host_parallelism():
    """Threads this process may really use: affinity mask and cgroup CPU quota next to os.cpu_count()."""
    out = {"cpu_count": os.cpu_count() or 1}
    try:
        out["affinity"] = len(os.sched_getaffinity(0))
    except Exception:
        out["affinity"] = None
    quota = None
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()
        quota = None if q == "max" else float(q) / float(per)
    except Exception:
        try:
            q = float(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read()); per = float(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            quota = None if q <= 0 else q / per
        except Exception:
            pass
    out["cgroup_cpu_quota"] = quota
    eff = out["affinity"] or out["cpu_count"]
    if quota:
        eff = min(eff, quota)
    out["effective"] = eff
    return out


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""

    def __init__(self, index):
        self.index = index; self.samples = []; self.reasons = set(); self.max_mhz = None; self._stop = False; self._t = None

    def _run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        while not self._stop:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q, "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip().split(",")
                self.samples.append(float(out[0])); self.max_mhz = float(out[1])
                for n, v in zip(names, out[2:]):
                    if v.strip().lower().startswith("active"):
                        self.reasons.add(n)
            except Exception:
                pass
            time.sleep(0.15)

    def start(self):
        self._t = threading.Thread(target=self._run, daemon=True); self._t.start()

    def stop(self):
        self._stop = True
        if self._t:
            self._t.join(timeout=6)
        return {"sm_mhz": float(np.median(self.samples)) if self.samples else None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(self.samples)}


# ------------------------------------------------------------------------------------------------ workloads
def _instance_spec(config, g):
    """(pose seed, gait, cmd_vel, phase) of global instance g (SURVEY 8d)."""
    if config == 1:
        return SEED + g, "trot", (0.2, 0.0, 0.0, 0.0), 0.0
    if config == 2:
        p = g % 1024
        vx = np.linspace(-0.5, 0.5, 32)[p // 32]; wz = np.linspace(-0.5, 0.5, 32)[p % 32]
        return SEED + (g // 1024) % 8, "trot", (float(vx), 0.0, 0.0, float(wz)), 0.0
    gait = GAIT_NAMES[g % 4]
    return SEED + g, gait, (0.2, 0.0, 0.0, 0.0), float(np.random.default_rng(SEED + g).uniform(0.0, GAIT_PERIOD[gait]))


def _gen_range(args):
    config, lo, hi = args
    from hunter_bipedal_control_b200 import scenarios as S
    n = hi - lo
    x0 = np.zeros((n, 22)); x_ref = np.zeros((n, HORIZON_N + 1, 22)); swing = np.zeros((n, HORIZON_N + 1, 24)); mode = np.zeros((n, HORIZON_N + 1), dtype=np.int32)
    compacts = []
    for i in range(n):
        seed, gait, cmd, phase = _instance_spec(config, lo + i)
        x0[i] = S.random_initial_states(1, seed)[0]
        x_ref[i], swing[i], mode[i], c = S.make_reference(x0[i], cmd, gait, HORIZON_N, DT, phase=phase)
        compacts.append(c)
    return x0, x_ref, swing, mode, compacts


def workload(B, seed_offset=0, with_compact=False, config=1):
    """Instances [seed_offset, seed_offset + B) of the given config: x0, node-sampled references, rbd measurement (+ compact references)."""
    from hunter_bipedal_control_b200 import scenarios as S
    lo = seed_offset
    nproc = min(os.cpu_count() or 1, 32, max(1, B // 256))
    if nproc > 1:
        import multiprocessing as mp
        chunks = [(config, lo + B * k // nproc, lo + B * (k + 1) // nproc) for k in range(nproc)]
        with mp.get_context("fork").Pool(nproc) as pool:
            parts = pool.map(_gen_range, chunks)
        x0, x_ref, swing, mode = (np.concatenate([p[j] for p in parts]) for j in range(4))
        compacts = [c for p in parts for c in p[4]]
    else:
        x0, x_ref, swing, mode, compacts = _gen_range((config, lo, lo + B))
    rbd = S.consistent_rbd(x0, np.random.default_rng(SEED + seed_offset), 0.0)
    if with_compact:
        return x0, x_ref, swing, mode, rbd, S.pack_references(compacts, 1.05 * HORIZON_N * DT)
    return x0, x_ref, swing, mode, rbd


def workload_desc(config, B):
    if config == 1:
        return "configs[1]: %d Hunter instances per GPU, trot gait, N=100 dt=10 ms, randomised initial base pose (seed 20240901+i)" % B
    if config == 2:
        return "configs[2]: %d Hunter instances per GPU, walking mode, trot schedule, cmd_vel grid vx x wz in [-0.5, 0.5]^2 (32 x 32) x 8 pose seeds, N=100 dt=10 ms" % B
    return ("configs[3]: %d Hunter instances per GPU, schedule i mod 4 in {stance, trot, standing_trot, flying_trot} with random phase, sorted by schedule "
            "inside the GPU, N=100 dt=10 ms" % B)


def cpu_control_steps(x0, x_ref, swing, mode, rbd, threads):
    """The oracle's control step on host threads; returns (seconds, torques)."""
    from oracle import hbo
    n = x0.shape[0]
    xt = np.zeros((n, HORIZON_N + 1, 22)); ut = np.zeros((n, HORIZON_N, 22))
    for i in range(n):
        xt[i], ut[i] = hbo.mpc_cold_start(HORIZON_N, DT, x0[i], mode[i])
    t = time.perf_counter()
    xt1, ut1, _ = hbo.mpc_iteration_batch(HORIZON_N, DT, x0, x_ref, swing, mode, xt, ut, threads=threads)
    al = T_POLICY / DT
    xd = (1 - al) * xt1[:, 0] + al * xt1[:, 1]; ud = (1 - al) * ut1[:, 0] + al * ut1[:, 1]
    sol, _ = hbo.wbc_solve_batch(xd, ud, rbd, mode[:, 0], np.zeros(n, dtype=np.uint8), 1e-8, threads=threads)
    return time.perf_counter() - t, sol[:, 28:]


def qp_sweep_states(B, seed=SEED):
    """Config-2-style random states for the raw QP sweep: modes {STANCE 50 %, L 25 %, R 25 %} (SURVEY 8d config 5)."""
    from hunter_bipedal_control_b200 import scenarios as S
    rng = np.random.default_rng(seed)
    mode = rng.choice(np.array([3, 3, 2, 1], dtype=np.int32), B)
    x = np.tile(S.INITIAL_STATE, (B, 1)) + rng.uniform(-.05, .05, (B, 22))
    u = np.zeros((B, 22))
    fl = np.stack([(mode == 2) | (mode == 3), (mode == 1) | (mode == 3), (mode == 2) | (mode == 3), (mode == 1) | (mode == 3)], axis=1)
    u[:, 2:12:3] = fl * (S.TOTAL_MASS * 9.81 / fl.sum(axis=1))[:, None]
    u[:, 12:] = rng.uniform(-.5, .5, (B, 10))
    rbd = S.consistent_rbd(x, rng, 0.02)
    return x, u, rbd, mode


# ------------------------------------------------------------------------------------------------ reference arm
def run_reference(args, rank, world):
    if rank != 0:
        return
    par = host_parallelism()
    cores = os.cpu_count() or 1
    if args.config == 4:
        from oracle import hbo
        n = max(8 * cores, 64)
        x, u, rbd, mode = qp_sweep_states(n)
        H = np.zeros((n, 38, 38)); g = np.zeros((n, 38)); A = np.zeros((n, 60, 38)); lb = np.full((n, 60), -1e20); ub = np.full((n, 60), 1e20)
        for i in range(n):
            Hi, gi, Ai, lbi, ubi = hbo.wbc_assemble(x[i], u[i], rbd[i], int(mode[i]), False)
            m = Ai.shape[0]
            H[i] = Hi; g[i] = gi; A[i, :m] = Ai; lb[i, :m] = lbi; ub[i, :m] = ubi
        for _ in range(args.warmup):
            hbo.wbc_qp_batch(H[:cores], g[:cores], A[:cores], lb[:cores], ub[:cores], 1e-8, threads=cores)
        t = time.perf_counter()
        for _ in range(args.steps):
            hbo.wbc_qp_batch(H, g, A, lb, ub, 1e-8, threads=cores)
        total = time.perf_counter() - t
        val = n * args.steps / total
        line = {"impl": "reference", "metric": "WeightedWbc QPs/sec (38 variables, 56-60 rows), raw QP sweep", "value": val, "unit": "QPs/s", "n_gpus": args.gpus,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total / args.steps, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                "config": {"workload": "configs[4]: raw WeightedWbc QPs; %d-problem sample per step" % n,
                           "note": "CPU interior-point restatement (oracle port); qpOASES itself is not available offline"},
                "cpu_baseline": {"value": val, "unit": "QPs/s", "cores": cores, "kind": "port", "sample": "%d QPs per bench step, all host threads" % n, "host_parallelism": par},
                "e2e": {"value": val, "unit": "QPs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line))
        return
    n = max(2 * cores, 8)
    data = workload(n, config=args.config)
    for _ in range(args.warmup):
        cpu_control_steps(*[d[:min(n, cores)] for d in data], threads=cores)
    ts = []
    for _ in range(args.steps):
        dt_, _ = cpu_control_steps(*data, threads=cores)
        ts.append(dt_)
    total = float(np.sum(ts))
    val = n * args.steps / total
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1e3 * total / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic",
            "config": {"workload": "%s; %d-instance sample per step" % (workload_desc(args.config, PER_GPU_BATCH[args.config]), n),
                       "note": "CPU restatement of the reference algorithm (oracle port); upstream OCS2+qpOASES binaries cannot be built offline"},
            "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": "port", "sample": "%d control steps per bench step, all host threads" % n,
                             "host_parallelism": par},
            "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------ configs[4]: raw QP sweep
def run_qp_sweep(args, rank, world, local):
    import torch
    import ctypes as C
    import hunter_bipedal_control_b200 as hb
    if rank != 0:       # one GPU by definition (BASELINE configs[4]: 1 x B200)
        return
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    sizes = [2 ** k for k in range(10, 21, 2)]
    if args.batch:
        sizes = [s for s in sizes if s <= args.batch] or [args.batch]
    Bmax = max(sizes)
    ctx = hb.Context(horizon_N=1, dt=DT, max_batch=Bmax, device=local)     # WBC-only context: the MPC node records are never allocated
    lib = hb.load_library()
    stream = torch.cuda.ExternalStream(ctx.stream_handle, device=dev)
    x, u, rbd, mode = qp_sweep_states(Bmax)
    to = lambda a, dt_=torch.float64: torch.from_numpy(np.ascontiguousarray(a)).to(dev, dtype=dt_)
    d_x, d_u, d_rbd, d_mode = to(x), to(u), to(rbd), to(mode, torch.int32)
    f8 = dict(dtype=torch.float64, device=dev)
    d_H = torch.empty((Bmax, 38, 38), **f8); d_g = torch.empty((Bmax, 38), **f8); d_A = torch.empty((Bmax, 60, 38), **f8)
    d_lb = torch.empty((Bmax, 60), **f8); d_ub = torch.empty((Bmax, 60), **f8); d_m = torch.empty(Bmax, dtype=torch.int32, device=dev)
    d_sol = torch.empty((Bmax, 38), **f8); d_st = torch.empty(Bmax, dtype=torch.int32, device=dev); d_it = torch.empty(Bmax, dtype=torch.int32, device=dev)
    P = lambda t: C.c_void_p(t.data_ptr())
    ck = lambda rc: (_ for _ in ()).throw(RuntimeError("C ABI call failed: %d" % rc)) if rc else None
    ck(lib.hb_wbc_assemble_batch_dev(ctx._h, Bmax, P(d_x), P(d_u), P(d_rbd), P(d_mode), None, P(d_H), P(d_g), P(d_A), P(d_lb), P(d_ub), P(d_m)))
    ctx.sync()
    sampler = ClockSampler(local); sampler.start()
    sweep = []
    l0 = ctx.launch_count
    launches_timed = 0
    for B in sizes:
        def raw():
            ck(lib.hb_wbc_qp_rows_batch_dev(ctx._h, B, 38, 60, P(d_m), P(d_H), P(d_g), P(d_A), P(d_lb), P(d_ub), P(d_sol), P(d_st), P(d_it)))

        def fused():
            ck(lib.hb_wbc_solve_batch_dev(ctx._h, B, P(d_x), P(d_u), P(d_rbd), P(d_mode), None, P(d_sol), P(d_st)))
        res = {"B": B}
        for name, fn in (("raw", raw), ("fused", fused)):
            for _ in range(max(args.warmup, 3)):
                fn()
            ctx.sync()
            e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            for _ in range(args.steps):
                fn()
            e1.record(stream)
            ctx.sync(); torch.cuda.synchronize(dev)
            ms = e0.elapsed_time(e1) / args.steps
            launches_timed += args.steps
            solved = float((d_st[:B] == 0).double().mean().item())      # unsolved QPs take WeightedWbc's fallback (previous solution) in the product
            res[name] = {"qps": B / (ms * 1e-3), "ms_per_step": ms, "solved_fraction": solved}
            if name == "raw":
                it = d_it[:B].to(torch.float64)
                res[name]["mean_iters"] = float(it.mean().item()); res[name]["max_iters"] = int(it.max().item())
                # interior-point iterations per QP: {iterations: QPs}; the kernel's latency is (slowest warp per SM) x (per-iteration chain)
                hist = torch.bincount(d_it[:B].to(torch.int64))
                res[name]["iters_hist"] = {str(i): int(c) for i, c in enumerate(hist.tolist()) if c}
        sweep.append(res)
    # parity of the two device paths on the largest batch (same optimum: torques to 1e-4 relative)
    raw_tau = None
    ck(lib.hb_wbc_qp_rows_batch_dev(ctx._h, sizes[0], 38, 60, P(d_m), P(d_H), P(d_g), P(d_A), P(d_lb), P(d_ub), P(d_sol), P(d_st), P(d_it))); ctx.sync()
    raw_tau = d_sol[:sizes[0], 28:].cpu().numpy()
    ck(lib.hb_wbc_solve_batch_dev(ctx._h, sizes[0], P(d_x), P(d_u), P(d_rbd), P(d_mode), None, P(d_sol), P(d_st))); ctx.sync()
    fused_tau = d_sol[:sizes[0], 28:].cpu().numpy()
    fused_vs_raw = float(np.abs(raw_tau - fused_tau).max() / max(1.0, np.abs(raw_tau).max()))
    # end to end through the host-pointer call hb_wbc_qp_batch (pinned host buffers): 30.4 KB per QP cross PCIe
    Be = min(2 ** 14, Bmax)
    hH = d_H[:Be].cpu().pin_memory(); hg = d_g[:Be].cpu().pin_memory(); hA = d_A[:Be].cpu().pin_memory(); hlb = d_lb[:Be].cpu().pin_memory(); hub = d_ub[:Be].cpu().pin_memory()
    hx = torch.zeros((Be, 38), dtype=torch.float64).pin_memory(); hst = torch.zeros(Be, dtype=torch.int32).pin_memory(); hit = torch.zeros(Be, dtype=torch.int32).pin_memory()

    def e2e():
        ck(lib.hb_wbc_qp_batch(ctx._h, Be, 38, 60, P(hH), P(hg), P(hA), P(hlb), P(hub), P(hx), P(hst), P(hit)))
    for _ in range(2):
        e2e()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        e2e()
    e2e_s = (time.perf_counter() - t0) / args.steps
    clocks = sampler.stop()
    peaks, src = load_peaks()
    top = sweep[-1]
    ach = top["B"] * BYTES_PER_RAW_QP / (top["raw"]["ms_per_step"] * 1e-3) / 1e9
    line = {"metric": "WeightedWbc QPs/sec (38 variables, 56-60 rows), raw QP sweep", "value": top["raw"]["qps"], "unit": "QPs/s", "n_gpus": 1, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": top["raw"]["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic",
            "config": {"workload": "configs[4]: WBC-only raw QP sweep, B = %s WeightedWbc problems in the qpOASES layout (H 38x38, A 60x38 allocated, 56-60 rows used), "
                                   "assembled on the device from config-2-style random states, modes {STANCE 50 %%, L 25 %%, R 25 %%}" % sizes,
                       "l2": "inputs of one launch (%.0f MB at the largest B) exceed the 126 MB L2 from B = 4096 on" % (top["B"] * BYTES_PER_RAW_QP / 1e6)},
            "sweep": sweep, "fused_vs_raw_torque_rel_diff": fused_vs_raw,
            "e2e": {"value": Be / e2e_s, "unit": "QPs/s", "h2d_bytes_per_step": int((hH.numel() + hg.numel() + hA.numel() + hlb.numel() + hub.numel()) * 8),
                    "d2h_bytes_per_step": int(hx.numel() * 8 + hst.numel() * 4 + hit.numel() * 4), "ms_per_step": e2e_s * 1e3, "B": Be,
                    "call": "hb_wbc_qp_batch: H, g, A, lbA, ubA in; x, status, iterations out"},
            "gpu_launches": int(launches_timed),
            "roofline": {"bound": "hbm", "kernel": "qp_batch_kernel", "achieved": ach, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": ach / peaks["hbm_gbs"],
                         "peak_source": src, "traffic": None, "note": "compute/latency-bound interior point (SURVEY 8d: FP64 ceiling ~2e7 QP/s, HBM ceiling 2.6e8 QP/s)"},
            "clocks": clocks}
    if not args.no_cpu_baseline:
        from oracle import hbo
        cores = os.cpu_count() or 1
        n = max(4 * cores, 32)
        H, g, A, lb, ub = (t[:n].cpu().numpy() for t in (d_H, d_g, d_A, d_lb, d_ub))
        mrows = d_m[:n].cpu().numpy()
        for i in range(n):      # rows beyond m_rows[i] are unconstrained for the fixed-shape CPU call
            A[i, mrows[i]:] = 0.0; lb[i, mrows[i]:] = -1e20; ub[i, mrows[i]:] = 1e20
        t0 = time.perf_counter(); xo, sto = hbo.wbc_qp_batch(H, g, A, lb, ub, 1e-8, threads=cores); t_all = time.perf_counter() - t0
        t0 = time.perf_counter(); hbo.wbc_qp_batch(H[:4], g[:4], A[:4], lb[:4], ub[:4], 1e-8, threads=1); t_one = (time.perf_counter() - t0) / 4
        ck(lib.hb_wbc_qp_rows_batch_dev(ctx._h, n, 38, 60, P(d_m), P(d_H), P(d_g), P(d_A), P(d_lb), P(d_ub), P(d_sol), P(d_st), P(d_it))); ctx.sync()
        err = float(np.abs(xo[:, 28:] - d_sol[:n, 28:].cpu().numpy()).max() / max(1.0, np.abs(xo[:, 28:]).max()))
        line["cpu_baseline"] = {"value": n / t_all, "unit": "QPs/s", "cores": cores, "kind": "port", "host_parallelism": host_parallelism(),
                                "sample": "%d QPs of the same sweep, all host threads; single-thread %.1f QPs/s; qpOASES itself is not available offline" % (n, 1.0 / t_one),
                                "single_thread_value": 1.0 / t_one, "torque_rel_err_vs_gpu": err}
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------ configs[1..3]
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", type=int, default=1, choices=[1, 2, 3, 4], help="BASELINE.json configs[k]")
    ap.add_argument("--batch", type=int, default=0, help="instances per GPU (default: the config's size)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--torch-gather", action="store_true", help="multi-GPU: gather with torch.distributed instead of hb_shard_gather_dev")
    ap.add_argument("--e2e-chunks", type=int, default=0, help="chunks of the host-pointer cycle (0 = library default)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step as DIR/<name>.npy (configs[1..3])")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "b200" or args.config == 4):
        ap.error("--dump-outputs applies to configs[1..3] of the b200 path")
    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1")); local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    args.warmup = max(args.warmup, 3)
    import torch
    import hunter_bipedal_control_b200 as hb
    from hunter_bipedal_control_b200 import sharding
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device visible; the product path has no CPU fallback")
    if args.config == 4:
        run_qp_sweep(args, rank, world, local)
        return
    cfg = args.config
    dist = None
    if world > 1:
        import torch.distributed as dist
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    B = args.batch or PER_GPU_BATCH[cfg]
    total_B = B * world
    lo, hi = sharding.partition(total_B, world, rank)
    x0, x_ref, swing, mode, rbd, refs = workload(B, seed_offset=lo, with_compact=True, config=cfg)     # instance index = global index
    import ctypes as C
    perm = inv = None
    if cfg == 3:      # instances sorted by mode schedule inside the GPU (warp-uniform control flow); outputs are un-permuted before the gather
        perm, inv = sharding.sort_by_schedule(mode)
        x0, x_ref, swing, mode, rbd = x0[perm], x_ref[perm], swing[perm], mode[perm], rbd[perm]
        sorted_refs = (hb.HbReference * B)()
        for k in range(B):
            C.memmove(C.addressof(sorted_refs[k]), C.addressof(refs[int(perm[k])]), C.sizeof(hb.HbReference))
        refs = sorted_refs
    ctx = hb.Context(horizon_N=HORIZON_N, dt=DT, max_batch=B, device=local, e2e_chunks=args.e2e_chunks)
    stream = torch.cuda.ExternalStream(ctx.stream_handle, device=dev)
    comm_stream = torch.cuda.Stream(device=dev) if world > 1 else None
    # the gather behind the C ABI (hb_shard_*: un-permute + NCCL all-gather on the shard's own stream); torch.distributed only carries the
    # 128-byte communicator id and the barriers. `--torch-gather` keeps the round-1 path (dist.all_gather issued from Python).
    shard = None
    if world > 1 and not args.torch_gather:
        uid_t = torch.zeros(sharding.SHARD_ID_BYTES, dtype=torch.uint8, device=dev)
        if rank == 0:
            uid_t.copy_(torch.frombuffer(bytearray(sharding.unique_id()), dtype=torch.uint8))
        dist.broadcast(uid_t, 0)
        shard = sharding.Shard(ctx, bytes(uid_t.cpu().numpy().tobytes()), world, rank, total_B, max_row_doubles=10)
        assert (shard.lo, shard.hi) == (lo, hi)
    to = lambda a, dt_=torch.float64: torch.from_numpy(np.ascontiguousarray(a)).to(dev, dtype=dt_)
    d_x0, d_xref, d_swing, d_rbd = to(x0), to(x_ref), to(swing), to(rbd)
    d_mode = to(mode, torch.int32)
    d_inv = to(inv, torch.int64) if inv is not None else None
    d_inv32 = to(inv, torch.int32) if inv is not None else None
    d_xt0 = torch.zeros((B, HORIZON_N + 1, 22), dtype=torch.float64, device=dev); d_ut0 = torch.zeros((B, HORIZON_N, 22), dtype=torch.float64, device=dev)
    ctx.mpc_cold_start_dev(d_x0, d_mode, d_xt0, d_ut0)
    ctx.sync()
    d_xt = d_xt0.clone(); d_ut = d_ut0.clone()
    d_info = torch.zeros((B, 7), dtype=torch.float64, device=dev)
    d_sol = torch.zeros((B, 38), dtype=torch.float64, device=dev); d_tau = torch.zeros((B, 10), dtype=torch.float64, device=dev)
    d_st = torch.zeros(B, dtype=torch.int32, device=dev)
    d_out = [torch.zeros((B, 10), dtype=torch.float64, device=dev) for _ in range(2)]      # gather sources (instance order), double buffered
    gathered = [None]
    step_no = [0]

    def step_device():
        with torch.cuda.stream(stream):
            d_xt.copy_(d_xt0, non_blocking=True); d_ut.copy_(d_ut0, non_blocking=True)   # every step starts from the initializer's cold start
        ctx.control_step_dev(T_POLICY, d_x0, d_xref, d_swing, d_mode, d_rbd, d_xt, d_ut, d_info, d_sol, d_tau, d_st)
        if shard is not None:
            gathered[0] = shard.gather(d_tau, d_inv32)      # asynchronous: pack on the compute stream, all-gather + compaction on the shard's stream
        elif world > 1:
            buf = d_out[step_no[0] & 1]
            step_no[0] += 1
            with torch.cuda.stream(stream):
                if d_inv is not None:
                    torch.index_select(d_tau, 0, d_inv, out=buf)       # back to instance order
                else:
                    buf.copy_(d_tau, non_blocking=True)
                ev = torch.cuda.Event(); ev.record(stream)
            # the NCCL gather runs on a side stream behind the event: the next step's kernels do not wait for it
            comm_stream.wait_event(ev)
            with torch.cuda.stream(comm_stream):
                gathered[0] = sharding.gather_to_rank0(buf, total_B, world, rank, dist)

    def barrier():
        if world > 1:
            if shard is not None:
                shard.wait(block_host=True)
            comm_stream.synchronize()
            dist.barrier()
        ctx.sync(); torch.cuda.synchronize(dev)

    # ---------------- device-resident measurement
    for _ in range(args.warmup):
        step_device()
    barrier()
    ctx.profile_enable(True)
    l0 = ctx.launch_count
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ev0 = torch.cuda.Event(enable_timing=True); ev1 = torch.cuda.Event(enable_timing=True)
    barrier()
    ev0.record(stream)
    for _ in range(args.steps):
        step_device()
    if shard is not None:
        shard.wait()                         # the compute stream waits for the last gather: the timed region ends when it has landed
    elif world > 1:
        stream.wait_stream(comm_stream)
    ev1.record(stream)
    barrier()
    ms = ev0.elapsed_time(ev1)
    launches = ctx.launch_count - l0
    prof = ctx.profile_read()
    ctx.profile_enable(False)
    if args.dump_outputs and rank == 0:
        info = d_info.cpu().numpy().view(hb.INFO_DTYPE)[:, 0]          # hb_solve_info records -> columns alpha ... armijo, status, n_trials
        outs = {"xt": d_xt.cpu().numpy(), "ut": d_ut.cpu().numpy(), "info": np.stack([info[n] for n in hb.INFO_DTYPE.names], axis=1),
                "sol": d_sol.cpu().numpy(), "tau": d_tau.cpu().numpy(), "status": d_st.cpu().numpy()}
        if inv is not None:                 # back to instance order (configs[3])
            outs = {k: v[inv] for k, v in outs.items()}
        dump_outputs(args.dump_outputs, outs, np.arange(lo, hi))
    gather_ok = None
    if world > 1 and rank == 0:
        if shard is not None:
            g_all = shard.to_host(gathered[0], 10)
            mine = d_tau.cpu().numpy() if inv is None else d_tau.cpu().numpy()[inv]
            gather_ok = bool(g_all.shape[0] == total_B and np.isfinite(g_all).all() and np.array_equal(g_all[lo:hi], mine))
        else:
            gather_ok = bool(gathered[0] is not None and gathered[0].shape[0] == total_B and torch.isfinite(gathered[0]).all().item())
    # ---------------- end-to-end through the host-pointer C ABI, pinned host buffers, copies inside the timed region.
    # e2e      : hb_resident_cycle_batch -- the closed-loop call: t0 / x0 / compact references / rbd in, info / WBC solution / torques out;
    #            reference expansion and the initializer cold start run on the device, the primal solution stays resident.
    # e2e_full : hb_control_step_batch -- node-sampled references and the full state / input trajectories cross PCIe both ways (configs[1] only).
    pin = lambda a: torch.from_numpy(np.ascontiguousarray(a)).pin_memory()
    h_x0, h_rbd = pin(x0), pin(rbd)
    ref_bytes = C.sizeof(refs)
    h_refs = torch.empty(ref_bytes, dtype=torch.uint8).pin_memory()
    C.memmove(h_refs.data_ptr(), C.addressof(refs), ref_bytes)
    h_t0 = torch.zeros(B, dtype=torch.float64).pin_memory()
    h_info = torch.zeros((B, 7), dtype=torch.float64).pin_memory(); h_sol = torch.zeros((B, 38), dtype=torch.float64).pin_memory()
    h_tau = torch.zeros((B, 10), dtype=torch.float64).pin_memory(); h_st = torch.zeros(B, dtype=torch.int32).pin_memory()
    lib = hb.load_library()
    P = lambda t: C.c_void_p(t.data_ptr())

    def step_e2e():
        rc = lib.hb_resident_cycle_batch(ctx._h, B, 1, C.c_double(T_POLICY), P(h_t0), P(h_x0), P(h_refs), P(h_rbd), P(h_info), P(h_sol), P(h_tau), P(h_st))
        assert rc == 0, rc

    for _ in range(2):
        step_e2e()
    barrier()
    _td = d_tau.cpu().numpy()
    e2e_tau_diff = float(np.abs(h_tau.numpy() - _td).max() / max(1e-300, np.abs(_td).max()))     # same work as the device-resident step
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step_e2e()
    barrier()
    e2e_s = time.perf_counter() - t0
    ref_up = ctx.last_reference_upload_bytes            # only the used entries of the fixed-capacity hb_reference structs cross PCIe
    h2d = (h_t0.numel() + h_x0.numel() + h_rbd.numel()) * 8 + ref_up
    d2h = (h_info.numel() + h_sol.numel() + h_tau.numel()) * 8 + h_st.numel() * 4
    extra = {}
    plan_s = full_s = 0.0
    full_h2d = (x0.size + x_ref.size + swing.size + rbd.size + d_xt0.numel() + d_ut0.numel()) * 8 + mode.size * 4
    if cfg == 1:
        # e2e_plan_cycle: hb_resident_plan_cycle_batch -- plan inputs (t0, x0, cmd_vel, gait; 352 B per instance) and rbd in; foot positions, the
        # reference planner (gait tiling, swing planner, IK joint references), expansion, cold start, solve, WBC all on the device.
        ins = hb.make_plan_inputs(np.zeros(B), HORIZON_N * DT, x0, (0.2, 0.0, 0.0, 0.0), None, "trot", 0.1)
        plan_bytes = C.sizeof(ins)
        h_ins = torch.empty(plan_bytes, dtype=torch.uint8).pin_memory()
        C.memmove(h_ins.data_ptr(), C.addressof(ins), plan_bytes)
        h_ps = torch.zeros(B, dtype=torch.int32).pin_memory()

        def step_plan():
            rc = lib.hb_resident_plan_cycle_batch(ctx._h, B, 1, C.c_double(T_POLICY), P(h_ins), P(h_rbd), P(h_info), P(h_sol), P(h_tau), P(h_st), P(h_ps))
            assert rc == 0, rc

        for _ in range(2):
            step_plan()
        barrier()
        plan_ok = bool((h_ps.numpy() == 0).all() and (h_st.numpy() == 0).all())
        t0 = time.perf_counter()
        for _ in range(args.steps):
            step_plan()
        barrier()
        plan_s = time.perf_counter() - t0
        plan_h2d = plan_bytes + h_rbd.numel() * 8
        plan_d2h = (h_info.numel() + h_sol.numel() + h_tau.numel()) * 8 + h_st.numel() * 4 + h_ps.numel() * 4
        # every full-trajectory step gets its own pre-initialised in/out trajectory buffers (cold start): no host-side reset in the timed region
        h_xref, h_swing, h_mode = pin(x_ref), pin(swing), pin(mode)
        n_e2e = args.steps + 2
        h_xts = [d_xt0.cpu().pin_memory() for _ in range(n_e2e)]; h_uts = [d_ut0.cpu().pin_memory() for _ in range(n_e2e)]
        h_xt, h_ut = h_xts[0], h_uts[0]
        e2e_i = [0]

        def step_e2e_full():
            xt_, ut_ = h_xts[e2e_i[0]], h_uts[e2e_i[0]]
            e2e_i[0] += 1
            rc = lib.hb_control_step_batch(ctx._h, B, C.c_double(T_POLICY), P(h_x0), P(h_xref), P(h_swing), P(h_mode), P(h_rbd), P(xt_), P(ut_), P(h_info),
                                           P(h_sol), P(h_tau), P(h_st))
            assert rc == 0, rc

        for _ in range(2):
            step_e2e_full()
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            step_e2e_full()
        barrier()
        full_s = time.perf_counter() - t0
        full_d2h = (h_xt.numel() + h_ut.numel() + h_info.numel() + h_sol.numel() + h_tau.numel()) * 8 + h_st.numel() * 4
    clocks = sampler.stop() if rank == 0 else None
    # ---------------- max over ranks
    if world > 1:
        t = torch.tensor([ms, e2e_s * 1e3, full_s * 1e3, plan_s * 1e3], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms, e2e_ms, full_ms, plan_ms = float(t[0]), float(t[1]), float(t[2]), float(t[3])
    else:
        e2e_ms, full_ms, plan_ms = e2e_s * 1e3, full_s * 1e3, plan_s * 1e3
    ok = bool((d_st == 0).all().item())
    accepted = float((d_info[:, 0] > 0).double().mean().item())
    if rank == 0:
        peaks, src = load_peaks()
        value = total_B * args.steps / (ms * 1e-3)
        e2e_val = total_B * args.steps / (e2e_ms * 1e-3)
        mpc_names = [n for n in prof if n.startswith("mpc_")]
        top = max(mpc_names, key=lambda n: prof[n]["ms"])     # dominant kernel of the step
        bk = prof[top]
        bk_ms = bk["ms"] / max(1, bk["launches"])
        ach = B * BYTES_PER_MPC_SOLVE / (bk_ms * 1e-3) / 1e9 if bk_ms > 0 else None
        step_ms = ms / args.steps
        traffic = None
        try:   # dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed ncu --set full capture (same workload, 1024 instances)
            tj = None
            for name in ("r02_traffic.json", "r01_traffic.json"):
                pth = os.path.join(ROOT, "profiles", name)
                if os.path.exists(pth):
                    tj = json.load(open(pth)); break
            traffic = tj[KERNEL_OF[top]]["dram_bytes"] * B / tj[KERNEL_OF[top]]["instances"]
        except Exception:
            pass
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": step_ms,
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                "config": {"workload": workload_desc(cfg, B) + ", one SQP iteration from the initializer cold start + policy eval at 2 ms + WeightedWbc QP",
                           "instances_total": total_B,
                           "parallelism": ("instances sharded in contiguous blocks, NCCL all-gather of torques on a side stream (%s)" % ("hb_shard_gather_dev, C ABI" if shard is not None else "torch.distributed")) if world > 1 else "single GPU",
                           "l2": "per-step working set (node records %.0f MB + references/trajectories %.0f MB) exceeds the 126 MB L2" % (B * HORIZON_N * (1200 + 2320 + 368) * 8 / 1e6, full_h2d / 1e6)},
                "e2e": {"value": e2e_val, "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h), "ms_per_step": e2e_ms / args.steps,
                        "call": "hb_resident_cycle_batch(cold_start=1): t0, x0, compact references (packed: %d of %d bytes), rbd in; info, WBC solution, torques, status out" % (ref_up, ref_bytes),
                        "torque_max_rel_diff_vs_device_path": e2e_tau_diff},
                "gpu_launches": int(launches),
                "kernel_ms_per_step": {k: v["ms"] / args.steps for k, v in prof.items()},
                "roofline": {"bound": "hbm", "kernel": top, "achieved": ach, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                             "frac": (ach / peaks["hbm_gbs"]) if ach else None, "peak_source": src, "traffic": traffic,
                             "share_of_step": bk_ms / step_ms if step_ms > 0 else None,
                             "note": "latency/FP64-bound path: the HBM fraction is small by construction (SURVEY 8d); see roofline_fp64"},
                "roofline_fp64": {"achieved_tflops": value / world * FLOPS_PER_SOLVE / 1e12, "peak_tflops_nominal": FP64_NOMINAL_TFLOPS,
                                  "frac": value / world * FLOPS_PER_SOLVE / 1e12 / FP64_NOMINAL_TFLOPS},
                "clocks": clocks, "all_converged": ok, "line_search_accepted_fraction": accepted}
        if cfg == 1:
            line["e2e_plan_cycle"] = {"value": total_B * args.steps / (plan_ms * 1e-3), "unit": UNIT, "h2d_bytes_per_step": int(plan_h2d), "d2h_bytes_per_step": int(plan_d2h),
                                      "ms_per_step": plan_ms / args.steps, "all_planned_and_solved": plan_ok,
                                      "call": "hb_resident_plan_cycle_batch(cold_start=1): plan inputs + rbd in; reference planner (P1, P3, P4, P5) on the device; same gait / command as the workload"}
            line["e2e_full_trajectories"] = {"value": total_B * args.steps / (full_ms * 1e-3), "unit": UNIT, "h2d_bytes_per_step": int(full_h2d),
                                             "d2h_bytes_per_step": int(full_d2h), "ms_per_step": full_ms / args.steps,
                                             "call": "hb_control_step_batch: node-sampled references and full trajectories both ways"}
        if world > 1:
            line["gather"] = {"rows_at_rank0": total_B, "finite": gather_ok, "unpermuted_before_gather": cfg == 3}
        if cfg == 3:
            line["config"]["schedule_mix"] = {g: int(sum(1 for i in range(lo, hi) if i % 4 == k)) for k, g in enumerate(GAIT_NAMES)}
        if not args.no_cpu_baseline and world == 1:     # reported on rank 0 at N = 1 only
            cores = os.cpu_count() or 1
            n = max(cores, 4)
            data = [d[:n] for d in (x0, x_ref, swing, mode, rbd)]
            t_all, tau_cpu = cpu_control_steps(*data, threads=cores)
            t_one, _ = cpu_control_steps(*[d[:2] for d in data], threads=1)
            err = float(np.abs(tau_cpu - d_tau[:n].cpu().numpy()).max() / max(1.0, np.abs(tau_cpu).max()))
            line["cpu_baseline"] = {"value": n / t_all, "unit": UNIT, "cores": cores, "kind": "port", "host_parallelism": host_parallelism(),
                                    "sample": "%d control steps of the same workload, all host threads; single-thread %.2f solves/s" % (n, 2 / t_one),
                                    "single_thread_value": 2 / t_one, "torque_rel_err_vs_gpu": err}
        print(json.dumps(line))
    if shard is not None:
        shard.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
