#!/usr/bin/env python
"""bench.py — CUP2D hot path on B200: Mcell-updates/s (advect+diffuse+Poisson iter) at 8192^2.

One "step" = one full time step of the hot path on a uniform grid without bodies:
    dt control (umax reduction) -> RK2 (two fused WENO5 advect-diffuse stages) -> Poisson RHS ->
    K BiCGSTAB iterations (K fixed, tolerance 0, like the reference's first 10 steps with its
    hard-coded cap, main.cpp:7028-7030 / cuda.cu:438) -> pressure correction.
cell-updates per step = cells * (2 stage sweeps + K Poisson iterations)   [the metric's own definition]

    python bench.py [--gpus N] [--steps K] [--warmup W] [--level L] [--poisson-iters K] [--impl reference]
                    [--dump-outputs DIR]

--dump-outputs DIR writes what the last timed step handed back (u, v, p and the step's dt, iterations, residual) as .npy
files, so that two builds run with the same arguments (hence the same seeded inputs) can be compared output for output.

N > 1: launched by torchrun, one rank per GPU; the 8192^2 grid is split into contiguous Hilbert ranges
(strong scaling); halos and Krylov dots go over NVLink peer memory inside the library's kernels.
`--impl reference` times the reference's own CPU code (oracle/_ref/ref_harness: unmodified main.cpp
operators under OpenMP on all host cores; its GPU-only Poisson solver is replaced by the CPU restatement
of cuda.cu) on a bounded sample of the same workload.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

HARNESS = os.path.join(ROOT, "oracle", "_ref", "ref_harness")          # main.cpp + CPU restatement of cuda.cu
HARNESS_GPU = os.path.join(ROOT, "oracle", "_ref", "ref_harness_gpu")  # main.cpp + the reference's own cuda.cu

# algorithmic bytes per cell per launch (DESIGN.md "Kernels"; SURVEY.md §8(d))
ALG_BYTES = {
    "advect_stage_kernel": 48.0,      # read V_in 16 + read V_old 16 + write V_out 16 (stage 1 aliases in/old: 32)
    "umax_kernel": 16.0,
    "pressure_rhs_kernel": 40.0,      # no bodies: vel 16 + pold 8 read; tmp 8 + pres 8 written (+ udef 16 + chi 8 with bodies)
    "pressure_correct_kernel": 56.0,  # x 8 + pold 8 + vel 16 read; pres 8 + vel 16 written
    "k_init": 56.0,                   # b, x0 read; x, r, rhat, p, nu written
    "k_pupdate": 40.0,                # r, p, nu read; p, z written
    "k_spmv<0>": 24.0,                # z, rhat read; nu written
    "k_r_update": 32.0,               # r, nu read; r, z_r written (the x half-step is deferred to k_final)
    "k_spmv<1>": 24.0,                # z, r read; t written
    "k_final": 64.0,                  # x, z_p, z_r, r, t, rhat read; x, r written
}


def load_traffic():
    """measured DRAM bytes per cell per launch of each kernel (ncu --set full, profiles/traffic.json)"""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    return json.load(open(p)) if os.path.exists(p) else {}


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks/throttle reasons sampled while the timed region runs."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.rows = []
        self.proc = None
        self.idx = gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.idx), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def gpu_visible():
    try:
        return subprocess.run(["nvidia-smi", "-L"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL).returncode == 0
    except Exception:
        return False


def usable_cpus():
    """host threads this process may really use: scheduler affinity, capped by the cgroup CPU quota (a 1-GPU lease on
    a 128-core box is typically given a slice; os.cpu_count() ignores both and oversubscribes OpenMP)"""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()
        if quota != "max":
            n = max(1, min(n, int(float(quota) / float(period) + 0.5)))
    except Exception:
        pass
    return max(1, n)


def run_harness_time(binary, level, reps, kiter, threads, timeout=None):
    env = dict(os.environ, OMP_NUM_THREADS=str(threads), OMP_PROC_BIND="false", OMP_WAIT_POLICY="active")
    out = subprocess.run([binary, "time", str(level), str(reps), str(kiter)], env=env, check=True,
                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, timeout=timeout).stdout
    return json.loads(out.strip().splitlines()[-1])


def _composite(t, kiter, which=None):
    """cells*(2+K) / (2 t_stage + t_rhs + K t_iter + t_correct) in Mcell-updates/s; which = 0/1/2 picks min/median/max times"""
    g = (lambda k: t[k]) if which is None else (lambda k: t["min_med_max"][k][which])
    step_s = 2 * g("t_stage") + g("t_rhs") + kiter * g("t_poisson_iter") + g("t_correct")
    return t["cells"] * (2 + kiter) / step_s / 1e6, step_s


def cpu_composite(level, reps, kiter):
    """The reference's own path on a bounded sample.  Operators = unmodified main.cpp under OpenMP on the host threads this
    process may use.  The reference has no CPU Poisson solver (cuda.cu is its only one), so `value` always uses the CPU
    restatement of cuda.cu for the Poisson iterations (one fixed definition: the figure never switches solver), and the
    composite with the reference's own GPU solver on this box's B200 is reported beside it as `with_reference_gpu_solver`."""
    threads = usable_cpus()
    run_harness_time(HARNESS, 3, 1, 1, threads, timeout=120)           # warm: binary and OpenMP runtime paged in
    t = run_harness_time(HARNESS, level, reps, kiter, threads, timeout=900)
    val, step_s = _composite(t, kiter)
    N = t["N"]
    spread = {"min": _composite(t, kiter, 2)[0], "median": _composite(t, kiter, 1)[0], "max": _composite(t, kiter, 0)[0]}
    out = {
        "value": val, "unit": "Mcell-updates/s", "cores": t["threads"], "kind": "reference",
        "sample": f"{N}x{N} uniform grid (L={level}), Taylor-Green, median of {t.get('reps', reps)} reps per operator after one warm-up; "
                  f"operators = unmodified reference main.cpp under OpenMP on {t['threads']} threads (affinity/cgroup-limited); "
                  f"Poisson iteration = CPU restatement of cuda.cu (the reference has no CPU solver); "
                  f"composite = 2 stages + RHS + {kiter} iterations + correction",
        "sample_cells": t["cells"], "ms_per_step": step_s * 1e3, "value_min_median_max": spread,
        "stage_Mcells_s": t["cells"] / t["t_stage"] / 1e6,
        "poisson_iter_Mcells_s": t["cells"] / t["t_poisson_iter"] / 1e6 if t["t_poisson_iter"] > 0 else None,
        "poisson_solver": "cpu_restatement",
        "operator_seconds_min_med_max": t.get("min_med_max"),
    }
    # named extra: the same composite with the reference's own cuda.cu (cuSPARSE/cuBLAS) iterating on the B200
    extra = {"unavailable": "no GPU visible or reference GPU binary not built"}
    if os.path.exists(HARNESS_GPU) and gpu_visible():
        try:
            run_harness_time(HARNESS_GPU, 3, 1, 1, threads, timeout=600)   # warm: first load of cuBLAS/cuSPARSE can take minutes on a fresh box
            tg = run_harness_time(HARNESS_GPU, level, reps, kiter, threads, timeout=900)
            vg, sg = _composite(tg, kiter)
            extra = {"value": vg, "unit": "Mcell-updates/s", "ms_per_step": sg * 1e3,
                     "poisson_iter_Mcells_s": tg["cells"] / tg["t_poisson_iter"] / 1e6,
                     "value_min_median_max": {"min": _composite(tg, kiter, 2)[0], "median": _composite(tg, kiter, 1)[0],
                                              "max": _composite(tg, kiter, 0)[0]},
                     "poisson_solver": "reference cuda.cu on 1 B200 (host<->device copies of x,b per solve included, as the reference does)"}
        except Exception as e:
            extra = {"unavailable": f"{type(e).__name__}: {e}"[:200]}
    out["with_reference_gpu_solver"] = extra
    return out


def multi_gpu_parity(cup2d_b200, np, torch, dist, rank, world, local_rank, K):
    """Before anything is timed: 256^2, 2 steps with dt control and K Krylov iterations each, on the SAME ranks that are
    about to be timed (peer-memory halo pulls, pushed Krylov halos, in-kernel all-reduce, CUDA-graph replay), against
    the same steps on ONE GPU (rank 0, same library; that path is pinned to the reference's goldens and to the oracle by
    tests/test_gpu_parity.py, which the driver runs on the same box).  L-inf over the whole field; > 1e-9 fails the run."""
    L = 5
    N = 8 << L
    x = (np.arange(N) + 0.5) / N
    X, Y = np.meshgrid(x, x)
    rng = np.random.default_rng(5)
    u = np.sin(2 * np.pi * X) * np.cos(2 * np.pi * Y) + 0.05 * rng.uniform(-1, 1, (N, N))
    v = -np.cos(2 * np.pi * X) * np.sin(2 * np.pi * Y) + 0.05 * rng.uniform(-1, 1, (N, N))
    p = np.cos(2 * np.pi * X) * np.cos(2 * np.pi * Y)

    def run(sim, nsteps=3):
        sim.upload("vel", u, v)
        sim.upload("pres", p)
        info = []
        for _ in range(nsteps):      # step 1 is launched kernel by kernel, steps 2 and 3 build and replay the two step graphs
            sim.step_enqueue(max_iter=K, max_restarts=0)
            info.append(sim.step_result())
        return info

    sim = cup2d_b200.Simulation(L, nu=1e-3, cfl=0.5, device=local_rank, rank=rank, nranks=world)
    sim.attach_peers(dist)
    info = run(sim)
    parts_v, parts_p = [None] * world, [None] * world
    dist.all_gather_object(parts_v, sim.download_blocks("vel"))
    dist.all_gather_object(parts_p, sim.download_blocks("pres"))
    nhalo = int(sim.lib.cup2d_nblocks_halo(sim._h))
    order, nbx, nby = sim.order, sim.nbx, sim.nby
    sim.close()
    out = [None]
    if rank == 0:
        one = cup2d_b200.Simulation(L, nu=1e-3, cfl=0.5, device=local_rank)
        info1 = run(one)
        ru, rv = one.download("vel")
        rp = one.download("pres")
        one.close()
        gu, gv = cup2d_b200.from_blocks(np.concatenate(parts_v), order, nbx, nby, 2)
        gp = cup2d_b200.from_blocks(np.concatenate(parts_p), order, nbx, nby, 1)
        out[0] = {"Linf_u": float(np.abs(gu - ru).max()), "Linf_v": float(np.abs(gv - rv).max()),
                  "Linf_p": float(np.abs(gp - rp).max()), "dt_rel": float(max(abs(a[0] - b[0]) / b[0] for a, b in zip(info, info1))),
                  "ranks": world, "grid": f"{N}x{N}", "steps": len(info), "poisson_iters": K, "halo_blocks_rank0": nhalo,
                  "against": "the same steps on one GPU through the same C ABI (single-GPU path pinned to the reference goldens "
                             "and the oracle by tests/test_gpu_parity.py); tools/multi_gpu_check.py compares with the oracle directly",
                  "tolerance": 1e-9}
    dist.broadcast_object_list(out, src=0)
    return out[0]


DUMP_CELLS = 1 << 20   # at most this many cells per field in --dump-outputs; larger grids are sampled (u, v, p, index: <= 32 MB)


def dump_outputs(path, np, dist, rank, order_loc, nbx, vel, pres, result):
    """Write u.npy, v.npy, p.npy (float64) at the cells of cell_index.npy (flat index iy*N+ix of the global grid: every cell,
    or the distinct cells among DUMP_CELLS fixed seeded draws) and step.npy = [dt, iterations, residual] of the last step.
    vel, pres: this rank's blocks in the reference layout; every rank calls this, rank 0 writes."""
    N = nbx * 8
    cells = N * N
    idx = np.arange(cells) if cells <= DUMP_CELLS else np.unique(np.random.default_rng(0).integers(0, cells, DUMP_CELLS))
    gy, gx = np.divmod(idx, N)
    where = np.full((nbx, nbx), -1, dtype=np.int64)   # global block (j, i) -> local block, -1 on other ranks
    where[order_loc[:, 1], order_loc[:, 0]] = np.arange(len(order_loc))
    b = where[gy // 8, gx // 8]
    mine = np.flatnonzero(b >= 0)
    cell = (b[mine] * 8 + gy[mine] % 8) * 8 + gx[mine] % 8
    uv = vel.reshape(-1, 2)[cell]
    parts = [(mine, uv[:, 0], uv[:, 1], pres[cell])]
    if dist is not None:
        gathered = [None] * dist.get_world_size()
        dist.all_gather_object(gathered, parts[0])
        parts = gathered
    if rank != 0:
        return
    out = {k: np.full(len(idx), np.nan) for k in ("u", "v", "p")}
    for pos, u, v, p in parts:
        out["u"][pos], out["v"][pos], out["p"][pos] = u, v, p
    if cells <= DUMP_CELLS:
        out = {k: a.reshape(N, N) for k, a in out.items()}
    out["cell_index"] = idx.astype(np.float64)
    out["step"] = np.array(result, dtype=np.float64)
    os.makedirs(path, exist_ok=True)
    for k, a in out.items():
        np.save(os.path.join(path, k + ".npy"), a)


# FP64 instructions the advect stage executes per cell (DFMA + DMUL + DADD of the ncu instruction mix; round 1: 189)
ADVECT_FP64_PER_CELL = 152.4


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=4)
    ap.add_argument("--level", type=int, default=10, help="uniform level: grid = (8*2^L)^2; 10 = 8192^2")
    ap.add_argument("--poisson-iters", type=int, default=10)
    ap.add_argument("--impl", default="cup2d_b200", choices=["cup2d_b200", "reference"])
    ap.add_argument("--cpu-level", type=int, default=9, help="grid level of the bounded CPU sample (9 = 4096^2, SURVEY 8(d))")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-pipeline", action="store_true", help="skip the pipelined end-to-end figure")
    ap.add_argument("--no-graph", action="store_true", help="launch every kernel from the host instead of replaying the step graph")
    ap.add_argument("--profile-steps", type=int, default=5, help="steps of the separate, event-instrumented pass (per-kernel table)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the fields and result of the last timed step to DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to the cup2d_b200 arm only")

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    K = args.poisson_iters
    L = args.level
    N = 8 << L
    cells = N * N
    warmup = max(4, args.warmup)   # step 1 runs kernel by kernel, steps 2 and 3 capture the two step graphs, step 4 replays
    config = {"workload": f"{N}x{N} uniform block grid (level {L}, {(1 << L) ** 2} blocks of 8x8, Hilbert order), "
                          f"Taylor-Green + seeded perturbation, nu=1e-4, CFL=0.5, free-slip box, no bodies",
              "step": f"dt control (umax reduction + dt rule, on the device) + RK2 WENO5 advect-diffuse + Poisson RHS + {K} BiCGSTAB "
                      f"iterations (tol 0) + pressure correction; one CUDA-graph launch per step, no host synchronisation inside the timed region",
              "cell_updates_per_step": f"cells*(2+{K})", "poisson_iters": K,
              "partition": f"{world} contiguous Hilbert range(s), halo + dots over NVLink peer memory" if world > 1 else "single GPU",
              "cache": "inputs larger than L2 (each field >= 0.5 GB vs 126 MB L2)" if L >= 9 else "L2-resident at this size"}

    if args.impl == "reference":
        if rank != 0:
            return
        try:
            cb = cpu_composite(args.cpu_level, args.steps, K)
        except Exception as ex:  # the reference harness could not be run on this box
            print(json.dumps({"impl": "reference", "unavailable": f"reference harness failed: {type(ex).__name__}: {ex}"[:300]}))
            return
        Ns = 8 << args.cpu_level
        rconfig = dict(config)
        rconfig["workload"] = (f"SAMPLE {Ns}x{Ns} uniform block grid (level {args.cpu_level}) of the {N}x{N} workload: same fields, same "
                               f"operators, same composite; CPU throughput per cell is size-independent at this size (memory-bound, "
                               f"working set >> last-level cache)")
        rconfig["step"] = (f"2 RK stages (computeA<KernelAdvectDiffuse> + update) + pressure_rhs + pressure_rhs1 + {K} BiCGSTAB "
                           f"iterations + pressure correction, each operator timed separately (median of {args.steps} reps) and composed")
        line = {"impl": "reference", "metric": "Mcell-updates/s (advect+diffuse+Poisson iter)", "value": cb["value"],
                "unit": "Mcell-updates/s", "n_gpus": 0, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": cb["ms_per_step"], "higher_is_better": True, "scaling": "strong",
                "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": rconfig,
                "cpu_baseline": cb,
                "e2e": {"value": cb["value"], "unit": "Mcell-updates/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line))
        return

    import numpy as np
    import torch
    import cup2d_b200

    if not torch.cuda.is_available():
        sys.exit("bench.py: no CUDA device; cup2d_b200 has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dist = None
    parity = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        parity = multi_gpu_parity(cup2d_b200, np, torch, dist, rank, world, local_rank, K)
        if max(parity["Linf_u"], parity["Linf_v"], parity["Linf_p"]) > parity["tolerance"] or not (parity["dt_rel"] < 1e-12):
            if rank == 0:
                print(json.dumps({"error": "multi-GPU parity check failed; nothing timed", "parity": parity}))
            dist.barrier()
            dist.destroy_process_group()
            sys.exit(3)

    # ---- synthetic input (host, reference block layout) -------------------------------------------
    sim = cup2d_b200.Simulation(L, nu=1e-4, cfl=0.5, device=local_rank, rank=rank, nranks=world)
    if world > 1:
        sim.attach_peers(dist)
    if args.no_graph:
        sim.set_graph(False)
    order = sim.local_order
    bi = order[:, 0].astype(np.float64)[:, None, None]
    bj = order[:, 1].astype(np.float64)[:, None, None]
    ix = np.arange(8, dtype=np.float64)[None, None, :]
    iy = np.arange(8, dtype=np.float64)[None, :, None]
    X = (bi * 8 + ix + 0.5) / N
    Y = (bj * 8 + iy + 0.5) / N
    rng = np.random.default_rng(1234 + rank)
    nloc = len(order)
    vel_h = torch.empty(nloc * 128, dtype=torch.float64).pin_memory()
    pres_h = torch.empty(nloc * 64, dtype=torch.float64).pin_memory()
    v = vel_h.numpy().reshape(nloc, 8, 8, 2)
    v[..., 0] = np.sin(2 * np.pi * X) * np.cos(2 * np.pi * Y) + 0.01 * rng.uniform(-1, 1, (nloc, 8, 8))
    v[..., 1] = -np.cos(2 * np.pi * X) * np.sin(2 * np.pi * Y) + 0.01 * rng.uniform(-1, 1, (nloc, 8, 8))
    pres_h.numpy().reshape(nloc, 8, 8)[:] = 0.0
    vel_out = torch.empty_like(vel_h).pin_memory()
    pres_out = torch.empty_like(pres_h).pin_memory()
    del X, Y

    lib = sim.lib
    from cup2d_b200 import lib as _l
    H = sim._h
    stream = torch.cuda.ExternalStream(sim.stream, device=torch.device("cuda", local_rank))

    def upload():
        _l.check(lib.cup2d_field_upload(H, 0, vel_h.data_ptr()))
        _l.check(lib.cup2d_field_upload(H, 4, pres_h.data_ptr()))

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def allmax(x):
        if dist is None:
            return x
        t = torch.tensor([x], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def enqueue():   # one full step incl. dt control; returns at once (a single cudaGraphLaunch from the second step on)
        sim.step_enqueue(dt=0.0, max_iter=K, max_restarts=0)

    # ---- device-resident timing (`value`): profiling OFF, nothing but step launches inside the timed region ----
    upload()
    sim.sync()
    for _ in range(warmup):
        enqueue()
    dt0, it0, _ = sim.step_result()
    assert it0 == K
    barrier()
    l0 = sim.launch_count()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(args.steps):
        enqueue()
    e1.record(stream)
    barrier()
    ms = allmax(e0.elapsed_time(e1))
    clocks = sampler.stop() if rank == 0 else None
    launches = sim.launch_count() - l0
    dt_last, it_last, err_last = sim.step_result()
    if args.dump_outputs:
        _l.check(lib.cup2d_field_download(H, 0, vel_out.data_ptr()))
        _l.check(lib.cup2d_field_download(H, 4, pres_out.data_ptr()))
        dump_outputs(args.dump_outputs, np, dist, rank, order, sim.nbx, vel_out.numpy(), pres_out.numpy(),
                     (dt_last, it_last, err_last))
    ms_per_step = ms / args.steps
    value = cells * (2 + K) / (ms_per_step * 1e-3) / 1e6

    # ---- separate pass for the per-kernel table: same steps launched kernel by kernel, each bracketed by (pooled) events ----
    sim.profile(True)
    for _ in range(2):
        enqueue()       # fills the event pool, so that no event is created inside the measured steps
    sim.sync()
    sim.profile(True)   # drop the records of the two pool-filling steps
    barrier()
    ep0, ep1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ep0.record(stream)
    for _ in range(args.profile_steps):
        enqueue()
    ep1.record(stream)
    barrier()
    ms_prof_step = allmax(ep0.elapsed_time(ep1)) / args.profile_steps
    prof = sim.profile_read()
    sim.profile(False)
    sim.step_result()

    # ---- end-to-end through the C ABI with host buffers (`e2e`): upload, step, download in sequence, every step ----------
    e2e = None
    if not args.no_e2e:
        def e2e_step():
            upload()                                   # H2D from pinned memory: vel + pres
            sim.step(dt=0.0, max_iter=K, max_restarts=0)   # full step incl. dt control; waits for the result (dt, iterations, residual)
            _l.check(lib.cup2d_field_download(H, 0, vel_out.data_ptr()))   # D2H (synchronises the stream)
            _l.check(lib.cup2d_field_download(H, 4, pres_out.data_ptr()))
        for _ in range(3):
            e2e_step()
        barrier()
        t0 = time.perf_counter()
        e0.record(stream)
        for _ in range(args.steps):
            e2e_step()
        e1.record(stream)
        barrier()
        ms_e = allmax(e0.elapsed_time(e1)) / args.steps
        wall = (time.perf_counter() - t0) * 1e3
        e2e = {"value": cells * (2 + K) / (ms_e * 1e-3) / 1e6, "unit": "Mcell-updates/s",
               "h2d_bytes_per_step": int((vel_h.numel() + pres_h.numel()) * 8 * world),
               "d2h_bytes_per_step": int((vel_out.numel() + pres_out.numel()) * 8 * world),
               "ms_per_step": ms_e, "wall_ms_per_step": wall / args.steps, "mode": "blocking",
               "note": "every step: pinned-host vel+pres -> device, one full step (dt control included, result read back), "
                       "vel+pres -> pinned host, strictly in sequence: what a time-marching caller with host-resident fields gets"}

    # ---- the same work through the host-buffer pipeline (cup2d_pipe_*): upload(n+1) || step(n) || download(n-1).  Only
    # INDEPENDENT jobs can overlap like this (a time loop's step n+1 needs step n's result), so this is reported beside the
    # blocking figure, never instead of it.  Single rank only: the peer mappings of a multi-rank context are tied to its field buffers.
    if e2e is not None and world == 1 and not args.no_pipeline:
        try:
            outs = [(torch.empty_like(vel_h).pin_memory(), torch.empty_like(pres_h).pin_memory()) for _ in range(2)]
            njobs = args.steps

            def batch(n):
                return sim.pipelined_steps(((vel_h.data_ptr(), pres_h.data_ptr(), outs[j % 2][0].data_ptr(), outs[j % 2][1].data_ptr())
                                            for j in range(n)), dt=0.0, max_iter=K, max_restarts=0)
            batch(3)
            barrier()
            t0 = time.perf_counter()
            e0.record(stream)
            batch(njobs)
            e1.record(stream)           # every download has landed (pipe_wait), so this stamps the end of the batch
            barrier()
            ms_p = e0.elapsed_time(e1) / njobs
            wall_p = (time.perf_counter() - t0) * 1e3 / njobs
            same = all(torch.equal(o[0], vel_out) and torch.equal(o[1], pres_out) for o in outs)
            if same and ms_p > 0:
                e2e["pipelined"] = {"value": cells * (2 + K) / (ms_p * 1e-3) / 1e6, "ms_per_step": ms_p, "wall_ms_per_step": wall_p,
                                    "jobs": njobs, "verified_bit_identical_to_blocking_calls": True,
                                    "note": "independent jobs only: the three legs of successive jobs overlap on three streams "
                                            "(cup2d_pipe_*); pipeline fill and drain included"}
            else:
                e2e["pipelined"] = {"error": "pipelined results differ from the blocking calls; figure not reported"}
            del outs
        except Exception as ex:
            e2e["pipelined"] = {"error": repr(ex)[:300]}
    elif e2e is not None and world > 1:
        e2e["pipelined"] = {"unavailable": "multi-rank contexts export their field buffers to the peers (CUDA IPC); the pipeline "
                                           "trades buffers with the context, which would invalidate those mappings"}

    # ---- per-kernel roofline from the CUDA events of the instrumented pass ------------------------------
    peak, peak_src = load_peaks()
    cells_loc = nloc * 64
    kernels = []
    ksum = 0.0
    for name, (tot_ms, n) in prof.items():
        per = tot_ms / n
        ab = ALG_BYTES.get(name)
        gbs = cells_loc * ab / (per * 1e-3) / 1e9 if ab else None
        per_step = tot_ms / args.profile_steps
        ksum += per_step
        kernels.append({"kernel": name, "launches_per_step": n / args.profile_steps, "ms_per_launch": per,
                        "share_of_step": per_step / ms_per_step,
                        "alg_bytes_per_cell": ab, "achieved_GBs": gbs, "frac_hbm": gbs / peak if gbs else None})
    kernels.sort(key=lambda k: -k["share_of_step"])
    adv = next((k for k in kernels if k["kernel"] == "advect_stage_kernel"), None)
    top = kernels[0] if kernels else None
    roofline = None
    if top:
        tr = load_traffic().get(top["kernel"])
        roofline = {"kernel": top["kernel"], "bound": "hbm", "achieved": top["achieved_GBs"], "peak": peak,
                    "unit": "GB/s", "frac": top["frac_hbm"],
                    "traffic": tr * cells_loc if tr else None, "traffic_unit": "bytes per launch (ncu dram read+write, profiles/)",
                    "peak_source": peak_src,
                    "ms_per_launch": top["ms_per_launch"], "share_of_step": top["share_of_step"],
                    "timed": "CUDA events around every launch in a separate instrumented pass of the same steps (kernel-by-kernel launches)"}
    extra = {"timing_passes": {"value_pass_ms_per_step": ms_per_step, "instrumented_pass_ms_per_step": ms_prof_step,
                               "sum_of_kernel_ms_per_step": ksum, "outside_kernels_frac_of_value_pass": max(0.0, 1.0 - ksum / ms_per_step),
                               "note": "`value` comes from the pass with instrumentation off (one graph launch per step); the kernel table "
                                       "from the instrumented pass"}}
    if adv:
        # the north-star kernel: HBM fraction and the FP64-pipe bound it actually sits under
        gcell = cells_loc / (adv["ms_per_launch"] * 1e-3) / 1e9
        sm_mhz = (clocks or {}).get("sm_mhz") or 1920.0
        fp64_floor_ms = cells_loc * ADVECT_FP64_PER_CELL / 32.0 / (148 * 2 * sm_mhz * 1e6) * 1e3   # 2 FP64 warp-instr/clk/SM
        extra["advect_stage"] = {"Gcell_per_s": gcell, "achieved_GBs": adv["achieved_GBs"], "frac_hbm": adv["frac_hbm"],
                                 "ms_per_launch": adv["ms_per_launch"], "alg_bytes_per_cell": 48.0,
                                 "fp64_floor_ms": fp64_floor_ms, "frac_fp64_floor": fp64_floor_ms / adv["ms_per_launch"],
                                 "note": f"bound by the FP64 pipe, not HBM: {ADVECT_FP64_PER_CELL:g} FP64 instr/cell (ncu, profiles/r02g_advect_ncu.md) at 64 lanes/clk/SM; see DESIGN.md 3.1"}
        # SURVEY 8(d)(ii): one full RK2 step = the two fused stages (vold = vel is a pointer swap, not a copy)
        try:
            rk2_ms = adv["ms_per_launch"] * adv["launches_per_step"]
            extra["rk2_step"] = {"ms": rk2_ms, "Gcell_steps_per_s": cells_loc / (rk2_ms * 1e-3) / 1e9,
                                 "alg_bytes_per_cell": 80.0, "frac_hbm": cells_loc * 80.0 / (rk2_ms * 1e-3) / 1e9 / peak}
        except Exception:  # a derived figure must never cost the bench line
            pass
    it_ms = sum(k["ms_per_launch"] * k["launches_per_step"] for k in kernels
                if k["kernel"] in ("k_pupdate", "k_spmv<0>", "k_r_update", "k_spmv<1>", "k_final")) / max(K, 1)
    if it_ms > 0:
        gbs = cells_loc * 184.0 / (it_ms * 1e-3) / 1e9
        extra["poisson_iteration"] = {"ms_per_iteration": it_ms, "Gcell_iter_per_s": cells_loc / (it_ms * 1e-3) / 1e9,
                                      "alg_bytes_per_cell": 184.0, "achieved_GBs": gbs, "frac_hbm": gbs / peak,
                                      "note": "23 doubles/cell/iteration (SURVEY 8(d) budgets 25 = 200 B): the x half-step "
                                              "is deferred into k_final; with several ranks the halo rows of z are pushed by the producing "
                                              "kernel (no halo kernel in the loop)"}

    if rank != 0:
        if dist is not None:
            dist.barrier()
            dist.destroy_process_group()
        return

    cpu = None
    if world == 1 and not args.no_cpu_baseline and os.path.exists(HARNESS):
        try:
            cpu = cpu_composite(args.cpu_level, 5, K)
        except Exception as ex:  # the baseline is a reported figure, not a gate
            cpu = {"error": str(ex)}

    line = {"metric": "Mcell-updates/s (advect+diffuse+Poisson iter)", "value": value, "unit": "Mcell-updates/s",
            "n_gpus": world, "steps": args.steps, "warmup": warmup, "ms_per_step": ms_per_step,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": config, "e2e": e2e, "gpu_launches": int(launches), "clocks": clocks,
            "roofline": roofline, "kernels": kernels, "cpu_baseline": cpu, "dt": dt_last, "poisson_residual": err_last,
            "graph": not args.no_graph}
    if parity is not None:
        line["parity"] = parity
    line.update(extra)
    print(json.dumps(line))
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
