#!/usr/bin/env python
"""Benchmark of the batched MPC hot path (estimator -> target -> OCP -> input extraction).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K ...   # CPU arm: the oracle port on all host cores

Workload at N=1 (BASELINE.json configs[1]): Ex_NMPC - nonlinear CSTR NMPC with EKF, horizon 50, Mx=10,
batch 4 096 instances with perturbed initial states (SURVEY.md 8(d) C2).  With N>1 every rank runs its
own 4 096 instances (weak scaling, no data-path collective); NCCL only gathers the closed-loop inputs and
solver statistics after the timed region.  One JSON line is printed by rank 0.
"""
import argparse
import json
import multiprocessing as mp
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")     # keep stdout to the ONE JSON line (NCCL prints its version banner)

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

BATCH_PER_GPU = 4096
DEFAULT_GROUPS = 2         # instance groups of the fused step (mpcb_set_groups); MPCB_GROUPS overrides.  Measured with the
#                            device-driven solve (profiles/r02_groups_sweep*.txt): 1 group 687k, 2 groups 697k, 4 groups 584k, 8 groups 505k steps/s
SEED_X0, SEED_NOISE = 20240419, 7
X0_SCALE = np.array([0.02, 0.002, 0.02])
METRIC = "batched MPC steps/sec (Ex_NMPC CSTR, N=50, FP64)"


def _problem():
    import __graft_entry__ as entry
    return entry._problem("nmpc_cstr")


def _workload(prob, B, nsteps, rank=0):
    rng = np.random.default_rng(SEED_X0 + 1000003 * rank)
    # 2 % on concentration and level, 0.2 % on temperature: a 2 % (6.5 K) temperature offset makes the optimal
    # first move drain the tank to its 0.5 bound, after which measurement noise puts y_0 outside [ymin, ymax]
    # and the reference's own NLP is infeasible (its Y_0 row only involves the fixed x_0, Control_Calc.py:128-151)
    x0 = prob.x0_p * (1 + X0_SCALE * rng.uniform(-1, 1, (B, prob.nxp)))
    noise = np.sqrt(1e-7) * np.random.default_rng(SEED_NOISE + rank).standard_normal((nsteps, B, prob.ny))
    return x0, noise


# ---------------------------------------------------------------------------------------------
# CPU arm: used for `cpu_baseline` and for `--impl reference`.  Two implementations are timed on the box's host cores,
# each on a bounded sample of the SAME workload (same x0 distribution and noise), each over CONSECUTIVE closed-loop steps
# of every instance after that instance's own cold-start steps (the first step has a different warm start,
# MPC_code.py:740-756, and more iterations):
#   * "cxx"   - oracle/cxx_loop.cpp: the host build (g++ -O3 -march=native -fopenmp) of this repo's solver sources,
#               OpenMP over instances on all cores.  Same algorithm as the kernels, ~15x faster than the NumPy port: the
#               strongest CPU implementation available here, hence the one the reference arm reports.
#   * "numpy" - oracle/closed_loop.py: the independent NumPy/LAPACK restatement (dense KKT), one process per core.
# Neither is IPOPT: CasADi/IPOPT cannot be installed here or on the GPU box (profiles/r02_casadi_probe.txt).
# ---------------------------------------------------------------------------------------------
CPU_WARM_STEPS = 5            # per-instance cold-start steps excluded from the CPU timings


def cxx_throughput(n_inst, nsteps, rank=0):
    """(instance-steps/s, threads, wall seconds) of the C++/OpenMP closed loop for `nsteps` timed steps per instance."""
    from oracle.cxx_baseline import CxxLoop, range_bounds_of
    prob, ss, ocp = _problem()
    loop = CxxLoop("nmpc_cstr", prob, ss, ocp, range_bounds_of(ocp))
    x0, noise = _workload(prob, n_inst, CPU_WARM_STEPS + nsteps, rank)
    t0 = time.time()
    v, r = loop.throughput(x0, noise, CPU_WARM_STEPS)
    return v, int(r["threads"]), time.time() - t0


_ORACLE = {}


def _oracle_init():
    for var in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):
        os.environ[var] = "1"                         # one core per worker process
    sys.path.insert(0, ROOT)
    from oracle import cmodel
    from oracle.closed_loop import OracleLoop
    prob, ss, ocp = _problem()
    _ORACLE["loop"] = OracleLoop(prob, ss, ocp, cmodel.build("nmpc_cstr", prob, ocp, ss))


def _oracle_worker(args):
    """Closed loop of one instance; returns the seconds spent in the steps after the cold-start ones."""
    x0, noise, nwarm = args
    loop = _ORACLE["loop"]
    t_mark = []
    rec = loop.run(Nsim=noise.shape[0], x0_p=x0, x0_m=x0, noise=noise, on_step=lambda k: t_mark.append(time.time()))
    t_end = time.time()
    return t_end - t_mark[nwarm], int(np.sum(rec["ITER_DYN"]))


class OraclePool:
    """Worker processes (spawned, so no BLAS thread state is inherited), each holding the NumPy oracle."""

    def __init__(self, cores):
        self.cores = cores
        self.pool = mp.get_context("spawn").Pool(cores, initializer=_oracle_init)
        prob, _, _ = _problem()
        x0, noise = _workload(prob, cores, 1)
        self.pool.map(_oracle_worker, [(x0[i], noise[:, i, :], 0) for i in range(cores)], chunksize=1)   # build / import
        self.prob = prob

    def throughput(self, n_inst, nsteps):
        """Closed-loop instance-steps per second over all workers (timed steps / per-core busy time)."""
        x0, noise = _workload(self.prob, n_inst, CPU_WARM_STEPS + nsteps)
        jobs = [(x0[i], noise[:, i, :], CPU_WARM_STEPS) for i in range(n_inst)]
        t0 = time.time()
        res = self.pool.map(_oracle_worker, jobs, chunksize=1)
        wall = time.time() - t0
        busy = sum(r[0] for r in res) / self.cores
        return n_inst * nsteps / busy, wall

    def close(self):
        self.pool.close(); self.pool.join()


def cpu_baselines(cores, cxx_inst_per_core=16, cxx_steps=60, numpy_steps=20):
    """The two CPU figures of one bench line (bounded: ~30 core-seconds of C++ work, ~70 core-seconds of NumPy work)."""
    v, threads, wall = cxx_throughput(cxx_inst_per_core * cores, cxx_steps)
    cxx = {"value": v, "unit": "steps/s", "cores": threads, "kind": "port",
           "sample": "%d instances x %d consecutive closed-loop steps after %d cold-start steps each, same workload; host build of "
                     "this repo's solver sources (same algorithm, C++, g++ -O3 -fopenmp over instances; %.1f s wall = %.0f core-seconds); "
                     "not IPOPT" % (cxx_inst_per_core * cores, cxx_steps, CPU_WARM_STEPS, wall, wall * threads)}
    pool = OraclePool(cores)
    v2, wall2 = pool.throughput(cores, numpy_steps)
    pool.close()
    npy = {"value": v2, "unit": "steps/s", "cores": cores, "kind": "port",
           "sample": "%d instances x %d consecutive closed-loop steps after %d cold-start steps each, one process per core (%.1f s); "
                     "independent NumPy/LAPACK dense-KKT oracle (the parity checker), not IPOPT" % (cores, numpy_steps, CPU_WARM_STEPS, wall2)}
    return cxx, npy


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    n_inst, nsteps = 4 * cores, 20          # per bench step: every instance runs 5 cold-start + 20 timed consecutive steps
    samples, threads = [], cores
    for _ in range(args.warmup):
        cxx_throughput(n_inst, nsteps)
    t0 = time.time()
    for _ in range(args.steps):
        v, threads, _ = cxx_throughput(n_inst, nsteps)
        samples.append(v)
    wall = time.time() - t0
    value = float(np.mean(samples))
    sample = ("per bench step: %d instances x %d consecutive closed-loop steps after %d cold-start steps each; host build of this "
              "repo's solver sources (same algorithm, C++, OpenMP over instances); not IPOPT" % (n_inst, nsteps, CPU_WARM_STEPS))
    pool = OraclePool(cores)
    v2, wall2 = pool.throughput(cores, 20)
    pool.close()
    emit({
        "impl": "reference", "metric": METRIC, "value": value, "unit": "steps/s", "n_gpus": 0, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * wall / max(args.steps, 1), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": _config(max(1, args.gpus)),
        "cpu_baseline": {"value": value, "unit": "steps/s", "cores": threads, "kind": "port", "sample": sample},
        "cpu_baseline_numpy": {"value": v2, "unit": "steps/s", "cores": cores, "kind": "port",
                               "sample": "%d instances x 20 consecutive steps after %d cold-start steps, one process per core "
                                         "(%.1f s); independent NumPy/LAPACK oracle" % (cores, CPU_WARM_STEPS, wall2)},
        "e2e": {"value": value, "unit": "steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0})


def _config(world):
    """`config` of BOTH arms, key for key: the workload (the CPU arm times a bounded sample of it, described in its
    `cpu_baseline.sample`; GPU-arm specifics - instance groups, cache note - are top-level keys of its line)."""
    return {"workload": "Ex_NMPC (configs[1]): CSTR NMPC + EKF + target, N=50, Mx=10, closed loop with plant and measurement "
                        "noise; x0 perturbed 2%%/0.2%%/2%% (seed %d)" % SEED_X0,
            "batch_per_gpu": BATCH_PER_GPU, "global_batch": world * BATCH_PER_GPU,
            "parallelism": "instances sharded, %d rank(s)" % world}


# ---------------------------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------------------------
def _clock_sampler(path):
    q = ("timestamp,index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    try:
        return subprocess.Popen(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader,nounits", "-lms", "50"],
                                stdout=open(path, "w"), stderr=subprocess.DEVNULL)
    except Exception:
        return None


def _parse_clocks(path, gpu_index, windows):
    """Median SM clock and throttle reasons of the samples that fall inside the timed windows [(t0, t1), ...]."""
    import datetime
    sm, smax, reasons, n_all = [], 0.0, set(), 0
    try:
        for line in open(path):
            f = [x.strip() for x in line.split(",")]
            if len(f) < 10 or not f[1].isdigit() or int(f[1]) != gpu_index:
                continue
            n_all += 1
            try:
                ts = datetime.datetime.strptime(f[0], "%Y/%m/%d %H:%M:%S.%f").timestamp()
            except ValueError:
                continue
            if not any(a - 0.05 <= ts <= b + 0.05 for a, b in windows):
                continue
            sm.append(float(f[2])); smax = max(smax, float(f[3]))
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[6:10]):
                if val.lower().startswith("active"):
                    reasons.add(name)
    except Exception:
        pass
    return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": smax or None, "reasons": sorted(reasons),
            "samples": len(sm), "samples_total": n_all}


def stage_flops(cp):
    """Algorithmic FLOPs of one stage's derivative evaluation (DAG op counts; see DESIGN.md 'FLOP accounting')."""
    p, f = cp.prob, cp.flops
    nx, nz = p.nx, p.nx + p.nu
    nzp = nz * (nz + 1) // 2
    mx = cp.library.dims.Mx
    per_sub = 4 * (f["mdl_f"] + f["mdl_f_vjp"] + f["mdl_f_sh"]) + 13 * nx + 15 * nx + 13 * nx * (nz + 1) + 4 * nzp
    return mx * per_sub + f.get("mdl_post", 0) + f["ocp_cost_d"] + f.get("ocp_out_d", 0) + 2 * nx


def first_eval_enabled(cp):
    """True when the library evaluates the first tick of a solve to first order (MPCB_EVAL_FIRST, csrc/mpcb_ocp.cuh)."""
    D = cp.build["gen"]["defines"]
    if "-DMPCB_EVAL_FIRST=0" in os.environ.get("MPCB_EXTRA_FLAGS", ""):
        return False
    return bool(D.get("MPCB_DYN_RK4")) and not D.get("MPCB_CONTFORM") and not D.get("MPCB_DENSE_SH")


def stage_flops_first(cp):
    """Algorithmic FLOPs of a FIRST-tick stage evaluation (k_ocp_eval_first: one forward sensitivity sweep, no adjoint /
    second-order sweep - every multiplier is zero there)."""
    p, f = cp.prob, cp.flops
    nx, nz = p.nx, p.nx + p.nu
    mx = cp.library.dims.Mx
    per_sub = 4 * f["mdl_f_s"] + 13 * nx + 13 * nx * nz
    return mx * per_sub + f.get("mdl_post", 0) + f["ocp_cost_d"] + f.get("ocp_out_d", 0) + 2 * nx


def stage_bytes(cp):
    """Algorithmic HBM bytes of one stage's derivative evaluation: x,u,x+,lam,ym,s in; A,B,c,H,grad,G,g,partials out."""
    p = cp.prob
    nx, nu, ng = p.nx, p.nu, cp.library.dims.ng
    nz = nx + nu
    rd = nz + nx + nx + 2 * ng + (p.nd + 1 + p.npx + p.npy + 2 * nz)
    wr = nx * nx + nx * nu + nx + nz * (nz + 1) // 2 + nz + ng * nz + ng + 2
    return 8 * (rd + wr)


def kkt_bytes(cp):
    """Algorithmic HBM bytes of one instance's KKT step (k_ocp_kkt): the stage records read by the backward sweep, the
    record / forward-record heads read by the forward sweep, the record tails read by the stage-parallel pass, the forward
    records written and read, the step and new multipliers written (layout: csrc/mpcb_ocp.cuh R_* / FREC_*)."""
    D = cp.build["gen"]["defines"]
    p = cp.prob
    nxa = p.nx + D["MPCB_NAUG"]; nu = p.nu; nza = nxa + nu; ng = D["MPCB_NG"]; ngs = max(ng, 1); N = p.N
    r_gl = nxa * nza + nxa + nza * nza
    r_bwd = r_gl + 3 * nza + ngs * nza + 4 * ngs
    rec = r_bwd + 2 * nza + 4 * ngs + 10
    frec = nu * nxa + nu + nxa * nxa + nxa
    per_stage = r_bwd + (nxa * nza + nxa) + (nu * nxa + nu) + (rec - r_gl) + 2 * frec + nza + nxa + 2 * ng
    return 8 * N * per_stage


def run_gpu(args):
    import torch
    import torch.distributed as dist
    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        raise SystemExit("bench.py --gpus %d needs %d ranks: launch it with `python -m torch.distributed.run --nnodes=1 "
                         "--nproc-per-node %d --master-addr 127.0.0.1 bench.py --gpus %d ...` (WORLD_SIZE is %d)"
                         % (args.gpus, args.gpus, args.gpus, args.gpus, world))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    from mpc_code_b200.mpc_loop import CompiledProblem
    prob, ss, ocp = _problem()
    cp = CompiledProblem(prob, "nmpc_cstr")
    B, K, W = BATCH_PER_GPU, args.steps, args.warmup
    total = W + K
    x0, noise = _workload(prob, B, total, rank)
    ctl = cp.controller(B)
    noise_dev = torch.as_tensor(noise, device=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    # ---------------- device-resident closed loop (value) ----------------
    clock_file = os.path.join(tempfile.gettempdir(), "mpcb_clocks_%d.csv" % os.getpid())
    sampler = _clock_sampler(clock_file) if rank == 0 and not os.environ.get("MPCB_BENCH_NOSAMPLER") else None
    windows = []
    # The problem set-up leaves ~10^6 live Python objects (the symbolic expression graphs).  A generation-2 garbage
    # collection walking them takes 20-110 ms and showed up as outlier steps every ~12 steps of the timed loop; freeze
    # them into the permanent generation (they stay alive anyway) so that collections during the loop are cheap.
    import gc
    gc.collect(); gc.freeze()
    if sampler is not None:                 # let nvidia-smi finish its NVML start-up (it stalls launches) before timing
        t_wait = time.time()
        while time.time() - t_wait < 5.0 and (not os.path.exists(clock_file) or os.path.getsize(clock_file) == 0):
            time.sleep(0.05)
        time.sleep(0.2)
    ctl.reset(x0_p=x0, x0_m=x0)
    # records are written into buffers allocated BEFORE the timed region: growing torch's caching allocator inside it
    # (one new 2 MB segment every ~12 steps of cloned outputs) means a cudaMalloc, seen as 10-100 ms outlier steps
    ys = torch.empty(total, B, prob.ny, device=dev, dtype=torch.float64)
    us = torch.empty(total, B, prob.nu, device=dev, dtype=torch.float64)
    st_dyn = torch.empty(K, B, device=dev, dtype=torch.int32); it_dyn = torch.empty_like(st_dyn); st_ss = torch.empty_like(st_dyn)
    # instance groups: sub-batches queued on their own streams by this one thread (no polling threads since round 2: the
    # solve is a device-driven CUDA graph), so the number of groups no longer depends on the host's core count
    groups = int(os.environ.get("MPCB_GROUPS", DEFAULT_GROUPS))
    ctl.h.set_groups(groups)
    for k in range(W):
        o = ctl.step_fused(noise_dev[k]); ys[k].copy_(o["Yp"]); us[k].copy_(o["U"])
    launches0 = ctl.h.launches
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(K + 1)]
    barrier()
    t_w0 = time.time()
    ev[0].record()
    for k in range(K):
        o = ctl.step_fused(noise_dev[W + k])
        ev[k + 1].record()
        ys[W + k].copy_(o["Yp"]); us[W + k].copy_(o["U"])
        st_dyn[k].copy_(o["STATUS_DYN"]); it_dyn[k].copy_(o["ITER_DYN"]); st_ss[k].copy_(o["STATUS_SS"])
    barrier()
    windows.append((t_w0, time.time()))
    # what the caller of the timed path received from its last step (the buffers behind `o` are reused by the runs below)
    last = {key: val.clone() for key, val in o.items() if isinstance(val, torch.Tensor)} if args.dump_outputs else None
    elapsed_ms = ev[0].elapsed_time(ev[K])
    launches = ctl.h.launches - launches0
    step_ms = np.array([ev[k].elapsed_time(ev[k + 1]) for k in range(K)])
    t_all = torch.tensor([elapsed_ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t_all, op=dist.ReduceOp.MAX)
    elapsed_max = float(t_all.item())
    value = world * B * K / (elapsed_max * 1e-3)

    # ---------------- kernel timing: the same W+K steps replayed WITHOUT groups and with event brackets around every launch
    # (with groups the kernels of different groups overlap and a per-kernel duration is not attributable) ----------------
    ctl.h.set_groups(1)
    ctl.reset(x0_p=x0, x0_m=x0)
    for k in range(W):
        ctl.step_fused(noise_dev[k])
    ctl.h.set_profiling(True)
    barrier()
    t_w0 = time.time()
    for k in range(K):
        ctl.step_fused(noise_dev[W + k])
    barrier()
    windows.append((t_w0, time.time()))
    prof = ctl.h.profile()
    ctl.h.set_profiling(False)
    ctl.h.set_groups(groups)

    # ---------------- end to end through the public API with host buffers (e2e) ----------------
    y_host = ys.cpu().pin_memory()                      # recorded plant measurements, [W+K, B, ny]
    u_host = torch.empty(total, B, prob.nu, dtype=torch.float64).pin_memory()
    y_dev = torch.empty(B, prob.ny, device=dev, dtype=torch.float64)
    ctl.reset(x0_p=x0, x0_m=x0)
    for k in range(W):
        y_dev.copy_(y_host[k], non_blocking=True); o = ctl.step_fused(y_meas=y_dev); u_host[k].copy_(o["U"], non_blocking=True)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_w0 = time.time()
    e0.record()
    for k in range(W, total):
        y_dev.copy_(y_host[k], non_blocking=True)                    # H2D of this step's measurement
        o = ctl.step_fused(y_meas=y_dev)
        u_host[k].copy_(o["U"], non_blocking=True)                   # D2H of the computed inputs
        torch.cuda.current_stream(dev).synchronize()                 # the caller needs u_k before the next sample
    e1.record()
    barrier()
    windows.append((t_w0, time.time()))
    if sampler is not None:
        time.sleep(0.1)
        sampler.terminate(); sampler.wait()
    t_e2e = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t_e2e, op=dist.ReduceOp.MAX)
    e2e_value = world * B * K / (float(t_e2e.item()) * 1e-3)
    replay_err = float((u_host[W:].to(dev) - us[W:]).abs().max().item())

    # ---------------- statistics gathered over NCCL (the only collective; off the timed path) ----------------
    from mpc_code_b200.sharding import gather_instances, reduce_stats
    stats = reduce_stats(st_dyn, it_dyn)
    u_all = gather_instances(us[W:].contiguous(), world * B)         # closed-loop inputs of all ranks, [K, N*B, nu]
    assert u_all.shape[1] == world * B
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---------------- roofline of the dominant kernel (stage derivatives, class ocp_eval) ----------------
    kms = prof["ms"]; kl = prof["launches"]
    dom = max(("ocp_eval", "ocp_kkt", "ocp_trial", "target", "estimate"), key=lambda c: kms[c])
    f_stage, b_stage = stage_flops(cp), stage_bytes(cp)
    eval_s = kms["ocp_eval"] * 1e-3
    evals = prof["eval_instances"] * prob.N                           # stage evaluations done in the timed region
    fp64_peak = ctl.h.dfma_peak_tflops()
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak, hbm_src = (peaks["hbm_gbs"], "measured (MEASURED_PEAKS.json)") if "hbm_gbs" in peaks else (6650.0, "fallback")
    # the first tick of every solve (one per instance and step) is the cheaper first-order kernel, counted with its own FLOPs
    evals_first = B * K * prob.N if first_eval_enabled(cp) else 0
    flops_total = (evals - evals_first) * f_stage + evals_first * stage_flops_first(cp)
    ach_tf = flops_total / eval_s / 1e12 if eval_s > 0 else 0.0
    ach_gb = evals * b_stage / eval_s / 1e9 if eval_s > 0 else 0.0
    traffic, traffic_src = None, None
    try:        # DRAM bytes of the kernel from the committed ncu capture, scaled to the average launch of THIS run
        tr = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))["k_ocp_eval"]
        traffic = tr["dram_bytes_per_full_launch"] / tr["stage_evals_per_full_launch"] * evals / max(kl["ocp_eval"], 1)
        traffic_src = tr["source"]
    except Exception:
        pass
    # second and third kernels by time: the KKT step (HBM traffic of the stage records) and the target solve (latency)
    kkt_b = kkt_bytes(cp)
    kkt_s = kms["ocp_kkt"] * 1e-3
    kkt_gb = prof["eval_instances"] * kkt_b / kkt_s / 1e9 if kkt_s > 0 else 0.0
    kkt_traffic = None
    try:
        trk = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))["k_ocp_kkt"]
        kkt_traffic = trk["dram_bytes_per_full_launch"] / trk["instances_per_full_launch"] * prof["eval_instances"] / max(kl["ocp_kkt"], 1)
    except Exception:
        pass
    roofline_others = {
        "k_ocp_kkt": {"bound": "hbm", "achieved": kkt_gb, "peak": hbm_peak, "unit": "GB/s", "frac": kkt_gb / hbm_peak,
                      "traffic": kkt_traffic, "algorithmic_bytes_per_instance": kkt_b, "avg_launch_ms": kms["ocp_kkt"] / max(kl["ocp_kkt"], 1),
                      "note": "N-sequential Riccati sweep, one warp per instance, records streamed by cp.async.bulk (TMA) into a "
                              "shared-memory ring; issue slots ~50 % busy, so neither HBM nor latency alone binds it"},
        "k_target": {"bound": "latency", "avg_launch_ms": kms["target"] / max(kl["target"], 1),
                     "note": "one thread per instance (9-13 sequential IPM iterations of one RK4 sweep + a 12 x 12 LDL'): 128 warps on "
                             "148 SMs, 3 % occupancy by construction; see DESIGN.md section 6"},
    }
    roofline = {
        "kernel": "k_ocp_eval", "bound": "fp64", "achieved": ach_tf, "peak": fp64_peak, "unit": "TFLOP/s",
        "frac": ach_tf / fp64_peak if fp64_peak else None, "traffic": traffic, "traffic_unit": "bytes per launch (average launch)",
        "traffic_source": traffic_src, "algorithmic_bytes_per_launch": b_stage * evals / max(kl["ocp_eval"], 1),
        "peak_source": "FP64 FMA micro-benchmark run in this process (mpcb_dfma_peak); MEASURED_PEAKS.json has no FP64 entry",
        "note": "kernel class ocp_eval: k_ocp_eval plus, for the first tick of every solve, k_ocp_eval_first (first-order sweep, "
                "counted with its own FLOPs); time and FLOPs are summed over both",
        "flops_per_stage_eval": f_stage, "stage_evals": int(evals), "stage_evals_first_order": int(evals_first),
        "flops_per_first_order_stage_eval": stage_flops_first(cp) if evals_first else None, "kernel_ms_total": kms["ocp_eval"],
        "kernel_launches": kl["ocp_eval"], "avg_launch_ms": kms["ocp_eval"] / max(kl["ocp_eval"], 1),
        "hbm": {"achieved": ach_gb, "peak": hbm_peak, "unit": "GB/s", "frac": ach_gb / hbm_peak, "bytes_per_stage_eval": b_stage,
                "peak_source": hbm_src},
        "kernel_time_share": {c: kms[c] / max(sum(kms.values()), 1e-12) for c in kms}, "dominant_by_time": dom,
        "line_search_trials_per_iteration": prof["trial_instances"] / max(prof["eval_instances"], 1),
    }

    # ---------------- CPU baselines beside it (bounded samples) ----------------
    cpu_baseline = cpu_numpy = None
    if world == 1 and not args.no_cpu_baseline:
        cpu_baseline, cpu_numpy = cpu_baselines(os.cpu_count() or 1)
    clocks = _parse_clocks(clock_file, local, windows)
    out = {
        "metric": METRIC, "value": value, "unit": "steps/s", "n_gpus": world, "steps": K, "warmup": W,
        "ms_per_step": elapsed_max / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic",
        "config": _config(world), "instance_groups_per_gpu": groups,
        "cache": "per-step working set %.0f MB per GPU > 126 MB L2 (no flush needed)" % (B * cp_ws_bytes(cp) / 1e6),
        "p50_step_latency_ms": float(np.median(step_ms)), "p99_step_latency_ms": float(np.percentile(step_ms, 99)),
        "slowest_steps": [[int(i), float(step_ms[i])] for i in np.argsort(-step_ms)[:3]],
        "e2e": {"value": e2e_value, "unit": "steps/s", "h2d_bytes_per_step": B * prob.ny * 8, "d2h_bytes_per_step": B * prob.nu * 8,
                "replay_max_abs_du": replay_err},
        "gpu_launches": int(launches),
        "roofline": roofline, "roofline_others": roofline_others, "cpu_baseline": cpu_baseline, "cpu_baseline_numpy": cpu_numpy, "clocks": clocks,
        "solver_stats": stats,
    }
    if last is not None:
        dump_outputs(args.dump_outputs, last)
    emit(out)
    if world > 1:
        dist.destroy_process_group()


def cp_ws_bytes(cp):
    """Per-instance bytes touched per step (solver workspace incl. stage records + caller buffers), see DESIGN.md 5."""
    d = cp.library.dims
    nz = d.nx + d.nu
    rec = nz * d.nx + d.nx + nz * nz + 7 * nz + d.ng * (nz + 10) + 10
    return 8 * (d.N * (rec + 20 + 4 * d.nx + 6 * d.ng) + 5 * d.nw + d.npar)


def dump_outputs(path, outputs):
    """``<path>/<name>.npy`` for every output of one fused step (rank 0's instances; [B, ...] float64, integer status
    and iteration counts included as float64): 0.7 MB at B = 4096, so nothing is sampled."""
    os.makedirs(path, exist_ok=True)
    for key, val in outputs.items():
        np.save(os.path.join(path, key + ".npy"), val.detach().cpu().numpy().astype(np.float64))


_JSON_FD = None


def emit(record):
    line = (json.dumps(record) + "\n").encode()
    if _JSON_FD is None:
        sys.stdout.write(line.decode()); sys.stdout.flush()
    else:
        os.write(_JSON_FD, line)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the arrays the last timed step returned as DIR/<name>.npy, to compare two builds "
                         "output for output on the same seeded workload")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the CUDA path (--impl b200)")
    # stdout carries exactly ONE line, the JSON record: everything else that libraries write to file descriptor 1 (NCCL
    # prints its version banner there) is sent to stderr, and the record goes to the saved descriptor at the end
    global _JSON_FD
    sys.stdout.flush()
    _JSON_FD = os.dup(1)
    os.dup2(2, 1)
    if args.impl == "reference":
        run_reference(args)
    else:
        if args.warmup < 3:
            args.warmup = 3
        run_gpu(args)


if __name__ == "__main__":
    main()
