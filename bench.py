"""bench.py -- rollout env-steps/s and CEM-iteration latency of the B200-native CEM planner.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--global-batch G] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

--dump-outputs DIR writes what the last timed step returned (the new mean and covariance, the per-sample costs, thetadot
and theta) as DIR/<name>.npy in float32.  The inputs are fixed constants and PRNGKey(0), so two builds run with the same
arguments can be compared array for array.

One "step" = one full CEM iteration of the planner hot path (sample -> projection filter ->
Bernstein evaluation -> T-step rollout of every sample -> cost -> elite top-k [+ NCCL all-gather
merge] -> mean/covariance update).
  default            BASELINE.json config 2 per GPU: 4096 samples x 100 steps on every GPU (weak scaling, global
                     batch = 4096 * N).  The same run also times BASELINE config 5 -- a 65536-sample global batch
                     sharded over the N GPUs (strong scaling) -- and reports it under "config5".
  --global-batch G   the headline itself is the strong-scaling configuration: G samples over N GPUs.
  value   env-steps/s with all inputs resident in HBM, CUDA-event timed, max over ranks
  e2e     the same through the public API (`cem_planner.compute_cem`, maxiter_cem=1) with HOST numpy
          inputs: pinned H2D of the tick inputs and D2H of the results inside the timed region
  roofline  FP32-FMA roofline of the rollout kernel (dominant kernel), timed live with CUDA events;
          flop per env-step = the op count of the CPU restatement (profiles/r2_flop_count.json)
  cpu_baseline  the in-repo CPU restatement of the same CEM iteration (oracle: numpy planner algebra + C rollout,
          float32 build, OpenMP over samples) on the host cores of the same box -- NOT the reference's MJX
          (jax / mujoco cannot be installed here)
`--impl reference` times that CPU restatement as the reference arm: the whole 4096-sample CEM iteration, same
seeds, same configuration (see DESIGN.md section 7).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

B_PER_GPU, T, DT = 4096, 100, 0.05
B_CONFIG5 = 65536
W_POS, W_ROT, W_COL, ELITE, PROJ_IT = 20.0, 3.0, 80.0, 0.05, 10
Q0 = np.array([1.5, -1.8, 1.75, -1.25, -1.6, 0.0])
TP, TR = np.array([-0.3, -0.3, 0.5]), np.array([0.0, 1.0, 0.0, 0.0])
HBM_BYTES_PER_ENV_STEP = 48.0    # theta + thetadot written per env-step (SURVEY.md 8d)
METRIC = "rollout env-steps/sec (CEM iteration, UR5e+Hand-E scene, 4096 samples x 100 steps per GPU)"


def flop_per_env_step():
    """Algorithmic work F_A per env-step: counted by the instrumented CPU restatement (oracle -DORACLE_COUNT,
    tools/count_flops.py) on this bench's own inputs and frozen in profiles/r2_flop_count.json / BASELINE.md section 4."""
    try:
        with open(os.path.join(ROOT, "profiles", "r2_flop_count.json")) as f:
            d = json.load(f)
        return float(d["flop_per_env_step"]), "counted (profiles/r2_flop_count.json)"
    except Exception:
        return 8.0e4, "provisional estimate of SURVEY.md 8d (no counter output found)"


class ClockSampler(threading.Thread):
    def __init__(self, gpu):
        super().__init__(daemon=True)
        self.gpu, self.rows, self.stop = gpu, [], False

    def run(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        while not self.stop:
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i", str(self.gpu)],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            time.sleep(0.1)

    def summary(self):
        sm = [float(r[0]) for r in self.rows if r[0].replace('.', '').isdigit()]
        mx = [float(r[1]) for r in self.rows if r[1].replace('.', '').isdigit()]
        reasons = set()
        for r in self.rows:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(self.rows)}


# ---------------------------------------------------------------------------------------------- CPU arm
class CpuCem:
    """One CEM iteration of the CPU restatement (`oracle/`), the same pipeline and the same inputs as the GPU arm:
    jax.random normal draws of PRNGKey(0)'s first split (numpy threefry) -> xi = mu + chol(cov + 0.003 I) z ->
    projection filter (dense float32 matrices, as the reference writes it) -> Bernstein evaluation -> rollout of every sample (C,
    float32, OpenMP over samples; the [B,T,187] distance tensor materialised like the reference does) -> cost ->
    stable argsort top-k -> mean / covariance.  numpy's BLAS and OpenMP use `nthreads` threads."""

    def __init__(self, B, Th, nthreads, maxiter_projection=PROJ_IT):
        from manipulator_mujoco_b200 import jax_prng
        from manipulator_mujoco_b200.mjcf import load_model
        from oracle import jax_random_ref
        from oracle.oracle import Oracle
        from oracle.planner_ref import PlannerRef
        self.B, self.T, self.nthreads = B, Th, nthreads
        self.pr = PlannerRef(6, B, Th, DT, ELITE, W_POS, W_ROT, W_COL, maxiter_projection).astype(np.float32)   # reference arithmetic: float32
        self.ora = Oracle(load_model(), DT, dtype="f32")
        self.warm = self.ora.initial_warmstart()
        self.key = jax_prng.split(jax_prng.PRNGKey(0))[0]
        self._prng, self._jr = jax_prng, jax_random_ref
        try:
            from threadpoolctl import threadpool_limits
            self._limit = lambda: threadpool_limits(limits=nthreads)
        except Exception:
            import contextlib
            self._limit = contextlib.nullcontext

    def normal(self, n):
        """jax.random.normal(key, (n,)) in the partitionable counter layout, vectorised (oracle/jax_random_ref.py holds
        the scalar restatement the tests pin; the mapping bits -> uniform -> erf_inv is that module's)."""
        x0, x1 = self._prng.threefry2x32(self.key, np.zeros(n, np.uint32), np.arange(n, dtype=np.uint32))
        bits = x0 ^ x1
        f = ((bits >> np.uint32(9)) | np.uint32(0x3F800000)).view(np.float32) - np.float32(1)
        lo = np.nextafter(np.float32(-1), np.float32(0))
        u = np.maximum(lo, (f * (np.float32(1) - lo) + lo).astype(np.float32))
        return (np.float32(np.sqrt(2)) * self._jr.erfinv32(u)).astype(np.float32)

    def iteration(self, chunk=1024):
        pr, B, Th = self.pr, self.B, self.T
        with self._limit():
            f32 = np.float32
            z = self.normal(B * pr.nvar).reshape(B, pr.nvar)
            xi = pr.compute_xi_samples(z, np.zeros(pr.nvar, f32), 10 * np.identity(pr.nvar, dtype=f32)).astype(f32)
            st = pr.state_term(Q0, np.zeros(6), np.zeros(6), B).astype(f32)
            xif = pr.compute_projection_filter(xi, st)
            td = xif @ pr.A_thetadot.T
            cost = np.empty(B)
            theta = np.empty((B, 6 * Th))
            for lo in range(0, B, chunk):                       # bounds the [chunk, T, 187] float64 distance tensor
                hi = min(B, lo + chunk)
                th, ep, er, col = self.ora.rollout(td[lo:hi], Q0, np.zeros(6), warm=self.warm, nthreads=self.nthreads,
                                                   want_collision=True)
                theta[lo:hi] = th
                cost[lo:hi] = pr.compute_cost_batch_vec(ep, er, col, TP, TR)[0]
            xi_e, idx, cost_e = pr.compute_ellite_samples(cost, xi)
            mean, cov = pr.compute_mean_cov(cost_e.astype(f32), np.zeros(pr.nvar, f32), 10 * np.identity(pr.nvar, dtype=f32), xi_e)
        return mean, cov, cost, td

    def timed(self, reps):
        ts = []
        for _ in range(reps):
            t0 = time.perf_counter()
            self.iteration()
            ts.append(time.perf_counter() - t0)
        return ts


def run_reference(args):
    """Reference arm: the CPU restatement of the whole CEM iteration on all host cores, same configuration and seeds as
    the GPU arm (each step = the full 4096-sample iteration, nothing extrapolated)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    B = args.batch_per_gpu
    cem = CpuCem(B, T, cores)
    small = CpuCem(256, T, cores)
    for _ in range(args.warmup):
        small.iteration()
    times = cem.timed(args.steps)
    tot = sum(times)
    val = B * T * args.steps / tot
    sample = (f"the full step: {B} samples x {T} steps, one CEM iteration (jax.random draws, dense projection filter x{PROJ_IT}, "
              f"C rollout float32 + [B,T,187] distances, cost, argsort top-k, mean/cov), all {cores} host threads")
    line = {"metric": METRIC, "value": val, "unit": "env-steps/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1e3 * tot / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "impl": "reference",
            "config": {"workload": f"UR5e+Hand-E scene A (ur5e_hande_mjx/scene.xml constants), {B} samples x {T} steps, dt={DT}, "
                                   f"order-10 Bernstein, {PROJ_IT} projection iterations, elite {ELITE}, 1 CEM iteration per step",
                       "global_batch": B, "horizon": T,
                       "note": "the reference's MJX/JAX cannot be installed in this image (BASELINE.md section 2); this arm is the in-repo CPU "
                               "restatement of the same path (oracle/: numpy float64 planner algebra + oracle/mjstep.c float32 rollout with "
                               "OpenMP), on rank 0's host cores only whatever N is; warm-up steps run a 256-sample batch"},
            "cpu_baseline": {"value": val, "unit": "env-steps/s", "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": val, "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


def cpu_baseline_record():
    """cpu_baseline of our own line: two full 4096-sample CEM iterations on all cores (about 10 s), plus BASELINE.md
    section 3's promised C1-configuration numbers (B=100, T=16) at one thread and at all cores."""
    cores = os.cpu_count() or 1
    cem = CpuCem(B_PER_GPU, T, cores)
    CpuCem(256, T, cores).iteration()
    ts = cem.timed(2)
    rec = {"value": B_PER_GPU * T * len(ts) / sum(ts), "unit": "env-steps/s", "cores": cores, "kind": "port",
           "sample": f"2 full CEM iterations of the same workload ({B_PER_GPU} samples x {T} steps; oracle/: numpy planner algebra + "
                     f"mjstep.c float32 rollout, OpenMP; {sum(ts):.1f} s)"}
    c1 = {}
    for name, nt in (("threads_1", 1), (f"threads_{cores}", cores)):
        c = CpuCem(100, 16, nt)
        c.iteration()
        t1 = c.timed(5)
        c1[name] = 100 * 16 * len(t1) / sum(t1)
    rec["c1_config_env_steps_per_s"] = c1
    return rec


# ---------------------------------------------------------------------------------------------- GPU arm
DUMP_BYTES = 60 * 10 ** 6          # array data of --dump-outputs: under 64 MB with the .npy headers


def dump_outputs(out_dir, whole, per_sample):
    """Write `whole` and `per_sample` (name -> numpy array; the latter with one row per sample) as out_dir/<name>.npy.  When
    they exceed DUMP_BYTES, only a fixed, seeded subset of the sample rows is written, and its row indices as sample_rows.npy.
    Returns {name: shape} of what was written."""
    os.makedirs(out_dir, exist_ok=True)
    out = dict(whole)
    n = len(next(iter(per_sample.values())))
    row_bytes = sum(a.nbytes for a in per_sample.values()) // n
    room = DUMP_BYTES - sum(a.nbytes for a in whole.values())
    if row_bytes * n > room:
        rows = np.sort(np.random.default_rng(0).choice(n, room // (row_bytes + 8), replace=False))
        per_sample = {k: a[rows] for k, a in per_sample.items()}
        out["sample_rows"] = rows.astype(np.float64)
    out.update(per_sample)
    for k, a in out.items():
        np.save(os.path.join(out_dir, k + ".npy"), a)
    return {k: list(a.shape) for k, a in out.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch-per-gpu", type=int, default=B_PER_GPU)
    ap.add_argument("--global-batch", type=int, default=0, help="strong scaling: this many samples over all GPUs (BASELINE config 5: 65536)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-config5", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the last timed step's outputs as DIR/<name>.npy (rank 0's samples when sharded; --impl ours only)")
    args = ap.parse_args()
    if args.impl == "reference" and args.dump_outputs is not None:
        ap.error("--dump-outputs writes the outputs of --impl ours; the reference arm has none to write")
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.gpus != world and world > 1:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}")
    torch.cuda.set_device(local)
    dev = torch.device(f"cuda:{local}")
    pg = None
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
        pg = dist.group.WORLD
    from manipulator_mujoco_b200 import cem_planner, jax_prng
    import contextlib
    import io
    flush = torch.empty(256 * 1024 * 1024 // 4, device=dev)            # > 126 MB L2

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def max_over_ranks(x):
        t = torch.tensor([x], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def all_ranks(x):
        t = torch.tensor([x], device=dev, dtype=torch.float64)
        if world == 1:
            return [float(x)]
        out = torch.empty(world, device=dev, dtype=torch.float64)
        dist.all_gather_into_tensor(out, t)
        return [float(v) for v in out.cpu()]

    def timed(fn, k):
        """Event times of k calls of fn, and what the last call returned (earlier results are dropped at once, so the
        allocator sees the same pattern in every step)."""
        evs, last = [], None
        for i in range(k):
            flush.fill_(1.0)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            if i == k - 1:
                last = fn()
            else:
                fn()
            b.record()
            evs.append((a, b))
        torch.cuda.synchronize(dev)
        return [a.elapsed_time(b) for a, b in evs], last

    z6 = torch.zeros(6, device=dev)
    q0 = torch.as_tensor(Q0, dtype=torch.float32, device=dev)
    tp = torch.as_tensor(TP, dtype=torch.float32, device=dev)
    tr = torch.as_tensor(TR, dtype=torch.float32, device=dev)

    def measure(Bg, with_e2e, with_kernel, with_outputs=False):
        """Device-resident CEM iteration (+ optionally the public-API tick and the rollout kernel alone) at global batch Bg.
        with_outputs: also return, on the host, what the last timed iteration computed."""
        Bl = Bg // world
        with contextlib.redirect_stdout(io.StringIO()):
            pl = cem_planner(num_dof=6, num_batch=Bg, num_steps=T, timestep=DT, maxiter_cem=1, num_elite=ELITE, w_pos=W_POS, w_rot=W_ROT,
                             w_col=W_COL, maxiter_projection=PROJ_IT, device=dev, process_group=pg)
        pl.cache_normal_draws = False      # the timed step draws its normals like the reference's cem_iter does (mjx_planner.py:315)
        lib, h = pl._lib, pl._h
        state_term = torch.cat([q0, z6, z6, z6, z6]).unsqueeze(0).expand(Bl, 30).contiguous()
        mean0 = torch.zeros(pl.nvar, device=dev)
        cov0 = 10 * torch.eye(pl.nvar, device=dev)
        key1 = jax_prng.split(pl.key)[0]                                   # compute_cem's key (mjx_planner.py:388)

        def device_step():
            carry = (q0, z6, tp, tr, mean0, cov0, key1, state_term)
            return pl.cem_iter(carry, None)

        # W warm-up steps; with several GPUs a few more, untimed: NCCL sets its channels up lazily over the first collectives
        for _ in range(args.warmup + (8 if world > 1 else 0)):
            device_step()
        barrier()
        l0 = lib.cemk_launch_count(h)
        ms, last = timed(device_step, args.steps)
        barrier()
        res = {"pl": pl, "Bl": Bl, "launches": lib.cemk_launch_count(h) - l0, "ms_all": [round(v, 4) for v in ms]}
        if with_outputs:
            carry, (cost, cost_g, cost_r, cost_c, thetadot, theta) = last
            host = lambda t: t.detach().float().cpu().numpy()
            res["outputs"] = ({"xi_mean": host(carry[4]), "xi_cov": host(carry[5])},
                              {n: host(t) for n, t in (("cost", cost), ("cost_g", cost_g), ("cost_r", cost_r), ("cost_c", cost_c),
                                                       ("thetadot", thetadot), ("theta", theta))})
        del last
        res["tot_ms"] = max_over_ranks(sum(ms))
        res["value"] = Bg * T * args.steps / (res["tot_ms"] * 1e-3)
        if with_e2e:
            xi_mean_host = np.zeros(pl.nvar, dtype=np.float64)

            def e2e_step():
                return pl.compute_cem(xi_mean_host, Q0, np.zeros(6), np.zeros(6), TP, TR)

            for _ in range(max(args.warmup, 3)):                           # (the third tick captures the CUDA graph)
                e2e_step()
            barrier()
            e2e_ms = []
            for _ in range(args.steps):
                flush.fill_(1.0)
                torch.cuda.synchronize(dev)
                t0 = time.perf_counter()
                e2e_step()                                   # returns after its own stream synchronisation
                e2e_ms.append((time.perf_counter() - t0) * 1e3)
            barrier()
            res["e2e_tot_ms"] = max_over_ranks(sum(e2e_ms))
            res["e2e_value"] = Bg * T * args.steps / (res["e2e_tot_ms"] * 1e-3)
            res["overflow_samples"] = int(pl.overflow_samples)
        if with_kernel:
            xi, _ = pl.compute_xi_samples(key1, mean0, cov0)
            xi_f, thetadot = pl._project(xi, state_term, True)

            def rollout_only():
                pl._rollout(thetadot, q0, z6, tp, tr, False)

            for _ in range(2):
                rollout_only()
            res["roll_ms"] = float(np.mean(timed(rollout_only, args.steps)[0]))
            res["roll_ms_by_rank"] = all_ranks(res["roll_ms"])
            # this rank's own event time per iteration (includes its wait inside the all-gather for the slowest rank)
            res["iter_ms_by_rank"] = all_ranks(sum(ms) / args.steps)
        return res

    Bg_main = args.global_batch if args.global_batch > 0 else args.batch_per_gpu * world
    if Bg_main % world:
        raise SystemExit("--global-batch must be divisible by the number of GPUs")
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    main_res = measure(Bg_main, True, True, with_outputs=args.dump_outputs is not None and rank == 0)
    c5 = None
    if not args.no_config5 and args.global_batch == 0 and B_CONFIG5 % world == 0:
        c5 = measure(B_CONFIG5, False, False)
    if rank == 0:
        sampler.stop = True
        sampler.join(timeout=2)
    pl, Bl = main_res["pl"], main_res["Bl"]
    roll_avg = main_res["roll_ms"]
    steps_per_s_kernel = Bl * T / (roll_avg * 1e-3)
    prop = torch.cuda.get_device_properties(dev)
    peaks = {}
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            peaks = json.load(f)
    except Exception:
        pass
    sm_max = peaks.get("sm_max_mhz", 1965.0)
    fp32_nominal = prop.multi_processor_count * 128 * 2 * sm_max * 1e6 / 1e12
    import ctypes as C
    meas = C.c_double(0.0)
    pl._lib.cemk_fp32_fma_peak(pl._h, C.byref(meas))
    fp32_peak = meas.value if meas.value > 0 else fp32_nominal
    F_A, F_A_source = flop_per_env_step()
    achieved = steps_per_s_kernel * F_A / 1e12

    def shutdown():
        """Drop the captured graphs (they hold NCCL kernels) before the communicator goes; never let teardown hang the run."""
        sys.stdout.flush()
        if world > 1:
            threading.Timer(30.0, lambda: os._exit(0)).start()
            main_res["pl"].close()
            if c5 is not None:
                c5["pl"].close()
            torch.cuda.synchronize(dev)
            dist.destroy_process_group()
            os._exit(0)

    if rank != 0:
        shutdown()
        return
    traffic = None
    try:
        with open(os.path.join(ROOT, "profiles", "r2_final_k_rollout_metrics.json")) as f:
            traffic = float(json.load(f)["dram_traffic_bytes_per_launch"]) if Bl == B_PER_GPU else None
    except Exception:
        pass
    strong = args.global_batch > 0
    line = {
        "metric": METRIC, "value": main_res["value"], "unit": "env-steps/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": main_res["tot_ms"] / args.steps, "higher_is_better": True, "scaling": "strong" if strong else "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"UR5e+Hand-E scene A (ur5e_hande_mjx/scene.xml constants), {Bl} samples/GPU x {T} steps, dt={DT}, "
                               f"order-10 Bernstein, {PROJ_IT} projection iterations, elite {ELITE}, 1 CEM iteration per step",
                   "global_batch": Bg_main, "horizon": T, "parallelism": f"sample-sharded x{world}", "l2": "flushed (256 MB write) before every timed step"},
        "cem_iter_latency_ms": main_res["tot_ms"] / args.steps, "ms_per_step_rank0": main_res["ms_all"],
        "e2e": {"value": main_res["e2e_value"], "unit": "env-steps/s", "ms_per_step": main_res["e2e_tot_ms"] / args.steps,
                "h2d_bytes_per_step": int(pl.h2d_bytes), "d2h_bytes_per_step": int(pl.d2h_bytes),
                "cuda_graph": pl._graph is not None, "contact_overflow_samples": main_res["overflow_samples"]},
        "gpu_launches": int(main_res["launches"]),
        "roofline": {"bound": "fp32", "kernel": "k_rollout", "achieved": achieved, "peak": fp32_peak, "unit": "TFLOP/s",
                     "frac": achieved / fp32_peak, "traffic": traffic,
                     "peak_source": "FP32 FMA throughput measured live by cemk_fp32_fma_peak (8 independent register chains/thread); "
                                    f"nominal {prop.multi_processor_count} SMs x 128 lanes x 2 x {sm_max} MHz = {fp32_nominal:.1f} TFLOP/s (MEASURED_PEAKS.json holds no FP32 figure)",
                     "peak_nominal": fp32_nominal,
                     "flop_per_env_step": F_A, "flop_per_env_step_source": F_A_source, "kernel_ms": roll_avg,
                     "kernel_env_steps_per_s": steps_per_s_kernel,
                     "hbm_gbs": steps_per_s_kernel * HBM_BYTES_PER_ENV_STEP / 1e9, "hbm_peak_gbs": peaks.get("hbm_gbs")},
        "per_rank": {"k_rollout_ms": {"min": min(main_res["roll_ms_by_rank"]), "max": max(main_res["roll_ms_by_rank"]),
                                      "all": [round(v, 4) for v in main_res["roll_ms_by_rank"]]},
                     "iteration_ms": {"min": min(main_res["iter_ms_by_rank"]), "max": max(main_res["iter_ms_by_rank"]),
                                      "all": [round(v, 4) for v in main_res["iter_ms_by_rank"]]}},
        "clocks": sampler.summary(),
    }
    if c5 is not None:
        line["config5"] = {"workload": f"BASELINE config 5: {B_CONFIG5}-sample CEM iteration sharded over {world} GPU(s) ({c5['Bl']} samples/GPU, "
                                       f"strong scaling), T={T}", "value": c5["value"], "unit": "env-steps/s",
                           "ms_per_step": c5["tot_ms"] / args.steps, "scaling": "strong", "gpu_launches": int(c5["launches"])}
    if not args.no_cpu_baseline:
        line["cpu_baseline"] = cpu_baseline_record()
    if args.dump_outputs is not None:
        line["dumped_outputs"] = dump_outputs(args.dump_outputs, *main_res["outputs"])
    print(json.dumps(line))
    shutdown()


if __name__ == "__main__":
    main()
