#!/usr/bin/env python
"""Benchmark of the GP+ hot path on B200: MLL + gradient evaluations per second at N=16384, D=10,
Matern-5/2, FP64 (BASELINE.json configs[3]).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--n 16384] [--dump-outputs DIR]

A *step* is one evaluation of the negative log marginal likelihood and its gradient w.r.t. all 13
hyper-parameters on the full training set: fused covariance build, blocked DMMA Cholesky, triangular
inverse, alpha / log|K|, K^-1, fused gradient reduction.  Under torchrun every rank owns one GPU and
evaluates its own restarts (the path shards over independent restarts: weak scaling, no data-path
collective); ``value`` is the whole-job rate.

One JSON line is printed by rank 0 (see the keys at the bottom of ``main``).
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")  # before any CUDA context exists (see gpplus_b200/__init__.py)

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "gp-plus_b200"))

import bench_workloads as W  # noqa: E402

N_HEADLINE = W.N_HEADLINE
D = W.D
LOG2PI = 1.8378770664093453
GOLDEN = os.path.join(ROOT, "tests", "golden", "c4_n%d_matern52.json")

METRIC = "MLL+grad evals/sec (N=16k, fp64)"


def bench_config(n):
    """The ``config`` object of the JSON line -- byte-identical in both arms (ours / --impl reference)."""
    return {"workload": "synthetic exact GP N=%d D=10 Matern-5/2 FP64 MLL+gradient (bench_workloads.c4_workload)" % n,
            "points": "the 65 seeded prior draws of a 64-restart fit (torch.manual_seed(0); SURVEY 8(d)), cycled",
            "l2": "inputs larger than L2: each step streams three %.1f GiB work matrices" % (8.0 * n * n / 2 ** 30)}


def step_theta(thetas, k, rank=0):
    """theta of timed step k on ``rank``: prior draw 1 + (k + 8 rank) mod 65 (index 0 of ``thetas`` is theta_init)."""
    return thetas[1 + (k + 8 * rank) % W.N_PRIOR_DRAWS]


def dump_outputs(dirname, arrays):
    """``--dump-outputs``: every array of the last timed step as DIR/<name>.npy in float64, so that two builds can be
    compared output for output (the inputs are seeded: the same arguments give the same inputs)."""
    os.makedirs(dirname, exist_ok=True)
    for name, v in arrays.items():
        np.save(os.path.join(dirname, name + ".npy"), np.asarray(v, dtype=np.float64))


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, device):
        self.device, self.rows, self.proc = device, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.device), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def stop(self, t0, t1):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for t, line in self.rows:
            if t < t0 or t > t1 + 0.2:
                continue
            f = [s.strip() for s in line.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def measure_fp64_peak(device):
    """FP64 GEMM peak of this GPU, measured live the way MEASURED_PEAKS.json measures bf16: cuBLAS through
    torch.matmul on 8192^3, best of 10 (MEASURED_PEAKS.json has no FP64 entry)."""
    import torch
    a = torch.randn(8192, 8192, dtype=torch.float64, device="cuda:%d" % device)
    b = torch.randn(8192, 8192, dtype=torch.float64, device="cuda:%d" % device)
    best = 1e9
    for i in range(12):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        torch.matmul(a, b)
        e1.record()
        e1.synchronize()
        if i >= 2:
            best = min(best, e0.elapsed_time(e1))
    del a, b
    torch.cuda.empty_cache()
    return 2.0 * 8192 ** 3 / (best * 1e-3) / 1e12


def oracle_full_size(n, theta_list, threads=None, warm=True):
    """Wall seconds of REAL oracle MLL+gradient evaluations at the full size ``n`` (no extrapolation): the CPU
    restatement of the reference's torch path (oracle/gp_oracle.mll: dense float64 K, torch Cholesky, autograd), on
    ``threads`` host threads.  Returns ([seconds per evaluation], [oracle results], threads used)."""
    import torch
    from oracle import gp_oracle as O
    if threads:
        torch.set_num_threads(threads)
    if warm:  # page in torch / MKL before the clock starts
        O.mll(W.c4_oracle_problem(1024), W.c4_natural(theta_list[0]), want_grad=True)
    prob = W.c4_oracle_problem(n)
    secs, outs = [], []
    for th in theta_list:
        t0 = time.time()
        outs.append(O.mll(prob, W.c4_natural(th), want_grad=True))
        secs.append(time.time() - t0)
    return secs, outs, torch.get_num_threads()


# ------------------------------------------------------------------------------------------------
def run_reference(args):
    """The reference arm: the reference's own CPU torch path for this workload.  The reference itself cannot be
    imported where the benchmark runs (gpytorch / botorch are not installed, and the GP-Plus checkout is not part of
    this repository), so the CPU restatement in oracle/ -- pinned to the reference's own code by
    tests/test_reference_pin.py -- is timed (kind "port") with every host thread, at the FULL size, for exactly
    ``--steps`` evaluations (about 25 s each at N=16384 on 16 cores)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    thetas = W.c4_theta_points(W.c4_model(256))
    secs = []
    for k in range(args.steps):
        s, outs, threads = oracle_full_size(args.n, [step_theta(thetas, k)], cores, warm=(k == 0))
        secs += s
    steps_run = len(secs)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, outs[0])
    rate = steps_run / sum(secs)
    line = {
        "impl": "reference", "metric": METRIC, "value": rate, "unit": "evals/s",
        "n_gpus": args.gpus, "steps": steps_run, "warmup": 0, "steps_requested": args.steps,
        "warmup_requested": args.warmup,
        "ms_per_step": 1e3 * sum(secs) / steps_run, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic",
        "config": bench_config(args.n),
        "cpu_baseline": {"value": rate, "unit": "evals/s", "cores": threads, "kind": "port",
                         "sample": "%d real oracle MLL+grad evaluation(s) at the full N=%d on the first timed theta "
                                   "points (%s s each); no extrapolation" % (
                                       steps_run, args.n, ", ".join("%.1f" % v for v in secs))},
        "e2e": {"value": rate, "unit": "evals/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def check_parity(n, results_by_index):
    """Compare engine results at the golden theta points with the committed oracle output (N=16384 only)."""
    path = GOLDEN % n
    if not os.path.exists(path):
        return None
    gold = json.load(open(path))
    rel_nll, rel_grad, pts = 0.0, 0.0, []
    for pt in gold["points"]:
        out = results_by_index.get(pt["index"])
        if out is None:
            continue
        g = np.concatenate([out["d_w"], [out["d_sigma_f2"]], out["d_noise"], out["d_beta"]])
        gr = np.concatenate([np.asarray(pt["d_w"]), [pt["d_sigma_f2"]], np.asarray(pt["d_noise"]), np.asarray(pt["d_beta"])])
        rel_nll = max(rel_nll, abs(out["nll"] - pt["nll"]) / abs(pt["nll"]))
        rel_grad = max(rel_grad, float(np.max(np.abs(g - gr)) / np.max(np.abs(gr))))
        pts.append(pt["index"])
    par = {"rel_nll": rel_nll, "rel_grad": rel_grad, "points": pts, "tol_nll": 1e-9, "tol_grad": 1e-8,
           "against": "tests/golden/c4_n%d_matern52.json (CPU oracle at the full size; point 1 is the first timed theta)" % n}
    if not (rel_nll <= 1e-9 and rel_grad <= 1e-8):
        raise SystemExit("bench.py: parity check FAILED against the committed oracle output: %s" % json.dumps(par))
    return par


def _other_denominators(ach_all, ach_largest):
    """The same achieved INT8 rate against the driver-measured tensor peak: MEASURED_PEAKS.json has a cuBLAS bf16 number
    only; dense INT8 is nominally 2x bf16 on this part (4.5 vs 2.25 P), so 2 x bf16_tflops is the library-GEMM-grade
    INT8 yardstick next to the raw issue rate used for `frac`."""
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        mp = json.load(open(path))
        bf = float(mp["bf16_tflops"])
        sus = float(mp.get("bf16_tflops_sustained", bf))
    except Exception:
        return None
    return {"measured_bf16_tflops_burst": bf, "measured_bf16_tflops_sustained": sus,
            "frac_of_2x_measured_bf16_burst": ach_all / (2.0 * bf), "frac_of_2x_measured_bf16_sustained": ach_all / (2.0 * sus),
            "largest_launch_frac_of_2x_measured_bf16_burst": ach_largest / (2.0 * bf),
            "nominal_int8_tops": 4500.0, "frac_of_nominal": ach_all / 4500.0,
            "source": "MEASURED_PEAKS.json (driver-written: torch.matmul bf16 8192^3)"}


def run_ours(args):
    import torch
    import torch.distributed as dist
    from gpplus_b200 import _engine as E
    from gpplus_b200.models.gpregression import set_default_device
    from gpplus_b200.optim.mll_scipy import MLLObjective

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available() or E.device_count() < 1:
        raise SystemExit("bench.py: no CUDA device -- the engine has no CPU path")
    torch.cuda.set_device(local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    set_default_device(local)

    n = args.n
    model = W.c4_model(n)
    thetas = W.c4_theta_points(model)
    obj = MLLObjective(model, True, [0, 0])
    eng = model._get_engine()

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident arm: X, y already in HBM, one gpp_mll_grad per step -------------------------------
    for k in range(args.warmup):
        eng.mll_grad(W.c4_natural(step_theta(thetas, -1 - k, rank)), want_grad=True)
    hypers = [W.c4_natural(step_theta(thetas, k, rank)) for k in range(args.steps)]
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
        time.sleep(0.3)
    barrier()
    st0 = eng.stats()
    l0 = E.launch_count()
    t0 = time.time()
    stage = {k: 0.0 for k in ("covariance", "cholesky", "trtri", "solve", "lauum", "gradient", "total")}
    first_out = None
    for k in range(args.steps):
        out = eng.mll_grad(hypers[k], want_grad=True)
        if k == 0:
            first_out = out
        tm = eng.timings()  # CUDA events recorded on the engine's own stream inside the call
        for s in stage:
            stage[s] += tm[s]
    barrier()
    t1 = time.time()
    launches = E.launch_count() - l0
    st1 = eng.stats()
    clocks = sampler.stop(t0, t1) if rank == 0 else None
    # two clocks, both max over ranks: wall time between the barriers (what `value` uses: it contains everything a
    # caller pays) and the device time of the K steps from CUDA events recorded on the engine's own stream
    both = torch.tensor([t1 - t0, stage["total"] * 1e-3], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(both, op=dist.ReduceOp.MAX)
    elapsed, device_elapsed = float(both[0]), float(both[1])
    value = world * args.steps / elapsed
    for s in stage:
        stage[s] /= args.steps

    # ---- end-to-end arm: the public API call (MLLObjective.fun), theta from host memory, result to host ----
    # fit_model_scipy's restart workers call the objective through the validated native layout (gpp_objective);
    # that is the call timed here.  MLLObjective.fun (torch path, +1.4 ms of host work) returns the same values.
    objective = obj.fun_fast if obj.enable_fast_path() else obj.fun
    for k in range(min(2, args.warmup)):
        objective(step_theta(thetas, -1 - k, rank))
    barrier()
    t0 = time.time()
    for k in range(args.steps):
        f, g = objective(step_theta(thetas, k, rank))
    barrier()
    e2e_elapsed = torch.tensor([time.time() - t0], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(e2e_elapsed, op=dist.ReduceOp.MAX)
    e2e_value = world * args.steps / float(e2e_elapsed)
    h2d = 8 * (eng.dq + eng.n_combo * eng.dz + eng.n_noise + eng.n_mean + 2)
    d2h = 8 * (4 + eng.dq + eng.n_noise + eng.n_mean) + 4
    if args.dump_outputs and rank == 0:
        # the last step of each timed arm: gpp_mll_grad's result dictionary, and (value, gradient) of the objective
        dump_outputs(args.dump_outputs, dict(out, objective_value=f, objective_grad=g))

    # ---- the sharded workloads of the metric's second half, in the same torchrun world (every rank takes part) ----
    extra = {}
    if not args.no_extras:
        model.release_engine()
        eng = None
        barrier()
        extra["fit_c2"] = fit_core(args, world, rank, local, "c2", 0)
        barrier()
        extra["acq_c5"] = acq_core(args, world, rank, local, steps=3)
        barrier()

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- parity at the timed points + the SURVEY 8(d) protocol over all 65 prior draws (rank 0, untimed region) ----
    if eng is None:
        eng = model._get_engine()
    results = {1: first_out, 0: eng.mll_grad(W.c4_natural(thetas[0]), want_grad=True),
               2: eng.mll_grad(W.c4_natural(thetas[2]), want_grad=True)}
    parity = check_parity(n, results)
    t_init = []
    for _ in range(3):
        eng.mll_grad(W.c4_natural(thetas[0]), want_grad=True)
        t_init.append(eng.timings()["total"])
    per_draw, retried = [], []
    sa = eng.stats()
    for k in range(1, 1 + (0 if args.no_prior_sweep else W.N_PRIOR_DRAWS)):
        s_before = eng.stats()["jitter_retries"]
        tq = time.time()
        try:
            eng.mll_grad(W.c4_natural(thetas[k]), want_grad=True)
            ok = True
        except (E.NotPSDError, E.NanError):
            ok = False
        ms = 1e3 * (time.time() - tq)
        r = eng.stats()["jitter_retries"] - s_before
        (retried if (r > 0 or not ok) else per_draw).append((ms, r))
    sb = eng.stats()
    clean = [m for m, _ in per_draw]
    n_retry = sum(r for _, r in retried)
    prior_draws = None if args.no_prior_sweep else {
        "n": W.N_PRIOR_DRAWS, "median_ms": statistics.median(clean) if clean else None,
        "mean_ms": sum(clean) / len(clean) if clean else None, "draws_needing_jitter": len(retried),
        "retries": int(sb["jitter_retries"] - sa["jitter_retries"]), "early_outs": int(sb["early_outs"] - sa["early_outs"]),
        "ms_per_retry": ((sum(m for m, _ in retried) - len(retried) * statistics.median(clean)) / n_retry)
        if (n_retry > 0 and clean) else None,
        "theta_init_ms": statistics.median(t_init),
        "note": "wall ms per evaluation at every seeded prior draw; evaluations that needed the jitter ladder are "
                "counted separately (a failed rung costs covariance + factorisation only: the status is read back "
                "before the inverse / K^-1 / gradient are enqueued)"}

    # ---- roofline of the dominant kernel -------------------------------------------------------------------------
    # The three O(N^3) stages (factorisation trailing updates, L^-1, K^-1) run either on the INT8-sliced tcgen05 GEMM
    # (oz_gemm_kernel; default from N = 3072) or on the FP64 DMMA GEMM (dgemm_dmma_kernel; GPP_FP64=dmma).
    fp64_mode = eng.fp64_mode()
    peak = measure_fp64_peak(local)
    n3 = float(n) ** 3
    tensor_ms = stage["cholesky"] + stage["trtri"] + stage["lauum"]
    if tensor_ms <= 0.0:  # CUDA-graph replay (N <= 2048): only the total is timed
        tensor_ms = stage["total"]
        for k in ("cholesky", "trtri", "lauum", "covariance", "gradient"):
            stage[k] = stage[k] or float("nan")
    achieved = n3 / (tensor_ms * 1e-3) / 1e12  # N^3/3 (potrf) + N^3/3 (trtri) + N^3/3 (lauum) algorithmic flops

    def _traffic(name):
        tpath = os.path.join(ROOT, "profiles", name)
        if os.path.exists(tpath):
            try:
                return json.load(open(tpath)).get("dram_bytes_per_launch")
            except Exception:
                return None
        return None

    stage_extra = {
        "stages_ms": stage,
        # the leading part of L^-1 runs on a low-priority stream behind the factorisation (trtri_early), so the
        # event split between "cholesky" and "trtri" is not a split of work; their sum is (GPP_OVERLAP_INV=0
        # separates them)
        "stage_tflops": {"cholesky_plus_trtri": 2 * n3 / 3 / ((stage["cholesky"] + stage["trtri"]) * 1e-3) / 1e12,
                         "lauum": n3 / 3 / (stage["lauum"] * 1e-3) / 1e12},
        "hbm_stage_gbs": {"covariance": 4.0 * n * (n + 1) / (stage["covariance"] * 1e-3) / 1e9,
                          "gradient": 4.0 * n * (n + 1) / (stage["gradient"] * 1e-3) / 1e9},
    }
    if fp64_mode == E.FP64_INT8:
        peak_i8 = E.probe_i8(256, 4096, local)     # raw tcgen05 kind::i8 issue rate, whole GPU, measured live
        peak_i8_n128 = E.probe_i8(128, 4096, local)
        pairs = 28.0                                # int8 multiply-adds per FP64-equivalent multiply-add
        kinv_pairs = {7: 28.0, 6: 21.0, 5: 15.0}.get(int(os.environ.get("GPP_OZ_KINV_LEVELS", "7")), 28.0)  # K^-1 product
        ops_eval = (2.0 * pairs + kinv_pairs) * n3 / 3.0   # potrf + trtri with 28 plane pairs, K^-1 with 28 (21 with GPP_OZ_KINV_LEVELS=6)
        ach_i8 = ops_eval / (tensor_ms * 1e-3) / 1e12
        roofline = {
            "bound": "tensor", "kernel": "oz_gemm_kernel (tcgen05.mma kind::i8 M=N=128 K=32, TMA-fed, int32 TMEM "
                                         "accumulators; 7 digit planes per operand, 28 plane pairs)",
            "achieved": ach_i8, "peak": peak_i8, "unit": "TOP/s (int8)", "frac": ach_i8 / peak_i8,
            "traffic": _traffic("oz_gemm_traffic.json"),
            "peak_source": "measured live: gpp_probe_i8 (tcgen05.mma kind::i8 M=128 N=256 issued back to back on "
                           "resident operands, 148 SMs); the N=128 shape the kernel uses issues at %.0f TOP/s; "
                           "MEASURED_PEAKS.json has no INT8 entry (nominal 4500)" % peak_i8_n128,
            "algorithmic_ops_per_eval": ops_eval,
            "basis": "all O(N^3) work of one step: N^3 FP64-equivalent flops (potrf + trtri + lauum, N^3/3 each) = "
                     "(28 + 28 + %d) N^3 / 3 int8 ops actually issued (28 plane pairs per product; K^-1, which only feeds the "
                     "gradient trace, can run with 21: GPP_OZ_KINV_LEVELS=6), over the CUDA-event time of those three stages (digit-plane splits, DMMA "
                     "panel chain, leaf kernels and launch gaps included)" % kinv_pairs,
            "largest_launch": {"what": "K^-1 = L^-T L^-1: transposed digit-plane split + one oz_gemm launch, %d plane pairs" % kinv_pairs,
                               "algorithmic_ops": kinv_pairs * n3 / 3, "ms": stage["lauum"],
                               "achieved": kinv_pairs * n3 / 3 / (stage["lauum"] * 1e-3) / 1e12,
                               "frac": kinv_pairs * n3 / 3 / (stage["lauum"] * 1e-3) / 1e12 / peak_i8},
            "other_denominators": _other_denominators(ach_i8, kinv_pairs * n3 / 3 / (stage["lauum"] * 1e-3) / 1e12),
            "fp64_equivalent": {"achieved_tflops": achieved, "fp64_tensor_peak_tflops": peak,
                                "ratio_to_fp64_tensor_peak": achieved / peak,
                                "peak_source": "torch.matmul f64 8192^3 best of 10 (cuBLAS DGEMM), measured live"},
        }
    else:
        roofline = {
            "bound": "tensor", "kernel": "dgemm_dmma_kernel (FP64 DMMA m8n8k4)", "achieved": achieved, "peak": peak,
            "unit": "TFLOP/s", "frac": achieved / peak, "traffic": _traffic("dgemm_traffic.json"),
            "peak_source": "measured live: torch.matmul f64 8192^3 best of 10 (cuBLAS); MEASURED_PEAKS.json has no FP64 entry",
            "algorithmic_flops_per_eval": n3,
            "basis": "all launches of the kernel in one step: N^3 algorithmic flops (potrf + trtri + lauum, N^3/3 each) over "
                     "the CUDA-event time of those three stages (leaf kernels and launch gaps included); `traffic` is the "
                     "ncu DRAM read+write of the single largest launch (LAUUM, N^3/3 flops), see profiles/dgemm_traffic.json",
            "largest_launch": {"what": "LAUUM K^-1 = L^-T L^-1, one launch", "algorithmic_flops": n3 / 3,
                               "ms": stage["lauum"], "achieved": n3 / 3 / (stage["lauum"] * 1e-3) / 1e12,
                               "frac": n3 / 3 / (stage["lauum"] * 1e-3) / 1e12 / peak},
        }
    roofline.update(stage_extra)

    # ---- the exact-DMMA arm of the same evaluation (IEEE FP64 products on mma.sync), rank 0, outside the timed region ----
    exact_dmma = None
    if fp64_mode == E.FP64_INT8 and not args.no_dmma_arm:
        model.release_engine()
        eng = None
        prev = E.set_fp64_mode(E.FP64_DMMA)
        try:
            eng2 = model._get_engine()
            eng2.mll_grad(W.c4_natural(thetas[2]), want_grad=True)
            res2, tms, st2 = {}, [], {k: 0.0 for k in ("cholesky", "trtri", "lauum")}
            for k in (1, 0, 2):
                res2[k] = eng2.mll_grad(W.c4_natural(thetas[k]), want_grad=True)
                tm = eng2.timings()
                tms.append(tm["total"])
                for q in st2:
                    st2[q] += tm[q] / 3.0
            par2 = check_parity(n, res2)
            t2 = sum(st2.values())
            exact_dmma = {"ms_per_step": statistics.median(tms), "value": 1e3 / statistics.median(tms), "unit": "evals/s",
                          "steps": 3, "parity": {"rel_nll": par2["rel_nll"], "rel_grad": par2["rel_grad"]},
                          "roofline": {"kernel": "dgemm_dmma_kernel (FP64 DMMA m8n8k4)", "achieved": n3 / (t2 * 1e-3) / 1e12,
                                       "peak": peak, "unit": "TFLOP/s", "frac": n3 / (t2 * 1e-3) / 1e12 / peak,
                                       "stages_ms": st2},
                          "int8_vs_dmma_rel_nll": abs(res2[1]["nll"] - first_out["nll"]) / abs(res2[1]["nll"]),
                          "note": "same engine with GPP_FP64=dmma (gpp_set_fp64_mode(0)): every product in IEEE FP64 on the "
                                  "DMMA tensor cores; device ms per evaluation from CUDA events"}
        finally:
            E.set_fp64_mode(prev)
            model.release_engine()

    # ---- CPU baseline: the oracle on this box's host cores, ONE real full-size evaluation (N=1 runs only) ----
    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        cores = os.cpu_count() or 1
        secs, outs, threads = oracle_full_size(n, [thetas[1]], cores)
        cpu = {"value": 1.0 / secs[0], "unit": "evals/s", "cores": threads, "kind": "port",
               "sample": "1 real oracle MLL+grad evaluation at the full N=%d on the first timed theta (%.1f s); no "
                         "extrapolation" % (n, secs[0]),
               "oracle_vs_engine_rel_nll": abs(outs[0]["nll"] - first_out["nll"]) / abs(outs[0]["nll"])}

    line = {
        "metric": METRIC, "value": value, "unit": "evals/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * elapsed / args.steps,
        "device_ms_per_step": 1e3 * device_elapsed / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "fp64_arithmetic": ("int8-sliced: FP64 operands cut into 7 signed base-256 digit planes per power-of-two-scaled row, "
                            "exact integer products on tcgen05 kind::i8, FP64 recombination and accumulation (results "
                            "within 1e-12 of the DMMA arm, see parity / exact_dmma)") if fp64_mode == E.FP64_INT8
        else "IEEE FP64 products on DMMA (mma.sync m8n8k4)",
        "config": bench_config(n),
        "parallelism": "independent restarts, one per GPU (no data-path collective)",
        "nll_first_step": first_out["nll"],
        "jitter_retries_in_timed_region": int(st1["jitter_retries"] - st0["jitter_retries"]),
        "e2e": {"value": e2e_value, "unit": "evals/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "api": "the objective fit_model_scipy hands to scipy: theta (host, float64) -> float32 cast, raw->natural "
                       "transforms, device evaluation, priors and chain rule (gpp_objective) -> (value, gradient) on "
                       "the host"},
        "gpu_launches": launches,
        "clocks": clocks,
        "roofline": roofline,
        "cpu_baseline": cpu,
        "parity": parity,
        "prior_draws": prior_draws,
        "exact_dmma": exact_dmma,
        "extra": extra,
    }
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


# ------------------------------------------------------------------------------------------------
# secondary workloads (not the driver's default line): BASELINE configs[1] and configs[4]
def _dist_setup():
    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    return world, rank, local


def _c2_problem():
    """Borehole mixed-variable emulation with a categorical latent map (Example 02): n=500, two categorical
    inputs x 5 levels, weighted rough-RBF kernel."""
    import torch
    from gpplus_b200.preprocessing import train_test_split_normalizeX
    from gpplus_b200.test_functions import borehole_mixed_variables
    from gpplus_b200.utils import set_seed
    set_seed(4)
    qd = {0: 5, 5: 5}
    X, y = borehole_mixed_variables(n=2000, qual_dict=qd, random_state=4)
    Xtr, Xte, ytr, yte = train_test_split_normalizeX(X, y, test_size=0.75, qual_dict=qd)
    return Xtr, ytr, Xte, yte, qd


def fit_core(args, world, rank, local, fit_config, maxiter):
    """64-restart multi-start MAP fit (fit_model_scipy, L-BFGS-B, reference defaults) in the current process group:
    restarts are claimed from the cross-rank work queue.  Returns the result dictionary on every rank."""
    import torch
    from gpplus_b200 import _engine as E
    from gpplus_b200.models import GP_Plus
    from gpplus_b200.optim import fit_model_scipy
    from gpplus_b200.optim.mll_scipy import _sample_from_prior
    options = {"maxiter": maxiter} if maxiter > 0 else {}
    if fit_config == "c4":
        X, y = W.c4_workload(args.n)
        Xtr, ytr = torch.from_numpy(X[: args.n - 256]), torch.from_numpy(y[: args.n - 256])
        Xte, yte = torch.from_numpy(X[args.n - 256:]), torch.from_numpy(y[args.n - 256:])
        model = GP_Plus(Xtr, ytr, dtype=torch.float64, quant_correlation_class="Matern52Kernel")
        what = "synthetic wing N=%d D=10 Matern-5/2, %d restarts (+1), L-BFGS-B%s" % (
            Xtr.shape[0], args.restarts, " maxiter=%d" % maxiter if maxiter > 0 else " reference defaults")
    else:
        Xtr, ytr, Xte, yte, qd = _c2_problem()
        model = GP_Plus(Xtr, ytr, qual_dict=qd, dtype=torch.float64)
        what = "borehole mixed-variable, n=%d, 2 categorical x 5 levels, rough-RBF x latent map, %d restarts (+1), " \
               "L-BFGS-B reference defaults" % (Xtr.shape[0], args.restarts)
    torch.manual_seed(0)
    theta0 = [_sample_from_prior(model) for _ in range(args.restarts + 1)]

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            import torch.distributed as dist
            dist.barrier()

    cold = None
    if fit_config == "c4":
        fit_model_scipy(model, num_restarts=0, theta0_list=theta0[:world], options={"maxiter": 1})  # warm-up
    else:
        # first fit of this shape in the process: includes creating the engine handles (up to 64 per GPU) and
        # capturing their CUDA graphs; the handles are then parked in the library's pool and the SECOND, timed fit
        # reuses them -- the steady state of BO / continuation loops, which refit the same shape many times
        sync_all()
        tc = time.time()
        fit_model_scipy(model, add_prior=True, num_restarts=args.restarts, theta0_list=theta0, options=options)
        torch.cuda.synchronize()
        cold = torch.tensor([time.time() - tc], dtype=torch.float64, device="cuda")
        if world > 1:
            import torch.distributed as dist
            dist.all_reduce(cold, op=dist.ReduceOp.MAX)
        cold = float(cold)
        model = GP_Plus(Xtr, ytr, qual_dict=qd, dtype=torch.float64)
    sync_all()
    l0 = E.launch_count()
    t0 = time.time()
    res, best = fit_model_scipy(model, add_prior=True, num_restarts=args.restarts, theta0_list=theta0, options=options)
    torch.cuda.synchronize()
    dt = torch.tensor([time.time() - t0], dtype=torch.float64, device="cuda")
    mine = torch.tensor([float(sum(1 for r in res if not isinstance(r, Exception) and
                                   getattr(r, "message", "") != "gathered from another rank"))],
                        dtype=torch.float64, device="cuda")
    per_rank = [mine.clone() for _ in range(world)]
    if world > 1:
        import torch.distributed as dist
        dist.all_reduce(dt, op=dist.ReduceOp.MAX)
        dist.all_gather(per_rank, mine)
    dt = float(dt)
    nfev = sum(int(r.nfev) for r in res if not isinstance(r, Exception))
    failed = sum(1 for r in res if isinstance(r, Exception))
    mu = model.predict(Xte, return_std=False)
    rrmse = float(torch.sqrt(torch.mean((mu - yte) ** 2)) / yte.std())
    model.release_engine()
    return {"metric": "64-restart fit time", "value": dt, "unit": "s", "n_gpus": world, "higher_is_better": False,
            "scaling": "strong", "dtype": "f64", "data": "synthetic", "config": {"workload": what},
            "objective_evals": nfev, "evals_per_s": nfev / dt, "failed_starts": failed,
            "best_neg_log_posterior": float(best), "test_rrmse": rrmse,
            "restarts_run_per_rank": [int(float(v)) for v in per_rank],
            "first_fit_s": cold,
            "protocol": "value = second fit of the same shape in the process (engine handles reused from the pool); "
                        "first_fit_s = the first one, handle creation and graph capture included",
            "gpu_launches_rank0": E.launch_count() - l0}


def run_fit(args):
    """``--workload fit``: the 64-restart fit alone (configs[1] by default, ``--fit-config c4`` for configs[3])."""
    from gpplus_b200.models.gpregression import set_default_device
    if args.impl == "reference":
        return run_fit_reference(args)
    world, rank, local = _dist_setup()
    set_default_device(local)
    out = fit_core(args, world, rank, local, args.fit_config, args.maxiter)
    if rank == 0:
        print(json.dumps(out), flush=True)
    if world > 1:
        import torch.distributed as dist
        dist.destroy_process_group()


def run_fit_reference(args):
    """CPU arm of the fit workload: the model-level oracle (the reference's torch path restated) driven by the same
    scipy L-BFGS-B, from the same starts, on a bounded number of restarts; scaled to restarts+1 runs spread over
    the host cores the way joblib(n_jobs=-1) would."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    import torch
    from scipy.optimize import minimize
    from gpplus_b200.models import GP_Plus
    from gpplus_b200.optim.mll_scipy import _sample_from_prior
    from oracle import gpplus_oracle as GO
    Xtr, ytr, Xte, yte, qd = _c2_problem()
    model = GP_Plus(Xtr, ytr, qual_dict=qd, dtype=torch.float64)
    torch.manual_seed(0)
    theta0 = [_sample_from_prior(model) for _ in range(args.restarts + 1)]
    spec = {"X": Xtr.numpy(), "y": ytr.numpy(), "qual_dict": qd, "kernel": "Rough_RBF"}
    torch.set_num_threads(1)  # one restart per core, as loky workers do
    sample = min(3, len(theta0))
    t0 = time.time()
    nfev = 0
    for th in theta0[:sample]:
        try:
            r = minimize(lambda x: GO.neg_log_posterior(spec, x), th, jac=True, method="L-BFGS-B",
                         options={"ftol": 1e-6, "gtol": 1e-5, "maxfun": 5000, "maxiter": 2000})
            nfev += int(r.nfev)
        except Exception:
            pass
    dt = time.time() - t0
    cores = os.cpu_count() or 1
    waves = -(-(args.restarts + 1) // cores)
    est = dt / sample * waves
    print(json.dumps({
        "impl": "reference", "metric": "64-restart fit time", "value": est, "unit": "s", "higher_is_better": False,
        "config": {"workload": "borehole mixed-variable, n=%d, %d restarts (+1)" % (Xtr.shape[0], args.restarts)},
        "cpu_baseline": {"value": est, "unit": "s", "cores": cores, "kind": "port",
                         "sample": "%d sequential single-thread oracle L-BFGS-B runs (%.1f s, %d evals), scaled to "
                                   "ceil(%d/%d) waves of one run per core" % (sample, dt, nfev, args.restarts + 1, cores)}
    }), flush=True)


def acq_core(args, world, rank, local, steps):
    """MFBO borehole (Example 04): predictive mean/variance + cost-aware acquisition + arg-max over M candidates,
    candidates sharded over the ranks of the current process group.  Returns the result dictionary on every rank."""
    import torch
    from gpplus_b200.bayesian_optimizations import (acquisition_table_argmax, prepare_candidate_table,
                                                    score_prepared, to_device)
    from gpplus_b200.models import GP_Plus
    from gpplus_b200.optim import fit_model_scipy
    from gpplus_b200.preprocessing.normalizeX import standard
    from gpplus_b200.test_functions.multi_fidelity import BH_MAX, BH_MIN, Borehole_MF_BO
    from scipy.stats.qmc import Sobol, scale
    np.random.seed(0)
    torch.manual_seed(0)
    qd = {8: 5}
    U, y = Borehole_MF_BO(True, {"0": 5, "1": 5, "2": 50, "3": 5, "4": 50})
    U, umean, ustd = standard(torch.tensor(U), qd)
    model = GP_Plus(U, torch.tensor(y).reshape(-1), qual_dict=qd, dtype=torch.float64, multiple_noise=False)
    fit_model_scipy(model, num_restarts=8, bounds=True)
    M = args.candidates
    cand = scale(Sobol(d=8, seed=1).random(M), l_bounds=BH_MIN, u_bounds=BH_MAX)
    cand = (cand - umean.numpy()) / ustd.numpy()
    src = np.random.RandomState(1).randint(0, 5, size=(M, 1)).astype(np.float64)
    table = np.hstack([cand, src])
    costs = [1000.0, 100.0, 10.0, 100.0, 10.0]
    ytr = torch.tensor(y).reshape(-1)
    best = [float(ytr[U[:, -1] == i].min()) for i in range(5)]
    acquisition_table_argmax(model, table[:4096], best, costs, maximize=False)  # warm-up
    torch.cuda.synchronize()

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            import torch.distributed as dist
            dist.barrier()

    # end-to-end arm: candidate table in HOST memory (ordering, level lookup, H2D, scoring, arg-max over ranks);
    # timed from PINNED host memory (the bench contract's e2e definition) and from a pageable numpy array
    table_pinned = torch.from_numpy(table).pin_memory()
    acquisition_table_argmax(model, table_pinned, best, costs, maximize=False)
    e2e_times, pageable_times = [], []
    for _ in range(max(1, steps)):
        sync_all()
        t0 = time.time()
        score_p, idx_p, order_p = acquisition_table_argmax(model, table, best, costs, maximize=False)
        sync_all()
        pageable_times.append(time.time() - t0)
        sync_all()
        t0 = time.time()
        score, idx, order = acquisition_table_argmax(model, table_pinned, best, costs, maximize=False)
        sync_all()
        e2e_times.append(time.time() - t0)
    assert idx_p == idx and score_p == score, "pinned and pageable tables disagree"
    # device-resident arm: this rank's chunk prepared once and already in HBM when the timed region starts
    prep = to_device(prepare_candidate_table(model, table, 5), local)
    score_prepared(model, prep, best, costs, maximize=False)
    dev_times = []
    for _ in range(max(3, steps)):
        sync_all()
        t0 = time.time()
        score_d, idx_d = score_prepared(model, prep, best, costs, maximize=False)
        sync_all()
        dev_times.append(time.time() - t0)
    assert idx_d == idx and score_d == score, "device-resident and host paths disagree"
    both = torch.tensor([min(e2e_times), min(dev_times), min(pageable_times)], dtype=torch.float64, device="cuda")
    if world > 1:
        import torch.distributed as dist
        dist.all_reduce(both, op=dist.ReduceOp.MAX)
    dt_e2e, dt_dev, dt_pageable = float(both[0]), float(both[1]), float(both[2])
    n_tr = int(U.shape[0])
    model.release_engine()
    return {
        "metric": "acquisition candidates/sec (predict mean/var + AF + arg-max)", "value": M / dt_dev,
        "unit": "candidates/s", "n_gpus": world, "higher_is_better": True, "scaling": "strong", "dtype": "f64",
        "data": "synthetic", "ms_per_step": 1e3 * dt_dev,
        "config": {"workload": "MFBO borehole, n_train=%d, 5 sources, %d Sobol candidates split in contiguous "
                               "chunks over the ranks; value: chunks resident in HBM" % (n_tr, M)},
        "e2e": {"value": M / dt_e2e, "unit": "candidates/s", "ms_per_step": 1e3 * dt_e2e,
                "h2d_bytes_per_step": int(M * 9 * 8), "d2h_bytes_per_step": 16,
                "from_pageable_numpy_ms": 1e3 * dt_pageable,
                "api": "bayesian_optimizations.acquisition_table_argmax(model, table) with the table in PINNED host "
                       "memory: H2D of the whole table, source-major ordering and level lookup on the device, fused "
                       "predict+AF+arg-max, arg-max over ranks"},
        "best": {"score": score, "index": int(idx), "table_row": int(order[int(idx)])}}


def run_acq(args):
    """``--workload acq``: BASELINE configs[4] alone."""
    from gpplus_b200.models.gpregression import set_default_device
    world, rank, local = _dist_setup()
    set_default_device(local)
    out = acq_core(args, world, rank, local, args.steps)
    if rank == 0:
        print(json.dumps(out), flush=True)
    if world > 1:
        import torch.distributed as dist
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--n", "--size", dest="n", type=int, default=N_HEADLINE,
                    help="training-set size (use --size under torchrun: its own parser claims the prefix --n)")
    ap.add_argument("--workload", default="mll", choices=["mll", "fit", "acq"],
                    help="mll (default, the headline metric) | fit: 64-restart fit of BASELINE configs[1] | "
                         "acq: predictive mean/var + acquisition arg-max over --candidates (configs[4])")
    ap.add_argument("--restarts", type=int, default=64)
    ap.add_argument("--maxiter", type=int, default=0, help="fit workload: cap on L-BFGS-B iterations (0 = reference default)")
    ap.add_argument("--fit-config", default="c2", choices=["c2", "c4"],
                    help="fit workload: c2 = borehole mixed n=500 (configs[1]); c4 = synthetic N=--n D=10 Matern-5/2 (configs[3])")
    ap.add_argument("--candidates", type=int, default=1000000)
    ap.add_argument("--no-extras", action="store_true",
                    help="mll workload: skip extra.fit_c2 / extra.acq_c5 (the sharded workloads of the metric's second half)")
    ap.add_argument("--no-cpu-baseline", action="store_true", help="mll workload: skip the full-size CPU oracle evaluation")
    ap.add_argument("--no-dmma-arm", action="store_true", help="mll workload: skip the exact-DMMA arm of the same evaluation")
    ap.add_argument("--no-prior-sweep", action="store_true",
                    help="mll workload: skip the untimed sweep over all 65 prior draws (profiling runs)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="mll workload: write what the last timed step computed to DIR/<name>.npy (float64, a few "
                         "hundred bytes in all)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.workload != "mll":
        ap.error("--dump-outputs applies to the mll workload only")
    if args.warmup < 3 and args.impl == "ours" and args.workload == "mll":
        args.warmup = 3
    if args.workload == "fit":
        run_fit(args)
    elif args.workload == "acq":
        run_acq(args)
    elif args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
