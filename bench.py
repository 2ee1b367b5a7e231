#!/usr/bin/env python
"""bench.py -- BioEn optimisation hot path on B200: gradient (f+g) evaluations per second and time to optimum.

Workload (BASELINE.json `metric`): log-weights method, synthetic "generic data" (SURVEY.md 8d: seed 12345,
sig_exp 0.5, sig_sim 1, uniform w0, G = 0), N = 1e6 structures x M = 1e3 observables per GPU, theta = 10, fp64.
One "step" = one evaluation of the log-posterior AND its gradient at a fresh point (2 passes over yTilde).

  value            steps / device time, yTilde + all vectors resident in HBM (CUDA events, max over ranks)
  e2e              the same through the C ABI with HOST vectors (bioen_b200_eval): every step copies g from pinned
                   host memory to the device and reads the objective and the gradient back
  roofline         the dominant kernel (stream_pass_kernel, one pass over yTilde = M*N*8 algorithmic bytes per
                   launch), timed live with CUDA events around every launch inside the timed region
  time_to_optimum  device L-BFGS (BioEn defaults) from x0 = 0; `.reference` = what the reference arm of the same
                   round-end run measured on the same problem (seconds, fmin, iterations) and the fmin difference;
                   `.coefficient_space_update` = the same with the opt-in 2-kernel L-BFGS update
  dropin_time_to_optimum  host NumPy arrays in -> optimum out through the reference-facing entry points
                   (c_bioen.bioen_opt_lbfgs_logw, optimize.log_weights.find_optimum)
  cpu_baseline     the reference's own OpenMP C kernels (oracle/_ref) on the host cores, bounded column sample
  extra_workloads  the other BASELINE configs, measured after the timed region: the forces method on the same matrix,
                   the 32-theta batched scan (config 4), the opt-in fp32 storage, config 2 (500 x 1e5), the ala5
                   shape (config 1); at N > 1 the strong-scaled config 3 and a config-5 shard (5000 x 1.25e6) per GPU
  sharded_checks   N > 1: the sharded result through the fused peer-memory exchange vs NCCL, identical f on all ranks,
                   f against an independent recombination (1e-12)

N > 1 (torchrun): the structure axis is sharded, every rank holds N = 1e6 columns (weak scaling), ONE exchange of
M+5 doubles per objective half and one of 4 scalars per gradient half, issued from inside the producing kernels over
NVLink peer memory (`run_info.exchange` = "p2p"; "nccl" when peer mapping is unavailable or BIOEN_B200_P2P=0);
`value` counts 1e6-structure evaluations per second summed over ranks.  `--strong` splits --structures over the GPUs.

`--impl reference` runs the UNMODIFIED reference C (BioEn's OpenMP kernels + liblbfgs, oracle/_ref) on the host cores
on the full problem: f+g evaluations/s (mean over the steps) and liblbfgs to the optimum.  No GPU code on that path.
"""
import argparse
import ctypes
import json
import os
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SEED = 12345
SIG_EXP, SIG_SIM = 0.5, 1.0
THETA = 10.0
METRIC = "grad_evals_per_s"


def unit(args):
    return ("evals/s (one evaluation = objective + gradient of the %s method over an N=%d x M=%d block of yTilde; "
            "summed over GPUs)" % (args.method, args.n, args.m))


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    # long spellings: under torchrun a bare `--m` is swallowed by the launcher's own abbreviation matching
    ap.add_argument("--m", "--observables", dest="m", type=int, default=1000)
    ap.add_argument("--n", "--structures", dest="n", type=int, default=1000000, help="structures PER GPU")
    ap.add_argument("--method", default="logw", choices=["logw", "forces"])
    ap.add_argument("--cpu-cols", type=int, default=200000, help="columns of the CPU-baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--strong", action="store_true",
                    help="strong scaling: --structures is the TOTAL N, split over the GPUs (default: weak, N per GPU)")
    ap.add_argument("--no-optimum", action="store_true")
    ap.add_argument("--no-numa", action="store_true", help="N > 1: do not bind each rank to its GPU's NUMA node")
    ap.add_argument("--no-extra", action="store_true", help="skip the extra_workloads records (other BASELINE configs)")
    ap.add_argument("--no-find-optimum", action="store_true", help="skip the public-API find_optimum timing")
    ap.add_argument("--no-dropin", action="store_true", help="skip the host-matrix drop-in call (needs M*N*8 B of host RAM)")
    ap.add_argument("--unfused-forces", action="store_true", help="forces: four tile passes instead of two fused")
    ap.add_argument("--only-cfg5", action="store_true",
                    help="N > 1: run only the BASELINE config-5 record (N=1e7 x M=5000 over 4 or 8 GPUs; a 50 GB shard "
                         "per GPU otherwise) and print it as the line's extra_workloads")
    ap.add_argument("--theta-scan", type=int, default=0, metavar="K",
                    help="BASELINE config 4: K theta values (log-spaced 1e3..1e-1) minimised together; prints the "
                         "batched-evaluation line instead of the single-theta one")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one returned (objective.npy, gradient.npy and the "
                         "point x.npy, float64; rank 0's block for N > 1) to DIR, to compare two builds output for output")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl == "reference" or args.theta_scan or args.only_cfg5):
        ap.error("--dump-outputs applies to the single-theta B200 workload only")
    return args


def observations(M):
    """YTrue / sigma and YTilde of the generic-data recipe (the M-vectors are tiny: host NumPy)."""
    rng = np.random.default_rng(SEED)
    ytrue = rng.standard_normal(M)
    yobs = ytrue + SIG_EXP * rng.standard_normal(M)
    return ytrue / SIG_EXP, yobs / SIG_EXP


def measured_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as fh:
            return float(json.load(fh)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def profiled_traffic(method, M, N):
    """dram__bytes_read + dram__bytes_write per launch of the dominant kernel from the committed `ncu --set full`
    capture of this same workload (profiles/), or None when the workload differs from the profiled one."""
    if (M, N) != (1000, 1000000):
        return None
    name = "r2_ncu_full_stream_pass.csv" if method == "logw" else "r1_ncu_full_fused_team_pass.csv"
    try:
        import csv
        with open(os.path.join(ROOT, "profiles", name)) as fh:
            rows = list(csv.reader(fh))
        hdr, units = rows[0], rows[1]
        ri, wi = hdr.index("dram__bytes_read.sum"), hdr.index("dram__bytes_write.sum")
        scale = {"Gbyte": 1e9, "Mbyte": 1e6, "Kbyte": 1e3, "byte": 1.0}
        vals = [float(r[ri]) * scale[units[ri]] + float(r[wi]) * scale[units[wi]] for r in rows[2:] if r]
        return sum(vals) / len(vals)
    except Exception:
        return None


class ClockSampler:
    """SM clock + throttle reasons sampled with NVML during the timed region."""

    def __init__(self, index):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._t = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def _run(self):
        nv = self.nv
        names = {"hw_slowdown": 0x8, "sw_thermal_slowdown": 0x20, "hw_thermal_slowdown": 0x40,
                 "sw_power_cap": 0x4, "hw_power_brake_slowdown": 0x80}
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                for k, bit in names.items():
                    if r & bit:
                        self.reasons.add(k)
            except Exception:
                pass
            self._stop.wait(0.05)

    def __enter__(self):
        if self.nv:
            self._t = threading.Thread(target=self._run, daemon=True)
            self._t.start()
        return self

    def __exit__(self, *exc):
        self._stop.set()
        if self._t:
            self._t.join()

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["unavailable"]}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


# ----------------------------------------------------------------------------------------------------------
# shared by both arms
# ----------------------------------------------------------------------------------------------------------
def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def workload_config(args, world):
    """`config` of the JSON line: IDENTICAL for the B200 arm and the reference arm of one launch (the arms differ in
    `run_info`, not here)."""
    n_local = args.n if not args.strong else None
    n_total = args.n if args.strong else args.n * world
    alg = float(args.m) * args.n * 8.0
    return {
        "workload": "%s f+g evaluation, synthetic generic data N=%d x M=%d per GPU (yTilde %.1f GB fp64), theta=%g"
                    % (args.method, args.n, args.m, alg / 1e9, THETA) if not args.strong else
                    "%s f+g evaluation, synthetic generic data N=%d x M=%d in total, split over the GPUs, theta=%g"
                    % (args.method, args.n, args.m, THETA),
        "method": args.method, "m": args.m, "n_per_gpu": n_local, "n_total": n_total, "theta": THETA, "seed": SEED,
        "l2": "inputs (%.1f GB per block) larger than L2 (126 MB) / any host cache; every step evaluates a new point"
              % (alg / 1e9),
        "optimum": "L-BFGS from x0 = 0 with BioEn's defaults (linesearch=2, past=10, delta=1e-6, epsilon=1e-6, "
                   "ftol=1e-5, max_linesearch=100)",
    }


# the reference arm leaves its optimum here for the B200 arm of the same run (outside the tree, which may be read-only)
T2O_FILE = os.path.join(tempfile.gettempdir(), "bioen_b200_bench_reference_optimum.json")
DUMP_MAX_ELEMENTS = 3_000_000      # per dumped vector: x and gradient together stay under 64 MB


def _t2o_key(args):
    return "%s:%d:%d:%g:%d" % (args.method, args.m, args.n, THETA, SEED)


# ----------------------------------------------------------------------------------------------------------
# reference arm / cpu_baseline: the reference's OpenMP C kernels + liblbfgs on the host cores
# ----------------------------------------------------------------------------------------------------------
def host_generate(M, cols, col0=0):
    """The same synthetic matrix the B200 arm generates on the device (counter-based law, oracle/hostgen.c), built
    on the host cores; entries agree with the device's to 1-2 ulp."""
    from oracle import oracle as O
    lib = O.hostgen()
    try:   # torchrun exports OMP_NUM_THREADS=1 to its ranks; the generator should use the host's cores all the same
        ctypes.CDLL("libgomp.so.1").omp_set_num_threads(host_cores())
    except OSError:
        pass
    a, _ = observations(M)
    yT = np.empty((M, cols))
    lib.hostgen_generic_ytilde(yT.ctypes.data_as(ctypes.POINTER(ctypes.c_double)), cols, M, cols, SEED, col0,
                               a.ctypes.data_as(ctypes.POINTER(ctypes.c_double)), SIG_SIM / SIG_EXP)
    return yT


def available_ram():
    try:
        import psutil
        return int(psutil.virtual_memory().available)
    except Exception:
        return 0


def cpu_reference(M, N_full, steps, warmup, method, want_optimum, max_cols=None):
    """The reference C code (oracle/_ref: BioEn's OpenMP kernels + liblbfgs 1.10, unmodified) -- or the oracle port
    if _ref is absent -- on the host cores.  Runs on the FULL N_full-column problem when host RAM allows, else on
    a column sample with the rate scaled linearly in N (stated in `sample`).  Every timed step is one f+g
    evaluation at a new point; `value` is the MEAN rate over the steps.  Returns (evals/s, info, optimum|None)."""
    from oracle import oracle as O
    from oracle import ref
    cores = host_cores()
    _, YT = observations(M)
    cols = N_full
    need = lambda c, copies: int(copies * M * c * 8 * 1.05) + (2 << 30)
    if max_cols:
        cols = min(cols, max_cols)
    ram = available_ram()
    while ram and cols > 50000 and need(cols, 1) > ram:
        cols //= 2
    t0 = time.perf_counter()
    yT = host_generate(M, cols)
    gen_s = time.perf_counter() - t0
    G = np.zeros(cols)
    w0 = np.full(cols, 1.0 / cols)
    rng = np.random.default_rng(SEED + 7)
    x = (0.1 * rng.standard_normal(N_full))[:cols] if method == "logw" else 1e-3 * rng.standard_normal(M)
    x = np.ascontiguousarray(x)
    if ref.available():
        kind, used = "reference", cores
        ref.set_num_threads(cores)
        ref.set_fast_openmp_flag(1)      # the reference's fastest mode
        # the reference's transposed-cache option ("auto" = on up to 8 GiB, bioen/optimize/common.py:83-106): time
        # both where a second copy fits, keep the faster
        modes = [False] + ([True] if (not ram or need(cols, 2.2) < ram) else [])
        evs = [((ref.LogwEvaluator(G, yT, YT, THETA, caching=c) if method == "logw"
                 else ref.ForcesEvaluator(w0, yT, YT, THETA, caching=c)), c) for c in modes]
    else:
        kind, used = "port", 1
        evs = [((lambda v: O.logw_fg(v, G, yT, YT, THETA)) if method == "logw"
                else (lambda v: O.forces_fg(v, w0, yT, YT, THETA)), False)]
    best = None
    for ev, caching in evs:
        for k in range(max(1, warmup)):
            ev(x)
        times = []
        for k in range(steps):
            x[0] += 1e-9                 # a new point every step
            t0 = time.perf_counter()
            ev(x)
            times.append(time.perf_counter() - t0)
        if best is None or np.mean(times) < best[0]:
            best = (float(np.mean(times)), float(min(times)), caching)
    dt_mean, dt_best, caching = best
    scale = N_full / cols
    info = {"kind": kind, "cores": used, "ms_per_eval_mean": 1e3 * dt_mean * scale, "ms_per_eval_best": 1e3 * dt_best * scale,
            "host_generate_s": gen_s,
            "sample": ("the full problem: %d columns x %d rows (%.1f GB)" % (cols, M, M * cols * 8 / 1e9) if cols == N_full
                       else "%d of %d columns x %d rows (%.1f GB; host RAM %.0f GB), rate scaled by %d/%d (cost linear "
                            "in N)" % (cols, N_full, M, M * cols * 8 / 1e9, ram / 1e9, cols, N_full))
                      + "; mean of %d f+g evaluations at new points (mean %.1f ms, best %.1f ms), %d OpenMP threads, "
                        "fast_openmp=1, yTildeT cache %s (faster of on/off where both fit), built -O3 -march=x86-64-v3 "
                        "(the library is compiled off-box; the kernels are DRAM-bound, AVX-512 would not change them)"
                        % (steps, 1e3 * dt_mean, 1e3 * dt_best, used, "on" if caching else "off")}
    optimum = None
    if want_optimum and kind == "reference" and cols == N_full:
        x0 = np.zeros(cols if method == "logw" else M)
        t0 = time.perf_counter()
        if method == "logw":
            xo, fmin, code = ref.opt_lbfgs_logw(x0, G, yT, YT, THETA, caching=caching)
            its = ctypes.c_size_t.in_dll(ref.lib(), "iterations_lbfgs_logw").value
        else:
            xo, fmin, code = ref.opt_lbfgs_forces(x0, w0, yT, YT, THETA, caching=caching)
            its = ctypes.c_size_t.in_dll(ref.lib(), "iterations_lbfgs_forces").value
        secs = time.perf_counter() - t0
        try:   # the end point itself, for the B200 arm of the same run (it evaluates ITS objective there)
            os.makedirs(os.path.dirname(T2O_FILE), exist_ok=True)
            np.save(T2O_FILE[:-5] + "_x.npy", xo)
        except OSError:
            pass
        optimum = {"seconds": secs, "fmin": fmin, "code": int(code), "iterations": int(its),
                   "minimizer": "the reference's _opt_lbfgs_%s (liblbfgs 1.10, BioEn defaults) on the full problem, "
                                "%d OpenMP threads, yTildeT cache %s" % (method, used, "on" if caching else "off"),
                   "includes": "host arrays in, result out; the matrix (and its cached transpose) already in host RAM"}
    elif want_optimum:
        optimum = {"unavailable": "needs oracle/_ref and the full matrix in host RAM (%.0f GB available)" % (ram / 1e9)}
    return 1.0 / (dt_mean * scale), info, optimum


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    t_wall = time.perf_counter()
    value, info, optimum = cpu_reference(args.m, args.n, args.steps, args.warmup, args.method,
                                         want_optimum=not args.no_optimum and not args.strong)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": unit(args),
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 / value, "higher_is_better": True,
        "scaling": "strong" if args.strong else "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(args, args.gpus),
        "cpu_baseline": {"value": value, "unit": unit(args), "cores": info["cores"], "kind": info["kind"],
                         "sample": info["sample"]},
        "gpu_launches": 0,
        "run_info": {"ms_per_eval_mean": info["ms_per_eval_mean"], "ms_per_eval_best": info["ms_per_eval_best"],
                     "host_generate_s": info["host_generate_s"],
                     "note": "one host runs the blocks of all %d GPU(s) one after the other: the rate in N-column "
                             "blocks per second does not depend on n_gpus" % args.gpus},
    }
    # (the unit counts N-column blocks, so the host's rate is the same at every n_gpus)
    line["e2e"] = {"value": line["value"], "unit": unit(args), "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    if optimum:
        line["time_to_optimum"] = optimum
        if "fmin" in optimum:
            try:   # left for the B200 arm of the same round-end run (it asserts agreement of the two optima)
                os.makedirs(os.path.dirname(T2O_FILE), exist_ok=True)
                with open(T2O_FILE, "w") as fh:
                    json.dump({"key": _t2o_key(args), **optimum, "cores": info["cores"]}, fh)
            except OSError:
                pass
    line["wall_s"] = time.perf_counter() - t_wall
    emit(line)


# ----------------------------------------------------------------------------------------------------------
# B200 arm
# ----------------------------------------------------------------------------------------------------------
def roofline_hbm(M, N, pass_ms, step_ms, kernel, traffic=None, read_gbs=None):
    peak, peak_src = measured_peak()
    alg = float(M) * N * 8.0
    ach = alg / (pass_ms * 1e-3) / 1e9 if pass_ms > 0 else 0.0
    r = {"bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak, "traffic": traffic,
         "peak_source": peak_src, "kernel": kernel + " (one pass over yTilde)", "bytes_per_launch": alg,
         "ms_per_launch": pass_ms, "step_frac": (2 * alg) / (step_ms * 1e-3) / 1e9 / peak if step_ms > 0 else None}
    if kernel in ("persistent_eval_kernel", "slice_eval_kernel"):
        r["kernel"] = kernel + " (one launch per evaluation)"
        r["ms_per_launch_is"] = "the step time divided by the algorithmic passes of an evaluation (2 log-weights, " \
                                "4 forces on the tile path): the launch is not bracketed by events of its own"
    if read_gbs:
        r["read_only_stream"] = {"gbs": read_gbs, "frac_of_it": ach / read_gbs,
                                 "what": "plain 16-byte-load read kernel over the same yTilde, mean of 10 launches, "
                                         "measured in this run; `peak` is a copy (read+write) figure"}
    return r


def connect_problem(prob, rank, world, n_total, dev):
    """library-side communicator for this rank's block (NCCL id broadcast by torch.distributed)"""
    import torch
    import torch.distributed as dist
    from bioen_b200 import _lib
    idbuf = torch.zeros(128, dtype=torch.uint8, device=dev)
    if rank == 0:
        raw = ctypes.create_string_buffer(128)
        _lib.check(_lib.load().bioen_b200_nccl_unique_id(raw), "nccl_unique_id")
        idbuf.copy_(torch.frombuffer(bytearray(raw.raw), dtype=torch.uint8))
    dist.broadcast(idbuf, 0)
    prob.comm_init(bytes(idbuf.cpu().numpy().tobytes()), rank, world, n_total)


def timed_evals(prob, method, nvar, dev, warmup, steps, seed_shift=0, world=1):
    """device-resident timing of `steps` f+g evaluations; returns (total ms, mean pass ms, launches), max over ranks"""
    import torch
    import torch.distributed as dist
    rng = np.random.default_rng(SEED + 7 + seed_shift)
    x = torch.from_numpy((0.1 if method == 0 else 1e-3) * rng.standard_normal(nvar)).to(dev)
    g = torch.zeros_like(x)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
        torch.cuda.synchronize()
    ms, pass_ms, launches = prob.time_evals(x.data_ptr(), g.data_ptr(), warmup, steps, method)
    if world > 1:
        dist.barrier()
        torch.cuda.synchronize()
        t = torch.tensor([ms, pass_ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms, pass_ms = float(t[0]), float(t[1])
    return ms, pass_ms, int(launches)


def dump_outputs(out_dir, prob, x_dev, g_dev):
    """The result of the last timed step as a caller of the evaluation receives it: the objective, the gradient and
    the point they belong to.  Vectors longer than DUMP_MAX_ELEMENTS are reduced to a fixed, seeded sample of
    entries (the same entries for every build)."""
    from bioen_b200 import _lib
    f = ctypes.c_double()
    _lib.check(_lib.load().bioen_b200_fetch(prob._h, ctypes.byref(f), None), "fetch")
    x, g = x_dev.cpu().numpy(), g_dev.cpu().numpy()
    if x.size > DUMP_MAX_ELEMENTS:
        idx = np.sort(np.random.default_rng(SEED).choice(x.size, DUMP_MAX_ELEMENTS, replace=False))
        x, g = x[idx], g[idx]
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "objective.npy"), np.array([f.value]))
    np.save(os.path.join(out_dir, "gradient.npy"), g)
    np.save(os.path.join(out_dir, "x.npy"), x)


def gram_optimum(prob, nvar, barrier=None):
    """the same minimisation with the opt-in coefficient-space L-BFGS update (2 kernels, 1 exchange per iteration)"""
    prob.set_option(6, 1)
    try:
        if barrier:
            barrier()
        t0 = time.perf_counter()
        xo, fmin, code, info = prob.opt_lbfgs(np.zeros(nvar))
        if barrier:
            barrier()
        return {"seconds": time.perf_counter() - t0, "code": code, "fmin": fmin, "iterations": info["iterations"],
                "evaluations": info["evaluations"], "option": "BIOEN_B200_OPT_LBFGS_GRAM=1 (rounds differently from the "
                                                              "default two-loop recursion)"}
    finally:
        prob.set_option(6, 0)


def small_workload(name, M, N, local, dev, steps, warmup):
    """One BASELINE config that is not the headline: logw and forces f+g rates, roofline of the pass kernel and
    the device L-BFGS to the optimum, on a freshly generated synthetic problem (single GPU)."""
    import bioen_b200
    from bioen_b200.problem import FORCES, LOGW
    a, YT = observations(M)
    out = {"name": name, "m": M, "n": N, "ytilde_bytes": M * N * 8}
    with bioen_b200.Problem(shape=(M, N), device=local) as prob:
        prob.generate(SEED, 0, a, SIG_SIM / SIG_EXP)
        for mname, method in (("logw", LOGW), ("forces", FORCES)):
            if method == LOGW:
                prob.set_logw(np.zeros(N), YT, THETA)
            else:
                prob.set_forces(np.full(N, 1.0 / N), YT, THETA)
            nvar = N if method == LOGW else M
            ms, pass_ms, launches = timed_evals(prob, method, nvar, dev, warmup, steps)
            t0 = time.perf_counter()
            xo, fmin, code, info = prob.opt_lbfgs(np.zeros(nvar))
            secs = time.perf_counter() - t0
            rec = {"value": steps / (ms * 1e-3), "unit": "f+g evals/s", "ms_per_step": ms / steps, "gpu_launches": launches,
                   "roofline": roofline_hbm(M, N, pass_ms, ms / steps, prob.pass_kernel_name(method)),
                   "time_to_optimum": {"seconds": secs, "code": code, "fmin": fmin, "iterations": info["iterations"],
                                       "evaluations": info["evaluations"]},
                   "time_to_optimum_coefficient_space": gram_optimum(prob, nvar)}
            if prob.query(7) == 1:
                rec["roofline"]["note"] = ("yTilde (%.1f MB) is dealt column-wise into the CTAs' shared memory and read "
                                           "ONCE per evaluation (from L2 when resident there); every sweep runs out of "
                                           "shared memory, the HBM figure is nominal" % (M * N * 8 / 1e6))
            elif M * N * 8 <= 100e6:
                rec["roofline"]["note"] = ("yTilde (%.1f MB) is L2-resident: the second pass of a step is served from "
                                           "L2, the HBM figure is nominal" % (M * N * 8 / 1e6))
            out[mname] = rec
    return out


def run_b200(args):
    import torch
    import torch.distributed as dist
    import bioen_b200
    from bioen_b200 import _lib
    from bioen_b200.problem import FORCES, LOGW

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        raise SystemExit("bench.py: --gpus %d but WORLD_SIZE=%d (launch with torchrun for N>1)" % (args.gpus, world))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the B200 path has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    numa_cpus = None
    if world > 1 and not args.no_numa:
        from bioen_b200.dist import bind_to_gpu_numa
        numa_cpus = bind_to_gpu_numa(local)      # before the pinned host vectors of the e2e leg are allocated

    if args.only_cfg5:
        if world < 2:
            raise SystemExit("bench.py --only-cfg5 needs N > 1 GPUs (torchrun)")
        recs = cfg5_records(rank, world, local, dev, min(args.steps, 10), not args.no_optimum)
        if rank == 0:
            emit({"metric": METRIC, "n_gpus": world, "only": "config 5", "data": "synthetic", "dtype": "f64",
                  "extra_workloads": recs})
        dist.destroy_process_group()
        return
    M = args.m
    if args.strong:
        from bioen_b200.dist import shard_bounds
        lo, hi = shard_bounds(args.n, rank, world)
        N, col0 = hi - lo, lo
    else:
        N, col0 = args.n, rank * args.n
    method = LOGW if args.method == "logw" else FORCES
    nvar = N if method == LOGW else M
    a, YT = observations(M)
    n_total = args.n if args.strong else N * world

    prob = bioen_b200.Problem(shape=(M, N), device=local)
    if world > 1:
        connect_problem(prob, rank, world, n_total, dev)
    t0 = time.perf_counter()
    prob.generate(SEED, col0, a, SIG_SIM / SIG_EXP)          # this rank's columns of the global matrix
    gen_s = time.perf_counter() - t0
    if method == LOGW:
        prob.set_logw(np.zeros(N), YT, THETA)
    else:
        if args.unfused_forces:
            prob.set_option(1, 0)
        prob.set_forces(np.full(N, 1.0 / n_total), YT, THETA)

    # start point: non-uniform weights (SURVEY 8d parity point); replicated vector for forces
    rng = np.random.default_rng(SEED + 7 + (rank if method == LOGW else 0))
    x_host = torch.empty(nvar, dtype=torch.float64).pin_memory()
    g_host = torch.empty(nvar, dtype=torch.float64).pin_memory()
    x_np, g_np = x_host.numpy(), g_host.numpy()
    x_np[:] = (0.1 if method == LOGW else 1e-3) * rng.standard_normal(nvar)
    x_dev = x_host.to(dev)
    g_dev = torch.zeros_like(x_dev)
    torch.cuda.synchronize()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident timing ------------------------------------------------------------------------
    barrier()
    with ClockSampler(local) as clk:
        ms, pass_ms, launches = prob.time_evals(x_dev.data_ptr(), g_dev.data_ptr(), args.warmup, args.steps)
    barrier()
    t = torch.tensor([ms, pass_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms, pass_ms = float(t[0]), float(t[1])
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, prob, x_dev, g_dev)
    # what a plain read-only stream over the same resident matrix reaches on this device (outside the timed region):
    # the context for a roofline fraction above 1 against the read+write copy figure of MEASURED_PEAKS.json
    read_gbs = ctypes.c_double(0.0)
    _lib.check(_lib.load().bioen_b200_read_stream_peak(prob._h, 10, ctypes.byref(read_gbs)), "read_stream_peak")
    units = 1 if args.strong else world     # weak: every rank adds one N-block per evaluation
    value = units * args.steps / (ms * 1e-3)

    # ---- end to end: host vectors through the C ABI ------------------------------------------------------
    lib = _lib.load()
    f = ctypes.c_double()
    e2e_steps = args.steps
    for k in range(args.warmup):
        _lib.check(lib.bioen_b200_eval(prob._h, method, _lib.ptr(x_np), ctypes.byref(f), _lib.ptr(g_np)), "eval")
    barrier()
    t0 = time.perf_counter()
    for k in range(e2e_steps):
        x_np[0] += 1e-9          # a new point every step
        _lib.check(lib.bioen_b200_eval(prob._h, method, _lib.ptr(x_np), ctypes.byref(f), _lib.ptr(g_np)), "eval")
    barrier()
    e2e_s = time.perf_counter() - t0
    te = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_value = units * e2e_steps / float(te[0])

    # ---- cross-rank correctness of the sharded evaluation (N > 1): the same point through the peer-memory
    # exchange and through NCCL, and against an independent recombination of rank-local pieces
    checks = None
    if world > 1:
        checks = sharded_checks(prob, method, x_np, YT, N, n_total, dev, world)

    # ---- time to optimum (device L-BFGS, BioEn defaults) -----------------------------------------------
    optimum = None
    if not args.no_optimum:
        x0 = np.zeros(nvar)
        barrier()
        t0 = time.perf_counter()
        xo, fmin, code, info = prob.opt_lbfgs(x0)
        barrier()
        optimum = {"seconds": time.perf_counter() - t0, "code": code, "fmin": fmin,
                   "iterations": info["iterations"], "evaluations": info["evaluations"],
                   "objective_only_evaluations": info["gradients_skipped"],
                   "minimizer": "device L-BFGS (liblbfgs semantics, BioEn defaults: linesearch=2, past=10, "
                                "delta=1e-6, epsilon=1e-6)", "includes": "x0 H2D + result D2H; yTilde resident"}
        optimum["coefficient_space_update"] = gram_optimum(prob, nvar, barrier)
        try:   # the reference arm of the same run (it runs first) left its optimum of the same problem here
            with open(T2O_FILE) as fh:
                r = json.load(fh)
            if r.get("key") == _t2o_key(args) and world == 1:
                d = abs(fmin - r["fmin"]) / abs(r["fmin"])
                optimum["reference"] = {"seconds": r["seconds"], "fmin": r["fmin"], "code": r["code"],
                                        "iterations": r["iterations"], "cores": r.get("cores"),
                                        "fmin_rel_diff": d, "agrees_1e-8": bool(d <= 1e-8),
                                        "speedup": r["seconds"] / optimum["seconds"]}
                # sanity bound only: liblbfgs's stop rule leaves the log-weights end point of an N >= 1e5 problem
                # defined to ~1e-6 (the reference's own two reduction modes end 2.8e-7 apart at config 2, DESIGN 7)
                try:   # per-evaluation parity AT the reference's own optimum: the device objective at its end point
                    xr = np.load(T2O_FILE[:-5] + "_x.npy")
                    if xr.size == nvar:
                        f_at, g_at = prob.objective_and_gradient(xr)
                        optimum["reference"]["device_objective_at_reference_optimum"] = f_at
                        optimum["reference"]["objective_rel_diff_at_reference_optimum"] = abs(f_at - r["fmin"]) / abs(r["fmin"])
                        optimum["reference"]["device_gnorm_over_xnorm_at_reference_optimum"] = float(
                            np.linalg.norm(g_at) / max(1.0, np.linalg.norm(xr)))
                except (OSError, ValueError):
                    pass
                optimum["reference"]["note"] = ("north_star bar 1e-8; the reference's own fast_openmp 0/1 end points differ by "
                                                "~3e-7 on such problems (stop rule delta=1e-6), see DESIGN.md section 7")
                if d > 1e-4:
                    raise SystemExit("bench.py: device optimum %.12g differs from the reference's %.12g" % (fmin, r["fmin"]))
        except (OSError, ValueError, KeyError):
            pass

    # ---- the reference-facing call with HOST buffers: bioen.optimize.ext.c_bioen.bioen_opt_lbfgs_* ------------
    dropin = None
    if world == 1 and not args.no_dropin and not args.no_optimum and available_ram() > 1.3 * M * N * 8:
        from bioen_b200 import optimize
        from bioen_b200.optimize.ext import c_bioen
        yT_host = prob.download()                       # the same matrix, now a pageable NumPy array
        cfg = optimize.minimize.Parameters("lbfgs")
        cfg["verbose"] = False
        t0 = time.perf_counter()
        with bioen_b200.Problem(yT_host, device=local):
            upload_s = time.perf_counter() - t0
        t0 = time.perf_counter()
        if method == LOGW:
            xo2, fmin2 = c_bioen.bioen_opt_lbfgs_logw(np.zeros(N), np.zeros(N), yT_host, YT, THETA, cfg)
        else:
            xo2, fmin2 = c_bioen.bioen_opt_lbfgs_forces(np.zeros(M), np.full(N, 1.0 / N), yT_host, YT, THETA, cfg)
        total_s = time.perf_counter() - t0
        dropin = {"api": "c_bioen.bioen_opt_lbfgs_%s (host NumPy arrays in, result out; = the reference's Cython entry)"
                         % args.method, "seconds": total_s, "ytilde_upload_s": upload_s,
                  "h2d_bytes": M * N * 8 + (N + M) * 8, "fmin": fmin2,
                  "agrees_with_resident_run": bool(optimum and abs(fmin2 - optimum["fmin"]) <= 1e-8 * abs(fmin2))}
        # the public API: bioen_b200.optimize.log_weights.find_optimum, host arrays in -> the reference's tuple out
        if method == LOGW and not args.no_find_optimum:
            y_host = yT_host                             # y is yTilde: one resident matrix (see DESIGN 'post-processing')
            GI = np.zeros((N, 1))
            t0 = time.perf_counter()
            res = optimize.log_weights.find_optimum(GI, GI, y_host, yT_host, YT.reshape(1, -1), THETA, cfg)
            dropin["find_optimum_s"] = time.perf_counter() - t0
            dropin["find_optimum_fmin"] = float(res[4])
            if available_ram() > 1.3 * M * N * 8:
                y_host = 0.5 * yT_host               # a DIFFERENT m x n array (y = sigma * yTilde in BioEn's callers)
                t0 = time.perf_counter()
                res = optimize.log_weights.find_optimum(GI, GI, y_host, yT_host, YT.reshape(1, -1), THETA, cfg)
                dropin["find_optimum_distinct_y_s"] = time.perf_counter() - t0
                dropin["find_optimum_distinct_y_note"] = ("y.wopt is streamed through a 256 MB device buffer in row "
                                                          "chunks: no second resident matrix")
                del y_host
        del yT_host

    kernel = "stream_pass_kernel" if method == LOGW or args.unfused_forces else "fused_team_pass"
    cfgd = workload_config(args, world)
    line = {
        "metric": METRIC, "value": value, "unit": unit(args), "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
        "scaling": "strong" if args.strong else "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": cfgd,
        "run_info": {"n_local": N, "global_evals_per_s": args.steps / (ms * 1e-3), "generate_s": gen_s,
                     "exchange": prob.comm_mode(), "exchanges_per_evaluation": prob.exchanges_per_eval(method),
                     "host_cpus_bound_to_gpu_numa_node": len(numa_cpus) if numa_cpus else None},
        "roofline": roofline_hbm(M, N, pass_ms, ms / args.steps, kernel, profiled_traffic(args.method, M, N),
                                 read_gbs.value),
        "e2e": {"value": e2e_value, "unit": unit(args), "h2d_bytes_per_step": nvar * 8, "d2h_bytes_per_step": nvar * 8 + 512,
                "api": "bioen_b200_eval (C ABI, pinned host vectors; yTilde resident after one upload)"},
        "gpu_launches": int(launches),
        "clocks": clk.summary(),
    }
    line["roofline"]["traffic_source"] = "profiles/ (ncu --set full of this workload, mean per launch)"
    if optimum:
        line["time_to_optimum"] = optimum
    if dropin:
        line["dropin_time_to_optimum"] = dropin
    if checks:
        line["sharded_checks"] = checks
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        try:
            v, info, _ = cpu_reference(M, N, 5, 1, args.method, want_optimum=False, max_cols=args.cpu_cols)
            line["cpu_baseline"] = {"value": v, "unit": unit(args), "cores": info["cores"], "kind": info["kind"],
                                    "sample": info["sample"]}
        except Exception as e:  # the baseline is reported, never required for the GPU number
            line["cpu_baseline"] = {"value": None, "unit": unit(args), "cores": 0, "kind": "unavailable", "sample": str(e)}

    # ---- the other BASELINE configs, after the timed region of the headline workload --------------------------
    if not args.no_extra:
        extra = []
        es, ew = min(args.steps, 20), min(args.warmup, 3)
        # (a) the other method on the same resident matrix
        other = FORCES if method == LOGW else LOGW
        oname = "forces" if other == FORCES else "logw"
        if other == FORCES:
            prob.set_forces(np.full(N, 1.0 / n_total), YT, THETA)
        else:
            prob.set_logw(np.zeros(N), YT, THETA)
        ovar = M if other == FORCES else N
        oms, opass, olaunch = timed_evals(prob, other, ovar, dev, ew, es, seed_shift=(rank if other == LOGW else 0),
                                          world=world)
        rec = {"name": "config 3, %s method (same matrix, N=%d x M=%d per GPU)" % (oname, N, M),
               "value": units * es / (oms * 1e-3), "unit": "f+g evals/s (N-column blocks, summed over GPUs)",
               "ms_per_step": oms / es, "gpu_launches": olaunch,
               "roofline": roofline_hbm(M, N, opass, oms / es, prob.pass_kernel_name(other))}
        if not args.no_optimum:
            barrier()
            t0 = time.perf_counter()
            xo, fmin, code, info = prob.opt_lbfgs(np.zeros(ovar))
            barrier()
            rec["time_to_optimum"] = {"seconds": time.perf_counter() - t0, "code": code, "fmin": fmin,
                                      "iterations": info["iterations"], "evaluations": info["evaluations"]}
        extra.append(rec)
        # (b) config 4: the 32-theta L-curve batched on fp64 tensor cores, same matrix
        if not args.strong:
            extra.append(theta_scan_record(prob, LOGW, 32, M, N, n_total, YT, rank, world, local, dev,
                                           min(args.steps, 10), ew, not args.no_optimum))
        # (b') opt-in fp32 STORAGE of the same matrix (not parity-preserving, never the default): half the bytes
        if not args.strong:
            prob.set_option(7, 1)
            prob.set_logw(np.zeros(N), YT, THETA)
            fms, fpass, flaunch = timed_evals(prob, LOGW, N, dev, ew, es, seed_shift=rank, world=world)
            r32 = roofline_hbm(M, N, fpass, fms / es, prob.pass_kernel_name(LOGW))
            for k in ("achieved", "frac", "bytes_per_launch", "step_frac"):
                r32[k] = r32[k] / 2.0          # 4-byte entries: M*N*4 algorithmic bytes per pass
            extra.append({"name": "config 3, logw with OPT-IN fp32 storage of yTilde (fp64 arithmetic; results differ "
                                  "from the reference at the 1e-8 level -- not a parity path)",
                          "value": units * es / (fms * 1e-3), "unit": "f+g evals/s (N-column blocks, summed over GPUs)",
                          "ms_per_step": fms / es, "gpu_launches": flaunch, "roofline": r32})
        prob.close()
        # (c) configs 2 and 1 (ala5 shape): small, L2-resident problems, single GPU each (rank 0 reports)
        if world == 1:
            extra.append(small_workload("config 2: N=1e5 x M=500 (0.4 GB)", 500, 100000, local, dev, es, ew))
            extra.append(small_workload("config 1 shape (ala5): N=50001 x M=28 (11 MB)", 28, 50001, local, dev, es, ew))
        else:
            # (d) strong scaling of config 3 (N = 1e6 in total over the GPUs) and a config-5 shard per GPU
            extra.append(sharded_record("config 3 strong: N=1e6 x M=1e3 in total", 1000, 1000000, True, rank, world,
                                        local, dev, es, ew, not args.no_optimum))
            extra.extend(cfg5_records(rank, world, local, dev, es, not args.no_optimum))
        line["extra_workloads"] = extra
    else:
        prob.close()
    if rank == 0:
        emit(line)
    if world > 1:
        dist.destroy_process_group()


def cfg5_records(rank, world, local, dev, es, want_optimum):
    """BASELINE config 5 (N = 1e7 x M = 5000, 400 GB): the whole problem on 4 or 8 GPUs (100 / 50 GB per GPU), a 50 GB
    shard per GPU otherwise.  The forces leg keeps only the structure-major copy, so both legs need ONE copy of the
    shard per GPU."""
    import torch
    n_per = 10000000 // world if world in (4, 8) else 1250000
    need = 5000.0 * n_per * 8.0 * 1.06 + 4e9
    free_b, _tot = torch.cuda.mem_get_info(dev)
    if free_b < need:
        return []
    if world in (4, 8):
        name = "config 5: N=1e7 x M=5000 over %d GPUs (%d GB of yTilde per GPU)" % (world, round(5000 * n_per * 8 / 1e9))
    else:
        name = "config 5 shard: N=1.25e6 x M=5000 per GPU (50 GB per GPU)"
    return [sharded_record(name, 5000, n_per, False, rank, world, local, dev, min(es, 10), 2, want_optimum,
                           forces_structure_major_only=True)]


def sharded_checks(prob, method, x_np, YT, N, n_total, dev, world):
    """N > 1: (1) the exchange carried by the peer-memory kernel and by NCCL gives bit-identical f and gradient;
    (2) f equals an independent recombination -- rank-local pieces computed by the library WITHOUT its communicator
    semantics (weights download, local yTilde.w through the average entry point is itself sharded, so the pieces are
    formed on the host from the downloaded weights) summed with torch.distributed -- to 1e-12."""
    import torch
    import torch.distributed as dist
    out = {}
    f1, g1 = prob.objective_and_gradient(x_np)
    mode = prob.comm_mode()
    if mode == "p2p":
        prob.set_option(2, 0)
        f2, g2 = prob.objective_and_gradient(x_np)
        prob.set_option(2, 1)
        out["p2p_vs_nccl_bit_identical"] = bool(f1 == f2 and np.array_equal(g1, g2))
        out["p2p_vs_nccl_rel_diff"] = abs(f1 - f2) / abs(f1)
    # every rank must hold the same f
    fl = [torch.zeros(1, dtype=torch.float64, device=dev) for _ in range(world)]
    dist.all_gather(fl, torch.tensor([f1], dtype=torch.float64, device=dev))
    out["f_identical_on_all_ranks"] = bool(all(float(v) == f1 for v in fl))
    if method == 0:
        # independent recombination: global log-sum-exp and the prior from the rank-local g slices (torch collectives,
        # host arithmetic), chi^2 from the library's all-reduced averages
        mx = torch.tensor([x_np.max()], dtype=torch.float64, device=dev)
        dist.all_reduce(mx, op=dist.ReduceOp.MAX)
        e = np.exp(x_np - float(mx))
        parts = torch.tensor([e.sum(), (x_np * e).sum()], dtype=torch.float64, device=dev)
        dist.all_reduce(parts)
        S, gE = float(parts[0]), float(parts[1])
        w = e / S
        avg = prob.average(w)                           # all-reduced inside the library
        r = avg - YT
        # G = 0: prior = theta * (sum g w - log sum exp g + log n_total)
        f_host = THETA * (gE / S - (float(mx) + np.log(S)) + np.log(n_total)) + 0.5 * float(r @ r)
        out["f_vs_host_recombination_rel_diff"] = abs(f_host - f1) / abs(f_host)
        out["f_vs_host_recombination_ok_1e-12"] = bool(abs(f_host - f1) <= 1e-12 * abs(f_host))
    return out


def sharded_record(name, M, n_arg, strong, rank, world, local, dev, steps, warmup, want_optimum,
                   forces_structure_major_only=False):
    """A second sharded problem of the same job (strong-scaled config 3, or config 5): logw and forces f+g rates with
    the pass roofline, and the log-weights L-BFGS to the optimum.  forces_structure_major_only: the forces leg runs on
    a SECOND problem that holds only the structure-major copy of yTilde (generated directly in that layout, after the
    row-major problem of the log-weights leg is closed), so the peak is ONE copy of the shard per GPU, not two."""
    import bioen_b200
    import torch
    import torch.distributed as dist
    from bioen_b200.dist import shard_bounds
    from bioen_b200.problem import FORCES, LOGW
    if strong:
        lo, hi = shard_bounds(n_arg, rank, world)
        N, col0, n_total = hi - lo, lo, n_arg
    else:
        N, col0, n_total = n_arg, rank * n_arg, n_arg * world
    a, YT = observations(M)
    out = {"name": name, "m": M, "n_local": N, "n_total": n_total, "scaling": "strong" if strong else "weak"}
    prob = bioen_b200.Problem(shape=(M, N), device=local)
    try:
        connect_problem(prob, rank, world, n_total, dev)
        prob.generate(SEED, col0, a, SIG_SIM / SIG_EXP)
        units = 1 if strong else world
        for mname, method in (("logw", LOGW), ("forces", FORCES)):
            if method == LOGW:
                prob.set_logw(np.zeros(N), YT, THETA)
            else:
                if forces_structure_major_only:
                    prob.close()
                    torch.cuda.empty_cache()
                    prob = bioen_b200.Problem(shape=(M, N), device=local, structure_major_only=True)
                    connect_problem(prob, rank, world, n_total, dev)
                    prob.generate(SEED, col0, a, SIG_SIM / SIG_EXP)
                prob.set_forces(np.full(N, 1.0 / n_total), YT, THETA)
            nvar = N if method == LOGW else M
            ms, pass_ms, launches = timed_evals(prob, method, nvar, dev, warmup, steps,
                                                seed_shift=(rank if method == LOGW else 0), world=world)
            rec = {"value": units * steps / (ms * 1e-3), "unit": "f+g evals/s (%s, summed over GPUs)"
                   % ("the whole N" if strong else "N-column blocks"), "ms_per_step": ms / steps,
                   "gpu_launches": launches, "exchange": prob.comm_mode(),
                   "roofline": roofline_hbm(M, N, pass_ms, ms / steps, prob.pass_kernel_name(method)),
                   "ytilde_bytes_resident_per_gpu": prob.query(8)}
            if method == FORCES and forces_structure_major_only:
                rec["layout"] = "structure-major copy only (BIOEN_B200_OPT_STRUCTURE_MAJOR_ONLY)"
            if want_optimum and (method == LOGW or M <= 1000):
                dist.barrier()
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                xo, fmin, code, info = prob.opt_lbfgs(np.zeros(nvar))
                dist.barrier()
                rec["time_to_optimum"] = {"seconds": time.perf_counter() - t0, "code": code, "fmin": fmin,
                                          "iterations": info["iterations"], "evaluations": info["evaluations"]}

                def _bar():
                    dist.barrier()
                    torch.cuda.synchronize()
                rec["time_to_optimum_coefficient_space"] = gram_optimum(prob, nvar, _bar)
            out[mname] = rec
    finally:
        prob.close()
    return out


def theta_scan_record(prob, meth, K, M, N, n_total, YT, rank, world, local, dev, steps, warmup, want_optimum):
    """BASELINE config 4 on the resident matrix: K theta values batched (skinny fp64 GEMMs on tensor cores)."""
    import torch
    import torch.distributed as dist
    from bioen_b200 import _lib
    lib = _lib.load()
    forces = meth == 1
    nvar = M if forces else N
    if forces:
        prob.set_forces(np.full(N, 1.0 / n_total), YT, THETA)
    else:
        prob.set_logw(np.zeros(N), YT, THETA)
    thetas = np.geomspace(1e3, 1e-1, K)
    rng = np.random.default_rng(SEED + 7 + (0 if forces else rank))
    X0 = np.ascontiguousarray((1e-3 if forces else 0.1) * rng.standard_normal((K, nvar)))
    peak_tf = ctypes.c_double()
    _lib.check(lib.bioen_b200_dmma_peak(local, ctypes.byref(peak_tf)), "dmma_peak")
    ms, gemm_ms, launches = ctypes.c_float(), ctypes.c_float(), ctypes.c_longlong()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    barrier()
    _lib.check(lib.bioen_b200_time_scan_evals(prob._h, meth, K, _lib.ptr(thetas), _lib.ptr(X0), warmup, steps,
                                              ctypes.byref(ms), ctypes.byref(gemm_ms), ctypes.byref(launches)),
               "time_scan_evals")
    barrier()
    t = torch.tensor([ms.value, gemm_ms.value], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    tot_ms, g_ms = float(t[0]), float(t[1])
    KP = (K + 7) // 8 * 8
    flops = 2.0 * M * N * KP
    ach = flops / (g_ms * 1e-3) / 1e12
    hbm_peak, _ = measured_peak()
    rec = {"name": "config 4: theta L-curve scan, K=%d theta values batched, N=%d x M=%d per GPU (%s)"
                   % (K, N, M, "forces" if forces else "logw"),
           "value": world * K * steps / (tot_ms * 1e-3), "unit": "problem f+g evals/s (summed over K and GPUs)",
           "ms_per_step": tot_ms / steps, "gpu_launches": int(launches.value),
           "roofline": {"bound": "tensor", "achieved": ach, "peak": peak_tf.value, "unit": "TFLOP/s",
                        "frac": ach / peak_tf.value, "traffic": None,
                        "peak_source": "measured in this run: register-resident mma.sync.m8n8k4.f64 loop (no fp64 "
                                       "figure in MEASURED_PEAKS.json)",
                        "kernel": "batched_gemm_kernel (one pass over yTilde for all K)", "flops_per_launch": flops,
                        "ms_per_launch": g_ms,
                        "hbm_frac_same_launch": (M * N * 8.0) / (g_ms * 1e-3) / 1e9 / hbm_peak}}
    if want_optimum:
        barrier()
        t0 = time.perf_counter()
        X, fmin, codes, info = prob.theta_scan(thetas, x0=np.zeros(nvar), method=meth)
        barrier()
        rec["time_to_optimum"] = {"seconds": time.perf_counter() - t0, "rounds": info["rounds"],
                                  "codes": [int(c) for c in codes],
                                  "evaluations_total": int(info["evaluations"].sum()),
                                  "fmin_first_last": [float(fmin[0]), float(fmin[-1])]}
    return rec


def run_theta_scan(args):
    """BASELINE.json config 4: the L-curve -- K problems, one yTilde stream per pass for all of them.  With
    N > 1 GPUs the structure axis is sharded (N per GPU, weak scaling) and the per-problem scalars are all-reduced."""
    import torch
    import torch.distributed as dist
    import bioen_b200
    from bioen_b200 import _lib
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the B200 path has no CPU fallback")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        raise SystemExit("bench.py: --gpus %d but WORLD_SIZE=%d (launch with torchrun for N>1)" % (args.gpus, world))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    M, N, K = args.m, args.n, args.theta_scan
    n_total = N * world
    a, YT = observations(M)
    prob = bioen_b200.Problem(shape=(M, N), device=local)
    lib = _lib.load()
    if world > 1:
        idbuf = torch.zeros(128, dtype=torch.uint8, device=dev)
        if rank == 0:
            raw = ctypes.create_string_buffer(128)
            _lib.check(lib.bioen_b200_nccl_unique_id(raw), "nccl_unique_id")
            idbuf.copy_(torch.frombuffer(bytearray(raw.raw), dtype=torch.uint8))
        dist.broadcast(idbuf, 0)
        prob.comm_init(bytes(idbuf.cpu().numpy().tobytes()), rank, world, n_total)
    prob.generate(SEED, rank * N, a, SIG_SIM / SIG_EXP)
    forces = args.method == "forces"
    meth = 1 if forces else 0
    nvar = M if forces else N
    if forces:
        prob.set_forces(np.full(N, 1.0 / n_total), YT, THETA)
    else:
        prob.set_logw(np.zeros(N), YT, THETA)
    thetas = np.geomspace(1e3, 1e-1, K)
    rng = np.random.default_rng(SEED + 7 + (0 if forces else rank))
    X0 = np.ascontiguousarray((1e-3 if forces else 0.1) * rng.standard_normal((K, nvar)))
    peak_tf = ctypes.c_double()
    _lib.check(lib.bioen_b200_dmma_peak(local, ctypes.byref(peak_tf)), "dmma_peak")
    ms, gemm_ms, launches = ctypes.c_float(), ctypes.c_float(), ctypes.c_longlong()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    barrier()
    with ClockSampler(local) as clk:
        _lib.check(lib.bioen_b200_time_scan_evals(prob._h, meth, K, _lib.ptr(thetas), _lib.ptr(X0), args.warmup, args.steps,
                                                  ctypes.byref(ms), ctypes.byref(gemm_ms), ctypes.byref(launches)),
                   "time_scan_evals")
    barrier()
    t = torch.tensor([ms.value, gemm_ms.value], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    tot_ms, g_ms = float(t[0]), float(t[1])
    KP = (K + 7) // 8 * 8
    flops = 2.0 * M * N * KP
    ach = flops / (g_ms * 1e-3) / 1e12
    hbm_peak, _ = measured_peak()
    line = {
        "metric": "theta_scan_problem_evals_per_s", "value": world * K * args.steps / (tot_ms * 1e-3),
        "unit": "f+g evaluations/s of N=%d x M=%d blocks, summed over K problems and GPUs (%s)" % (N, M, args.method),
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": tot_ms / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": "theta L-curve scan (%s method), K=%d theta values batched, N=%d x M=%d per GPU, skinny "
                               "fp64 GEMMs on tensor cores (DMMA)" % (args.method, K, N, M), "K": K,
                   "method": args.method, "n_total": n_total,
                   "l2": "inputs (%.1f GB) larger than L2" % (M * N * 8 / 1e9)},
        "roofline": {"bound": "tensor", "achieved": ach, "peak": peak_tf.value, "unit": "TFLOP/s",
                     "frac": ach / peak_tf.value, "traffic": None,
                     "peak_source": "measured in this run: register-resident mma.sync.m8n8k4.f64 loop (no fp64 figure "
                                    "in MEASURED_PEAKS.json)",
                     "kernel": "batched_gemm_kernel (one pass over yTilde for all K)", "flops_per_launch": flops,
                     "ms_per_launch": g_ms,
                     "hbm_frac_same_launch": (M * N * 8.0) / (g_ms * 1e-3) / 1e9 / hbm_peak},
        "gpu_launches": int(launches.value), "clocks": clk.summary(),
    }
    if not args.no_optimum:
        barrier()
        t0 = time.perf_counter()
        X, fmin, codes, info = prob.theta_scan(thetas, x0=np.zeros(nvar), method=meth)
        barrier()
        line["time_to_optimum"] = {"seconds": time.perf_counter() - t0, "rounds": info["rounds"],
                                   "codes": [int(c) for c in codes], "iterations": [int(i) for i in info["iterations"]],
                                   "evaluations_total": int(info["evaluations"].sum()),
                                   "fmin_first_last": [float(fmin[0]), float(fmin[-1])],
                                   "includes": "K x n start vectors H2D, results D2H; yTilde resident"}
    prob.close()
    if rank == 0:
        emit(line)
    if world > 1:
        dist.destroy_process_group()


_REAL_STDOUT = None


def _claim_stdout():
    """Everything libraries print to fd 1 (NCCL's version banner, liblbfgs-style progress prints) goes to stderr;
    the one JSON line is written to the real stdout by emit()."""
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)


def emit(line):
    sys.stdout.flush()
    os.write(_REAL_STDOUT if _REAL_STDOUT is not None else 1, (json.dumps(line) + "\n").encode())


def main():
    args = parse()
    _claim_stdout()
    if args.theta_scan and args.impl != "reference":
        return run_theta_scan(args)
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
