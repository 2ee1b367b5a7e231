"""Batched replicate minimisations: reference outputs and timings.

    python scripts/replicates_probe.py --dump DIR
        theta_scan outputs (X, fmin, codes, iterations) of seeded problems -- log-weights 100 x 20 000 and forces
        300 x 4 000, K = 11, line searches 2 and 0 -- written to DIR/theta_scan_<method>_ls<k>.npz; opt_lbfgs
        outputs (x, fmin, code, iterations, evaluations) of the same problems at theta = 1, at most 300 iterations,
        for line searches 0-3 with
        the single-CTA, speculative-trial and Gram update options each on and off, to DIR/opt_lbfgs_<method>.npz; and
        both minimisers on a log-weights 8 x 40 problem whose backtracking searches end in
        LBFGSERR_INCREASEGRADIENT, to DIR/increase_gradient.npz.  Two builds that must compute the same minimisations
        give identical files.

    python scripts/replicates_probe.py --time DIR
        prints the device name and power limit, then times (host clock around work that ends in a device
        synchronise, after warm-up):
          1. one batched f+g evaluation of K = 32 problems without per-problem inputs and with every input the
             method takes (YTilde, row weights, and w0 for forces) at 500 x 1e5 and 1000 x 1e6, both methods;
          2. a 256-replicate observable bootstrap and a 5-fold x 16-theta cross-validation (forces) at the ala5
             shape (28 x 50 001) and at 500 x 1e5, against sequential single-problem opt_lbfgs runs on explicitly
             rescaled problems.
        Records go to stdout and DIR/replicates_probe.jsonl.
"""
import argparse
import itertools
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

OPT_LBFGS_GRAM, OPT_LBFGS_SMALL, OPT_LBFGS_SPECULATIVE = 6, 9, 10   # bioen_b200_set_option
THETAS = np.array([1000.0, 300.0, 100.0, 30.0, 10.0, 3.0, 1.0, 0.3, 100.0, 10.0, 55.0])


def dump(out):
    import bioen_b200
    from bioen_b200.problem import FORCES, LOGW
    from oracle import oracle as O
    os.makedirs(out, exist_ok=True)
    for name, M, N, meth in (("logw", 100, 20000, LOGW), ("forces", 300, 4000, FORCES)):
        P = O.synthetic_problem(M, N, seed=M + N)
        w0 = np.random.default_rng(7).random(N) + 0.2
        w0 /= w0.sum()
        with bioen_b200.Problem(P["yTilde"]) as p:
            if meth == LOGW:
                p.set_logw(P["G"], P["YTilde"], 1.0)
            else:
                p.set_forces(w0, P["YTilde"], 1.0)
            for ls in (2, 0):
                X, fmin, codes, info = p.theta_scan(THETAS, method=meth, linesearch=ls)
                np.savez(os.path.join(out, "theta_scan_%s_ls%d.npz" % (name, ls)), X=X, fmin=fmin, codes=codes,
                         iterations=info["iterations"])
                print("%s ls=%d: codes %s iterations %s" % (name, ls, list(codes), list(info["iterations"])), flush=True)
            res = {}
            x0 = P["GInit"] if meth == LOGW else np.zeros(M)
            for ls in range(4):
                for small, spec, gram in itertools.product((1, 0), repeat=3):
                    for opt, v in ((OPT_LBFGS_SMALL, small), (OPT_LBFGS_SPECULATIVE, spec), (OPT_LBFGS_GRAM, gram)):
                        p.set_option(opt, v)
                    x, fmin, code, info = p.opt_lbfgs(x0, method=meth, linesearch=ls, max_iterations=300)
                    key = "ls%d_small%d_spec%d_gram%d" % (ls, small, spec, gram)
                    res.update({key + "_x": x, key + "_fmin": fmin, key + "_code": code,
                                key + "_iterations": info["iterations"], key + "_evaluations": info["evaluations"]})
            np.savez(os.path.join(out, "opt_lbfgs_%s.npz" % name), **res)
            print("%s opt_lbfgs: codes %s" % (name, sorted({int(v) for k, v in res.items() if k.endswith("_code")})),
                  flush=True)
    P = O.synthetic_problem(8, 40, seed=5)
    thetas = np.array([0.01, 1.0, 100.0])
    with bioen_b200.Problem(P["yTilde"]) as p:
        p.set_logw(P["G"], P["YTilde"], 1.0)
        X, fmin, codes, info = p.theta_scan(thetas, x0=P["GInit"], linesearch=1)
        res = dict(scan_X=X, scan_fmin=fmin, scan_codes=codes, scan_iterations=info["iterations"])
        for q, th in enumerate(thetas):
            p.set_theta(th)
            x, f, code, info = p.opt_lbfgs(P["GInit"], linesearch=1)
            res.update({"opt%d_x" % q: x, "opt%d_fmin" % q: f, "opt%d_code" % q: code})
        np.savez(os.path.join(out, "increase_gradient.npz"), **res)
        print("increase_gradient: scan codes %s" % list(codes))


def emit(out, rec):
    print(json.dumps(rec), flush=True)
    with open(os.path.join(out, "replicates_probe.jsonl"), "a") as fh:
        fh.write(json.dumps(rec) + "\n")


def device_facts():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def make_problem(M, N, seed):
    """Device-generated synthetic yTilde (bench.py's recipe) and its YTilde, w0."""
    import bioen_b200
    rng = np.random.default_rng(seed)
    ytrue = rng.standard_normal(M)
    YT = (ytrue + 0.5 * rng.standard_normal(M)) / 0.5
    p = bioen_b200.Problem(shape=(M, N))
    p.generate(seed, 0, ytrue / 0.5, 1.0 / 0.5)
    return p, YT, np.full(N, 1.0 / N)


def time_evals(p, method, K, planes, x0, warmup, steps):
    """ms per batched f+g evaluation of K problems (CUDA events over `steps` evaluations after `warmup`)"""
    import ctypes as C
    from bioen_b200 import _lib
    thetas = np.geomspace(1e3, 1e-1, K)
    arrs = {k: np.ascontiguousarray(v) for k, v in planes.items()}
    b = _lib.bioen_b200_batch(K, _lib.ptr(thetas), *(_lib.ptr(arrs[k]) if k in arrs else None
                                                      for k in ("YTilde", "row_weights", "w0")))
    ms, gemm_ms, launches = C.c_float(), C.c_float(), C.c_longlong()
    _lib.check(p._lib.bioen_b200_time_batch_evals(p._ctx, method, C.byref(b), _lib.ptr(x0), warmup, steps,
                                                  C.byref(ms), C.byref(gemm_ms), C.byref(launches)), "time_batch_evals")
    return ms.value / steps


def time_planes(out, reps=3, steps=20):
    from bioen_b200.problem import FORCES, LOGW
    K = 32
    for M, N in ((500, 100000), (1000, 1000000)):
        p, YT, w0 = make_problem(M, N, 12345)
        rng = np.random.default_rng(1)
        for method in (LOGW, FORCES):
            if method == LOGW:
                p.set_logw(np.zeros(N), YT, 1.0)
            else:
                p.set_forces(w0, YT, 1.0)
            n = M if method == FORCES else N
            x0 = np.ascontiguousarray((1e-3 if method == FORCES else 0.1) * rng.standard_normal((K, n)))
            planes = dict(YTilde=YT + rng.standard_normal((K, M)),
                          row_weights=rng.multinomial(M, np.full(M, 1.0 / M), size=K).astype(float))
            if method == FORCES:
                planes["w0"] = w0 * rng.multinomial(N, np.full(N, 1.0 / N), size=K)
            t = {"none": [], "planes": []}
            for r in range(reps):                      # alternate the two variants
                t["none"].append(time_evals(p, method, K, {}, x0, 3, steps))
                t["planes"].append(time_evals(p, method, K, planes, x0, 3, steps))
            a, b = np.median(t["none"]), np.median(t["planes"])
            plane_bytes = 8.0 * K * (2 * M + (3 * N if method == FORCES else 0))   # YTilde, c once; w0 thrice
            emit(out, dict(what="batched f+g evaluation, K=32", M=M, N=N, method="forces" if method else "logw",
                           ms_no_planes=t["none"], ms_planes=t["planes"], median_no_planes=a, median_planes=b,
                           gap_percent=100.0 * (b - a) / a, plane_reads_bytes_estimate=plane_bytes,
                           matrix_bytes=8.0 * M * N))
        p.close()


def time_helpers(out, seq_limit):
    """256-replicate observable bootstrap and 5-fold x 16-theta cross-validation (forces, the ala5 notebook's
    L-BFGS settings) against sequential single-problem opt_lbfgs runs on explicitly rescaled, re-uploaded
    matrices.  The sequential timing covers min(seq_limit, all) runs and is scaled to all of them."""
    import bioen_b200
    from bioen_b200 import _lib, replicates
    cfg = dict(epsilon=1e-5, ftol=1e-4, max_iterations=20000)
    theta = 10.0
    for M, N in ((28, 50001), (500, 100000)):
        rng = np.random.default_rng(3)
        ytrue = rng.standard_normal(M)
        y = ytrue[:, None] + rng.standard_normal((M, N))
        yT = np.ascontiguousarray(y / 0.5)
        YT = (ytrue + 0.5 * rng.standard_normal(M)) / 0.5
        w0 = np.full(N, 1.0 / N)
        with bioen_b200.Problem(yT) as p:
            p.set_forces(w0, YT, theta)
            p.batch_minimize(theta, row_weights=np.ones((2, M)), max_iterations=5)      # warm-up
            t0 = time.perf_counter()
            bs = replicates.bootstrap(p, 256, "observables", theta, seed=1, **cfg)
            t_bs = time.perf_counter() - t0
            thetas = np.geomspace(1e3, 1e-1, 16)
            t0 = time.perf_counter()
            cv = replicates.cross_validate(p, thetas, folds=5, seed=1, **cfg)
            t_cv = time.perf_counter() - t0

        def sequential(weights, th):
            """opt_lbfgs per problem on yTilde and YTilde rescaled by sqrt(c) (fresh upload each time)"""
            runs = min(seq_limit, len(weights))
            with bioen_b200.Problem(yT) as q:
                q.set_forces(w0, YT, theta)
                q.opt_lbfgs(np.zeros(M), max_iterations=5)
                t0 = time.perf_counter()
                for r in range(runs):
                    s = np.sqrt(weights[r])
                    blk = np.ascontiguousarray(yT * s[:, None])
                    _lib.check(q._lib.bioen_b200_upload_ytilde(q._ctx, _lib.ptr(blk), N), "upload_ytilde")
                    q.set_forces(w0, YT * s, th[r])
                    q.opt_lbfgs(np.zeros(M), **cfg)
                return (time.perf_counter() - t0) * len(weights) / runs, runs

        seq_bs, n_bs = sequential(bs["counts"].astype(float), np.full(256, theta))
        fold = cv["fold"]
        wcv = np.array([(fold != f).astype(float) for t in range(16) for f in range(5)])
        seq_cv, n_cv = sequential(wcv, np.repeat(thetas, 5))
        emit(out, dict(what="observable bootstrap, 256 replicates, forces", M=M, N=N, batched_s=t_bs,
                       sequential_s=seq_bs, sequential_runs_timed=n_bs, speedup=seq_bs / t_bs,
                       codes={int(c): int(v) for c, v in zip(*np.unique(bs["codes"], return_counts=True))}))
        emit(out, dict(what="cross-validation, 5 folds x 16 thetas, forces", M=M, N=N, batched_s=t_cv,
                       sequential_s=seq_cv, sequential_runs_timed=n_cv, speedup=seq_cv / t_cv,
                       codes={int(c): int(v) for c, v in zip(*np.unique(cv["codes"], return_counts=True))}))


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--dump", metavar="DIR")
    ap.add_argument("--time", metavar="DIR")
    ap.add_argument("--seq-limit", type=int, default=32,
                    help="sequential baseline: time at most this many runs and scale to all of them")
    args = ap.parse_args()
    if args.dump:
        dump(args.dump)
    if args.time:
        os.makedirs(args.time, exist_ok=True)
        emit(args.time, dict(device=device_facts()))
        time_planes(args.time)
        time_helpers(args.time, args.seq_limit)


if __name__ == "__main__":
    main()
