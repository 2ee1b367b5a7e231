"""Cost of the per-problem row-affine planes of the batched engine, and the batched theta series with nuisance
refits against the sequential one.

    python scripts/nuisance_batch_probe.py DIR [--reps 5] [--steps 20]

prints the device name, power limit and maximum SM clock, then measures
  (a) one batched f+g evaluation of K = 32 problems without and with row_scale / row_offset planes (CUDA events over
      `steps` evaluations after 3 warm-up ones, bioen_b200_time_batch_evals; the two variants alternate `reps`
      times) at 500 x 1e5 and 1000 x 1e6 (device-generated yTilde), both methods;
  (b) 16 thetas x 4 weight <-> nuisance iterations, log-weights, end to end (host clock around work that ends in a
      device synchronise): nuisance.theta_series against the sequential path -- per theta a fresh upload of the
      start matrix, a fresh NuisanceRefit, and per iteration find_optimum(problem=...) then NuisanceRefit.update --
      on the reference's DEER test data (tests/golden/nuisance_deer.npz, 462 x 10) and on a synthetic 500 x 1e5
      problem with four DEER blocks, one scattering block and fixed rows.
Records go to stdout and DIR/nuisance_batch_probe.jsonl.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def emit(out, rec):
    print(json.dumps(rec), flush=True)
    with open(os.path.join(out, "nuisance_batch_probe.jsonl"), "a") as fh:
        fh.write(json.dumps(rec) + "\n")


def device_facts():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def time_evals(p, method, K, planes, x0, steps):
    """ms per batched f+g evaluation of K problems"""
    from bioen_b200 import _lib
    thetas = np.geomspace(1e3, 1e-1, K)
    arrs = {k: np.ascontiguousarray(v) for k, v in planes.items()}
    b = _lib.bioen_b200_batch(K, _lib.ptr(thetas), *(_lib.ptr(arrs[k]) if k in arrs else None
                                                      for k in p._PLANES))
    ms, gemm_ms, launches = C.c_float(), C.c_float(), C.c_longlong()
    _lib.check(p._lib.bioen_b200_time_batch_evals(p._ctx, method, C.byref(b), _lib.ptr(x0), 3, steps,
                                                  C.byref(ms), C.byref(gemm_ms), C.byref(launches)), "time_batch_evals")
    return ms.value / steps


def plane_cost(out, reps, steps):
    import bioen_b200
    from bioen_b200.problem import FORCES, LOGW
    K = 32
    for M, N in ((500, 100000), (1000, 1000000)):
        rng = np.random.default_rng(M)
        ytrue = rng.standard_normal(M)
        YT = (ytrue + 0.5 * rng.standard_normal(M)) / 0.5
        with bioen_b200.Problem(shape=(M, N)) as p:
            p.generate(12345, 0, ytrue / 0.5, 1.0 / 0.5)
            planes = dict(row_scale=rng.uniform(0.5, 1.5, (K, M)), row_offset=rng.standard_normal((K, M)))
            for method in (LOGW, FORCES):
                if method == LOGW:
                    p.set_logw(np.zeros(N), YT, 1.0)
                else:
                    p.set_forces(np.full(N, 1.0 / N), YT, 1.0)
                n = M if method == FORCES else N
                x0 = np.ascontiguousarray((1e-3 if method == FORCES else 0.1) * rng.standard_normal((K, n)))
                t = {"none": [], "planes": []}
                for r in range(reps):
                    t["none"].append(time_evals(p, method, K, {}, x0, steps))
                    t["planes"].append(time_evals(p, method, K, planes, x0, steps))
                a, b = float(np.median(t["none"])), float(np.median(t["planes"]))
                emit(out, dict(what="batched f+g evaluation, K=32", M=M, N=N, method="forces" if method else "logw",
                               ms_no_planes=t["none"], ms_planes=t["planes"], median_no_planes=a,
                               median_planes=b, gap_percent=100.0 * (b - a) / a,
                               plane_bytes=8.0 * K * 2 * M, matrix_bytes=8.0 * M * N))


def synthetic(M_deer=(100, 100, 100, 100), M_sc=60, M_fixed=40, N=100000, seed=7):
    """base matrix, blocks (start values) and YTilde: four DEER blocks, one scattering block, fixed rows"""
    from bioen_b200 import nuisance as NU
    rng = np.random.default_rng(seed)
    M = sum(M_deer) + M_sc + M_fixed
    base = np.empty((M, N))
    err = np.full(M, 0.2)
    blocks, r0 = [], 0
    wtrue = rng.random(N) ** 4
    wtrue /= wtrue.sum()
    for q, rows in enumerate(M_deer):
        t = np.linspace(0.0, 3.0, rows)[:, None]
        base[r0:r0 + rows] = np.exp(-t * rng.uniform(0.5, 3.0, N)[None, :]) / err[r0:r0 + rows, None]
        blocks.append((NU.DEER, r0, r0 + rows, 0.3 + 0.05 * q))
        r0 += rows
    qv = np.linspace(0.01, 0.5, M_sc)[:, None]
    base[r0:r0 + M_sc] = 3000.0 * np.exp(-(qv * rng.uniform(5.0, 15.0, N)[None, :]) ** 2 / 3.0) / err[r0:r0 + M_sc, None]
    blocks.append((NU.SCATTERING, r0, r0 + M_sc, 3e-4))
    r0 += M_sc
    err[r0:] = 0.5
    base[r0:] = rng.standard_normal((M_fixed, N)) / 0.5
    blocks.append((NU.FIXED, r0, M, None))
    true = [NU.Block(k, a, b, err=err[a:b], exp_fit=np.ones(b - a), value=v) for k, a, b, v in blocks]
    Y = NU.proc_sim(base, true) @ wtrue + rng.standard_normal(M)
    start = [NU.Block(k, a, b, err=err[a:b], exp_fit=None if k == NU.FIXED else Y[a:b] * err[a:b],
                      value=None if v is None else 1.2 * v, name="b%d" % q) for q, (k, a, b, v) in enumerate(blocks)]
    return base, start, Y


def series(out, name, base, blocks, Y, thetas, lbfgs):
    import bioen_b200
    from bioen_b200 import _lib, nuisance as NU, optimize
    M, N = base.shape
    its = 4
    G = np.zeros(N)
    y0 = NU.proc_sim(base, blocks)
    starts = {b.name: b.value for b in blocks if b.kind != NU.FIXED}
    with bioen_b200.Problem(y0) as p:
        p.set_logw(G, Y, 1.0)
        p.batch_minimize([1.0, 2.0], max_iterations=3)                     # warm-up
        t0 = time.perf_counter()
        res = NU.theta_series(p, blocks, thetas, its, x0=G, **lbfgs)
        t_batch = time.perf_counter() - t0
        cfg = optimize.minimize.Parameters("lbfgs")
        cfg["verbose"] = False
        cfg["params"].update(lbfgs)
        YT = Y.reshape(1, -1)
        Gc = G.reshape(-1, 1)
        fmin_seq, val_seq = np.full((its, 16), np.nan), {k: np.full((its + 1, 16), np.nan) for k in starts}
        t0 = time.perf_counter()
        for t, theta in enumerate(thetas):
            _lib.check(p._lib.bioen_b200_upload_ytilde(p._ctx, _lib.ptr(y0), N), "upload_ytilde")
            for b in blocks:
                if b.kind != NU.FIXED:
                    b.value = starts[b.name]
                    val_seq[b.name][0, t] = b.value
            refit = NU.NuisanceRefit(p, blocks)
            for it in range(its):
                try:
                    r = optimize.log_weights.find_optimum(Gc, Gc, y0, y0, YT, float(theta), cfg, problem=p)
                except RuntimeError:
                    break
                fmin_seq[it, t] = r[4]
                w = r[0].ravel().copy()
                w[w == 0.0] = 1e-150
                for k, v in refit.update(w).items():
                    val_seq[k][it + 1, t] = v
        t_seq = time.perf_counter() - t0
        for b in blocks:
            if b.kind != NU.FIXED:
                b.value = starts[b.name]
    ok = np.isfinite(fmin_seq) & np.isin(res["codes"], (0, 1, 2))
    dv = max(float(np.nanmax(np.abs(res["values"][k][1:][ok] / val_seq[k][1:][ok] - 1.0))) for k in starts)
    emit(out, dict(what="theta series, 16 thetas x 4 iterations, log-weights", problem=name, M=M, N=N,
                   thetas=[float(thetas[0]), float(thetas[-1])], lbfgs=lbfgs,
                   batched_s=t_batch, sequential_s=t_seq, speedup=t_seq / t_batch,
                   max_rel_fmin_diff=float(np.max(np.abs(res["fmin"][ok] / fmin_seq[ok] - 1.0))),
                   max_rel_value_diff=dv, compared=int(ok.sum()),
                   codes={int(c): int(v) for c, v in zip(*np.unique(res["codes"], return_counts=True))}))


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("out")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--steps", type=int, default=20)
    args = ap.parse_args()
    os.makedirs(args.out, exist_ok=True)
    from bioen_b200 import nuisance as NU
    emit(args.out, dict(device=device_facts()))
    plane_cost(args.out, args.reps, args.steps)
    d = np.load(os.path.join(ROOT, "tests", "golden", "nuisance_deer.npz"))
    blocks = [NU.Block("deer", 0, d["raw"].shape[0], err=d["err"], exp_fit=d["exp_fit"],
                       value=float(d["wf_values"][0]), name="deer")]
    series(args.out, "reference DEER test data", NU.base_matrix(d["raw"], d["err"]), blocks, d["YTilde"].ravel(),
           np.geomspace(100.0, 0.5, 16), dict(epsilon=1e-7, delta=1e-10, max_iterations=20000))
    base, blocks, Y = synthetic()
    series(args.out, "synthetic, 4 DEER + 1 scattering block + fixed rows", base, blocks, Y,
           np.geomspace(1000.0, 10.0, 16), dict(epsilon=1e-7, delta=1e-10, max_iterations=20000))


if __name__ == "__main__":
    main()
