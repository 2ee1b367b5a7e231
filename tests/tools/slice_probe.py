"""Diagnostic (GPU box): device-timed f+g evaluations of small problems on the three launch paths -- stand-alone
kernels (0), persistent kernel (1), shared-memory slice kernel (2)."""
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
import torch  # noqa: E402

import bioen_b200  # noqa: E402

dev = torch.device("cuda", 0)
steps = int(os.environ.get("STEPS", "200"))
shapes = ((28, 50001), (808, 10), (808, 100), (64, 64), (100, 20000), (500, 2049), (1000, 777), (40, 76000))
if os.environ.get("SLICE_PROBE_SHAPES"):      # e.g. "28x50001,808x10"
    shapes = tuple(tuple(int(v) for v in s.split("x")) for s in os.environ["SLICE_PROBE_SHAPES"].split(","))
only = [int(v) for v in os.environ.get("SLICE_PROBE_PATHS", "2,1,0").split(",")]
for (M, N) in shapes:
    rng = np.random.default_rng(1)
    a = rng.standard_normal(M)
    YT = a + rng.standard_normal(M)
    with bioen_b200.Problem(shape=(M, N)) as p:
        p.generate(12345, 0, a, 2.0)
        for mode in only:
            p.set_option(5, 1 if mode else 0)
            p.set_option(8, 1 if mode == 2 else 0)
            if mode == 2 and p.query(7) != 1:
                print("M=%d N=%d: not slice-eligible" % (M, N), flush=True)
                continue
            for meth, name in ((0, "logw"), (1, "forces")):
                if meth == 0:
                    p.set_logw(np.zeros(N), YT, 10.0)
                else:
                    p.set_forces(np.full(N, 1.0 / N), YT, 10.0)
                n = N if meth == 0 else M
                x = torch.from_numpy((0.1 if meth == 0 else 1e-3) * rng.standard_normal(n)).to(dev)
                g = torch.zeros_like(x)
                ms, pass_ms, launches = p.time_evals(x.data_ptr(), g.data_ptr(), 5, steps, meth)
                print("M=%d N=%d %-6s path=%d (%s): %.2f us per f+g evaluation, %d launches" %
                      (M, N, name, mode, p.pass_kernel_name(meth), 1e3 * ms / steps, launches // steps), flush=True)
        # whole minimisations (host loop included)
        import time
        for mode in [m for m in only if m]:
            p.set_option(5, 1)
            p.set_option(8, 1 if mode == 2 else 0)
            if mode == 2 and p.query(7) != 1:
                continue
            p.set_forces(np.full(N, 1.0 / N), YT, 10.0)
            for small, spec, zc in ((1, 1, 1), (1, 1, 0), (0, 0, 0)):
                p.set_option(9, small)
                p.set_option(10, spec)
                p.set_option(12, zc)
                best = 1e9
                for _ in range(3):
                    t0 = time.perf_counter()
                    x, fmin, code, info = p.opt_lbfgs(np.zeros(M))
                    best = min(best, time.perf_counter() - t0)
                print("M=%d N=%d forces L-BFGS path=%d small-update=%d speculative=%d zero-copy-fetch=%d: %.3f ms (%d it, "
                      "%d evals, code %d, fmin %.10g)" % (M, N, mode, small, spec, zc, best * 1e3, info["iterations"],
                                                          info["evaluations"], code, fmin), flush=True)
            p.set_option(9, 1)
            p.set_option(10, 1)
            p.set_option(12, 1)
