"""Device-resident BioEn problem: yTilde uploaded once, evaluations and minimisers run in HBM.

Thin object wrapper over the handle API of libbioen_b200.so (include/bioen_b200.h part 2).  The reference has
no such object -- its C entry points take host pointers on every call (bioen/optimize/ext/c_bioen.pyx) -- but
every reference call maps onto one method here, and `bioen_b200.optimize` uses it so that a whole
`find_optimum` (and a whole theta series) performs exactly one host->device copy of the M x N matrix.
"""
import ctypes as C

import numpy as np

from . import _lib

LOGW, FORCES = 0, 1

LBFGS_DEFAULTS = dict(linesearch=2, max_iterations=5000, delta=1e-6, epsilon=1e-6, ftol=1e-5, gtol=0.9,
                      wolfe=0.9, past=10, max_linesearch=100)  # bioen/optimize/config/bioen_optimize.yaml:33-46
GSL_DEFAULTS = dict(algorithm=2, step_size=0.01, tol=0.001, max_iterations=5000)  # ...yaml:20-31
LBFGS_OK = (0, 1, 2)       # c_bioen.pyx:120
GSL_OK = (0, -2, 27)       # c_bioen.pyx:112-116


def device_count():
    return int(_lib.load().bioen_b200_device_count())


def lbfgs_strerror(code):
    return _lib.load().lbfgs_strerror(int(code)).decode()


def gsl_strerror(code):
    return _lib.load().bioen_gsl_error(int(code)).decode()


class _PinnedOwner:
    def __init__(self, ptr):
        self.ptr = ptr

    def __del__(self):
        try:
            _lib.load().bioen_b200_host_free(C.c_void_p(self.ptr))
        except Exception:
            pass


def pinned_empty(shape, dtype=np.float64):
    """NumPy array in page-locked host memory (freed with the array): fill yTilde into it and the upload runs as one
    asynchronous copy at PCIe speed instead of being staged through pageable memory."""
    shape = tuple(int(v) for v in np.atleast_1d(shape))
    nbytes = int(np.prod(shape)) * np.dtype(dtype).itemsize
    ptr = _lib.load().bioen_b200_host_alloc(max(nbytes, 1))
    if not ptr:
        raise RuntimeError("bioen_b200_host_alloc failed: " + _lib.last_error())
    buf = (C.c_char * max(nbytes, 1)).from_address(ptr)
    buf._bioen_owner = _PinnedOwner(ptr)     # the ctypes buffer is the base of every NumPy view: freed with the last one
    return np.frombuffer(buf, dtype=dtype, count=int(np.prod(shape))).reshape(shape)


_PROBE_MAX = 1 << 18   # entries of x up to which objective() keeps a copy for gradient()


class Problem:
    """yTilde (m x n, this rank's columns when sharded) resident on one GPU."""

    def __init__(self, yTilde=None, shape=None, device=0, structure_major_only=False):
        """structure_major_only=True: the device keeps ONLY the structure-major copy of yTilde that the fused forces
        kernels read (half the memory of the default forces set-up; forces method only, 256 <= M <= ~5500)."""
        self._lib = _lib.load()
        self._h = None
        if yTilde is not None:
            yT = _lib.mat(yTilde)
            if yT.ndim != 2:
                raise ValueError("yTilde must be a 2-d array")
            shape = yT.shape
        if shape is None:
            raise ValueError("either yTilde or shape is required")
        self.m, self.n = int(shape[0]), int(shape[1])
        self.device = int(device)
        self._h = self._lib.bioen_b200_create(self.m, self.n, self.device)
        if not self._h:
            msg = _lib.last_error()
            _lib.clear_pending()
            raise RuntimeError("bioen_b200_create failed: " + msg)
        self.method = None
        self.YTilde = None      # host copies of the data set_logw / set_forces put on the device (replicates.py)
        self.w0 = None
        self.nranks = 1
        if structure_major_only:
            _lib.check(self._lib.bioen_b200_set_option(self._ctx, 11, 1), "set_option")
        if yTilde is not None:
            _lib.check(self._lib.bioen_b200_upload_ytilde(self._ctx, _lib.ptr(yT), self.n), "upload_ytilde")

    # ---- lifetime -----------------------------------------------------------------------------------
    @property
    def _ctx(self):
        if not getattr(self, "_h", None):
            raise RuntimeError("bioen_b200.Problem: used after close()")
        return self._h

    def close(self):
        cached = getattr(self, "_y_cache", None)
        if cached is not None:
            self._y_cache = None
            cached[1].close()
        if getattr(self, "_h", None):
            self._lib.bioen_b200_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def like(self, y):
        """A problem on the same device holding another matrix (e.g. y for the post-processing y.wopt)."""
        return Problem(y, device=self.device)

    # ---- data ---------------------------------------------------------------------------------------
    def adopt(self, dev_ptr, ld):
        """Use a matrix already on the device (e.g. a torch tensor's data_ptr()); caller keeps ownership."""
        _lib.check(self._lib.bioen_b200_adopt_ytilde(self._ctx, C.c_void_p(int(dev_ptr)), int(ld)), "adopt_ytilde")

    def upload_rows(self, row0, rows):
        """Chunked upload: rows[row0 : row0 + len(rows)] of yTilde (2-d, n columns).  For `Problem(shape=...)`
        objects whose matrix arrives block by block (e.g. read from disk); call before set_logw / set_forces."""
        blk = _lib.mat(rows)
        if blk.ndim != 2 or blk.shape[1] != self.n:
            raise ValueError("rows must be a (k, n) block")
        _lib.check(self._lib.bioen_b200_upload_rows(self._ctx, int(row0), blk.shape[0], _lib.ptr(blk), self.n),
                   "upload_rows")

    def generate(self, seed, col_offset, ytrue_over_sigma, inv_sigma):
        a = _lib.vec(ytrue_over_sigma)
        if a.size != self.m:
            raise ValueError("ytrue_over_sigma must have m entries")
        _lib.check(self._lib.bioen_b200_generate_ytilde(self._ctx, int(seed), int(col_offset), _lib.ptr(a),
                                                        float(inv_sigma)), "generate_ytilde")

    def download(self, row0=0, nrows=None, col0=0, ncols=None):
        nrows = self.m - row0 if nrows is None else nrows
        ncols = self.n - col0 if ncols is None else ncols
        out = np.empty((nrows, ncols), dtype=np.float64)
        _lib.check(self._lib.bioen_b200_download_ytilde(self._ctx, row0, nrows, col0, ncols, _lib.ptr(out)),
                   "download_ytilde")
        return out

    def set_logw(self, G, YTilde, theta):
        G, Y = _lib.vec(G), _lib.vec(YTilde)
        if G.size != self.n or Y.size != self.m:
            raise ValueError("G must have n and YTilde m entries")
        _lib.check(self._lib.bioen_b200_set_logw(self._ctx, _lib.ptr(G), _lib.ptr(Y), float(theta)), "set_logw")
        self.method = LOGW
        self.YTilde, self.w0 = Y.copy(), None

    def set_forces(self, w0, YTilde, theta):
        w0, Y = _lib.vec(w0), _lib.vec(YTilde)
        if w0.size != self.n or Y.size != self.m:
            raise ValueError("w0 must have n and YTilde m entries")
        _lib.check(self._lib.bioen_b200_set_forces(self._ctx, _lib.ptr(w0), _lib.ptr(Y), float(theta)), "set_forces")
        self.method = FORCES
        self.YTilde, self.w0 = Y.copy(), w0.copy()

    def set_option(self, option, value):
        """Tuning switches of include/bioen_b200.h (1 = fused two-pass forces kernels, default on)."""
        _lib.check(self._lib.bioen_b200_set_option(self._ctx, int(option), int(value)), "set_option")

    def set_theta(self, theta):
        self._lib.bioen_b200_set_theta(self._ctx, float(theta))

    def comm_init(self, unique_id, rank, nranks, n_total):
        _lib.check(self._lib.bioen_b200_comm_init(self._ctx, unique_id, rank, nranks, int(n_total)), "comm_init")
        self.nranks = int(nranks)

    def comm_init_local(self, group, rank, nranks, n_total):
        """Join an in-process group (one host thread per rank; blocks until all `nranks` contexts have joined)."""
        _lib.check(self._lib.bioen_b200_comm_init_local(self._ctx, int(group), int(rank), int(nranks), int(n_total)),
                   "comm_init_local")
        self.nranks = int(nranks)

    def comm_mode(self):
        """How the per-evaluation exchanges travel: 'single', 'nccl' or 'p2p' (peer-memory kernel over NVLink)."""
        return ("single", "nccl", "p2p")[self._lib.bioen_b200_comm_mode(self._ctx)]

    # ---- evaluations --------------------------------------------------------------------------------
    def _dim(self, method):
        return self.m if method == FORCES else self.n

    def _method(self, method):
        """The method an evaluation runs for: the one whose data is set; an explicit mismatch is an error (G and w0
        share device storage, so the other method's data is gone)."""
        if self.method is None:
            raise RuntimeError("bioen_b200.Problem: call set_logw or set_forces first")
        if method is not None and method != self.method:
            raise ValueError("bioen_b200.Problem: %s data is set; call %s first" % (
                ("log-weights", "set_forces") if self.method == LOGW else ("forces", "set_logw")))
        return self.method

    def objective(self, x, method=None):
        method = self._method(method)
        x = _lib.vec(x)
        if x.size != self._dim(method):
            raise ValueError("wrong length of the variable vector")
        f = C.c_double()
        _lib.check(self._lib.bioen_b200_eval(self._ctx, method, _lib.ptr(x), C.byref(f), None), "eval")
        # remembered so that gradient(x) at this same point runs the gradient half only (SciPy asks f, then fprime);
        # for long vectors the copy + compare would cost what it saves
        self._probe = (method, x.copy()) if x.size <= _PROBE_MAX else None
        return f.value

    def objective_and_gradient(self, x, method=None):
        method = self._method(method)
        x = _lib.vec(x)
        if x.size != self._dim(method):
            raise ValueError("wrong length of the variable vector")
        f = C.c_double()
        g = np.empty(x.size, dtype=np.float64)
        _lib.check(self._lib.bioen_b200_eval(self._ctx, method, _lib.ptr(x), C.byref(f), _lib.ptr(g)), "eval")
        return f.value, g

    def gradient(self, x, method=None):
        method = self._method(method)
        probe, self._probe = getattr(self, "_probe", None), None
        if probe is not None and probe[0] == method:
            x = _lib.vec(x)
            if x.size == probe[1].size and np.array_equal(x, probe[1]):
                g = np.empty(x.size, dtype=np.float64)
                status = self._lib.bioen_b200_grad_continue(self._ctx, method, _lib.ptr(g))
                if status == 0:
                    return g
                if status != 2:         # 2: the device state has moved on -> full evaluation below
                    _lib.check(status, "grad_continue")
        return self.objective_and_gradient(x, method)[1]

    def weights(self, x, method=None):
        """w (n,) and, for the log-weights method, s = sum_j exp(g_j) (None for forces)."""
        method = self._method(method)
        x = _lib.vec(x)
        w = np.empty(self.n, dtype=np.float64)
        s = C.c_double()
        _lib.check(self._lib.bioen_b200_weights(self._ctx, method, _lib.ptr(x), _lib.ptr(w), C.byref(s)), "weights")
        return w, (s.value if method == LOGW else None)

    def average(self, w):
        """avg (m,) = yTilde . w with the resident matrix."""
        w = _lib.vec(w)
        if w.size != self.n:
            raise ValueError("w must have n entries")
        out = np.empty(self.m, dtype=np.float64)
        _lib.check(self._lib.bioen_b200_average(self._ctx, _lib.ptr(w), _lib.ptr(out)), "average")
        return out

    def affine_rows(self, scale, offset):
        """In-place on the device: yTilde_ij <- scale_i * yTilde_ij + offset_i (refitted nuisance parameters, see
        bioen_b200.nuisance).  Evaluations and minimisers afterwards see the transformed matrix."""
        scale, offset = _lib.vec(scale), _lib.vec(offset)
        if scale.size != self.m or offset.size != self.m:
            raise ValueError("scale and offset must have m entries")
        _lib.check(self._lib.bioen_b200_affine_rows(self._ctx, _lib.ptr(scale), _lib.ptr(offset)), "affine_rows")

    def chi2_residuals(self, w, scale=None, offset=None, YTilde=None):
        """Residuals r_i = scale_i * (yTilde . w)_i + offset_i * sum(w) - YTilde_i of the resident matrix seen through
        a row-affine transform (default: identity), with ONE row pass on the device; chi^2 = 0.5 * r.r.  A nuisance
        parameter that acts affinely on the rows is scanned with this at O(M) cost per trial value."""
        w = _lib.vec(w)
        avg = self.average(w)
        sw = float(w.sum())
        scale = np.ones(self.m) if scale is None else _lib.vec(scale)
        offset = np.zeros(self.m) if offset is None else _lib.vec(offset)
        r = scale * avg + offset * sw
        return r if YTilde is None else r - _lib.vec(YTilde)

    def average_streamed(self, y, w, chunk_bytes=256 << 20):
        """y . w for a HOST matrix y (m' x n) that is needed once (the post-processing yopt = y . wopt of find_optimum,
        bioen/optimize/log_weights.py:612-613): y is streamed through a device buffer of `chunk_bytes` in row chunks
        and each chunk is reduced by the row-pass kernel (256 MB chunks measured fastest and steadiest: 0.77-0.80 s for
        8 GB against 0.50 s for a whole-matrix upload), so no second resident copy of an M x N matrix is allocated
        (8 GB at config 3) and a y larger than the free HBM works too."""
        yv = _lib.mat(y)
        w = _lib.vec(w)
        if yv.ndim != 2 or yv.shape[1] != self.n or w.size != self.n:
            raise ValueError("y must be (m', n) and w (n,)")
        mp = yv.shape[0]
        rows = max(1, min(mp, int(chunk_bytes) // (8 * self.n)))
        out = np.empty(mp, dtype=np.float64)
        with Problem(shape=(rows, self.n), device=self.device) as q:
            for r0 in range(0, mp, rows):
                blk = yv[r0:r0 + rows]
                if blk.shape[0] < rows:                      # ragged tail: pad to the buffer's shape
                    pad = np.zeros((rows, self.n))
                    pad[:blk.shape[0]] = blk
                    blk = pad
                _lib.check(self._lib.bioen_b200_upload_ytilde(q._ctx, _lib.ptr(blk), self.n), "upload_ytilde")
                out[r0:r0 + rows] = q.average(w)[:min(rows, mp - r0)]
        return out

    def forces_from_weights(self, w, gradient=True):
        """Reference semantics of _bioen_log_posterior_forces/_grad_...: objective (, gradient) for GIVEN w."""
        w = _lib.vec(w)
        f = C.c_double()
        g = np.empty(self.m, dtype=np.float64) if gradient else None
        _lib.check(self._lib.bioen_b200_forces_from_weights(self._ctx, _lib.ptr(w), C.byref(f),
                                                            _lib.ptr(g) if gradient else None), "forces_from_weights")
        return (f.value, g) if gradient else f.value

    # ---- minimisers ---------------------------------------------------------------------------------
    def opt_lbfgs(self, x0, method=None, verbose=0, **cfg):
        """Device-resident L-BFGS (liblbfgs semantics).  Returns (x, fmin, code, info)."""
        method = self._method(method)
        p = dict(LBFGS_DEFAULTS)
        p.update(cfg)
        c = _lib.lbfgs_config_params(**{k: p[k] for k, _ in _lib.lbfgs_config_params._fields_})
        v = _lib.visual_params(0, int(bool(verbose)))
        x0 = _lib.vec(x0)
        x = np.empty_like(x0)
        fmin = C.c_double()
        info = (C.c_int * 4)()
        code = self._lib.bioen_b200_opt_lbfgs(self._ctx, method, _lib.ptr(x0), _lib.ptr(x), c, v, C.byref(fmin), info)
        if code == -2000:
            raise RuntimeError("bioen_b200_opt_lbfgs failed: " + _lib.last_error())
        return x, fmin.value, code, dict(iterations=info[0], evaluations=info[1], gradients_skipped=info[2])

    def opt_gsl(self, x0, method=None, verbose=0, **cfg):
        """Device-resident GSL-style minimisers.  Returns (x, fmin, status, info)."""
        method = self._method(method)
        p = dict(GSL_DEFAULTS)
        p.update(cfg)
        c = _lib.gsl_config_params(float(p["step_size"]), float(p["tol"]), int(p["max_iterations"]),
                                   int(p["algorithm"]))
        v = _lib.visual_params(0, int(bool(verbose)))
        x0 = _lib.vec(x0)
        x = np.empty_like(x0)
        fmin = C.c_double()
        info = (C.c_int * 4)()
        code = self._lib.bioen_b200_opt_gsl(self._ctx, method, _lib.ptr(x0), _lib.ptr(x), c, v, C.byref(fmin), info)
        if code == -2000:
            raise RuntimeError("bioen_b200_opt_gsl failed: " + _lib.last_error())
        return x, fmin.value, code, dict(iterations=info[0], gradient_evaluations=info[1], f_only_evaluations=info[2],
                                          gradient_half_only=info[3])

    def theta_scan(self, thetas, x0=None, method=None, verbose=0, **cfg):
        """Minimise the problem for up to 32 theta values TOGETHER (lockstep L-BFGS, batched fp64 tensor-core
        evaluations).  x0: (n,) shared start or (K, n), n = N for log-weights, M for forces.  Returns
        (X (K, n), fmin (K,), codes (K,), info dict).  Call set_logw / set_forces first (their theta is ignored)."""
        method = self.method if method is None else method
        if method is None:
            raise RuntimeError("theta_scan: log-weights data not set / forces data not set (call set_logw or "
                               "set_forces first)")
        n = self._dim(method)
        thetas = _lib.vec(thetas)
        K = thetas.size
        if x0 is None:
            x0 = np.zeros(n)
        x0 = np.asarray(x0, dtype=np.float64)
        X0 = np.ascontiguousarray(np.broadcast_to(x0.reshape(-1, n) if x0.size != n else x0.reshape(1, n), (K, n)))
        p = dict(LBFGS_DEFAULTS)
        p.update(cfg)
        c = _lib.lbfgs_config_params(**{k: p[k] for k, _ in _lib.lbfgs_config_params._fields_})
        v = _lib.visual_params(0, int(bool(verbose)))
        X = np.empty((K, n), dtype=np.float64)
        fmin = np.empty(K, dtype=np.float64)
        codes = (C.c_int * K)()
        info = (C.c_int * (2 * K))()
        stats = np.zeros(4, dtype=np.float64)
        _lib.check(self._lib.bioen_b200_theta_scan(self._ctx, method, K, _lib.ptr(thetas), _lib.ptr(X0), _lib.ptr(X), c, v,
                                                   _lib.ptr(fmin), codes, info, _lib.ptr(stats)), "theta_scan")
        return X, fmin, np.array(codes[:]), dict(iterations=np.array(info[0::2]), evaluations=np.array(info[1::2]),
                                                 rounds=int(stats[0]), gemm_launches=int(stats[1]),
                                                 seconds=float(stats[2]))

    # ---- batched replicates: K <= 32 problems with per-problem YTilde, observable weights, w0, row transform --------
    _PLANES = ("YTilde", "row_weights", "w0", "row_scale", "row_offset")

    def _batch(self, method, thetas, X, YTilde, row_weights, w0, row_scale=None, row_offset=None):
        """The bioen_b200_batch of a call and the arrays it points to: thetas (K,), X (K, n), and (K, M) / (K, N)
        planes or None.  A scalar theta and single vectors are broadcast; K comes from whichever argument has rows."""
        n = self._dim(method)
        args = [("thetas", np.asarray(thetas, dtype=np.float64), 0), ("x", np.asarray(X, dtype=np.float64), n),
                ("YTilde", YTilde, self.m), ("row_weights", row_weights, self.m), ("w0", w0, self.n),
                ("row_scale", row_scale, self.m), ("row_offset", row_offset, self.m)]
        args = [(name, None if a is None else np.asarray(a, dtype=np.float64), width) for name, a, width in args]
        Ks = {a.shape[0] for name, a, width in args if a is not None and a.ndim == (1 if width == 0 else 2)} - {1}
        if len(Ks) > 1:
            raise ValueError("per-problem arguments disagree on the number of problems: %s" % sorted(Ks))
        K = Ks.pop() if Ks else 1
        if not 1 <= K <= 32:
            raise ValueError("a batch holds 1..32 problems, got %d" % K)
        out = {}
        for name, a, width in args:
            if a is None:
                out[name] = None
                continue
            want = (K,) if width == 0 else (K, width)
            if a.shape not in (want, want[1:], (1,) + want[1:]):
                raise ValueError("%s must have shape %s or %s, got %s" % (name, want[1:] or "()", want, a.shape))
            out[name] = np.ascontiguousarray(np.broadcast_to(a, want))
        b = _lib.bioen_b200_batch(K, _lib.ptr(out["thetas"]), *(None if out[k] is None else _lib.ptr(out[k])
                                                                   for k in self._PLANES))
        return K, n, b, out

    def batch_minimize(self, thetas, x0=None, YTilde=None, row_weights=None, w0=None, method=None, verbose=0,
                       row_scale=None, row_offset=None, **cfg):
        """Minimise up to 32 problems that share yTilde TOGETHER (the theta scan's lockstep L-BFGS and batched fp64
        tensor-core evaluations).  Per problem k, optionally: YTilde[k] (M,) in place of the shared YTilde,
        observable weights row_weights[k] (M,) >= 0 with chi^2 = 1/2 sum_i c_i r_i^2, (forces only) reference
        weights w0[k] (N,) >= 0, and a row-affine transform row_scale[k], row_offset[k] (M,) (finite; default ones
        and zeros): problem k is the one of the matrix row_scale[k][:, None] * yTilde + row_offset[k][:, None], e.g.
        nuisance parameters (bioen_b200.nuisance.theta_series), while the resident matrix stays as it is.  Scalars /
        single vectors are broadcast.  Returns (X (K, n), fmin (K,), codes (K,), info) like theta_scan; info also
        holds averages (K, M) = yTilde . w of the RESIDENT matrix (problem k's own averages are
        row_scale[k] * averages[k] + row_offset[k]), chi2 (K,) and kl (K,) at the returned points (NaN when the
        L-BFGS parameters are refused)."""
        method = self._method(method)
        K, n, b, a = self._batch(method, thetas, np.zeros(self._dim(method)) if x0 is None else x0, YTilde,
                                 row_weights, w0, row_scale, row_offset)
        p = dict(LBFGS_DEFAULTS)
        p.update(cfg)
        c = _lib.lbfgs_config_params(**{k: p[k] for k, _ in _lib.lbfgs_config_params._fields_})
        v = _lib.visual_params(0, int(bool(verbose)))
        X = np.empty((K, n), dtype=np.float64)
        fmin, chi2, kl = np.empty(K), np.empty(K), np.empty(K)
        avg = np.empty((K, self.m), dtype=np.float64)
        codes = (C.c_int * K)()
        info = (C.c_int * (2 * K))()
        stats = np.zeros(4, dtype=np.float64)
        _lib.check(self._lib.bioen_b200_batch_minimize(self._ctx, method, C.byref(b), _lib.ptr(a["x"]), _lib.ptr(X), c, v,
                                                       _lib.ptr(fmin), codes, info, _lib.ptr(stats), _lib.ptr(avg),
                                                       _lib.ptr(chi2), _lib.ptr(kl)), "batch_minimize")
        return X, fmin, np.array(codes[:]), dict(iterations=np.array(info[0::2]), evaluations=np.array(info[1::2]),
                                                 rounds=int(stats[0]), gemm_launches=int(stats[1]),
                                                 seconds=float(stats[2]), averages=avg, chi2=chi2, kl=kl)

    def batch_evaluate(self, X, thetas, YTilde=None, row_weights=None, w0=None, gradient=True, method=None,
                       row_scale=None, row_offset=None):
        """One batched evaluation of up to 32 problems (arguments as batch_minimize) at the points X (K, n).
        Returns (f (K,), grad (K, n) or None, dict(averages (K, M), chi2 (K,), kl (K,))); averages as batch_minimize:
        yTilde . w of the resident matrix."""
        method = self._method(method)
        K, n, b, a = self._batch(method, thetas, X, YTilde, row_weights, w0, row_scale, row_offset)
        f, chi2, kl = np.empty(K), np.empty(K), np.empty(K)
        g = np.empty((K, n), dtype=np.float64) if gradient else None
        avg = np.empty((K, self.m), dtype=np.float64)
        _lib.check(self._lib.bioen_b200_batch_eval(self._ctx, method, C.byref(b), _lib.ptr(a["x"]), _lib.ptr(f),
                                                   _lib.ptr(g) if gradient else None, _lib.ptr(avg), _lib.ptr(chi2),
                                                   _lib.ptr(kl)), "batch_eval")
        return f, g, dict(averages=avg, chi2=chi2, kl=kl)

    # ---- device-pointer entry points (bench.py) -----------------------------------------------------------
    def time_evals(self, x_dev_ptr, grad_dev_ptr, warmup, steps, method=None):
        method = self.method if method is None else method
        ms, pass_ms, launches = C.c_float(), C.c_float(), C.c_longlong()
        _lib.check(self._lib.bioen_b200_time_evals(self._ctx, method, C.c_void_p(int(x_dev_ptr)),
                                                   C.c_void_p(int(grad_dev_ptr)), warmup, steps, C.byref(ms),
                                                   C.byref(pass_ms), C.byref(launches)), "time_evals")
        return ms.value, pass_ms.value, launches.value

    def query(self, what):
        return int(self._lib.bioen_b200_query(self._ctx, int(what)))

    def pass_kernel_name(self, method=None):
        """Name of the kernel that streams yTilde for `method` (bench.py's roofline record)."""
        method = self.method if method is None else method
        if self.query(7) == 1:
            return "slice_eval_kernel"
        if self.query(3):
            return "persistent_eval_kernel"
        return "fused_team_pass" if (method == FORCES and self.query(0)) else "stream_pass_kernel"

    def exchanges_per_eval(self, method=None):
        method = self.method if method is None else method
        return self.query(2 if method == FORCES else 1)

    def kernels_launched(self):
        return int(self._lib.bioen_b200_kernels_launched(self._ctx))

    def debug_read(self, what, count):
        """Device vectors an evaluation leaves behind (tests): 1 weights, 2 averages, 3 / 4 the forces method's
        per-structure vectors (E_j or x_j; guarded log-ratio)."""
        out = np.empty(int(count), dtype=np.float64)
        _lib.check(self._lib.bioen_b200_debug_read(self._ctx, int(what), _lib.ptr(out), int(count)), "debug_read")
        return out

    def scalars(self):
        out = np.empty(64, dtype=np.float64)
        _lib.check(self._lib.bioen_b200_debug_read(self._ctx, 0, _lib.ptr(out), 64), "debug_read")
        return out
