"""Pathway-seeded initialisation on the GPU -- `--manifolds-init` of the reference CLI (script/prmf_runner.py:272-334,
:1023-1064).  The reference loops over the init pathways and calls scipy.optimize.nnls twice for each, on the host.
Here every solve of one side runs in one batched device call (prmf_nnls_x): Lawson & Hanson's active-set method,
whose only work over all of X is the dual vector A^T (b - A x), computed by the same X streams as the inner step.
"""
import numpy as np

from . import _lib
from .engine import CudaEngine


def _is_cuda(X):
    return hasattr(X, "is_cuda") and X.is_cuda


def _check_X(X, x_dtype="f64"):
    """Shape and finiteness of X (host array or CUDA tensor), before any library call.  An "f32" solve also takes
    float32 X, whose values it keeps exactly."""
    if x_dtype not in ("f64", "f32"):
        raise ValueError('x_dtype must be "f64" or "f32", got %r' % (x_dtype,))
    if _is_cuda(X):
        import torch
        if X.dim() != 2:
            raise ValueError("Expected a 2D array, but the shape of X is %s" % (tuple(X.shape),))
        if X.dtype != torch.float64 and not (x_dtype == "f32" and X.dtype == torch.float32):
            raise ValueError("device X must be float64" + (" or float32" if x_dtype == "f32" else ""))
        if not bool(torch.isfinite(X).all()):
            raise ValueError("array must not contain infs or NaNs")
        return X, tuple(X.shape)
    X = np.asarray(X)
    if not (x_dtype == "f32" and X.dtype == np.float32):
        X = np.asarray(X, dtype=np.float64)
    if X.ndim != 2:
        raise ValueError("Expected a 2D array, but the shape of X is %s" % (X.shape,))
    if not np.isfinite(X).all():
        raise ValueError("array must not contain infs or NaNs")            # np.asarray_chkfinite in scipy's nnls
    return X, X.shape


def _device(X, device):
    if device is not None:
        return int(device)
    import torch
    if not torch.cuda.is_available():
        raise _lib.PrmfLibraryError("the NNLS initialisation needs a CUDA device (no CPU fallback)")
    return X.device.index if _is_cuda(X) and X.device.index is not None else torch.cuda.current_device()


def _engine(X, shape, k, device, x_dtype):
    if not (1 <= k <= 128):
        raise ValueError("between 1 and 128 problems per call, got %d" % k)
    eng = CudaEngine(shape[0], shape[0], shape[1], k, device=_device(X, device), x_dtype=x_dtype)
    eng.set_X(X)
    return eng


def _solve(eng, B, transpose, maxiter, stats=None, key=None):
    x, rnorm, status, iters = eng.nnls(B, transpose, maxiter)
    if stats is not None:
        stats[key] = iters.tolist()
    if (status == -1).any():
        raise RuntimeError("Maximum number of iterations reached.")          # scipy's message
    if (status < -1).any():
        raise _lib.PrmfLibraryError(eng.last_error)
    return x, rnorm


def nnls_x(X, B, *, transpose, maxiter=None, device=None, x_dtype="f64"):
    """x[:, c] = scipy.optimize.nnls(op(X), B[:, c], maxiter=maxiter)[0] for every column c, with op(X) = X.T when
    `transpose` and X otherwise; all columns share each pass over X.  X: (m, n) host array or CUDA float64 tensor;
    B: (n, k) when `transpose`, (m, k) otherwise, or a vector for k = 1.  Returns (x, rnorm) shaped like B's columns
    ((m, k) / (n, k) and (k,); vectors for a vector B).  Raises RuntimeError at the iteration limit, as scipy does, and
    PrmfLibraryError when a solution needs more passive columns than the device workspace holds.  x_dtype="f32" solves
    on X held in fp32 (float32 X is kept exactly, float64 X is rounded to fp32): bitwise the "f64" solve on
    X.astype(np.float32).astype(np.float64)."""
    X, shape = _check_X(X, x_dtype)
    B = np.asarray(B, dtype=np.float64)
    vector = B.ndim == 1
    if vector:
        B = B[:, None]
    rows = shape[1] if transpose else shape[0]
    if B.ndim != 2 or B.shape[0] != rows:
        raise ValueError("Incompatible dimensions: X %s, B %s, transpose=%s" % (shape, B.shape, bool(transpose)))
    if not np.isfinite(B).all():
        raise ValueError("array must not contain infs or NaNs")
    if maxiter is not None and int(maxiter) <= 0:
        maxiter = None                                                      # scipy: `if not maxiter: maxiter = 3 * n`
    with _engine(X, shape, B.shape[1], device, x_dtype) as eng:
        x, rnorm = _solve(eng, B, bool(transpose), maxiter)
    return (x[:, 0], rnorm[0]) if vector else (x, rnorm)


def pathway_init(X, Gs_init, nodelist, rel_weight=5, device=None, stats=None, x_dtype="f64"):
    """(U_init (m, k), V_init (n, k)) for the k = len(Gs_init) init pathways, equal to the reference's per-pathway
    pathway_to_vec -> nmf_init_u -> nmf_init_v -> v_new[on] = signal (script/prmf_runner.py:272-334, :1023-1064).
    X: (m, n) host array or CUDA float64 tensor; it is uploaded once.  Consumes no random numbers.  A dict passed as
    `stats` receives the iterations of every solve, as scipy counts them ("iterations_u", "iterations_v").  x_dtype="f32"
    takes float32 X as well and solves on X held in fp32, as `nnls_x` does."""
    X, (m, n) = _check_X(X, x_dtype)
    k = len(Gs_init)
    index = {node: i for i, node in enumerate(nodelist)}
    if len(nodelist) != n:
        raise ValueError("nodelist has %d entries, X has %d columns" % (len(nodelist), n))
    with _engine(X, (m, n), k, device, x_dtype) as eng:
        # column means of X: one X^T . ones product, summed on the device and divided by m here, as np.mean does
        eng.set_UV(U=np.ones((m, k)))
        mean = eng.project_t()[:, 0] / m
        V0 = np.empty((n, k))
        ons = []
        for c, G in enumerate(Gs_init):                                     # pathway_to_vec (:272-334)
            v = np.zeros((n,))
            for node in G.nodes():
                v[index[node]] = 1
            on = (v == 1)
            off = np.invert(on)
            v[off] = mean[off]
            v[on] = (np.sum(v[off]) * rel_weight) / np.sum(on)
            V0[:, c] = v / np.linalg.norm(v)
            ons.append(on)
        u, _ = _solve(eng, V0, True, None, stats, "iterations_u")          # nmf_init_u: nnls(X^T, v)
        U_init = np.empty((m, k))
        for c in range(k):
            U_init[:, c] = u[:, c] / np.linalg.norm(u[:, c]) ** 2
        v, _ = _solve(eng, U_init, False, None, stats, "iterations_v")     # nmf_init_v: nnls(X, u)
        V_init = np.empty((n, k))
        for c in range(k):
            V_init[:, c] = v[:, c] / np.linalg.norm(v[:, c]) ** 2
            V_init[ons[c], c] = V0[ons[c], c]                               # v_new[on] = signal
    return U_init, V_init
