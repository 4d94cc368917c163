"""Device engine: one `prmf_handle` (include/prmf_b200.h) per GPU, driven through ctypes.

The engine is the only thing the host solver (`prmf_b200.solver`) talks to for arithmetic.  It has no
CPU implementation: constructing it without a CUDA device or without libprmf_b200.so raises.
"""
import ctypes

import numpy as np

from . import _lib
from .pathways import PackedPathways

OBJ_KEYS = ("recon", "manifold", "ignore", "fro", "obj", "gamma", "delta", "recon_sq")


def _f64(a):
    a = np.ascontiguousarray(a, dtype=np.float64)
    return a


def _ptr(a):
    return a.ctypes.data_as(ctypes.c_void_p) if a is not None else None


class CudaEngine:
    """Owns the device-resident X row block, U, V, pathway tables and scratch of one rank."""

    def __init__(self, m_local, m_global, n, k, device=0, stream=None, x_dtype="f64"):
        """x_dtype: "f64" (parity mode, X streamed in fp64), "f32" (opt-in, single rank: X stored as exact fp32
        values and streamed through the fp64 kernels, bitwise what "f64" returns on X.astype(np.float64)) or "tf32"
        (opt-in: X stored as fp32 rounded to tf32, X.V and X^T.U on the tcgen05 tensor cores; everything else stays
        fp64)."""
        self.lib = _lib.load()
        self.m, self.m_global, self.n, self.k = int(m_local), int(m_global), int(n), int(k)
        self.P = 0
        if x_dtype not in _lib.X_DTYPES:
            raise ValueError("x_dtype must be one of %s" % sorted(_lib.X_DTYPES))
        self.x_dtype = x_dtype
        h = ctypes.c_void_p()
        rc = self.lib.prmf_create_ex(ctypes.byref(h), int(device), self.m, self.m_global, self.n, self.k,
                                     ctypes.c_void_p(stream) if stream else None, _lib.X_DTYPES[x_dtype])
        if rc != 0:
            msg = self.lib.prmf_last_error(None)
            raise _lib.PrmfLibraryError("prmf_create failed (%d): %s" % (rc, msg.decode() if msg else "?"))
        self.h = h
        self.device = int(device)
        self._keep = None

    # -- lifetime ------------------------------------------------------------------------------------
    def close(self):
        if getattr(self, "h", None):
            self.lib.prmf_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def _ck(self, rc):
        _lib.check(self.lib, self.h, rc)

    # -- data ----------------------------------------------------------------------------------------
    def set_X(self, X):
        """X: this rank's row block; a float64 numpy array (host) or a CUDA torch tensor.  "f32" and "tf32" engines
        also take float32 input, and round float64 input to fp32 (to tf32 in the tf32 mode) on the device."""
        x32 = self.x_dtype in ("tf32", "f32")
        if hasattr(X, "is_cuda") and X.is_cuda:
            import torch
            f32_ok = x32 and X.dtype == torch.float32
            if (X.dtype != torch.float64 and not f32_ok) or X.dim() != 2 or X.stride(1) != 1:
                raise ValueError("device X must be a 2-D float64 tensor with unit column stride"
                                 " (float32 is accepted by f32 and tf32 engines)")
            if tuple(X.shape) != (self.m, self.n):
                raise ValueError("X has shape %s, engine expects %s" % (tuple(X.shape), (self.m, self.n)))
            torch.cuda.current_stream(X.device).synchronize()
            if f32_ok:
                self._ck(self.lib.prmf_set_X_f32(self.h, ctypes.c_void_p(X.data_ptr()), int(X.stride(0)), 1))
            else:
                self._ck(self.lib.prmf_set_X_device(self.h, ctypes.c_void_p(X.data_ptr()), int(X.stride(0))))
            return
        X = np.asarray(X)
        if X.shape != (self.m, self.n):
            raise ValueError("X has shape %s, engine expects %s" % (X.shape, (self.m, self.n)))
        if x32 and X.dtype == np.float32 and X.strides[1] == 4 and X.strides[0] % 4 == 0:
            self._ck(self.lib.prmf_set_X_f32(self.h, _ptr(X), X.strides[0] // 4 if self.m > 0 else self.n, 0))
            return
        if X.dtype != np.float64 or X.strides[1] != 8 or X.strides[0] % 8 != 0:
            X = _f64(X)
        self._ck(self.lib.prmf_set_X(self.h, _ptr(X), X.strides[0] // 8 if self.m > 0 else self.n))

    @property
    def normX_sq(self):
        out = ctypes.c_double()
        self._ck(self.lib.prmf_get_normX_sq(self.h, ctypes.byref(out)))
        return out.value

    def set_pathways(self, packed):
        if not isinstance(packed, PackedPathways):
            raise TypeError("expected PackedPathways")
        if packed.n != self.n:
            raise ValueError("pathways were packed for n=%d, engine has n=%d" % (packed.n, self.n))
        self._ck(self.lib.prmf_set_pathways(self.h, packed.P, _ptr(packed.path_ptr), _ptr(packed.support_idx),
                                            _ptr(packed.row_ptr), _ptr(packed.col_local), _ptr(packed.w)))
        self.P = packed.P

    def set_UV(self, U=None, V=None):
        if U is not None:
            U = _f64(U)
            if U.shape != (self.m, self.k):
                raise ValueError("U has shape %s, expected %s" % (U.shape, (self.m, self.k)))
        if V is not None:
            V = _f64(V)
            if V.shape != (self.n, self.k):
                raise ValueError("V has shape %s, expected %s" % (V.shape, (self.n, self.k)))
        self._ck(self.lib.prmf_set_UV(self.h, _ptr(U), _ptr(V)))

    def get_UV(self, want_U=True, want_V=True):
        U = np.empty((self.m, self.k)) if want_U else None
        V = np.empty((self.n, self.k)) if want_V else None
        self._ck(self.lib.prmf_get_UV(self.h, _ptr(U), _ptr(V)))
        return U, V

    def set_active(self, pathway_of_factor):
        a = np.ascontiguousarray(pathway_of_factor, dtype=np.int32)
        if a.shape != (self.k,):
            raise ValueError("need one active pathway per factor")
        self._ck(self.lib.prmf_set_active(self.h, _ptr(a)))

    # -- compute -------------------------------------------------------------------------------------
    def step(self, n_steps, gamma, delta, tradeoff=None):
        """`n_steps` inner updates; returns (parts[n_steps, 8], gamma_next, delta_next)."""
        parts = np.empty((n_steps, _lib.OBJ_STRIDE))
        gd = np.empty(2)
        t = -1.0 if tradeoff is None else float(tradeoff)
        self._ck(self.lib.prmf_step(self.h, int(n_steps), float(gamma), float(delta), t, _ptr(parts), _ptr(gd)))
        return parts, float(gd[0]), float(gd[1])

    def step_async(self, n_steps, gamma, delta, tradeoff=None):
        t = -1.0 if tradeoff is None else float(tradeoff)
        self._ck(self.lib.prmf_step_async(self.h, int(n_steps), float(gamma), float(delta), t))

    def step_collect(self, n_steps):
        parts = np.empty((n_steps, _lib.OBJ_STRIDE))
        gd = np.empty(2)
        self._ck(self.lib.prmf_step_collect(self.h, int(n_steps), _ptr(parts), _ptr(gd)))
        return parts, float(gd[0]), float(gd[1])

    def scores(self):
        """(mass, quad_norm, quad_raw), each k x P, from the current V."""
        mass = np.empty((self.k, self.P)); qn = np.empty((self.k, self.P)); qr = np.empty((self.k, self.P))
        self._ck(self.lib.prmf_scores(self.h, _ptr(mass), _ptr(qn), _ptr(qr)))
        return mass, qn, qr

    def block_end(self, n_steps, want_scores=True, prefetch=True):
        """Collect a block enqueued by `step_async` with one host wait: (parts[n_steps, 8], gamma_next,
        delta_next, tables) where tables is (mass, quad_norm, quad_raw) or None.  `prefetch` lets the GPU start
        the next inner step's X.V pass while the host works on the tables (see prmf_block_end)."""
        parts = np.empty((n_steps, _lib.OBJ_STRIDE))
        gd = np.empty(2)
        tables = None
        if want_scores:
            tables = tuple(np.empty((self.k, self.P)) for _ in range(3))
        self._ck(self.lib.prmf_block_end(self.h, int(n_steps), _ptr(parts), _ptr(gd), 1 if want_scores else 0,
                                         _ptr(tables[0]) if tables else None, _ptr(tables[1]) if tables else None,
                                         _ptr(tables[2]) if tables else None, 1 if prefetch else 0))
        return parts, float(gd[0]), float(gd[1]), tables

    def project(self):
        """X_local . V for the current V (m_local x k): the pass-1 stream on its own (prmf_project)."""
        A = np.empty((self.m, self.k))
        self._ck(self.lib.prmf_project(self.h, _ptr(A)))
        return A

    def project_t(self):
        """X^T . U for the current U (n x k): the pass-2 stream on its own (prmf_project_t)."""
        B = np.empty((self.n, self.k))
        self._ck(self.lib.prmf_project_t(self.h, _ptr(B)))
        return B

    def nnls(self, B, transpose, maxiter=None):
        """scipy.optimize.nnls(op(X), B[:, c]) for every column c at once (prmf_nnls_x), op(X) = X^T when `transpose`
        (B: n x k, x: m x k) and X otherwise (B: m x k, x: n x k).  Returns (x, rnorm[k], status[k]) with status 1
        converged, -1 iteration limit, -2 passive-set capacity, -3 loss of positive definiteness, and iters[k], the
        iterations of each problem as scipy counts them.  U and V of the engine are unset afterwards: steps and
        projections raise until `set_UV` gives them again."""
        rows, cols = (self.n, self.m) if transpose else (self.m, self.n)
        B = _f64(B)
        if B.shape != (rows, self.k):
            raise ValueError("B has shape %s, expected %s" % (B.shape, (rows, self.k)))
        x = np.empty((cols, self.k))
        rnorm = np.empty(self.k)
        status = np.empty(self.k, dtype=np.int32)
        iters = np.empty(self.k, dtype=np.int32)
        self._ck(self.lib.prmf_nnls_x(self.h, 1 if transpose else 0, _ptr(B), int(maxiter or 0), _ptr(x), _ptr(rnorm),
                                      _ptr(status), _ptr(iters)))
        return x, rnorm, status, iters

    @property
    def last_error(self):
        msg = self.lib.prmf_last_error(self.h)
        return msg.decode() if msg else ""

    def snapshot_best(self):
        self._ck(self.lib.prmf_snapshot_best(self.h))

    def restore_best(self):
        self._ck(self.lib.prmf_restore_best(self.h))

    def residual_sq(self):
        out = ctypes.c_double()
        self._ck(self.lib.prmf_residual_sq(self.h, ctypes.byref(out)))
        return out.value

    def objective(self, gamma, delta):
        """Objective parts of the current state (explicit residual pass); a row like `step`'s."""
        out = np.empty(_lib.OBJ_STRIDE)
        self._ck(self.lib.prmf_objective(self.h, float(gamma), float(delta), _ptr(out)))
        return out

    # -- multi-GPU -----------------------------------------------------------------------------------
    def attach_comm(self, rank, nranks, unique_id):
        buf = (ctypes.c_uint8 * _lib.UNIQUE_ID_BYTES).from_buffer_copy(bytes(unique_id))
        self._ck(self.lib.prmf_comm_init(self.h, int(rank), int(nranks), buf))

    def p2p_export(self):
        buf = (ctypes.c_uint8 * _lib.IPC_HANDLE_BYTES)()
        self._ck(self.lib.prmf_p2p_export(self.h, buf))
        return bytes(buf)

    def p2p_attach(self, rank, nranks, handles):
        """handles: list of every rank's `p2p_export()` bytes, in rank order."""
        blob = b"".join(handles)
        buf = (ctypes.c_uint8 * len(blob)).from_buffer_copy(blob)
        self._ck(self.lib.prmf_p2p_attach(self.h, int(rank), int(nranks), buf))

    def p2p_finalize(self):
        """Collective: agree on the in-kernel exchange (call after `p2p_attach` succeeded on every rank)."""
        self._ck(self.lib.prmf_p2p_finalize(self.h))

    @property
    def exchange_mode(self):
        """"none" | "nccl" | "p2p-v-update" | "p2p-pass2" | "p2p-push-block": how the per-step sum over ranks is done."""
        return ("none", "nccl", "p2p-v-update", "p2p-pass2", "p2p-push-block")[int(self.lib.prmf_exchange_mode(self.h))]

    # -- introspection -------------------------------------------------------------------------------
    @property
    def launch_count(self):
        return int(self.lib.prmf_launch_count(self.h))

    def set_profiling(self, on):
        self._ck(self.lib.prmf_set_profiling(self.h, 1 if on else 0))

    def kernel_times(self, reset=True):
        """{phase: (total_ms, count)} for the phases of the inner step timed in profiling mode."""
        ms = (ctypes.c_double * _lib.N_PHASES)()
        n = (ctypes.c_int64 * _lib.N_PHASES)()
        self._ck(self.lib.prmf_kernel_times(self.h, 1 if reset else 0, ms, n))
        return {name: (float(ms[i]), int(n[i])) for i, name in enumerate(_lib.PHASES)}

    def inject_fault(self, kind):
        """Testing aid (prmf_debug_inject_fault): make the next persistent step launch wait for something that never comes."""
        self._ck(self.lib.prmf_debug_inject_fault(self.h, int(kind)))

    @property
    def stream(self):
        return self.lib.prmf_stream(self.h)


def _device_identity(eng):
    """Something that is equal exactly for ranks whose engines sit on the same physical GPU."""
    try:
        import torch
        return str(torch.cuda.get_device_properties(eng.device).uuid)
    except Exception:
        import os
        return "%s:%d" % (os.environ.get("CUDA_VISIBLE_DEVICES", ""), eng.device)


def nccl_unique_id():
    """128-byte NCCL unique id (rank 0 creates it and ships it to the other ranks)."""
    lib = _lib.load()
    nccl_load()
    buf = (ctypes.c_uint8 * _lib.UNIQUE_ID_BYTES)()
    rc = lib.prmf_comm_unique_id(buf)
    if rc != 0:
        raise _lib.PrmfLibraryError("prmf_comm_unique_id failed: %s" % lib.prmf_last_error(None).decode())
    return bytes(buf)


def nccl_load():
    """Bind the library to the NCCL instance torch already loaded (torch bundles libnccl.so.2)."""
    import glob
    import os
    lib = _lib.load()
    path = None
    try:
        import nvidia.nccl
        cands = glob.glob(os.path.join(os.path.dirname(nvidia.nccl.__path__[0] + "/"), "lib", "libnccl.so*"))
        if cands:
            path = cands[0]
    except Exception:
        pass
    rc = lib.prmf_nccl_load(path.encode() if path else None)
    if rc != 0:
        raise _lib.PrmfLibraryError("prmf_nccl_load failed: %s" % lib.prmf_last_error(None).decode())


def attach_collectives(eng, ctx, p2p=None):
    """Give the engine of a multi-rank run its communicators: NCCL (set-up reductions, and the per-step all-reduce of
    configurations that cannot use peer memory) and -- unless PRMF_P2P=0 -- the NVLink / CUDA-IPC peer buffers through
    which the per-step sum over ranks runs inside the kernels (pushed inside the persistent step kernel for k <= 10,
    pulled inside the V update otherwise).  Ranks that share one device, or PRMF_NCCL=0, skip NCCL altogether.
    Collective over `ctx`: call on every rank."""
    import os
    if ctx.world <= 1:
        return eng
    # NCCL refuses two ranks on one device; ranks that share a GPU (a one-GPU test box) -- or PRMF_NCCL=0 -- run on the
    # peer buffers alone: the per-step exchange lives in the persistent step kernel anyway, and the few set-up scalars
    # are summed through the same buffers (the library reports what it cannot do without a communicator)
    devices = ctx.all_gather_bytes(_device_identity(eng).encode())
    use_nccl = os.environ.get("PRMF_NCCL", "1") != "0" and len(set(devices)) == len(devices)
    if use_nccl:
        nccl_load()
        uid = ctx.broadcast_bytes(nccl_unique_id() if ctx.rank == 0 else None, src=0)
        eng.attach_comm(ctx.rank, ctx.world, uid)
    if p2p is None:
        p2p = os.environ.get("PRMF_P2P", "1") != "0"
    if not use_nccl and not (p2p and ctx.world <= 8):
        raise _lib.PrmfLibraryError("ranks share a device (or PRMF_NCCL=0): the run needs the peer-memory exchange (PRMF_P2P)")
    if p2p and ctx.world <= 8:
        handles = ctx.all_gather_bytes(eng.p2p_export())
        ok = True
        try:
            eng.p2p_attach(ctx.rank, ctx.world, handles)
        except _lib.PrmfLibraryError:
            ok = False
        # all ranks must agree, otherwise some would wait on flags nobody writes
        flags = ctx.all_gather_bytes(b"1" if ok else b"0")
        if not all(f == b"1" for f in flags):
            raise _lib.PrmfLibraryError("NVLink peer exchange could not be set up on every rank; "
                                        "rerun with PRMF_P2P=0 to use the NCCL all-reduce")
        eng.p2p_finalize()
    return eng
