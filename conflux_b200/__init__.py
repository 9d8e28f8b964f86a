"""conflux_b200 -- B200-native (sm_100a) implementation of CONFLUX's LU hot path.

Python mirror of the reference's driver-facing interface for this path (same names, argument meaning and
error behaviour; reference file:line relative to eth-cscs/conflux):

    lu_params(M, N, v[, Px, Py, Pz], comm)   src/conflux/lu/lu_params.hpp:401-409   sizes, grid, InitMatrix, data
    LU_rep(params, C, permutation) -> ms      src/conflux/lu/conflux_opt.hpp:343-346 the factorisation
    LU_solve(params, B_local) -> (X, ms)      (no counterpart in the reference) A X = B with those factors

All arithmetic happens in libconflux_b200.so (hand-written CUDA, include/conflux_b200.h is the C ABI);
this package is a thin ctypes host layer and never falls back to a CPU path.
"""
import ctypes

import numpy as np

from ._lib import ConfluxError, LIB_PATH, SYMBOLS, check, lib

__all__ = ["pinned_empty", "pinned_free", "Comm", "lu_params", "LU_rep", "LU_solve", "residual", "validate", "timeline", "auto_grid", "lu_dims", "init_matrix_host", "ConfluxError", "dbg", "cholesky", "chol_dims", "chol_auto_grid"]


def auto_grid(M, N, P):
    """lu_params::get_p_grid (lu_params.hpp:21-47)."""
    px, py, pz = ctypes.c_int(), ctypes.c_int(), ctypes.c_int()
    check(lib().cflx_auto_grid(int(M), int(N), int(P), ctypes.byref(px), ctypes.byref(py), ctypes.byref(pz)), "auto_grid")
    return px.value, py.value, pz.value


def lu_dims(M, N, v, Px, Py, Pz):
    """Padded sizes exactly as lu_params::initialize (lu_params.hpp:67-82)."""
    o = (ctypes.c_int * 8)()
    check(lib().cflx_lu_dims(int(M), int(N), int(v), int(Px), int(Py), int(Pz), o), "lu_dims")
    return dict(M=o[0], N=o[1], Ml=o[2], Nl=o[3], Nt=o[4], nlayr=o[5], Mt=o[6], P=o[7])


def init_matrix_host(M, N, v, Px, Py, Pz, rank, seed=42, out=None):
    """lu_params::InitMatrix, random branch (lu_params.hpp:364-375) for one rank."""
    d = lu_dims(M, N, v, Px, Py, Pz)
    if out is None:
        out = np.empty((d["Ml"], d["Nl"]), dtype=np.float64)
    check(lib().cflx_init_matrix_host(int(M), int(N), int(v), int(Px), int(Py), int(Pz), int(rank), int(seed),
                                      out.ctypes.data), "init_matrix_host")
    return out


def pinned_empty(shape, dtype=np.float64):
    """numpy array backed by page-locked host memory (cudaHostAlloc) -- staging for LU_rep's host->device copy."""
    n = int(np.prod(shape)) * np.dtype(dtype).itemsize
    p = ctypes.c_void_p()
    check(lib().cflx_host_alloc(n, ctypes.byref(p)), "host_alloc")
    buf = (ctypes.c_char * n).from_address(p.value)
    arr = np.frombuffer(buf, dtype=dtype).reshape(shape)
    _PINNED[arr.ctypes.data] = p
    return arr


_PINNED = {}


def pinned_free(arr):
    p = _PINNED.pop(arr.ctypes.data, None)
    if p is not None:
        lib().cflx_host_free(p)


class Comm:
    """Process-grid handle: the MPI_Comm of the reference.  One per rank (= per GPU)."""

    def __init__(self, world_size=1, rank=0, unique_id=None, device=0):
        self.world_size, self.rank, self.device = int(world_size), int(rank), int(device)
        self._h = ctypes.c_void_p()
        idbuf = None
        if unique_id is not None:
            idbuf = ctypes.create_string_buffer(bytes(unique_id), 128)
        check(lib().cflx_comm_create(self.world_size, self.rank, idbuf, self.device, ctypes.byref(self._h)), "comm_create")

    @staticmethod
    def unique_id():
        buf = ctypes.create_string_buffer(128)
        check(lib().cflx_get_unique_id(buf), "get_unique_id")
        return bytes(buf.raw)

    @classmethod
    def from_torch_distributed(cls, device=None):
        """Bootstrap over an initialised torch.distributed group (plumbing only): rank 0's NCCL id is broadcast."""
        import torch
        import torch.distributed as dist
        if not dist.is_initialized() or dist.get_world_size() == 1:
            return cls(1, 0, None, 0 if device is None else device)
        rank, world = dist.get_rank(), dist.get_world_size()
        obj = [cls.unique_id() if rank == 0 else None]
        dist.broadcast_object_list(obj, src=0)
        if device is None:
            device = rank % max(1, torch.cuda.device_count())
        return cls(world, rank, obj[0], device)

    def barrier(self):
        check(lib().cflx_comm_barrier(self._h), "comm_barrier")

    def close(self):
        if self._h:
            lib().cflx_comm_destroy(self._h)
            self._h = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class lu_params:
    """Mirror of conflux::lu_params<double> (lu_params.hpp:8-459): public fields M, N, P, Ml, Nl, Px, Py, Pz, v,
    nlayr, Mt, Nt, pi, pj, pk, rank, seed, data (Ml x Nl numpy array owned by the object), InitMatrix(),
    free_comms().  `comm` is a conflux_b200.Comm instead of an MPI_Comm."""

    def __init__(self, M, N, v, *grid_and_comm):
        if len(grid_and_comm) == 1:
            (comm,) = grid_and_comm
            Px = Py = Pz = -1
        elif len(grid_and_comm) == 4:
            Px, Py, Pz, comm = grid_and_comm
        else:
            raise TypeError("lu_params(M, N, v, comm) or lu_params(M, N, v, Px, Py, Pz, comm)")
        self.lu_comm = comm
        self.seed = 42
        self._h = ctypes.c_void_p()
        check(lib().cflx_lu_create(comm._h, int(M), int(N), int(v), int(Px), int(Py), int(Pz), ctypes.byref(self._h)),
              "lu_create")
        info = (ctypes.c_int * 16)()
        check(lib().cflx_lu_info(self._h, info), "lu_info")
        (self.M, self.N, self.Ml, self.Nl, self.Nt, self.nlayr, self.P, self.Px, self.Py, self.Pz, self.pi, self.pj,
         self.pk, self.rank, self.v) = list(info)[:15]
        self.Mt = self.M // self.v
        self.tA11x, self.tA11y = self.Ml // self.v, self.Nl // self.v
        self.use_collectives = self.v > 1024
        self.data = np.zeros((self.Ml, self.Nl), dtype=np.float64)
        self.InitMatrix()

    def InitMatrix(self):
        init_matrix_host(self.M, self.N, self.v, self.Px, self.Py, self.Pz, self.rank, self.seed, out=self.data)

    def free_comms(self):
        if self._h:
            lib().cflx_lu_destroy(self._h)
            self._h = ctypes.c_void_p()

    def __del__(self):
        try:
            self.free_comms()
        except Exception:
            pass


def LU_rep(gv, C=None, permutation=None, upload=True, next_data=None):
    """conflux::LU_rep<double>(gv, C, permutation) (conflux_opt.hpp:343-346): collective over gv.lu_comm, does not
    modify gv.data, fills C (Ml x Nl, L\\U of PA in the conflux layout, layer 0) and permutation (M ints) when they
    are given, returns the time of the main loop in ms (device-timed).

    upload=True copies gv.data to the device first; upload=False factors the input that is already there (the previous
    one, or the matrix a previous call streamed in through next_data).  next_data (page-locked array of gv.data's shape):
    the input of the NEXT factorisation, uploaded on a copy stream while this one runs (cflx_lu_queue_next_local)."""
    if upload:
        a = np.ascontiguousarray(gv.data, dtype=np.float64)
        check(lib().cflx_lu_set_local(gv._h, a.ctypes.data), "lu_set_local")
    if next_data is not None:
        assert next_data.dtype == np.float64 and next_data.flags.c_contiguous and next_data.size == gv.Ml * gv.Nl
        check(lib().cflx_lu_queue_next_local(gv._h, next_data.ctypes.data), "lu_queue_next_local")
    ms = ctypes.c_double()
    check(lib().cflx_lu_factor(gv._h, ctypes.byref(ms)), "lu_factor")
    if C is not None:
        assert C.dtype == np.float64 and C.flags.c_contiguous and C.size >= gv.Ml * gv.Nl
        if permutation is None:
            permutation = np.empty(gv.M, dtype=np.int32)
        check(lib().cflx_lu_get_factors(gv._h, C.ctypes.data, permutation.ctypes.data), "lu_get_factors")
    elif permutation is not None:
        assert permutation.dtype == np.int32 and permutation.size >= gv.M
        check(lib().cflx_lu_get_permutation(gv._h, permutation.ctypes.data), "lu_get_permutation")
    return ms.value


def LU_solve(gv, B_local, nrhs=None):
    """Solves A X = B with the factors of the last LU_rep (P A = L U, A the padded M x M matrix).  COLLECTIVE over
    gv.lu_comm, with the same number of right-hand sides on every rank.

    B_local: this rank's rows of B in A's row distribution, (Ml, nrhs) float64 C-contiguous (or (Ml,) for one
    right-hand side): global row g on grid row (g // v) % Px at local row (g // (v*Px))*v + g % v.  It is read on the
    ranks with pj == 0 and pk == 0; elsewhere it may be None, and then nrhs must be given.
    Returns (X_local, ms): X_local (Nl, nrhs) (or (Nl,)) holds X in A's column distribution -- global row g on every rank
    with pj == (g // v) % Py at local row (g // (v*Py))*v + g % v -- and ms is the device time of the solve proper."""
    vector = False
    if B_local is not None:
        assert B_local.dtype == np.float64 and B_local.flags.c_contiguous and B_local.ndim in (1, 2) \
            and B_local.shape[0] == gv.Ml
        vector = B_local.ndim == 1
        n = 1 if vector else B_local.shape[1]
        assert nrhs is None or nrhs == n
        nrhs = n
    if nrhs is None or nrhs < 1:
        raise ValueError("LU_solve: nrhs >= 1 is needed when B_local is None")
    X = np.empty((gv.Nl,) if vector else (gv.Nl, int(nrhs)), dtype=np.float64)
    ms = ctypes.c_double()
    check(lib().cflx_lu_solve(gv._h, int(nrhs), B_local.ctypes.data if B_local is not None else None, X.ctypes.data,
                              ctypes.byref(ms)), "lu_solve")
    return X, ms.value


def timeline(gv):
    """Per-region device time of the last LU_rep run under cflx_lu_set_profiling(gv._h, 1 or 2): dict(main={region: (ms,
    count)}, side={...}); region names are the reference's semiprof regions."""
    import json
    n = lib().cflx_lu_timeline(gv._h, None, 0)
    buf = ctypes.create_string_buffer(max(n, 2))
    check(lib().cflx_lu_timeline(gv._h, buf, n), "lu_timeline")
    return json.loads(buf.value.decode())


def validate(gv):
    """The reference's validation (examples/conflux_miniapp.cpp:349-500) of the last LU_rep on the GPU grid.
    COLLECTIVE over gv.lu_comm.  Returns (||PA - LU||_F, ||PA - LU||_F / ||A||_F), identical on every rank."""
    a, r = ctypes.c_double(), ctypes.c_double()
    check(lib().cflx_lu_validate(gv._h, ctypes.byref(a), ctypes.byref(r)), "lu_validate")
    return a.value, r.value


def residual(gv):
    """||PA - LU||_F / ||A||_F of the last LU_rep, computed on the GPU grid (collective)."""
    return validate(gv)[1]


class cholesky:
    """Mirror of the reference's CONFCHOX driver interface (src/conflux/cholesky/Cholesky.h:20-22):
        initialize(N, v, grid, comm) -> object;  obj.parallelCholesky() -> ms;  obj.finalize().
    grid = (0, 0, 0) and v = 0 select the reference's automatic choices (Cholesky.cpp:75-134).  `data` is this rank's share
    of the input (Ml x Nl, conflux tile layout), filled by the reference's generator (CholeskyIO.cpp:100-172)."""

    def __init__(self, N, v, grid, comm):
        self.comm = comm
        self._h = ctypes.c_void_p()
        g = tuple(int(x) for x in grid)
        check(lib().cflx_chol_create(comm._h, int(N), int(v), g[0], g[1], g[2], ctypes.byref(self._h)), "chol_create")
        info = (ctypes.c_int * 16)()
        check(lib().cflx_chol_info(self._h, info), "chol_info")
        (self.N, self.v, self.Kappa, self.Ml, self.Nl, self.l, self.P, self.PX, self.PY, self.PZ, self.px, self.py, self.pz,
         self.rank) = list(info)[:14]
        self.data = np.zeros((self.Ml, self.Nl))
        self.generateInputMatrixDistributed()

    @classmethod
    def initialize(cls, N, v, grid, comm):
        return cls(N, v, grid, comm)

    def generateInputMatrixDistributed(self):
        check(lib().cflx_chol_init_matrix_host(self.N, self.v, self.PX, self.PY, self.PZ, self.rank, self.data.ctypes.data),
              "chol_init_matrix_host")

    def parallelCholesky(self, upload=True):
        if upload:
            a = np.ascontiguousarray(self.data, dtype=np.float64)
            check(lib().cflx_chol_set_local(self._h, a.ctypes.data), "chol_set_local")
        ms = ctypes.c_double()
        check(lib().cflx_chol_factor(self._h, ctypes.byref(ms)), "chol_factor")
        return ms.value

    def local_factor(self):
        L = np.empty((self.Ml, self.Nl))
        check(lib().cflx_chol_get_local(self._h, L.ctypes.data), "chol_get_local")
        return L

    def validate(self):
        a, r = ctypes.c_double(), ctypes.c_double()
        check(lib().cflx_chol_validate(self._h, ctypes.byref(a), ctypes.byref(r)), "chol_validate")
        return a.value, r.value

    def finalize(self, clean=True):
        if self._h:
            lib().cflx_chol_destroy(self._h)
            self._h = ctypes.c_void_p()

    def __del__(self):
        try:
            self.finalize()
        except Exception:
            pass


def chol_dims(N, v, Px, Py, Pz):
    o = (ctypes.c_int * 6)()
    check(lib().cflx_chol_dims(int(N), int(v), int(Px), int(Py), int(Pz), o), "chol_dims")
    return dict(N=o[0], Kappa=o[1], Ml=o[2], Nl=o[3], l=o[4], P=o[5])


def chol_auto_grid(P, N):
    g = (ctypes.c_int * 3)()
    check(lib().cflx_chol_auto_grid(int(P), int(N), g), "chol_auto_grid")
    return tuple(g)


class dbg:
    """Single-kernel hooks (tests and micro-benchmarks)."""

    @staticmethod
    def gemm_tn(AT, B, C=None, alpha=1.0, beta=0.0, reps=1):
        AT = np.ascontiguousarray(AT, dtype=np.float64)
        B = np.ascontiguousarray(B, dtype=np.float64)
        K, M = AT.shape
        N = B.shape[1]
        D = np.empty((M, N))
        ms = ctypes.c_double()
        Cp = None
        if C is not None:
            C = np.ascontiguousarray(C, dtype=np.float64)
            Cp = C.ctypes.data
        check(lib().cflx_dbg_gemm_tn(M, N, K, AT.ctypes.data, B.ctypes.data, Cp, float(alpha), float(beta), D.ctypes.data,
                                     int(reps), ctypes.byref(ms)), "dbg_gemm_tn")
        return D, ms.value

    @staticmethod
    def panel(P, reps=1):
        P = np.ascontiguousarray(P, dtype=np.float64)
        n, v = P.shape
        perm = np.zeros(v, dtype=np.int32)
        A00 = np.zeros((v, v))
        LU = np.zeros((max(n, 1), v))
        ms = ctypes.c_double()
        check(lib().cflx_dbg_panel(n, v, P.ctypes.data, perm.ctypes.data, A00.ctypes.data, LU.ctypes.data, int(reps),
                                   ctypes.byref(ms)), "dbg_panel")
        return perm, A00, LU[:n], ms.value

    @staticmethod
    def trsm(A00, B=None, R=None):
        A00 = np.ascontiguousarray(A00, dtype=np.float64)
        v = A00.shape[0]
        X = Y = None
        n = B.shape[0] if B is not None else R.shape[1]
        if B is not None:
            B = np.ascontiguousarray(B, dtype=np.float64)
            X = np.empty_like(B)
        if R is not None:
            R = np.ascontiguousarray(R, dtype=np.float64)
            Y = np.empty_like(R)
        check(lib().cflx_dbg_trsm(n, v, A00.ctypes.data, B.ctypes.data if B is not None else None,
                                  X.ctypes.data if X is not None else None, R.ctypes.data if R is not None else None,
                                  Y.ctypes.data if Y is not None else None), "dbg_trsm")
        return X, Y

    @staticmethod
    def trsm_left_upper(A00, R):
        """X = U^-1 R with U = upper(A00) (v x v) and R (v x n): the diagonal-tile solve of LU_solve."""
        A00 = np.ascontiguousarray(A00, dtype=np.float64)
        R = np.ascontiguousarray(R, dtype=np.float64)
        v, n = R.shape
        X = np.empty_like(R)
        check(lib().cflx_dbg_trsm_left_upper(v, n, A00.ctypes.data, R.ctypes.data, X.ctypes.data), "dbg_trsm_left_upper")
        return X

    @staticmethod
    def potrf_tile(A, blocked=False):
        """Cholesky of one v x v tile (lower triangle of A referenced) by the factorisation's own tile kernels: the
        one-CTA kernel (blocked=False) or the 128-wide blocked path (blocked=True, v in 256/384/512).
        Returns (L, LT, info) with info = dpotrf's (1-based column of the first non-positive pivot, 0 = success)."""
        A = np.ascontiguousarray(A, dtype=np.float64)
        v = A.shape[0]
        L, LT, info = np.empty((v, v)), np.empty((v, v)), ctypes.c_int()
        check(lib().cflx_dbg_potrf_tile(v, int(bool(blocked)), A.ctypes.data, L.ctypes.data, LT.ctypes.data,
                                        ctypes.byref(info)), "dbg_potrf_tile")
        return L, LT, info.value

    @staticmethod
    def ozaki_gemm(AT, B, C=None, reps=1, want_planes=False):
        """D = C - AT^T @ B on the int8 tcgen05 path.  Returns dict(D, ms, split_ms[, pa, pb, ea, eb])."""
        AT = np.ascontiguousarray(AT, dtype=np.float64)
        B = np.ascontiguousarray(B, dtype=np.float64)
        K, M = AT.shape
        N = B.shape[1]
        D = np.empty((M, N))
        Cp = np.ascontiguousarray(C, dtype=np.float64) if C is not None else None
        pa = np.zeros((8, M, K), dtype=np.int8) if want_planes else None
        pb = np.zeros((8, N, K), dtype=np.int8) if want_planes else None
        ea = np.zeros(M, dtype=np.int32) if want_planes else None
        eb = np.zeros(N, dtype=np.int32) if want_planes else None
        ms, sms = ctypes.c_double(), ctypes.c_double()
        ptr = lambda a: a.ctypes.data if a is not None else None
        check(lib().cflx_dbg_ozaki_gemm(M, N, K, AT.ctypes.data, B.ctypes.data, ptr(Cp), D.ctypes.data, ptr(pa), ptr(pb), ptr(ea),
                                        ptr(eb), int(reps), ctypes.byref(ms), ctypes.byref(sms)), "dbg_ozaki_gemm")
        return dict(D=D, ms=ms.value, split_ms=sms.value, pa=pa, pb=pb, ea=ea, eb=eb)

    @staticmethod
    def push_pivots(A, pivot_rows, fnpr):
        """plan_moves + push_phase1..3 + gri update on one rank; returns (A_new, new_row -> old_row, extracted rows)."""
        A = np.array(A, dtype=np.float64, order="C")
        piv = np.ascontiguousarray(pivot_rows, dtype=np.int32)
        gri = np.zeros(A.shape[0], dtype=np.int32)
        a01 = np.zeros((max(1, len(piv)), A.shape[1]))
        check(lib().cflx_dbg_push_pivots(A.shape[0], A.shape[1], A.ctypes.data, len(piv), piv.ctypes.data, int(fnpr),
                                         gri.ctypes.data, a01.ctypes.data), "dbg_push_pivots")
        return A, gri, a01[:len(piv)]

    @staticmethod
    def umma_peak(which, n):
        """tera-MACs/s of back-to-back tcgen05.mma 128 x n x 32B-K: which 0 = kind::i8, 1 = kind::f16 (bf16)."""
        t = ctypes.c_double()
        check(lib().cflx_dbg_umma_peak(int(which), int(n), ctypes.byref(t)), "dbg_umma_peak")
        return t.value

    @staticmethod
    def fp64_peak_ex(which):
        """(burst, sustained) TFLOP/s of the DMMA (0) / DFMA (1) pipe."""
        a, b = ctypes.c_double(), ctypes.c_double()
        check(lib().cflx_dbg_fp64_peak_ex(int(which), ctypes.byref(a), ctypes.byref(b)), "dbg_fp64_peak_ex")
        return a.value, b.value

    @staticmethod
    def fp64_peak(which):
        tf = ctypes.c_double()
        check(lib().cflx_dbg_fp64_peak(int(which), ctypes.byref(tf)), "dbg_fp64_peak")
        return tf.value
