"""parmgmc_b200 -- B200-native sampling hot path of ParMGMC behind the reference's plugin surface.

This package is a thin ctypes mirror of the C ABI in ``include/parmgmc_b200.h`` (the drop-in
boundary).  All arithmetic runs in hand-written sm_100a kernels inside
``parmgmc_b200/lib/libparmgmc_b200.so``; there is no CPU or PyTorch fallback: if the library is
missing, or no CUDA device is visible, construction fails loudly.

Object model = the reference's (SURVEY.md section 8(b)):

    Context                     ParMGMCInitialize / the global PetscRandom (src/parmgmc.c)
    Mat.from_csr / .laplace     the Mat handed to KSPSetOperators (MatSeqAIJGetCSRAndMemType view,
                                or the DMDA generator src/problems.c:14-75 matrix-free)
    MCSOR                       include/parmgmc/mc_sor.h
    PC("mcgibbs"|"sorgibbs"|"gamgmc"|"cholsampler")   the PC plugins; options use the reference keys
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libparmgmc_b200.so")
HEADER_PATH = os.path.join(os.path.dirname(_HERE), "include", "parmgmc_b200.h")

SOR_FORWARD_SWEEP, SOR_BACKWARD_SWEEP, SOR_SYMMETRIC_SWEEP, SOR_LOCAL_FORWARD_SWEEP = 1, 2, 3, 4
COLORING_GREEDY, COLORING_LEXICOGRAPHIC, COLORING_PARITY = 0, 1, 2
NOISE_PHILOX, NOISE_INJECTED, NOISE_NONE = 0, 1, 2
PCRICHARDSON_CONVERGED_ITS = 4

ERR_NAMES = {1: "ARG", 2: "SUP", 3: "NO_DEVICE", 4: "CUDA", 5: "NOT_SPD", 6: "ORDER", 7: "NOISE", 8: "COLORING", 9: "COMM", 10: "CALLBACK"}


class PMGError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"parmgmc_b200 error {code} ({ERR_NAMES.get(code, '?')}): {msg}")
        self.code = code


SAMPLE_CB = C.CFUNCTYPE(C.c_int, C.c_int64, C.POINTER(C.c_double), C.c_int64, C.c_void_p)
DELETER = C.CFUNCTYPE(C.c_int, C.c_void_p)

_i64p = np.ctypeslib.ndpointer(np.int64, flags="C_CONTIGUOUS")
_i32p = np.ctypeslib.ndpointer(np.int32, flags="C_CONTIGUOUS")
_f64p = np.ctypeslib.ndpointer(np.float64, flags="C_CONTIGUOUS")
_vp = C.c_void_p

# name -> (restype, argtypes).  Kept in one table so tests can check it against the header.
SIGNATURES = {
    "pmg_version": (C.c_char_p, []),
    "pmg_last_error": (C.c_char_p, []),
    "pmg_device_count": (C.c_int, [C.POINTER(C.c_int)]),
    "pmg_ctx_create": (C.c_int, [C.c_int, C.POINTER(_vp)]),
    "pmg_ctx_destroy": (C.c_int, [_vp]),
    "pmg_ctx_set_stream": (C.c_int, [_vp, _vp]),
    "pmg_ctx_synchronize": (C.c_int, [_vp]),
    "pmg_ctx_set_seed": (C.c_int, [_vp, C.c_uint64]),
    "pmg_ctx_get_draw_counter": (C.c_int, [_vp, C.POINTER(C.c_uint64)]),
    "pmg_ctx_set_draw_counter": (C.c_int, [_vp, C.c_uint64]),
    "pmg_comm_unique_id": (C.c_int, [C.c_char_p]),
    "pmg_ctx_comm_init": (C.c_int, [_vp, C.c_int, C.c_int, C.c_char_p]),
    "pmg_ctx_comm_rank": (C.c_int, [_vp, C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "pmg_ctx_comm_p2p": (C.c_int, [_vp, C.POINTER(C.c_int)]),
    "pmg_mat_create_csr": (C.c_int, [_vp, C.c_int64, _i64p, _i32p, _f64p, C.POINTER(_vp)]),
    "pmg_mat_create_laplace": (C.c_int, [_vp, C.c_int, C.c_int64, C.c_int64, C.c_int64, C.c_double, C.c_int64, C.c_int64, C.POINTER(_vp)]),
    "pmg_mat_create_lrc": (C.c_int, [_vp, C.c_int, _f64p, _f64p, C.POINTER(_vp)]),
    "pmg_plan_sweep3d": (C.c_int, [C.c_int64, C.c_int64, C.c_int64, C.c_int64, C.c_int64, C.c_int, C.c_int, C.c_void_p, C.c_int64, C.POINTER(C.c_int64)]),
    "pmg_plan_sweep2d": (C.c_int, [C.c_int64, C.c_int64, C.c_int64, C.c_int64, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int64, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    "pmg_pc_set_qoi": (C.c_int, [_vp, C.c_void_p, C.c_int64, C.c_int]),
    "pmg_pc_get_qoi": (C.c_int, [_vp, C.c_void_p, C.POINTER(C.c_int64), C.c_int]),
    "pmg_pc_get_mean_var": (C.c_int, [_vp, C.c_void_p, C.c_void_p, C.POINTER(C.c_int64)]),
    "pmg_autocorrelation": (C.c_int, [_vp, C.c_int64, _f64p, _f64p]),
    "pmg_iact": (C.c_int, [_vp, C.c_int64, _f64p, C.POINTER(C.c_double), C.c_void_p, C.POINTER(C.c_int)]),
    "pmg_mat_create_csr_dist": (C.c_int, [_vp, C.c_int64, C.c_int64, C.c_int64, _i64p, _i64p, _f64p, C.POINTER(_vp)]),
    "pmg_mat_destroy": (C.c_int, [_vp]),
    "pmg_mat_get_size": (C.c_int, [_vp, C.POINTER(C.c_int64), C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    "pmg_mat_set_coloring": (C.c_int, [_vp, C.c_int, _i32p]),
    "pmg_mat_set_coloring_auto": (C.c_int, [_vp, C.c_int]),
    "pmg_mat_get_coloring": (C.c_int, [_vp, C.POINTER(C.c_int), _vp]),
    "pmg_mat_mult": (C.c_int, [_vp, _f64p, _f64p]),
    "pmg_mcsor_create": (C.c_int, [_vp, C.POINTER(_vp)]),
    "pmg_mcsor_destroy": (C.c_int, [_vp]),
    "pmg_mcsor_set_omega": (C.c_int, [_vp, C.c_double]),
    "pmg_mcsor_set_sweep_type": (C.c_int, [_vp, C.c_int]),
    "pmg_mcsor_get_sweep_type": (C.c_int, [_vp, C.POINTER(C.c_int)]),
    "pmg_mcsor_get_num_colors": (C.c_int, [_vp, C.POINTER(C.c_int)]),
    "pmg_mcsor_apply": (C.c_int, [_vp, _f64p, _f64p]),
    "pmg_mcsor_apply_dev": (C.c_int, [_vp, _vp, _vp]),
    "pmg_pc_create": (C.c_int, [_vp, C.c_char_p, C.POINTER(_vp)]),
    "pmg_pc_destroy": (C.c_int, [_vp]),
    "pmg_pc_reset": (C.c_int, [_vp]),
    "pmg_pc_set_operator": (C.c_int, [_vp, _vp]),
    "pmg_pc_set_option": (C.c_int, [_vp, C.c_char_p, C.c_char_p]),
    "pmg_pc_setup": (C.c_int, [_vp]),
    "pmg_pc_view": (C.c_int, [_vp, C.c_char_p, C.c_size_t]),
    "pmg_pc_apply_richardson": (C.c_int, [_vp, _vp, _f64p, C.c_int64, C.c_int, C.POINTER(C.c_int64), C.POINTER(C.c_int)]),
    "pmg_pc_apply_richardson_dev": (C.c_int, [_vp, _vp, _vp, C.c_int64, C.c_int, C.POINTER(C.c_int64), C.POINTER(C.c_int)]),
    "pmg_pc_apply": (C.c_int, [_vp, _f64p, _f64p]),
    "pmg_pc_set_sample_callback": (C.c_int, [_vp, SAMPLE_CB, _vp, DELETER]),
    "pmg_pc_mcgibbs_set_omega": (C.c_int, [_vp, C.c_double]),
    "pmg_pc_mcgibbs_set_sweep_type": (C.c_int, [_vp, C.c_int]),
    "pmg_pc_gamgmc_set_levels": (C.c_int, [_vp, C.c_int]),
    "pmg_pc_gamgmc_get_levels": (C.c_int, [_vp, C.POINTER(C.c_int)]),
    "pmg_pc_gamgmc_set_interpolation": (C.c_int, [_vp, C.c_int, C.c_int64, C.c_int64, _i64p, _i32p, _f64p]),
    "pmg_pc_gamgmc_get_level_info": (C.c_int, [_vp, C.c_int, C.POINTER(C.c_int64), C.POINTER(C.c_int64), C.POINTER(C.c_int)]),
    "pmg_pc_gamgmc_get_level_csr": (C.c_int, [_vp, C.c_int, _i64p, _i32p, _f64p]),
    "pmg_pc_set_noise_mode": (C.c_int, [_vp, C.c_int]),
    "pmg_pc_set_noise_tape": (C.c_int, [_vp, _f64p, C.c_int64]),
    "pmg_pc_noise_per_sample": (C.c_int, [_vp, C.POINTER(C.c_int64)]),
    "pmg_normal_fill": (C.c_int, [_vp, C.c_uint64, C.c_uint64, C.c_int64, C.c_int64, _f64p]),
    "pmg_pc_last_stats": (C.c_int, [_vp, C.POINTER(C.c_double), C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    "pmg_pc_profile": (C.c_int, [_vp, C.c_char_p, C.c_size_t, C.c_int]),
}

_lib = None


def _preload_nccl():
    """The library links libnccl.so.2.  When PyTorch is (or will be) in the same process its bundled,
    newer NCCL must be the one that gets loaded, otherwise `import torch` fails afterwards on missing
    symbols; a plain C host program just uses the system NCCL."""
    import importlib.util
    try:
        spec = importlib.util.find_spec("nvidia.nccl")
    except (ImportError, ValueError):
        spec = None
    if spec and spec.submodule_search_locations:
        for d in spec.submodule_search_locations:
            cand = os.path.join(d, "lib", "libnccl.so.2")
            if os.path.exists(cand):
                C.CDLL(cand, mode=C.RTLD_GLOBAL)
                return


def lib():
    """Load the CUDA extension.  No fallback: a missing library is an error."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                              "(nvcc, sm_100a). parmgmc_b200 has no CPU fallback.")
        _preload_nccl()
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)  # AttributeError if the library does not export what the header declares
            fn.restype, fn.argtypes = res, args
        _lib = L
    return _lib


def _check(rc):
    if rc:
        raise PMGError(rc, lib().pmg_last_error().decode())


def device_count() -> int:
    n = C.c_int()
    _check(lib().pmg_device_count(C.byref(n)))
    return n.value


def _f64(a):
    return np.ascontiguousarray(a, np.float64)


def _devptr(t):
    """device pointer of a torch CUDA tensor (float64, contiguous) or a raw int"""
    if t is None:
        return None
    if isinstance(t, int):
        return t
    assert t.is_cuda and t.is_contiguous() and str(t.dtype) == "torch.float64", "need a contiguous float64 CUDA tensor"
    return t.data_ptr()


class Context:
    """One GPU, one stream, one global noise stream (seed + draw counter)."""

    def __init__(self, device: int = 0, stream=None, seed: int | None = None):
        self._h = _vp()
        _check(lib().pmg_ctx_create(device, C.byref(self._h)))
        self.device = device
        if stream is not None:
            _check(lib().pmg_ctx_set_stream(self._h, _vp(stream)))
        if seed is not None:
            self.set_seed(seed)

    def set_seed(self, seed: int):
        _check(lib().pmg_ctx_set_seed(self._h, seed))

    @property
    def draw_counter(self) -> int:
        d = C.c_uint64()
        _check(lib().pmg_ctx_get_draw_counter(self._h, C.byref(d)))
        return d.value

    @draw_counter.setter
    def draw_counter(self, v: int):
        _check(lib().pmg_ctx_set_draw_counter(self._h, v))

    def synchronize(self):
        _check(lib().pmg_ctx_synchronize(self._h))

    def comm_init(self, rank: int, nranks: int, unique_id: bytes):
        _check(lib().pmg_ctx_comm_init(self._h, rank, nranks, unique_id))

    def comm_p2p(self) -> bool:
        """True when the slab halo exchange runs through peer memory (CUDA IPC mailboxes), False when through NCCL."""
        on = C.c_int()
        _check(lib().pmg_ctx_comm_p2p(self._h, C.byref(on)))
        return bool(on.value)

    def normal_fill(self, seed, call, row0, n):
        z = np.empty(n, np.float64)
        _check(lib().pmg_normal_fill(self._h, seed, call, row0, n, z))
        return z

    def close(self):
        if self._h:
            lib().pmg_ctx_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def partition_slabs(n_units: int, nranks: int, align: int = 2):
    """Contiguous slabs [lo, hi) of the slowest grid dimension, one per rank, in rank order: the row-block ownership
    ranges PETSc gives an MPIAIJ matrix (src/mc_sor.c:308-310), with every cut on a multiple of `align` so that coarse
    unit J and fine unit 2J have the same owner on the first coarsenings."""
    if nranks < 1 or n_units < nranks * align:
        raise ValueError(f"cannot split {n_units} units over {nranks} ranks with alignment {align}")
    per = (n_units // nranks) // align * align
    cuts = [r * per for r in range(nranks)] + [n_units]
    return [(cuts[r], cuts[r + 1]) for r in range(nranks)]


def comm_unique_id() -> bytes:
    buf = C.create_string_buffer(128)
    _check(lib().pmg_comm_unique_id(buf))
    return buf.raw


def plan_sweep3d(nx, ny, nz, slab=None, bz=64, nw=16):
    """Work list of the fused 3D sweep as an (items, 5) int32 array: strip, first row, first plane, end plane, narrow flag."""
    slo, shi = slab if slab is not None else (0, nz)
    cnt = C.c_int64()
    _check(lib().pmg_plan_sweep3d(nx, ny, nz, slo, shi, bz, nw, None, 0, C.byref(cnt)))
    out = np.empty((cnt.value, 5), np.int32)
    _check(lib().pmg_plan_sweep3d(nx, ny, nz, slo, shi, bz, nw, out.ctypes.data, cnt.value, C.byref(cnt)))
    return out


def plan_sweep2d(nx, ny, slab=None, by=64, restrict_mode=False, overlap=True):
    """Work list of the fused 2D sweep as ((items, 3) int32 array: strip, first row, end row; number of leading tiles that read no ghost row)."""
    slo, shi = slab if slab is not None else (0, ny)
    cnt, nh = C.c_int64(), C.c_int64()
    _check(lib().pmg_plan_sweep2d(nx, ny, slo, shi, by, int(restrict_mode), int(overlap), None, 0, C.byref(cnt), C.byref(nh)))
    out = np.empty((cnt.value, 3), np.int32)
    _check(lib().pmg_plan_sweep2d(nx, ny, slo, shi, by, int(restrict_mode), int(overlap), out.ctypes.data, cnt.value, C.byref(cnt), C.byref(nh)))
    return out, nh.value


def autocorrelation(ctx: "Context", x):
    """Autocorrelation (src/iact.c:17-46) on the device (cuFFT)."""
    x = _f64(x)
    acf = np.empty(x.size, np.float64)
    _check(lib().pmg_autocorrelation(ctx._h, x.size, x, acf))
    return acf


def iact(ctx: "Context", x):
    """IACT (src/iact.c:48-92): returns (tau, valid)."""
    x = _f64(x)
    tau, valid = C.c_double(), C.c_int()
    _check(lib().pmg_iact(ctx._h, x.size, x, C.byref(tau), None, C.byref(valid)))
    return tau.value, bool(valid.value)


class Mat:
    def __init__(self, ctx: Context, handle):
        self.ctx, self._h = ctx, handle

    @staticmethod
    def from_csr(ctx: Context, rowptr, col, val) -> "Mat":
        rowptr = np.ascontiguousarray(rowptr, np.int64)
        h = _vp()
        _check(lib().pmg_mat_create_csr(ctx._h, rowptr.size - 1, rowptr, np.ascontiguousarray(col, np.int32), _f64(val), C.byref(h)))
        return Mat(ctx, h)

    @staticmethod
    def from_csr_dist(ctx: Context, n_global, row_start, rowptr, col_global, val) -> "Mat":
        """This rank's rows [row_start, row_start + len(rowptr) - 1) with GLOBAL column indices (MPIAIJ-style; collective)."""
        rowptr = np.ascontiguousarray(rowptr, np.int64)
        h = _vp()
        _check(lib().pmg_mat_create_csr_dist(ctx._h, n_global, row_start, rowptr.size - 1, rowptr, np.ascontiguousarray(col_global, np.int64), _f64(val), C.byref(h)))
        return Mat(ctx, h)

    @staticmethod
    def laplace(ctx: Context, dim, nx, ny, nz=1, kappa=1.0, slab=None) -> "Mat":
        """MatAssembleShiftedLaplaceFD (src/problems.c:14-75) without assembling anything."""
        lo, hi = slab if slab is not None else (0, nz if dim == 3 else ny)
        h = _vp()
        _check(lib().pmg_mat_create_laplace(ctx._h, dim, nx, ny, nz, kappa, lo, hi, C.byref(h)))
        return Mat(ctx, h)

    @staticmethod
    def lrc(A: "Mat", B, S) -> "Mat":
        """MatCreateLRC(A, B, S, NULL): A + B diag(S) B^T with B dense n x k (src/mc_sor.c:565-595).  A is borrowed.

        On a distributed A (a slab or row-partitioned operator) the call is collective: B holds this rank's n_local rows and
        S must be bitwise identical on every rank (otherwise every rank raises PMGError).  B^T y is then reduced across ranks in
        rank order, so N GPUs agree with one GPU to rounding (not bitwise); woodbury and a stand-alone cholsampler refuse it."""
        B = np.asarray(B, np.float64)
        S = np.ascontiguousarray(S, np.float64)
        if B.ndim != 2 or B.shape[0] != A.n or B.shape[1] != S.size:
            raise ValueError("B must be n x k and S of length k")
        h = _vp()
        _check(lib().pmg_mat_create_lrc(A._h, int(S.size), np.ascontiguousarray(B.T).ravel(), S, C.byref(h)))  # column-major
        m = Mat(A.ctx, h)
        m._base = A  # keep the borrowed base alive
        return m

    @property
    def size(self):
        a, b, c = C.c_int64(), C.c_int64(), C.c_int64()
        _check(lib().pmg_mat_get_size(self._h, C.byref(a), C.byref(b), C.byref(c)))
        return a.value, b.value, c.value

    @property
    def n(self):
        return self.size[0]

    def set_coloring(self, color, ncolors=None):
        color = np.ascontiguousarray(color, np.int32)
        _check(lib().pmg_mat_set_coloring(self._h, int(color.max()) + 1 if ncolors is None else ncolors, color))

    def set_coloring_auto(self, policy=COLORING_GREEDY):
        _check(lib().pmg_mat_set_coloring_auto(self._h, policy))

    def get_coloring(self):
        k = C.c_int()
        color = np.empty(self.n, np.int32)
        _check(lib().pmg_mat_get_coloring(self._h, C.byref(k), color.ctypes.data))
        return k.value, color

    def mult(self, x):
        y = np.empty(self.n, np.float64)
        _check(lib().pmg_mat_mult(self._h, _f64(x), y))
        return y

    def close(self):
        if self._h:
            lib().pmg_mat_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class MCSOR:
    """include/parmgmc/mc_sor.h: MCSORCreate+SetUp / Apply / SetOmega / SetSweepType / GetNumColors."""

    def __init__(self, mat: Mat):
        self.mat, self._h = mat, _vp()
        _check(lib().pmg_mcsor_create(mat._h, C.byref(self._h)))

    def set_omega(self, omega):
        _check(lib().pmg_mcsor_set_omega(self._h, omega))

    def set_sweep_type(self, t):
        _check(lib().pmg_mcsor_set_sweep_type(self._h, t))

    def get_sweep_type(self):
        t = C.c_int()
        _check(lib().pmg_mcsor_get_sweep_type(self._h, C.byref(t)))
        return t.value

    def get_num_colors(self):
        t = C.c_int()
        _check(lib().pmg_mcsor_get_num_colors(self._h, C.byref(t)))
        return t.value

    def apply(self, b, y):
        """MCSORApply(mc, b, y): in place on the numpy array y."""
        assert y.dtype == np.float64 and y.flags.c_contiguous
        _check(lib().pmg_mcsor_apply(self._h, _f64(b), y))
        return y

    def apply_dev(self, b, y):
        _check(lib().pmg_mcsor_apply_dev(self._h, _devptr(b), _devptr(y)))

    def close(self):
        if self._h:
            lib().pmg_mcsor_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class PC:
    """A sampler with the reference's PC type string and option keys.

    >>> pc = PC(ctx, "gamgmc"); pc.set_operator(A); pc.set_options({"-gamgmc_pc_mg_levels": 9}); pc.setup()
    >>> pc.apply_richardson(b, y, its=100)   # KSPSolve with -ksp_type richardson -ksp_max_it 100
    """

    def __init__(self, ctx: Context, pc_type: str):
        self.ctx, self.type, self._h = ctx, pc_type, _vp()
        _check(lib().pmg_pc_create(ctx._h, pc_type.encode(), C.byref(self._h)))
        self._cb = self._del = None
        self.mat = None

    def set_operator(self, mat: Mat):
        _check(lib().pmg_pc_set_operator(self._h, mat._h))
        self.mat = mat

    def set_option(self, key: str, value=""):
        _check(lib().pmg_pc_set_option(self._h, key.encode(), str(value).encode()))

    def set_options(self, opts: dict):
        for k, v in opts.items():
            self.set_option(k, "" if v is None or v is True else v)

    def setup(self):
        _check(lib().pmg_pc_setup(self._h))

    def reset(self):
        _check(lib().pmg_pc_reset(self._h))

    def view(self) -> str:
        buf = C.create_string_buffer(8192)
        _check(lib().pmg_pc_view(self._h, buf, 8192))
        return buf.value.decode()

    def apply_richardson(self, b, y, its=1, guesszero=False):
        """PCApplyRichardson: `its` samples continuing the chain in the numpy array y (in place)."""
        assert y.dtype == np.float64 and y.flags.c_contiguous
        bb = None if b is None else _f64(b)
        outits, reason = C.c_int64(), C.c_int()
        _check(lib().pmg_pc_apply_richardson(self._h, None if bb is None else bb.ctypes.data, y, its, int(guesszero), C.byref(outits), C.byref(reason)))
        return outits.value, reason.value

    def apply_richardson_dev(self, b, y, its=1, guesszero=False):
        outits, reason = C.c_int64(), C.c_int()
        _check(lib().pmg_pc_apply_richardson_dev(self._h, _devptr(b), _devptr(y), its, int(guesszero), C.byref(outits), C.byref(reason)))
        return outits.value, reason.value

    def apply(self, x):
        y = np.empty(self.mat.n, np.float64)
        _check(lib().pmg_pc_apply(self._h, _f64(x), y))
        return y

    # ---- device-side SaveSample of examples/benchmark/main.cc:151-175 ----
    def set_qoi(self, meas, capacity, est_mean_and_var=False):
        """qoi[it] = <y, meas> after every sample (and Welford's mean / variance of the field), kept on the device."""
        if meas is None:
            _check(lib().pmg_pc_set_qoi(self._h, None, 0, 0))
            return
        m = _f64(meas)
        _check(lib().pmg_pc_set_qoi(self._h, m.ctypes.data, int(capacity), int(bool(est_mean_and_var))))

    def get_qoi(self, reset=False):
        cnt = C.c_int64()
        _check(lib().pmg_pc_get_qoi(self._h, None, C.byref(cnt), 0))
        out = np.empty(cnt.value, np.float64)
        _check(lib().pmg_pc_get_qoi(self._h, out.ctypes.data, C.byref(cnt), int(bool(reset))))
        return out

    def get_mean_var(self):
        n, seen = self.mat.n, C.c_int64()
        mean, var = np.empty(n, np.float64), np.empty(n, np.float64)
        _check(lib().pmg_pc_get_mean_var(self._h, mean.ctypes.data, var.ctypes.data, C.byref(seen)))
        return mean, var, seen.value

    def set_sample_callback(self, cb, deleter=None):
        """PCSetSampleCallback(pc, cb, ctx, deleter): cb(it, y) with y a read-only numpy view."""
        if cb is None:
            c_cb = C.cast(None, SAMPLE_CB)
        else:
            def tramp(it, yptr, n, _ctx):
                try:
                    r = cb(int(it), np.ctypeslib.as_array(yptr, shape=(n,)))
                    return int(r or 0)
                except Exception:  # noqa: BLE001 - surfaced as PMG_ERR_CALLBACK
                    import traceback
                    traceback.print_exc()
                    return 1
            c_cb = SAMPLE_CB(tramp)
        if deleter is None:
            c_del = C.cast(None, DELETER)
        else:
            def dtramp(_ctx):
                deleter()
                return 0
            c_del = DELETER(dtramp)
        keep = (self._cb, self._del)
        _check(lib().pmg_pc_set_sample_callback(self._h, c_cb, None, c_del))
        self._old = keep  # the previous deleter may just have run; keep its trampoline alive until now
        self._cb, self._del = c_cb, c_del

    def mcgibbs_set_omega(self, omega):
        _check(lib().pmg_pc_mcgibbs_set_omega(self._h, omega))

    def mcgibbs_set_sweep_type(self, t):
        _check(lib().pmg_pc_mcgibbs_set_sweep_type(self._h, t))

    def gamgmc_set_levels(self, levels):
        _check(lib().pmg_pc_gamgmc_set_levels(self._h, levels))

    def gamgmc_get_levels(self):
        k = C.c_int()
        _check(lib().pmg_pc_gamgmc_get_levels(self._h, C.byref(k)))
        return k.value

    def gamgmc_set_interpolation(self, level, nf, nc, rowptr, col, val):
        _check(lib().pmg_pc_gamgmc_set_interpolation(self._h, level, nf, nc, np.ascontiguousarray(rowptr, np.int64), np.ascontiguousarray(col, np.int32), _f64(val)))

    def gamgmc_level_info(self, level):
        n, nnz, k = C.c_int64(), C.c_int64(), C.c_int()
        _check(lib().pmg_pc_gamgmc_get_level_info(self._h, level, C.byref(n), C.byref(nnz), C.byref(k)))
        return n.value, nnz.value, k.value

    def gamgmc_level_csr(self, level):
        n, nnz, _ = self.gamgmc_level_info(level)
        rp, col, val = np.empty(n + 1, np.int64), np.empty(nnz, np.int32), np.empty(nnz, np.float64)
        _check(lib().pmg_pc_gamgmc_get_level_csr(self._h, level, rp, col, val))
        return rp, col, val

    def set_noise_mode(self, mode):
        _check(lib().pmg_pc_set_noise_mode(self._h, mode))

    def set_noise_tape(self, z):
        z = _f64(z).ravel()
        _check(lib().pmg_pc_set_noise_tape(self._h, z, z.size))

    def noise_per_sample(self) -> int:
        d = C.c_int64()
        _check(lib().pmg_pc_noise_per_sample(self._h, C.byref(d)))
        return d.value

    def last_stats(self):
        ms, l, u = C.c_double(), C.c_int64(), C.c_int64()
        _check(lib().pmg_pc_last_stats(self._h, C.byref(ms), C.byref(l), C.byref(u)))
        return {"ms": ms.value, "launches": l.value, "dof_updates": u.value}

    def profile(self, reset=True):
        """Per-kernel totals of the V-cycle since the last reset (enable with set_option("-pc_b200_profile", 1))."""
        import json
        buf = C.create_string_buffer(1 << 16)
        _check(lib().pmg_pc_profile(self._h, buf, len(buf), 1 if reset else 0))
        return json.loads(buf.value.decode())

    def close(self):
        if self._h:
            lib().pmg_pc_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
