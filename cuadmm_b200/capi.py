"""ctypes binding of include/cuadmm_b200.h (one thin class per opaque handle)."""
import ctypes as C
import os
import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("CUADMM_LIB_PATH") or os.path.join(_HERE, "lib", "libcuadmm_b200.so")   # override: A/B builds in experiments
if not os.path.exists(LIB_PATH):
    raise ImportError(
        f"{LIB_PATH} is missing: build it with `make` at the repo root (or "
        "`python -c 'import __graft_entry__ as g; g.build()'`). There is no pure-Python fallback.")
lib = C.CDLL(LIB_PATH, mode=C.RTLD_GLOBAL)

c_i32p = C.POINTER(C.c_int32)
c_i64p = C.POINTER(C.c_int64)
c_f64p = C.POINTER(C.c_double)
vp = C.c_void_p


class CuadmmError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"cuadmm error {code}: {msg}")
        self.code = code


lib.cuadmm_last_error.restype = C.c_char_p
lib.cuadmm_version.restype = C.c_char_p


def _check(rc):
    if rc != 0:
        raise CuadmmError(rc, lib.cuadmm_last_error().decode())


def _i32(a):
    return np.ascontiguousarray(a, dtype=np.int32)


def _i64(a):
    return np.ascontiguousarray(a, dtype=np.int64)


def _f64(a):
    return np.ascontiguousarray(a, dtype=np.float64)


def _p(a, t):
    return a.ctypes.data_as(t) if a is not None else None


def _types(types, nblk):
    """block cones as the C ABI takes them: nblk letters 's' (PSD), 'l' (nonnegative), 'u' (free); None stays None
    (every block PSD).  Accepts a string, bytes or a sequence of one-letter strings."""
    if types is None:
        return None
    t = types.encode() if isinstance(types, str) else bytes(types) if isinstance(types, (bytes, bytearray)) \
        else "".join(types).encode()
    if len(t) != nblk:
        raise ValueError(f"{len(t)} block types for {nblk} blocks")
    return t


def version():
    return lib.cuadmm_version().decode()


def device_count():
    lib.cuadmm_device_count.restype = C.c_int
    return lib.cuadmm_device_count()


def _sig(name, restype, *argtypes):
    f = getattr(lib, name)
    f.restype = restype
    f.argtypes = list(argtypes)
    return f


# ---------------------------------------------------------------- plan
_sig("cuadmm_plan_create", C.c_int, c_i32p, C.c_int64, C.c_int, C.POINTER(vp))
_sig("cuadmm_plan_create_typed", C.c_int, C.c_char_p, c_i32p, C.c_int64, C.c_int, C.POINTER(vp))
_sig("cuadmm_plan_destroy", None, vp)
_sig("cuadmm_plan_vec_len", C.c_int64, vp)
_sig("cuadmm_plan_nblk", C.c_int64, vp)
_sig("cuadmm_plan_num_sizes", C.c_int64, vp)
_sig("cuadmm_plan_sizes", C.c_int, vp, c_i32p, c_i32p, c_i32p)
_sig("cuadmm_plan_totals", C.c_int, vp, c_i64p)
_sig("cuadmm_plan_start_indices", C.c_int64, vp, C.c_int, c_i64p)
_sig("cuadmm_plan_maps", C.c_int, vp, c_i32p, c_i32p, c_i32p)
_sig("cuadmm_plan_partition", C.c_int, vp, C.c_int, c_i32p, c_f64p)
_sig("cuadmm_plan_set_jacobi", C.c_int, vp, C.c_double, C.c_int)
_sig("cuadmm_plan_set_warm_start", C.c_int, vp, C.c_int)
_sig("cuadmm_plan_set_rank_limit", C.c_int, vp, C.c_int)
_sig("cuadmm_eig_rank_mask", C.c_int, c_i32p, C.c_int64, C.c_int64, C.c_int64)
_sig("cuadmm_plan_last_ms", C.c_double, vp)
_sig("cuadmm_plan_last_launches", C.c_int64, vp)
_sig("cuadmm_project_psd", C.c_int, vp, vp, vp, vp)
_sig("cuadmm_project_psd_host", C.c_int, vp, c_f64p, c_f64p)
_sig("cuadmm_project_epilogue", C.c_int, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp)
_sig("cuadmm_project_psd_eig_host", C.c_int, vp, c_f64p, c_f64p, c_f64p, c_i32p)
_sig("cuadmm_svec_to_smat", C.c_int, vp, vp, vp, vp, vp)
_sig("cuadmm_smat_to_svec", C.c_int, vp, vp, vp, vp, vp)


class Plan:
    """Block plan + cone projection (cuadmm_plan_*, cuadmm_project_psd*).  types: one letter per block, 's' PSD,
    'l' nonnegative orthant, 'u' free (None: all 's')."""

    def __init__(self, blk, device=0, types=None):
        self.blk = _i32(blk)
        self.types = _types(types, len(self.blk))
        self.h = vp()
        if self.types is None:
            _check(lib.cuadmm_plan_create(_p(self.blk, c_i32p), len(self.blk), device, C.byref(self.h)))
        else:
            _check(lib.cuadmm_plan_create_typed(self.types, _p(self.blk, c_i32p), len(self.blk), device, C.byref(self.h)))
        self.device = device

    def close(self):
        if self.h:
            lib.cuadmm_plan_destroy(self.h)
            self.h = vp()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def vec_len(self):
        return lib.cuadmm_plan_vec_len(self.h)

    @property
    def nblk(self):
        return lib.cuadmm_plan_nblk(self.h)

    def sizes(self):
        k = lib.cuadmm_plan_num_sizes(self.h)
        s = np.zeros(k, np.int32); n = np.zeros(k, np.int32); lg = np.zeros(k, np.int32)
        _check(lib.cuadmm_plan_sizes(self.h, _p(s, c_i32p), _p(n, c_i32p), _p(lg, c_i32p)))
        return s, n, lg

    def totals(self):
        t = np.zeros(6, np.int64)
        _check(lib.cuadmm_plan_totals(self.h, _p(t, c_i64p)))
        return t

    def start_indices(self, which):
        k = lib.cuadmm_plan_start_indices(self.h, which, None)
        if k < 0:
            raise CuadmmError(k, lib.cuadmm_last_error().decode())
        out = np.zeros(k, np.int64)
        lib.cuadmm_plan_start_indices(self.h, which, _p(out, c_i64p))
        return out

    def maps(self):
        L = self.vec_len
        B = np.zeros(L, np.int32); M1 = np.zeros(L, np.int32); M2 = np.zeros(L, np.int32)
        _check(lib.cuadmm_plan_maps(self.h, _p(B, c_i32p), _p(M1, c_i32p), _p(M2, c_i32p)))
        return B, M1, M2

    def partition(self, nparts):
        owner = np.zeros(self.nblk, np.int32); cost = np.zeros(nparts, np.float64)
        _check(lib.cuadmm_plan_partition(self.h, nparts, _p(owner, c_i32p), _p(cost, c_f64p)))
        return owner, cost

    def set_jacobi(self, threshold, max_sweeps):
        _check(lib.cuadmm_plan_set_jacobi(self.h, threshold, max_sweeps))

    def set_warm_start(self, enable):
        _check(lib.cuadmm_plan_set_warm_start(self.h, 1 if enable else 0))

    def set_rank_limit(self, eig_rank):
        """fixed-rank projection: keep only the eig_rank largest eigenvalues of every block (0: off)"""
        _check(lib.cuadmm_plan_set_rank_limit(self.h, int(eig_rank)))

    def project_host(self, Xb):
        Xb = _f64(Xb)
        assert Xb.shape == (self.vec_len,)
        out = np.empty_like(Xb)
        _check(lib.cuadmm_project_psd_host(self.h, _p(Xb, c_f64p), _p(out, c_f64p)))
        return out

    def project_eig_host(self, Xb):
        Xb = _f64(Xb)
        out = np.empty_like(Xb)
        eig = np.zeros(int(self.blk.sum()), np.float64)
        sweeps = np.zeros(self.nblk, np.int32)
        _check(lib.cuadmm_project_psd_eig_host(self.h, _p(Xb, c_f64p), _p(out, c_f64p), _p(eig, c_f64p), _p(sweeps, c_i32p)))
        return out, eig, sweeps

    def project_device(self, d_in_ptr, d_out_ptr, stream=0):
        """device pointers (ints), e.g. torch tensor .data_ptr()"""
        _check(lib.cuadmm_project_psd(self.h, vp(d_in_ptr), vp(d_out_ptr), vp(stream)))

    def project_epilogue_device(self, d_Xb, d_Xproj, d_X, d_Rd1, d_C, d_S, d_SmC, d_sig, stream=0):
        """projection with the solver's fused epilogue: S = (Xproj - X)/sig - Rd1, SmC = S - C (S = 0 on 'u' blocks);
        device pointers (ints), d_sig a device scalar"""
        _check(lib.cuadmm_project_epilogue(self.h, vp(d_Xb), vp(d_Xproj), vp(d_X), vp(d_Rd1), vp(d_C), vp(d_S), vp(d_SmC),
                                           vp(d_sig), vp(stream)))

    def svec_to_smat_device(self, d_svec, d_large, d_small, stream=0):
        _check(lib.cuadmm_svec_to_smat(self.h, vp(d_svec), vp(d_large), vp(d_small), vp(stream)))

    def smat_to_svec_device(self, d_large, d_small, d_svec, stream=0):
        _check(lib.cuadmm_smat_to_svec(self.h, vp(d_large), vp(d_small), vp(d_svec), vp(stream)))

    @property
    def last_ms(self):
        return lib.cuadmm_plan_last_ms(self.h)

    @property
    def last_launches(self):
        return lib.cuadmm_plan_last_launches(self.h)


# ---------------------------------------------------------------- spmv
def _maybe(name, restype, *argtypes):
    try:
        return _sig(name, restype, *argtypes)
    except AttributeError:
        return None


_maybe("cuadmm_spmv_create", C.c_int, C.c_int64, C.c_int64, C.c_int64, c_i32p, c_i32p, c_f64p, C.c_int, C.POINTER(vp))
_maybe("cuadmm_spmv_destroy", None, vp)
_maybe("cuadmm_spmv", C.c_int, vp, C.c_double, vp, C.c_double, vp, vp)
_maybe("cuadmm_spmv_host", C.c_int, vp, C.c_double, c_f64p, C.c_double, c_f64p)
_maybe("cuadmm_normA_host", C.c_int, C.c_int64, c_i32p, c_f64p, c_f64p)
_maybe("cuadmm_csc_to_csr_host", C.c_int, C.c_int64, C.c_int64, C.c_int64, c_i32p, c_i32p, c_f64p, c_i32p, c_i32p, c_f64p)


class SpMV:
    """CSR y = alpha*A*x + beta*y (cuadmm_spmv_*)."""

    def __init__(self, rows, cols, rowptr, colind, val, device=0):
        self.rows, self.cols = int(rows), int(cols)
        self.rowptr, self.colind, self.val = _i32(rowptr), _i32(colind), _f64(val)
        self.h = vp()
        _check(lib.cuadmm_spmv_create(self.rows, self.cols, len(self.val), _p(self.rowptr, c_i32p),
                                      _p(self.colind, c_i32p), _p(self.val, c_f64p), device, C.byref(self.h)))

    def close(self):
        if self.h:
            lib.cuadmm_spmv_destroy(self.h)
            self.h = vp()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def apply_host(self, x, alpha=1.0, beta=0.0, y=None):
        x = _f64(x)
        y = np.zeros(self.rows) if y is None else _f64(y).copy()
        _check(lib.cuadmm_spmv_host(self.h, alpha, _p(x, c_f64p), beta, _p(y, c_f64p)))
        return y

    def apply_device(self, d_x, d_y, alpha=1.0, beta=0.0, stream=0):
        _check(lib.cuadmm_spmv(self.h, alpha, vp(d_x), beta, vp(d_y), vp(stream)))


def normA_host(col_ptrs, vals):
    """get_normA on host arrays: returns (normA, normalised vals)"""
    col_ptrs = _i32(col_ptrs); vals = _f64(vals).copy()
    m = len(col_ptrs) - 1
    normA = np.zeros(m)
    _check(lib.cuadmm_normA_host(m, _p(col_ptrs, c_i32p), _p(vals, c_f64p), _p(normA, c_f64p)))
    return normA, vals


def csc_to_csr_host(nrows, ncols, col_ptrs, row_ids, vals):
    col_ptrs, row_ids, vals = _i32(col_ptrs), _i32(row_ids), _f64(vals)
    nnz = len(vals)
    rp = np.zeros(nrows + 1, np.int32); ci = np.zeros(nnz, np.int32); v = np.zeros(nnz)
    _check(lib.cuadmm_csc_to_csr_host(nrows, ncols, nnz, _p(col_ptrs, c_i32p), _p(row_ids, c_i32p), _p(vals, c_f64p),
                                      _p(rp, c_i32p), _p(ci, c_i32p), _p(v, c_f64p)))
    return rp, ci, v


# ---------------------------------------------------------------- y-solve
_maybe("cuadmm_ysolve_create", C.c_int, C.c_int64, C.c_int64, C.c_int64, c_i32p, c_i32p, c_f64p, C.c_double, C.c_int, C.POINTER(vp))
_maybe("cuadmm_ysolve_destroy", None, vp)
_maybe("cuadmm_ysolve", C.c_int, vp, vp, vp, vp)
_maybe("cuadmm_ysolve_host", C.c_int, vp, c_f64p, c_f64p)
_maybe("cuadmm_ysolve_stats", C.c_int, vp, c_i64p)
_maybe("cuadmm_ysolve_perm", C.c_int, vp, c_i32p)
_maybe("cuadmm_debug_ysolve_paths", C.c_int, vp, c_i64p)

_SWEEP_PATHS = ("n_sub", "n_sub_pack", "n_sub_warp", "n_sub_cta", "pk_rows", "pk_n_heavy", "pk_has_ext", "collapsed",
                "max_chunks", "long_records", "levels", "narrow_phases", "wide_phases", "top_long_slots")


class YSolve:
    """y = (A A^T + eps I)^-1 rhs on the device (cuadmm_ysolve_*). A is CSR (m x vec_len)."""

    def __init__(self, m, vec_len, rowptr, colind, val, eps=1e-15, device=0):
        self.m = int(m)
        rowptr, colind, val = _i32(rowptr), _i32(colind), _f64(val)
        self.h = vp()
        _check(lib.cuadmm_ysolve_create(self.m, int(vec_len), len(val), _p(rowptr, c_i32p), _p(colind, c_i32p),
                                        _p(val, c_f64p), eps, device, C.byref(self.h)))

    def close(self):
        if self.h:
            lib.cuadmm_ysolve_destroy(self.h)
            self.h = vp()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def solve_host(self, rhs):
        rhs = _f64(rhs)
        y = np.zeros(self.m)
        _check(lib.cuadmm_ysolve_host(self.h, _p(rhs, c_f64p), _p(y, c_f64p)))
        return y

    def solve_device(self, d_rhs, d_y, stream=0):
        _check(lib.cuadmm_ysolve(self.h, vp(d_rhs), vp(d_y), vp(stream)))

    def stats(self):
        s = np.zeros(8, np.int64)
        _check(lib.cuadmm_ysolve_stats(self.h, _p(s, c_i64p)))
        return dict(nnz_AAt=int(s[0]), nnz_L=int(s[1]), levels=int(s[2]), dense_tail=int(s[3]),
                    launches=int(s[4]), bytes=int(s[5]), deficient=int(s[6]), subtrees=int(s[7]) // 100000,
                    subtree_depth=int(s[7]) % 100000)

    def paths(self):
        """the kernel paths a solve takes (cuadmm_debug_ysolve_paths): {"fwd": {...}, "bwd": {...}, "tail": {...}}"""
        s = np.zeros(32, np.int64)
        _check(lib.cuadmm_debug_ysolve_paths(self.h, _p(s, c_i64p)))
        sweep = lambda o: {k: int(s[o + i]) for i, k in enumerate(_SWEEP_PATHS)}
        return dict(fwd=sweep(0), bwd=sweep(14),
                    tail=dict(n_tail=int(s[28]), tiles_lower=int(s[29]), tiles_upper=int(s[30]),
                              postorder_fallback=int(s[31])))

    def perm(self):
        p = np.zeros(self.m, np.int32)
        _check(lib.cuadmm_ysolve_perm(self.h, _p(p, c_i32p)))
        return p


# ---------------------------------------------------------------- problem + solver
_maybe("cuadmm_problem_from_txt", C.c_int, C.c_char_p, C.c_int, C.POINTER(vp))
_maybe("cuadmm_problem_destroy", None, vp)
_maybe("cuadmm_problem_dims", C.c_int, vp, c_i64p)
_maybe("cuadmm_problem_array", vp, vp, C.c_int)
_maybe("cuadmm_solver_create", C.c_int, C.POINTER(vp))
_maybe("cuadmm_solver_destroy", None, vp)
_maybe("cuadmm_solver_set_verbose", C.c_int, vp, C.c_int)
_maybe("cuadmm_solver_init", C.c_int, vp, C.c_int, C.c_int, C.c_int64, C.c_int64,
       c_i32p, c_i32p, c_f64p, C.c_int64, c_i32p, c_f64p, C.c_int64, c_i32p, c_f64p, C.c_int64,
       c_i32p, C.c_int64, c_f64p, c_f64p, c_f64p, C.c_double)
_maybe("cuadmm_solver_solve", C.c_int, vp, C.c_int, C.c_double, C.c_int, C.c_int, C.c_int, C.c_int, C.c_double, C.c_int)
_maybe("cuadmm_solver_get_X", C.c_int, vp, c_f64p)
_maybe("cuadmm_solver_get_y", C.c_int, vp, c_f64p)
_maybe("cuadmm_solver_get_S", C.c_int, vp, c_f64p)
_maybe("cuadmm_solver_set_XyS", C.c_int, vp, c_f64p, c_f64p, c_f64p, C.c_double)
_maybe("cuadmm_solver_update_data", C.c_int, vp, c_i32p, c_f64p, C.c_int64, c_i32p, c_f64p, C.c_int64, C.c_int, C.c_double)
_maybe("cuadmm_solver_iter_num", C.c_int64, vp)
_maybe("cuadmm_solver_history", C.c_int, vp, C.c_int, c_f64p, C.c_int64)
_maybe("cuadmm_solver_set_infeasibility_check", C.c_int, vp, C.c_int, C.c_double)
_maybe("cuadmm_solver_stop_reason", C.c_int, vp)
_maybe("cuadmm_solver_certificate", C.c_int, vp, C.c_int, c_f64p, c_f64p)
_maybe("cuadmm_solver_infeasibility_stats", C.c_int, vp, c_f64p)
_maybe("cuadmm_solver_times", C.c_int, vp, c_f64p)
_maybe("cuadmm_solver_launches", C.c_int64, vp)
_maybe("cuadmm_solver_run_iterations", C.c_int, vp, C.c_int, C.c_int, C.c_int, c_f64p)
_maybe("cuadmm_solver_run_iterations_ex", C.c_int, vp, C.c_int, C.c_int, c_f64p)
_maybe("cuadmm_solver_ysolve_stats", C.c_int, vp, c_i64p)
_maybe("cuadmm_nccl_unique_id", C.c_int, C.c_char_p)
_maybe("cuadmm_unique_id", C.c_int, C.c_char_p)
_maybe("cuadmm_solver_set_device", C.c_int, vp, C.c_int)
_maybe("cuadmm_solver_set_distributed", C.c_int, vp, C.c_int, C.c_int, C.c_char_p)
_maybe("cuadmm_shard_create", C.c_int, c_i32p, C.c_int64, C.c_int, C.c_int, C.POINTER(vp))
_maybe("cuadmm_shard_create_typed", C.c_int, C.c_char_p, c_i32p, C.c_int64, C.c_int, C.c_int, C.POINTER(vp))
_maybe("cuadmm_shard_local_types", C.c_int, vp, C.c_char_p)
_maybe("cuadmm_solver_set_block_types", C.c_int, vp, C.c_char_p, C.c_int64)
_maybe("cuadmm_shard_destroy", None, vp)
_maybe("cuadmm_shard_info", C.c_int, vp, c_i64p)
_maybe("cuadmm_shard_maps", C.c_int, vp, c_i32p, c_i64p, c_i64p, c_i32p)
_maybe("cuadmm_shard_slice_csc", C.c_int64, vp, C.c_int64, c_i32p, c_i32p, c_f64p, c_i32p, c_i32p, c_f64p)
_maybe("cuadmm_solver_init_from_problem", C.c_int, vp, vp, C.c_int, C.c_int, C.c_double)


def nccl_unique_id():
    """kept for callers of the removed NCCL transport: the same 128 random bytes as unique_id()"""
    buf = C.create_string_buffer(128)
    _check(lib.cuadmm_nccl_unique_id(buf))
    return buf.raw


def eig_rank_mask(batch_size, mat_size, eig_rank):
    """get_eig_rank_mask of the reference (src/utils/get_eig_rank_mask.cu)"""
    mask = np.zeros(batch_size * mat_size, np.int32)
    _check(lib.cuadmm_eig_rank_mask(_p(mask, c_i32p), batch_size, mat_size, eig_rank))
    return mask


def unique_id():
    """128 random bytes: job id of the peer-memory transport (rank 0 creates it, the launcher broadcasts it)"""
    buf = C.create_string_buffer(128)
    _check(lib.cuadmm_unique_id(buf))
    return buf.raw


class Shard:
    """Block-level sharding of an SDP over `world` GPUs (cuadmm_shard_*; host logic only)."""

    def __init__(self, blk, world, rank, types=None):
        self.blk = _i32(blk)
        self.types = _types(types, len(self.blk))
        self.h = vp()
        if self.types is None:
            _check(lib.cuadmm_shard_create(_p(self.blk, c_i32p), len(self.blk), world, rank, C.byref(self.h)))
        else:
            _check(lib.cuadmm_shard_create_typed(self.types, _p(self.blk, c_i32p), len(self.blk), world, rank,
                                                 C.byref(self.h)))
        info = np.zeros(4, np.int64)
        _check(lib.cuadmm_shard_info(self.h, _p(info, c_i64p)))
        self.vec_len_local, self.nblk_local, self.vec_len, self.world = [int(x) for x in info]
        self.local_blk = np.zeros(self.nblk_local, np.int32)
        self.local_block_ids = np.zeros(self.nblk_local, np.int64)
        self.loc2glob = np.zeros(self.vec_len_local, np.int64)
        self.owner = np.zeros(len(self.blk), np.int32)
        _check(lib.cuadmm_shard_maps(self.h, _p(self.local_blk, c_i32p), _p(self.local_block_ids, c_i64p),
                                     _p(self.loc2glob, c_i64p), _p(self.owner, c_i32p)))
        buf = C.create_string_buffer(max(self.nblk_local, 1))
        _check(lib.cuadmm_shard_local_types(self.h, buf))
        self.local_types = buf.raw[:self.nblk_local].decode()

    def slice_csc(self, col_ptrs, row_ids, vals):
        col_ptrs, row_ids, vals = _i32(col_ptrs), _i32(row_ids), _f64(vals)
        ncols = len(col_ptrs) - 1
        ocp = np.zeros(ncols + 1, np.int32); ori = np.zeros(max(len(vals), 1), np.int32); ov = np.zeros(max(len(vals), 1))
        nnz = lib.cuadmm_shard_slice_csc(self.h, ncols, _p(col_ptrs, c_i32p), _p(row_ids, c_i32p), _p(vals, c_f64p),
                                         _p(ocp, c_i32p), _p(ori, c_i32p), _p(ov, c_f64p))
        if nnz < 0:
            raise CuadmmError(-1, lib.cuadmm_last_error().decode())
        return ocp, ori[:nnz], ov[:nnz]

    def close(self):
        if self.h:
            lib.cuadmm_shard_destroy(self.h)
            self.h = vp()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Problem:
    """Problem::from_txt (cuadmm_problem_*)."""
    _KINDS = {0: np.int32, 1: np.int32, 2: np.float64, 3: np.int32, 4: np.float64, 5: np.int32,
              6: np.float64, 7: np.int32, 8: np.float64, 9: np.float64, 10: np.float64}

    def __init__(self, prefix, warm_start=False):
        self.h = vp()
        _check(lib.cuadmm_problem_from_txt(prefix.encode(), int(warm_start), C.byref(self.h)))
        d = np.zeros(8, np.int64)
        _check(lib.cuadmm_problem_dims(self.h, _p(d, c_i64p)))
        self.vec_len, self.con_num, self.mat_num, self.At_nnz, self.b_nnz, self.C_nnz = [int(x) for x in d[:6]]
        self.has_warm = bool(d[6])

    @property
    def blk_types(self):
        """the blk.txt letter of every block ('s', 'l' or 'u'), as one string"""
        ptr = lib.cuadmm_problem_array(self.h, 11)
        return C.string_at(ptr, self.mat_num).decode() if ptr and self.mat_num else ""

    def array(self, which):
        n = {0: self.con_num + 1, 1: self.At_nnz, 2: self.At_nnz, 3: self.b_nnz, 4: self.b_nnz, 5: self.C_nnz,
             6: self.C_nnz, 7: self.mat_num, 8: self.vec_len, 9: self.con_num, 10: self.vec_len}[which]
        if which >= 8 and not self.has_warm:
            return None
        ptr = lib.cuadmm_problem_array(self.h, which)
        if not ptr or n == 0:
            return np.zeros(0, self._KINDS[which])
        t = C.c_int32 if self._KINDS[which] == np.int32 else C.c_double
        return np.ctypeslib.as_array(C.cast(ptr, C.POINTER(t)), shape=(n,)).copy()

    def close(self):
        if self.h:
            lib.cuadmm_problem_destroy(self.h)
            self.h = vp()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Solver:
    """Mirror of the reference's SDPSolver (include/cuadmm/solver.h:30-248): init / solve, then X, y, S
    and the info_* history.  Same argument names and meaning; errors raise CuadmmError."""
    HIST = dict(pobj=0, dobj=1, errRp=2, errRd=3, relgap=4, sig=5, bscale=6, Cscale=7)

    def __init__(self, verbose=False):
        self.h = vp()
        _check(lib.cuadmm_solver_create(C.byref(self.h)))
        _check(lib.cuadmm_solver_set_verbose(self.h, int(verbose)))
        self.vec_len = self.con_num = 0

    def close(self):
        if self.h:
            lib.cuadmm_solver_destroy(self.h)
            self.h = vp()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_device(self, device):
        _check(lib.cuadmm_solver_set_device(self.h, int(device)))

    def set_distributed(self, rank, world, job_id):
        """one process per GPU: call before init with the id rank 0 got from unique_id()"""
        _check(lib.cuadmm_solver_set_distributed(self.h, int(rank), int(world), job_id))

    def init(self, eig_stream_num_per_gpu, cpu_eig_thread_num, vec_len, con_num,
             At_csc_col_ptrs, At_csc_row_ids, At_csc_vals, b_indices, b_vals, C_indices, C_vals, blk_vals,
             X_vals=None, y_vals=None, S_vals=None, sig=1.0, blk_types=None):
        """blk_types: one letter per block, 's' PSD, 'l' nonnegative, 'u' free (None: all 's')"""
        cp, ri, av = _i32(At_csc_col_ptrs), _i32(At_csc_row_ids), _f64(At_csc_vals)
        bi, bv, ci, cv, blk = _i32(b_indices), _f64(b_vals), _i32(C_indices), _f64(C_vals), _i32(blk_vals)
        X = _f64(X_vals) if X_vals is not None else None
        y = _f64(y_vals) if y_vals is not None else None
        S = _f64(S_vals) if S_vals is not None else None
        self.vec_len, self.con_num = int(vec_len), int(con_num)
        if blk_types is not None:
            _check(lib.cuadmm_solver_set_block_types(self.h, _types(blk_types, len(blk)), len(blk)))
        _check(lib.cuadmm_solver_init(self.h, eig_stream_num_per_gpu, cpu_eig_thread_num, vec_len, con_num,
                                      _p(cp, c_i32p), _p(ri, c_i32p), _p(av, c_f64p), len(av),
                                      _p(bi, c_i32p), _p(bv, c_f64p), len(bv), _p(ci, c_i32p), _p(cv, c_f64p), len(cv),
                                      _p(blk, c_i32p), len(blk), _p(X, c_f64p), _p(y, c_f64p), _p(S, c_f64p), sig))

    def init_from_problem(self, prob, eig_stream_num_per_gpu=15, cpu_eig_thread_num=30, sig=1.0):
        self.vec_len, self.con_num = prob.vec_len, prob.con_num
        _check(lib.cuadmm_solver_init_from_problem(self.h, prob.h, eig_stream_num_per_gpu, cpu_eig_thread_num, sig))

    def solve(self, max_iter, stop_tol, sig_update_threshold=500, sig_update_stage_1=50, sig_update_stage_2=100,
              switch_admm=11000, sigscale=1.05, if_first=True):
        _check(lib.cuadmm_solver_solve(self.h, max_iter, stop_tol, sig_update_threshold, sig_update_stage_1,
                                       sig_update_stage_2, switch_admm, sigscale, int(if_first)))

    def _get(self, fn, n):
        out = np.zeros(n)
        _check(fn(self.h, _p(out, c_f64p)))
        return out

    @property
    def X(self):
        return self._get(lib.cuadmm_solver_get_X, self.vec_len)

    @property
    def y(self):
        return self._get(lib.cuadmm_solver_get_y, self.con_num)

    @property
    def S(self):
        return self._get(lib.cuadmm_solver_get_S, self.vec_len)

    @property
    def info_iter_num(self):
        return lib.cuadmm_solver_iter_num(self.h)

    def history(self, name):
        n = self.info_iter_num
        out = np.zeros(max(n, 1))
        _check(lib.cuadmm_solver_history(self.h, self.HIST[name], _p(out, c_f64p), n))
        return out[:n]

    STOP_REASONS = {0: "not solved", 1: "converged", 2: "max_iter", 3: "primal_infeasible", 4: "dual_infeasible"}

    def set_infeasibility_check(self, interval, eps=1e-7):
        """check for primal / dual infeasibility every `interval` iterations (0: off) at tolerance eps; applies from the
        next solve"""
        _check(lib.cuadmm_solver_set_infeasibility_check(self.h, int(interval), float(eps)))

    @property
    def stop_reason(self):
        """0 before the first solve, 1 converged, 2 max iterations, 3 primal infeasible, 4 dual infeasible"""
        return lib.cuadmm_solver_stop_reason(self.h)

    def certificate(self, which):
        """(vector, ratio) of the last solve: which 0 the primal infeasibility certificate y-bar (b'y-bar = 1), which 1
        the dual infeasibility certificate d (<C, d> = -1), in the caller's units"""
        out = np.zeros(max(self.con_num if which == 0 else self.vec_len, 1))
        ratio = np.zeros(1)
        _check(lib.cuadmm_solver_certificate(self.h, int(which), _p(out, c_f64p), _p(ratio, c_f64p)))
        return out[:self.con_num if which == 0 else self.vec_len], float(ratio[0])

    def infeasibility_stats(self):
        """what the checks of the last solve saw (cuadmm_solver_infeasibility_stats)"""
        t = np.zeros(8)
        _check(lib.cuadmm_solver_infeasibility_stats(self.h, _p(t, c_f64p)))
        return dict(checks=int(t[0]), primal_projections=int(t[1]), dual_projections=int(t[2]), min_primal_ratio=t[3],
                    min_dual_ratio=t[4], min_primal_guard=t[5], min_dual_guard=t[6], last_check_iter=int(t[7]))

    def times(self):
        t = np.zeros(8)
        _check(lib.cuadmm_solver_times(self.h, _p(t, c_f64p)))
        return dict(total=t[0], init=t[1], solve=t[2], projection=t[3], ysolve=t[4], spmv=t[5], update=t[6])

    @property
    def launches(self):
        return lib.cuadmm_solver_launches(self.h)

    def run_iterations(self, n, sgs=True, profile=False):
        """measurement hook: n iterations from the current state, stop test off; device ms by CUDA events"""
        out = np.zeros(4)
        _check(lib.cuadmm_solver_run_iterations(self.h, int(n), int(sgs), int(profile), _p(out, c_f64p)))
        return dict(total_ms=out[0], projection_ms=out[1], ysolve_ms=out[2], other_ms=out[3])

    def run_iterations_ex(self, n, sgs=True):
        """profiled pass with the finer stage breakdown (ms totals over the n iterations)"""
        out = np.zeros(8)
        _check(lib.cuadmm_solver_run_iterations_ex(self.h, int(n), int(sgs), _p(out, c_f64p)))
        return dict(total_ms=out[0], projection_ms=out[1], ysolve_ms=out[2], other_ms=out[3], k5_ms=out[4], k8_ms=out[5],
                    tail_gemv_ms=out[6])

    def set_XyS(self, X, y, S, sig):
        X, y, S = _f64(X), _f64(y), _f64(S)
        _check(lib.cuadmm_solver_set_XyS(self.h, _p(X, c_f64p), _p(y, c_f64p), _p(S, c_f64p), float(sig)))

    def update_data(self, b_idx, b_val, C_idx, C_val, keep_iterate=False, sig=1.0):
        """New b and C (sparse triplets, as in init) for the same A and blocks, keeping the factorisation, the projection
        plan and the iteration graphs; follow with solve(..., if_first=True).  keep_iterate=False: the next solve is
        that of a fresh init with these b, C and sig; True: it starts from the X, y, S the last solve returned."""
        arrs = []
        for name, idx, val in (("b", b_idx, b_val), ("C", C_idx, C_val)):
            i, v = np.asarray(idx), np.asarray(val)
            if i.ndim != 1 or v.ndim != 1 or len(i) != len(v):
                raise ValueError(f"{name}: indices and values must be 1-D of one length, got shapes {i.shape} and {v.shape}")
            if len(i) and (not np.issubdtype(i.dtype, np.integer) or i.min() < np.iinfo(np.int32).min
                           or i.max() > np.iinfo(np.int32).max):
                raise ValueError(f"{name}: indices must be int32 integers")
            arrs += [_i32(i), _f64(v)]
        bi, bv, ci, cv = arrs
        _check(lib.cuadmm_solver_update_data(self.h, _p(bi, c_i32p), _p(bv, c_f64p), len(bv), _p(ci, c_i32p),
                                             _p(cv, c_f64p), len(cv), int(bool(keep_iterate)), float(sig)))

    def get_into(self, X, y, S):
        """D2H of X, y, S into caller-provided (e.g. pinned) arrays"""
        _check(lib.cuadmm_solver_get_X(self.h, _p(X, c_f64p)))
        _check(lib.cuadmm_solver_get_y(self.h, _p(y, c_f64p)))
        _check(lib.cuadmm_solver_get_S(self.h, _p(S, c_f64p)))

    def ysolve_stats(self):
        s = np.zeros(8, np.int64)
        _check(lib.cuadmm_solver_ysolve_stats(self.h, _p(s, c_i64p)))
        return dict(nnz_AAt=int(s[0]), nnz_L=int(s[1]), levels=int(s[2]), dense_tail=int(s[3]),
                    launches=int(s[4]), bytes=int(s[5]), deficient=int(s[6]))


# ---------------------------------------------------------------- MEX-shaped entry
_maybe("cuadmm_solve_matlab_like", C.c_int, C.c_int, C.c_int, C.c_double, C.c_int64, C.c_int64,
       c_i64p, c_i64p, c_f64p, c_i64p, c_f64p, C.c_int64, c_i64p, c_f64p, C.c_int64, c_f64p, C.c_int64,
       c_f64p, c_f64p, c_f64p, C.c_double, C.c_int, C.c_int, C.c_int, C.c_int, C.c_double,
       c_f64p, c_f64p, c_f64p, c_i64p, c_f64p, c_f64p)


def solve_matlab_like(eig_stream_num_per_gpu, max_iter, stop_tol, At_jc, At_ir, At_pr, b_ir, b_pr, C_ir, C_pr, blk_vec,
                      X0, y0, S0, sig, sig_update_threshold=500, sig_update_stage_1=50, sig_update_stage_2=100,
                      switch_admm=11000, sigscale=1.05):
    """cuadmm_solve_matlab_like: the argument list of the reference's MEX gateway (MATLAB/cuadmm_MATLAB.cu:197-433):
    At_stack as MATLAB sparse (jc/ir size_t, pr double), b and C_stack as sparse columns, blk_vec as doubles,
    X0/y0/S0 dense.  Returns (X, y, S, info) with info = {iter_num, pobj, dobj, errRp, errRd, relgap, sig, bscale,
    Cscale, total_time} like the 10 x 2 info cell (:157-183)."""
    jc, ir, pr = _i64(At_jc), _i64(At_ir), _f64(At_pr)
    bi, bp, ci, cp = _i64(b_ir), _f64(b_pr), _i64(C_ir), _f64(C_pr)
    blk = _f64(blk_vec)
    con_num = len(jc) - 1
    vec_len = int(sum(int(n) * (int(n) + 1) // 2 for n in blk))
    X0, y0, S0 = _f64(X0), _f64(y0), _f64(S0)
    X = np.zeros(vec_len); y = np.zeros(con_num); S = np.zeros(vec_len)
    it = C.c_int64(0); tt = C.c_double(0.0)
    info = np.zeros(8 * (max_iter + 1))
    _check(lib.cuadmm_solve_matlab_like(eig_stream_num_per_gpu, max_iter, stop_tol, vec_len, con_num,
                                        _p(jc, c_i64p), _p(ir, c_i64p), _p(pr, c_f64p), _p(bi, c_i64p), _p(bp, c_f64p), len(bp),
                                        _p(ci, c_i64p), _p(cp, c_f64p), len(cp), _p(blk, c_f64p), len(blk),
                                        _p(X0, c_f64p), _p(y0, c_f64p), _p(S0, c_f64p), sig,
                                        sig_update_threshold, sig_update_stage_1, sig_update_stage_2, switch_admm, sigscale,
                                        _p(X, c_f64p), _p(y, c_f64p), _p(S, c_f64p), C.byref(it), _p(info, c_f64p), C.byref(tt)))
    n = int(it.value)
    H = info.reshape(8, max_iter + 1)
    names = ["pobj", "dobj", "errRp", "errRd", "relgap", "sig", "bscale", "Cscale"]
    out = {k: H[i, :n].copy() for i, k in enumerate(names)}
    out["iter_num"] = n
    out["total_time"] = float(tt.value)
    return X, y, S, out
