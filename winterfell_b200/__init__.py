"""winterfell_b200 — ctypes binding of the B200-native STARK proving hot path.

The product is the C-ABI shared library `libwinterfell_b200.so` (include/winterfell_b200.h) built
from winterfell_b200/csrc/*.cu for sm_100a. This module only loads it and wraps the entry points
for the tests and bench.py; it contains no arithmetic and no CPU fallback: if the library is not
built, or no CUDA device is present, creating a Context raises.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("WF_LIB_PATH") or os.path.join(_HERE, "libwinterfell_b200.so")  # WF_LIB_PATH: kernel experiments

P = 0xFFFFFFFF00000001
HASH_BLAKE3_256 = 0
HASH_RP64_256 = 1
HASH_RPJIVE64_256 = 2
HASH_BLAKE3_192 = 3
HASH_SHA3_256 = 4

WF_OK = 0

u64p = C.POINTER(C.c_uint64)
u8p = C.POINTER(C.c_uint8)
vp = C.c_void_p

FRI_COMMIT_FN = C.CFUNCTYPE(None, C.c_void_p, u8p)
FRI_DRAW_FN = C.CFUNCTYPE(None, C.c_void_p, u64p)
AUX_BUILDER = C.CFUNCTYPE(C.c_int, C.c_void_p, u64p, u64p)
AUX_SHARD_BUILDER = C.CFUNCTYPE(C.c_int, C.c_void_p, u64p, C.c_uint32, C.c_uint32, u64p)

_lib = None

# every symbol include/winterfell_b200.h declares: (name, restype, argtypes)
_SIGS = [
    ("wf_ctx_create", C.c_int, [C.POINTER(vp), C.c_int, vp]),
    ("wf_ctx_destroy", None, [vp]),
    ("wf_last_error", C.c_char_p, [vp]),
    ("wf_ctx_sync", C.c_int, [vp]),
    ("wf_ctx_launch_count", C.c_uint64, [vp]),
    ("wf_ctx_mem_stats", C.c_int, [vp, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]),
    ("wf_version", C.c_char_p, []),
    ("wf_ctx_set_profiling", C.c_int, [vp, C.c_int]),
    ("wf_ctx_stage_times", C.c_int, [vp, C.c_char_p, C.c_size_t, C.POINTER(C.c_float), C.POINTER(C.c_size_t)]),
    ("wf_mat_from_host_columns", C.c_int, [vp, C.POINTER(u64p), C.c_uint32, C.c_size_t, C.c_int, C.c_int, C.POINTER(vp)]),
    ("wf_mat_from_device_columns", C.c_int, [vp, vp, C.c_uint32, C.c_size_t, C.POINTER(vp)]),
    ("wf_mat_select_columns", C.c_int, [vp, vp, C.c_uint32, C.c_uint32, C.POINTER(vp)]),
    ("wf_mat_free", C.c_int, [vp, vp]),
    ("wf_mat_rows", C.c_size_t, [vp]),
    ("wf_mat_cols", C.c_uint32, [vp]),
    ("wf_mat_to_columns", C.c_int, [vp, vp, vp, C.c_int, C.c_int]),
    ("wf_mat_to_rows", C.c_int, [vp, vp, vp, C.c_int, C.c_int]),
    ("wf_mat_read_rows", C.c_int, [vp, vp, u64p, C.c_size_t, u64p, C.c_int]),
    ("wf_mat_interpolate", C.c_int, [vp, vp, C.POINTER(vp)]),
    ("wf_mat_evaluate", C.c_int, [vp, vp, C.POINTER(vp)]),
    ("wf_mat_lde", C.c_int, [vp, vp, C.c_uint32, C.POINTER(vp)]),
    ("wf_mat_lde_into", C.c_int, [vp, vp, C.c_uint32, vp]),
    ("wf_mat_wrap_device", C.c_int, [vp, vp, C.c_size_t, C.c_uint32, C.POINTER(vp)]),
    ("wf_trace_lde_from_host", C.c_int, [vp, C.POINTER(u64p), C.c_uint32, C.c_size_t, C.c_int, C.c_uint32, C.POINTER(vp), C.POINTER(vp)]),
    ("wf_mat_interpolate_with_offset", C.c_int, [vp, vp, C.c_uint64, C.POINTER(vp)]),
    ("wf_commit_rows", C.c_int, [vp, C.c_int, vp, C.POINTER(vp)]),
    ("wf_commit_rows_partitioned", C.c_int, [vp, C.c_int, vp, C.c_uint32, C.POINTER(vp)]),
    ("wf_tree_from_leaves", C.c_int, [vp, C.c_int, vp, C.c_size_t, C.c_int, C.POINTER(vp)]),
    ("wf_tree_free", C.c_int, [vp, vp]),
    ("wf_tree_root", C.c_int, [vp, vp, u8p]),
    ("wf_tree_num_leaves", C.c_size_t, [vp]),
    ("wf_tree_to_host", C.c_int, [vp, vp, u8p, u8p]),
    ("wf_tree_open_many", C.c_int, [vp, vp, u64p, C.c_size_t, u8p, u8p, C.POINTER(C.c_size_t)]),
    ("wf_fri_build_layers", C.c_int, [vp, C.c_int, vp, C.c_int, C.c_uint32, C.c_uint32, C.c_uint32, FRI_COMMIT_FN, FRI_DRAW_FN, vp, C.POINTER(vp)]),
    ("wf_fri_build_layers_default_channel", C.c_int, [vp, C.c_int, vp, C.c_int, C.c_uint32, C.c_uint32, C.c_uint32, u8p, C.c_size_t, C.POINTER(vp)]),
    ("wf_fri_num_layers", C.c_uint32, [vp]),
    ("wf_fri_remainder", C.c_size_t, [vp, u64p, C.c_size_t]),
    ("wf_fri_build_proof", C.c_int, [vp, vp, u64p, C.c_size_t, u8p, C.POINTER(C.c_size_t)]),
    ("wf_fri_free", C.c_int, [vp, vp]),
    ("wf_prove_fib", C.c_int, [vp, C.POINTER(u64p), C.c_int, C.c_uint32, C.c_uint32, u64p, C.POINTER(C.c_uint32), u8p, C.POINTER(C.c_size_t)]),
    ("wf_prove_air", C.c_int, [vp, u64p, C.c_size_t, C.POINTER(u64p), C.c_int, C.c_uint32, C.POINTER(C.c_uint32), u8p, C.POINTER(C.c_size_t)]),
    ("wf_prove_air_aux", C.c_int, [vp, u64p, C.c_size_t, C.POINTER(u64p), C.c_int, C.c_uint32, C.POINTER(C.c_uint32), AUX_BUILDER, vp,
                                   u8p, C.POINTER(C.c_size_t)]),
        ("wf_prove_air_aux_dyn", C.c_int, [vp, u64p, C.c_size_t, C.POINTER(u64p), C.c_int, C.c_uint32, C.POINTER(C.c_uint32), AUX_BUILDER, AUX_BUILDER, vp,
                                   u8p, C.POINTER(C.c_size_t)]),
    ("wf_eval_constraints", C.c_int, [vp, u64p, C.c_size_t, C.c_uint32, C.c_uint32, C.c_uint32, vp, vp, u64p, u64p, C.POINTER(vp)]),
    ("wf_composition_commit", C.c_int, [vp, C.c_int, vp, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.POINTER(vp), C.POINTER(vp), C.POINTER(vp)]),
    ("wf_composition_commit_partitioned", C.c_int, [vp, C.c_int, vp, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.POINTER(vp),
                                                    C.POINTER(vp), C.POINTER(vp)]),
    ("wf_mat_evaluate_at", C.c_int, [vp, vp, C.c_uint32, C.c_uint32, u64p, u64p, u64p, u64p]),
    ("wf_deep_compose", C.c_int, [vp, C.c_uint32, vp, vp, vp, C.c_uint32, u64p, u64p, u64p, u64p, C.POINTER(vp)]),
    ("wf_prove_fib_dev", C.c_int, [vp, vp, C.c_uint32, C.c_uint32, u64p, C.POINTER(C.c_uint32), u8p, C.POINTER(C.c_size_t)]),
    ("wf_grind", C.c_int, [vp, C.c_int, u8p, C.c_uint32, C.POINTER(C.c_uint64)]),
    ("wf_ntt_dev", C.c_int, [vp, vp, C.c_uint32, C.c_uint32, C.c_int]),
    ("wf_hash_rows_dev", C.c_int, [vp, C.c_int, vp, C.c_size_t, C.c_uint32, vp]),
    ("wf_merkle_dev", C.c_int, [vp, C.c_int, vp, C.c_size_t, vp]),
    ("wf_fri_fold_dev", C.c_int, [vp, vp, C.c_size_t, C.c_int, C.c_uint32, u64p, vp]),
    ("wf_field_ops_dev", C.c_int, [vp, vp, vp, C.c_size_t, vp]),
    ("wf_ext_ops_dev", C.c_int, [vp, C.c_uint32, vp, vp, C.c_size_t, vp]),
    ("wf_ctx_set_jit", C.c_int, [vp, C.c_int]),
    ("wf_ctx_jit_stats", C.c_int, [vp, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]),
    ("wf_jit_compile_air", C.c_int, [u64p, C.c_size_t, C.c_uint32, C.POINTER(C.c_size_t), C.c_char_p, C.c_size_t]),
    ("wf_air_check", C.c_int, [u64p, C.c_size_t, C.c_uint32, C.c_uint32, C.c_char_p, C.c_size_t]),
    ("wf_host_hash_elements", C.c_int, [C.c_int, u64p, C.c_size_t, u8p]),
    ("wf_host_merge", C.c_int, [C.c_int, u8p, u8p]),
    ("wf_host_merge_with_int", C.c_int, [C.c_int, u8p, C.c_uint64, u8p]),
    ("wf_host_mul", C.c_uint64, [C.c_uint64, C.c_uint64]),
    ("wf_host_mul_2exp", C.c_uint64, [C.c_uint64, C.c_uint32]),
    ("wf_host_mont_to_canonical", C.c_uint64, [C.c_uint64]),
    ("wf_host_canonical_to_mont", C.c_uint64, [C.c_uint64]),
    ("wf_host_write_usize", C.c_size_t, [C.c_uint64, u8p]),
    ("wf_host_coin_draw", C.c_int, [C.c_int, u64p, C.c_size_t, u8p, C.c_int, C.c_size_t, u64p]),
    ("wf_host_build_fib_trace", C.c_int, [C.c_uint32, C.c_size_t, u64p, u64p]),
    ("wf_host_sharded_opening_plan", C.c_long, [C.c_size_t, C.c_int, C.c_int, u64p, C.c_size_t, u64p, u64p, C.c_size_t]),
    ("wf_prove_fib_sharded", C.c_int, [vp, vp, C.POINTER(u64p), vp, C.c_int, C.c_uint32, C.c_uint32, u64p, C.POINTER(C.c_uint32), u8p,
                                       C.POINTER(C.c_size_t), C.POINTER(C.c_double)]),
    ("wf_host_shard_columns", C.c_int, [C.c_uint32, C.c_int, C.c_int, C.POINTER(C.c_uint32), C.POINTER(C.c_uint32)]),
    ("wf_prove_air_sharded", C.c_int, [vp, vp, u64p, C.c_size_t, C.POINTER(u64p), vp, C.c_int, C.c_uint32, C.POINTER(C.c_uint32), u8p,
                                       C.POINTER(C.c_size_t), C.POINTER(C.c_double)]),
    ("wf_prove_air_aux_sharded", C.c_int, [vp, vp, u64p, C.c_size_t, C.POINTER(u64p), vp, C.c_int, C.c_uint32, C.POINTER(C.c_uint32),
                                           AUX_SHARD_BUILDER, AUX_BUILDER, vp, u8p, C.POINTER(C.c_size_t), C.POINTER(C.c_double)]),
]


def declared_symbols():
    return [s[0] for s in _SIGS]


def lib():
    """Load the C-ABI library. Fails loudly when it has not been built (no fallback)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} is missing: build it with winterfell_b200/build.sh "
                "(python -c 'import __graft_entry__ as g; g.build()'). There is no CPU fallback.")
        L = C.CDLL(LIB_PATH)
        for name, res, args in _SIGS:
            fn = getattr(L, name)
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


class WfError(RuntimeError):
    pass


def _u64(a):
    a = np.ascontiguousarray(a, dtype=np.uint64)
    return a, a.ctypes.data_as(u64p)


def _u8(a):
    a = np.ascontiguousarray(a, dtype=np.uint8)
    return a, a.ctypes.data_as(u8p)


class Context:
    """One prover context per GPU (wf_ctx). `stream` is a raw cudaStream_t integer (0 = default)."""

    def __init__(self, device=0, stream=0):
        self.L = lib()
        h = vp()
        r = self.L.wf_ctx_create(C.byref(h), device, vp(stream))
        if r != WF_OK:
            raise WfError(f"wf_ctx_create failed ({r}): no usable CUDA device — this library has no CPU path")
        self.h = h

    def close(self):
        if getattr(self, "h", None):
            self.L.wf_ctx_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def check(self, r):
        if r != WF_OK:
            raise WfError(f"error {r}: {self.L.wf_last_error(self.h).decode()}")

    def sync(self):
        self.check(self.L.wf_ctx_sync(self.h))

    @property
    def launches(self):
        return self.L.wf_ctx_launch_count(self.h)

    def mem_stats(self):
        """(live_buffers, live_bytes, pooled_bytes): device buffers handed out and not yet freed, and bytes parked for reuse."""
        a, b, c = C.c_uint64(0), C.c_uint64(0), C.c_uint64(0)
        self.check(self.L.wf_ctx_mem_stats(self.h, C.byref(a), C.byref(b), C.byref(c)))
        return a.value, b.value, c.value

    # ---- matrices ----
    def mat_from_host_columns(self, cols, ext_degree=1, mont=False):
        """cols: [c, n*d] uint64 array (ColMatrix<E>: c columns of n elements of degree d)."""
        a = np.ascontiguousarray(cols, dtype=np.uint64)
        c = a.shape[0]
        n = a.shape[1] // ext_degree
        ptrs = (u64p * c)(*[a[j].ctypes.data_as(u64p) for j in range(c)])
        h = vp()
        self.check(self.L.wf_mat_from_host_columns(self.h, ptrs, c, n, ext_degree, int(mont), C.byref(h)))
        return Mat(self, h)

    def trace_lde_from_host(self, cols, log_blowup, mont=False):
        """cols: [ncols, n] uint64 host array (pinned for overlap). Returns (polys Mat, lde Mat)."""
        a = np.ascontiguousarray(cols, dtype=np.uint64)
        c, n = a.shape
        ptrs = (u64p * c)(*[a[j].ctypes.data_as(u64p) for j in range(c)])
        p, l = vp(), vp()
        self.check(self.L.wf_trace_lde_from_host(self.h, ptrs, c, n, int(mont), log_blowup, C.byref(p), C.byref(l)))
        self.sync()  # `a` may be a temporary: the asynchronous copies must finish before it is released
        return Mat(self, p), Mat(self, l)

    def mat_wrap_device(self, dptr, nrows, ncols):
        """Non-owning Mat over device memory in segment layout (the caller keeps the memory alive)."""
        h = vp()
        self.check(self.L.wf_mat_wrap_device(self.h, vp(dptr), nrows, ncols, C.byref(h)))
        return Mat(self, h)

    def mat_from_device_columns(self, dptr, ncols, nrows):
        h = vp()
        self.check(self.L.wf_mat_from_device_columns(self.h, vp(dptr), ncols, nrows, C.byref(h)))
        return Mat(self, h)

    def commit_rows(self, hash_id, mat, partition_size=0):
        h = vp()
        if partition_size:
            self.check(self.L.wf_commit_rows_partitioned(self.h, hash_id, mat.h, partition_size, C.byref(h)))
        else:
            self.check(self.L.wf_commit_rows(self.h, hash_id, mat.h, C.byref(h)))
        return Tree(self, h)

    def tree_from_leaves(self, hash_id, leaves):
        l_, lp = _u8(leaves)
        h = vp()
        self.check(self.L.wf_tree_from_leaves(self.h, hash_id, C.cast(lp, vp), l_.size // 32, 0, C.byref(h)))
        return Tree(self, h)

    def fri_build_layers_default(self, hash_id, mat, ext_degree, folding, rem_max_deg, blowup):
        roots = np.zeros((64, 32), dtype=np.uint8)
        h = vp()
        self.check(self.L.wf_fri_build_layers_default_channel(self.h, hash_id, mat.h, ext_degree, folding, rem_max_deg,
                                                              blowup, roots.ctypes.data_as(u8p), roots.size, C.byref(h)))
        f = Fri(self, h, ext_degree)
        return f, roots[: f.num_layers + 1].copy()

    # ---- stepwise pipeline (the seams of prover/src/lib.rs:195-223 and the steps between them) ----
    def eval_constraints(self, desc, log_n, blowup, ext, main_lde, aux_lde, coeffs, aux_rand=None):
        d_, dp = _u64(desc)
        c_, cp = _u64(coeffs)
        rp = None
        if aux_rand is not None:
            r_, rp = _u64(aux_rand)
        h = vp()
        self.check(self.L.wf_eval_constraints(self.h, dp, d_.size, log_n, blowup, ext, main_lde.h, aux_lde.h if aux_lde else None,
                                              cp, rp, C.byref(h)))
        return Mat(self, h)

    def composition_commit(self, hash_id, comp_trace, log_n, blowup, ext, num_cols):
        a, b, t = vp(), vp(), vp()
        self.check(self.L.wf_composition_commit(self.h, hash_id, comp_trace.h, log_n, blowup, ext, num_cols,
                                                C.byref(a), C.byref(b), C.byref(t)))
        return Mat(self, a), Mat(self, b), Tree(self, t)

    def evaluate_at(self, polys, ext, col_ext, z0, z1):
        a_, ap = _u64(z0)
        b_, bp = _u64(z1)
        ncols = polys.cols // col_ext
        o0 = np.zeros((ncols, ext), dtype=np.uint64)
        o1 = np.zeros((ncols, ext), dtype=np.uint64)
        self.check(self.L.wf_mat_evaluate_at(self.h, polys.h, ext, col_ext, ap, bp, o0.ctypes.data_as(u64p), o1.ctypes.data_as(u64p)))
        return o0, o1

    def deep_compose(self, ext, main_lde, aux_lde, cons_lde, log_n, z, coeffs, ood_cur, ood_next):
        z_, zp = _u64(z)
        c_, cp = _u64(coeffs)
        a_, ap = _u64(ood_cur)
        b_, bp = _u64(ood_next)
        h = vp()
        self.check(self.L.wf_deep_compose(self.h, ext, main_lde.h, aux_lde.h if aux_lde else None, cons_lde.h, log_n, zp, cp, ap, bp,
                                          C.byref(h)))
        return Mat(self, h)

    def prove_fib(self, trace, results, opts, mont=False, out_buf=None):
        """trace: [2k, n] uint64; results: [k]; opts: uint32[9] (see wf_prove_fib). Returns proof bytes.
        out_buf: optional preallocated uint8 array for the proof (a caller proving in a loop reuses one)."""
        a = np.ascontiguousarray(trace, dtype=np.uint64)
        c, n = a.shape
        ptrs = (u64p * c)(*[a[j].ctypes.data_as(u64p) for j in range(c)])
        r_, rp = _u64(results)
        o_ = np.ascontiguousarray(opts, dtype=np.uint32)
        buf = out_buf if out_buf is not None else np.zeros(1 << 23, dtype=np.uint8)
        cap = buf.size
        ln = C.c_size_t(cap)
        self.check(self.L.wf_prove_fib(self.h, ptrs, int(mont), c // 2, int(n).bit_length() - 1, rp,
                                       o_.ctypes.data_as(C.POINTER(C.c_uint32)), buf.ctypes.data_as(u8p), C.byref(ln)))
        return buf[: ln.value].tobytes()

    def prove_air(self, desc, trace, opts, mont=False):
        """desc: flat AIR description (see wf_prove_air); trace: [width, n] uint64. Returns proof bytes."""
        d_, dp = _u64(desc)
        a = np.ascontiguousarray(trace, dtype=np.uint64)
        c, n = a.shape
        ptrs = (u64p * c)(*[a[j].ctypes.data_as(u64p) for j in range(c)])
        o_ = np.ascontiguousarray(opts, dtype=np.uint32)
        cap = 1 << 23
        buf = np.zeros(cap, dtype=np.uint8)
        ln = C.c_size_t(cap)
        self.check(self.L.wf_prove_air(self.h, dp, d_.size, ptrs, int(mont), int(n).bit_length() - 1,
                                       o_.ctypes.data_as(C.POINTER(C.c_uint32)), buf.ctypes.data_as(u8p), C.byref(ln)))
        return buf[: ln.value].tobytes()

    def prove_air_aux(self, desc, trace, opts, builder, aux_width, num_rands, mont=False):
        """Multi-segment AIR (wf_prove_air_aux). builder(rand [num_rands, d] uint64) -> aux columns
        [aux_width, n, d] uint64, called on the host after the main commitment."""
        d_, dp = _u64(desc)
        a = np.ascontiguousarray(trace, dtype=np.uint64)
        c, n = a.shape
        ptrs = (u64p * c)(*[a[j].ctypes.data_as(u64p) for j in range(c)])
        o_ = np.ascontiguousarray(opts, dtype=np.uint32)
        d = int(o_[3])

        def cb(_user, rand_p, out_p):
            try:
                rand = (np.ctypeslib.as_array(rand_p, shape=(num_rands, d)).copy() if num_rands
                        else np.zeros((0, d), dtype=np.uint64))
                aux = np.ascontiguousarray(builder(rand), dtype=np.uint64).reshape(aux_width, n, d)
                np.ctypeslib.as_array(out_p, shape=(aux_width, n, d))[:] = aux
                return 0
            except Exception:  # must not unwind through the C caller
                import traceback
                traceback.print_exc()
                return 1

        cfn = AUX_BUILDER(cb)
        cap = 1 << 23
        buf = np.zeros(cap, dtype=np.uint8)
        ln = C.c_size_t(cap)
        self.check(self.L.wf_prove_air_aux(self.h, dp, d_.size, ptrs, int(mont), int(n).bit_length() - 1,
                                           o_.ctypes.data_as(C.POINTER(C.c_uint32)), cfn, None, buf.ctypes.data_as(u8p),
                                           C.byref(ln)))
        return buf[: ln.value].tobytes()

    def prove_air_aux_dyn(self, desc, trace, opts, builder, values_fn, aux_width, num_rands, num_values, mont=False):
        """wf_prove_air_aux_dyn: as prove_air_aux, plus values_fn(rand [num_rands, d], values [num_values, d]) -> values
        [num_values, d] = Air::get_aux_assertions(aux_rand_elements) (air/src/air/mod.rs:279)."""
        d_, dp = _u64(desc)
        a = np.ascontiguousarray(trace, dtype=np.uint64)
        c, n = a.shape
        ptrs = (u64p * c)(*[a[j].ctypes.data_as(u64p) for j in range(c)])
        o_ = np.ascontiguousarray(opts, dtype=np.uint32)
        d = int(o_[3])

        def guard(fn):
            def wrapped(*args):
                try:
                    fn(*args)
                    return 0
                except Exception:  # must not unwind through the C caller
                    import traceback
                    traceback.print_exc()
                    return 1
            return wrapped

        def cb_build(_user, rand_p, out_p):
            rand = np.ctypeslib.as_array(rand_p, shape=(num_rands, d)).copy()
            np.ctypeslib.as_array(out_p, shape=(aux_width, n, d))[:] = np.ascontiguousarray(builder(rand), dtype=np.uint64).reshape(aux_width, n, d)

        def cb_values(_user, rand_p, val_p):
            rand = np.ctypeslib.as_array(rand_p, shape=(num_rands, d)).copy()
            vals = np.ctypeslib.as_array(val_p, shape=(num_values, d))
            vals[:] = np.ascontiguousarray(values_fn(rand, vals.copy()), dtype=np.uint64).reshape(num_values, d)

        f1, f2 = AUX_BUILDER(guard(cb_build)), AUX_BUILDER(guard(cb_values))
        cap = 1 << 23
        buf = np.zeros(cap, dtype=np.uint8)
        ln = C.c_size_t(cap)
        self.check(self.L.wf_prove_air_aux_dyn(self.h, dp, d_.size, ptrs, int(mont), int(n).bit_length() - 1,
                                               o_.ctypes.data_as(C.POINTER(C.c_uint32)), f1, f2, None, buf.ctypes.data_as(u8p), C.byref(ln)))
        return buf[: ln.value].tobytes()

    def prove_fib_dev(self, d_trace, k, log_n, results, opts, out_buf=None):
        """trace resident on the device: column-major [2k][n] at raw pointer d_trace."""
        r_, rp = _u64(results)
        o_ = np.ascontiguousarray(opts, dtype=np.uint32)
        buf = out_buf if out_buf is not None else np.zeros(1 << 23, dtype=np.uint8)
        ln = C.c_size_t(buf.size)
        self.check(self.L.wf_prove_fib_dev(self.h, vp(d_trace), k, log_n, rp, o_.ctypes.data_as(C.POINTER(C.c_uint32)),
                                           buf.ctypes.data_as(u8p), C.byref(ln)))
        return buf[: ln.value].tobytes()

    def set_profiling(self, on):
        self.check(self.L.wf_ctx_set_profiling(self.h, int(on)))

    def stage_times(self):
        names = C.create_string_buffer(4096)
        ms = (C.c_float * 64)()
        cnt = C.c_size_t(64)
        self.check(self.L.wf_ctx_stage_times(self.h, names, 4096, ms, C.byref(cnt)))
        nm = [x for x in names.value.decode().split(",") if x]
        return [(nm[i], float(ms[i])) for i in range(cnt.value)]

    def grind(self, hash_id, seed: bytes, grinding):
        t_, tp = _u8(np.frombuffer(seed, dtype=np.uint8))
        nonce = C.c_uint64(0)
        self.check(self.L.wf_grind(self.h, hash_id, tp, grinding, C.byref(nonce)))
        return nonce.value

    # ---- plain device kernels (raw device pointers as integers) ----
    def ntt_dev(self, dptr, log_n, cols, inverse=False):
        self.check(self.L.wf_ntt_dev(self.h, vp(dptr), log_n, cols, int(inverse)))

    def hash_rows_dev(self, hash_id, d_rows, nrows, cols, d_digests):
        self.check(self.L.wf_hash_rows_dev(self.h, hash_id, vp(d_rows), nrows, cols, vp(d_digests)))

    def merkle_dev(self, hash_id, d_leaves, nleaves, d_nodes):
        self.check(self.L.wf_merkle_dev(self.h, hash_id, vp(d_leaves), nleaves, vp(d_nodes)))

    def field_ops_dev(self, d_a, d_b, n, d_out):
        self.check(self.L.wf_field_ops_dev(self.h, vp(d_a), vp(d_b), n, vp(d_out)))

    def set_jit(self, on):
        """constraint kernels compiled per AIR with NVRTC (default on) vs the built-in interpreter"""
        self.check(self.L.wf_ctx_set_jit(self.h, int(on)))

    def jit_stats(self):
        a, b, c = C.c_uint64(0), C.c_uint64(0), C.c_uint64(0)
        self.check(self.L.wf_ctx_jit_stats(self.h, C.byref(a), C.byref(b), C.byref(c)))
        return {"compiled": a.value, "cache_hits": b.value, "fallbacks": c.value}

    def ext_ops_dev(self, ext, d_a, d_b, n, d_out):
        self.check(self.L.wf_ext_ops_dev(self.h, ext, vp(d_a), vp(d_b), n, vp(d_out)))

    def fri_fold_dev(self, d_evals, length, ext_degree, folding, alpha, d_next):
        a_, ap = _u64(alpha)
        self.check(self.L.wf_fri_fold_dev(self.h, vp(d_evals), length, ext_degree, folding, ap, vp(d_next)))


class Mat:
    def __init__(self, ctx, h):
        self.ctx, self.h = ctx, h

    def free(self):
        if self.h:
            self.ctx.L.wf_mat_free(self.ctx.h, self.h)
            self.h = None

    @property
    def rows(self):
        return self.ctx.L.wf_mat_rows(self.h)

    @property
    def cols(self):
        return self.ctx.L.wf_mat_cols(self.h)

    def to_columns(self, mont=False):
        o = np.zeros((self.cols, self.rows), dtype=np.uint64)
        self.ctx.check(self.ctx.L.wf_mat_to_columns(self.ctx.h, self.h, vp(o.ctypes.data), 1, int(mont)))
        return o

    def to_rows(self, mont=False):
        o = np.zeros((self.rows, self.cols), dtype=np.uint64)
        self.ctx.check(self.ctx.L.wf_mat_to_rows(self.ctx.h, self.h, vp(o.ctypes.data), 1, int(mont)))
        return o

    def to_device_rows(self, dptr):
        self.ctx.check(self.ctx.L.wf_mat_to_rows(self.ctx.h, self.h, vp(dptr), 0, 0))

    def read_rows(self, positions, mont=False):
        p_, pp = _u64(positions)
        o = np.zeros((p_.size, self.cols), dtype=np.uint64)
        self.ctx.check(self.ctx.L.wf_mat_read_rows(self.ctx.h, self.h, pp, p_.size, o.ctypes.data_as(u64p), int(mont)))
        return o

    def _unary(self, fn, *extra):
        h = vp()
        self.ctx.check(fn(self.ctx.h, self.h, *extra, C.byref(h)))
        return Mat(self.ctx, h)

    def select_columns(self, first, count):
        return self._unary(self.ctx.L.wf_mat_select_columns, first, count)

    def interpolate(self):
        return self._unary(self.ctx.L.wf_mat_interpolate)

    def evaluate(self):
        return self._unary(self.ctx.L.wf_mat_evaluate)

    def lde_into(self, log_blowup, out):
        self.ctx.check(self.ctx.L.wf_mat_lde_into(self.ctx.h, self.h, log_blowup, out.h))

    def lde(self, log_blowup):
        return self._unary(self.ctx.L.wf_mat_lde, log_blowup)

    def interpolate_with_offset(self, offset):
        return self._unary(self.ctx.L.wf_mat_interpolate_with_offset, offset)


class Tree:
    def __init__(self, ctx, h):
        self.ctx, self.h = ctx, h

    def free(self):
        if self.h:
            self.ctx.L.wf_tree_free(self.ctx.h, self.h)
            self.h = None

    @property
    def num_leaves(self):
        return self.ctx.L.wf_tree_num_leaves(self.h)

    def root(self):
        o = np.zeros(32, dtype=np.uint8)
        self.ctx.check(self.ctx.L.wf_tree_root(self.ctx.h, self.h, o.ctypes.data_as(u8p)))
        return o.tobytes()

    def to_host(self):
        n = self.num_leaves
        lv = np.zeros((n, 32), dtype=np.uint8)
        nd = np.zeros((n, 32), dtype=np.uint8)
        self.ctx.check(self.ctx.L.wf_tree_to_host(self.ctx.h, self.h, lv.ctypes.data_as(u8p), nd.ctypes.data_as(u8p)))
        return lv, nd

    def open_many(self, positions):
        p_, pp = _u64(positions)
        k = p_.size
        lv = np.zeros((k, 32), dtype=np.uint8)
        cap = 64 + k * 40 * 33
        buf = np.zeros(cap, dtype=np.uint8)
        ln = C.c_size_t(cap)
        self.ctx.check(self.ctx.L.wf_tree_open_many(self.ctx.h, self.h, pp, k, lv.ctypes.data_as(u8p),
                                                    buf.ctypes.data_as(u8p), C.byref(ln)))
        return lv, buf[: ln.value].tobytes()


class Fri:
    def __init__(self, ctx, h, d):
        self.ctx, self.h, self.d = ctx, h, d

    def free(self):
        if self.h:
            self.ctx.L.wf_fri_free(self.ctx.h, self.h)
            self.h = None

    @property
    def num_layers(self):
        return self.ctx.L.wf_fri_num_layers(self.h)

    def remainder(self):
        buf = np.zeros(4096, dtype=np.uint64)
        n = self.ctx.L.wf_fri_remainder(self.h, buf.ctypes.data_as(u64p), buf.size)
        return buf[: n * self.d].copy()

    def build_proof(self, positions):
        p_, pp = _u64(positions)
        cap = 1 << 22
        buf = np.zeros(cap, dtype=np.uint8)
        ln = C.c_size_t(cap)
        self.ctx.check(self.ctx.L.wf_fri_build_proof(self.ctx.h, self.h, pp, p_.size, buf.ctypes.data_as(u8p), C.byref(ln)))
        return buf[: ln.value].tobytes()


# ---- host helpers (usable without a GPU) ----
def build_fib_trace(k, n, out=None):
    """FibSmall x k trace (examples/src/fibonacci/fib_small/prover.rs:37-53): ([2k, n] uint64, results [k]).
    `out`: optional preallocated [2k, n] uint64 array (e.g. a view of pinned memory)."""
    tr = out if out is not None else np.empty((2 * k, n), dtype=np.uint64)
    assert tr.shape == (2 * k, n) and tr.dtype == np.uint64 and tr.flags["C_CONTIGUOUS"]
    res = np.zeros(k, dtype=np.uint64)
    if lib().wf_host_build_fib_trace(k, n, tr.ctypes.data_as(u64p), res.ctypes.data_as(u64p)) != WF_OK:
        raise WfError("wf_host_build_fib_trace: bad arguments")
    return tr, res


def sharded_opening_plan(n_global, world, rank, positions):
    """(want, idx) of wf_host_sharded_opening_plan as uint64 arrays."""
    p_, pp = _u64(positions)
    cap = 64 * max(len(p_), 1) * 64
    want, idx = np.zeros(cap, dtype=np.uint64), np.zeros(cap, dtype=np.uint64)
    cnt = lib().wf_host_sharded_opening_plan(n_global, world, rank, pp, len(p_), want.ctypes.data_as(u64p), idx.ctypes.data_as(u64p), cap)
    if cnt < 0:
        raise WfError("wf_host_sharded_opening_plan: bad arguments")
    return want[:cnt].copy(), idx[:cnt].copy()


def shard_columns(width, world, rank):
    """(first, count): the trace columns rank `rank` of `world` owns in a sharded proof (wf_host_shard_columns)."""
    first, count = C.c_uint32(0), C.c_uint32(0)
    if lib().wf_host_shard_columns(width, world, rank, C.byref(first), C.byref(count)) != WF_OK:
        raise WfError(f"wf_host_shard_columns: bad arguments (width {width}, world {world}, rank {rank})")
    return first.value, count.value


def aux_shape(desc):
    """(aux width, number of random elements, number of aux assertion values) of a flat AIR description (wf_prove_air_aux);
    (0, 0, 0) without an aux segment or when the description is malformed (the library then refuses it)."""
    d = [int(v) for v in np.asarray(desc, dtype=np.uint64).reshape(-1)]
    p = 0

    def rd(k=1):
        nonlocal p
        if p + k > len(d):
            raise IndexError
        p += k
        return d[p - k]

    def degrees():
        for _ in range(rd()):
            rd()
            rd(rd())   # base, ncyc, cycles

    try:
        rd()                                     # width
        degrees()
        for _ in range(rd()):                    # periodic columns
            rd(rd())
        rd(rd())                                 # constants
        rd()                                     # registers
        rd(4 * rd())                             # program
        for _ in range(rd()):                    # assertions: column, first_step, stride, nvals, values
            rd(3)
            rd(rd())
        rd(rd())                                 # public inputs
        rd()                                     # exemptions
        if p == len(d):
            return 0, 0, 0
        aw, nr = rd(), rd()
        degrees()
        rd()
        rd(4 * rd())
        nv = 0
        for _ in range(rd()):                    # aux assertions: values in E, three words each
            rd(3)
            k = rd()
            rd(3 * k)
            nv += k
        return aw, nr, nv
    except IndexError:
        return 0, 0, 0


def host_hash_elements(hash_id, elems):
    e_, ep = _u64(np.asarray(elems, dtype=np.uint64).reshape(-1))
    o = np.zeros(32, dtype=np.uint8)
    lib().wf_host_hash_elements(hash_id, ep, e_.size, o.ctypes.data_as(u8p))
    return o.tobytes()


def host_merge(hash_id, a, b):
    t_, tp = _u8(np.frombuffer(a + b, dtype=np.uint8))
    o = np.zeros(32, dtype=np.uint8)
    lib().wf_host_merge(hash_id, tp, o.ctypes.data_as(u8p))
    return o.tobytes()


def host_merge_with_int(hash_id, seed, value):
    t_, tp = _u8(np.frombuffer(seed, dtype=np.uint8))
    o = np.zeros(32, dtype=np.uint8)
    lib().wf_host_merge_with_int(hash_id, tp, value, o.ctypes.data_as(u8p))
    return o.tobytes()


def air_check(desc, log_n, blowup):
    """The checks the proving entry points run on an AIR description, without a device. Returns (status, reason)."""
    d_, dp = _u64(desc)
    msg = C.create_string_buffer(512)
    rc = lib().wf_air_check(dp, d_.size, log_n, blowup, msg, 512)
    return rc, msg.value.decode(errors="replace")


def jit_compile_air(desc, ext):
    """Compiles the constraint kernel of an AIR description with NVRTC; needs no device. Returns (status, cubin bytes, log)."""
    d_, dp = _u64(desc)
    n = C.c_size_t(0)
    log = C.create_string_buffer(1 << 16)
    rc = lib().wf_jit_compile_air(dp, d_.size, ext, C.byref(n), log, 1 << 16)
    return rc, n.value, log.value.decode(errors="replace")
