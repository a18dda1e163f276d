"""ctypes binding of ``libb200repair.so`` (C ABI declared in ``include/b200repair.h``).

This is the only door into the hand-written sm_100a kernels.  There is no CPU fallback: if the
shared library is missing, or no CUDA device is usable, every engine entry point raises.
"""
import ctypes
import os
from ctypes import POINTER, byref, c_char_p, c_double, c_int, c_int32, c_int64, c_void_p

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_NAME = "libb200repair.so"
LIB_PATH = os.path.join(_HERE, LIB_NAME)

DR_OP = {"EQ": 0, "IQ": 1, "LT": 2, "GT": 3}


class NativeError(RuntimeError):
    pass


class dr_forest(ctypes.Structure):
    _fields_ = [
        ("n_seq", c_int32), ("n_trees", c_int32), ("n_nodes", c_int32), ("n_feat", c_int32),
        ("seq_tree_off", c_void_p), ("tree_node_off", c_void_p), ("node_thr", c_void_p),
        ("node_meta", c_void_p), ("baseline", c_void_p), ("feat_col", c_void_p),
        ("enc_lut_off", c_void_p), ("enc_lut", c_void_p), ("class_code", c_void_p),
        ("kind", c_int32), ("integral", c_int32), ("n_classes", c_int32),
    ]


class dr_forest_ranked(ctypes.Structure):
    _fields_ = [
        ("n_seq", c_int32), ("n_trees", c_int32), ("n_nodes", c_int32), ("n_leaves", c_int32),
        ("n_slots", c_int32), ("max_depth", c_int32), ("n_chunks", c_int32), ("layout", c_int32),
        ("chunk_tree_off", c_void_p), ("chunk_seq", c_void_p), ("chunk_node_off", c_void_p),
        ("chunk_leaf_off", c_void_p), ("chunk_hdr_off", c_void_p), ("tree_hdr", c_void_p),
        ("node_word", c_void_p), ("leaf_value", c_void_p), ("baseline", c_void_p), ("slot_col", c_void_p),
        ("rank_lut_off", c_void_p), ("rank_lut", c_void_p), ("slot_nan", c_void_p), ("class_code", c_void_p),
        ("n_classes", c_int32),
    ]


class dr_domain_target(ctypes.Structure):
    _fields_ = [("target", c_void_p), ("bitmap", c_void_p), ("hist_t", c_void_p), ("dom_t", c_int32),
                ("n_corr", c_int32), ("corr", c_void_p * 8), ("cooc", c_void_p * 8), ("tau", c_int64 * 8),
                ("dom_c", c_int32 * 8)]


class dr_gbdt_params(ctypes.Structure):
    _fields_ = [("n_rows", c_int32), ("n_features", c_int32), ("n_classes", c_int32), ("n_iter", c_int32),
                ("max_depth", c_int32), ("num_leaves", c_int32), ("min_data_in_leaf", c_int32),
                ("learning_rate", c_double), ("min_sum_hessian", c_double), ("qscale", c_double),
                ("reg_lambda", c_double), ("colsample_bytree", c_double), ("subsample", c_double),
                ("subsample_freq", c_int32), ("seed", c_int32)]


_PP = POINTER(c_void_p)
_SIGNATURES = {
    # name: (restype, argtypes)
    "dr_ctx_create": (c_int, [c_int, POINTER(c_void_p)]),
    "dr_ctx_destroy": (c_int, [c_void_p]),
    "dr_last_error": (c_char_p, [c_void_p]),
    "dr_abi_version": (c_int, []),
    "dr_launch_count": (c_int64, [c_void_p]),
    "dr_widen_u8": (c_int, [c_void_p, c_void_p, c_int64, c_void_p, c_void_p]),
    "dr_h2d_copy": (c_int, [c_void_p, _PP, _PP, POINTER(c_int64), c_int, c_int, c_void_p]),
    "dr_d2h_copy": (c_int, [c_void_p, _PP, _PP, POINTER(c_int64), c_int, c_int, c_void_p]),
    "dr_index_presence": (c_int, [c_void_p, c_void_p, c_int, c_void_p, c_int64, c_int64, c_int32, c_void_p, c_void_p]),
    "dr_index_remap": (c_int, [c_void_p, c_void_p, c_int, c_void_p, c_int64, c_int64, c_void_p, c_int32,
                               c_void_p, c_void_p]),
    "dr_ids_unique_i64": (c_int, [c_void_p, c_void_p, c_int64, POINTER(c_int), c_void_p]),
    "dr_gather_i64": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_void_p]),
    "dr_valid_bits": (c_int, [c_void_p, c_void_p, c_int64, c_void_p, c_void_p]),
    "dr_scan_hist": (c_int, [c_void_p, _PP, POINTER(c_int32), c_int, c_int64, _PP, c_void_p, c_void_p]),
    "dr_lut_scan": (c_int, [c_void_p, c_void_p, c_int64, c_void_p, c_int32, c_void_p, c_void_p]),
    "dr_quartiles": (c_int, [c_void_p, c_void_p, c_int64, POINTER(c_double), POINTER(c_int64), c_void_p]),
    "dr_range_flag": (c_int, [c_void_p, c_void_p, c_int64, c_double, c_double, c_void_p, c_void_p]),
    "dr_lof_workspace_bytes": (c_int64, [c_int64]),
    "dr_lof_flag": (c_int, [c_void_p, c_void_p, c_int64, c_int, c_int64, c_int64, c_void_p, c_void_p,
                            POINTER(c_int64), c_void_p, c_int64, c_void_p]),
    "dr_dc_const": (c_int, [c_void_p, _PP, POINTER(c_int32), POINTER(c_int32), c_int, c_int64, c_void_p, c_void_p]),
    "dr_dc_fd_build": (c_int, [c_void_p, _PP, POINTER(c_int64), c_int, c_void_p, c_int64, c_int64, c_void_p,
                               c_void_p, c_void_p]),
    "dr_dc_fd_flag": (c_int, [c_void_p, _PP, POINTER(c_int64), c_int, c_int64, c_int64, c_void_p, c_void_p,
                              c_void_p, c_void_p]),
    "dr_dc_hash_build": (c_int, [c_void_p, _PP, POINTER(c_int64), c_int, c_void_p, c_int64, c_int64, c_void_p,
                                 c_void_p, c_void_p, c_void_p]),
    "dr_dc_hash_flag": (c_int, [c_void_p, _PP, POINTER(c_int64), c_int, c_void_p, c_int, c_int64, c_int64, c_void_p,
                                c_void_p, c_void_p, c_void_p, c_void_p]),
    "dr_dc_lt_flag": (c_int, [c_void_p, _PP, POINTER(c_int64), c_int, c_void_p, c_int64, c_int64, c_void_p,
                              c_void_p, c_void_p]),
    "dr_bitmap_or": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_void_p]),
    "dr_bitmap_andnot": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_void_p]),
    "dr_bitmap_count": (c_int, [c_void_p, c_void_p, c_int64, POINTER(c_int64), c_void_p]),
    "dr_bitmap_count_many": (c_int, [c_void_p, _PP, c_int, c_int64, POINTER(c_int64), c_void_p]),
    "dr_bitmap_to_rows_async": (c_int, [c_void_p, c_void_p, c_int64, c_void_p, c_int64, c_void_p]),
    "dr_bitmaps_to_rows_many": (c_int, [c_void_p, _PP, c_int, c_int64, _PP, POINTER(c_int64), c_void_p]),
    "dr_bitmap_to_rows": (c_int, [c_void_p, c_void_p, c_int64, c_void_p, c_int64, POINTER(c_int64), c_void_p]),
    "dr_bitmap_rows_after_count": (c_int, [c_void_p, c_void_p, c_int64, c_void_p, c_int64, c_void_p]),
    "dr_tile_null_bitmaps": (c_int, [c_void_p, c_void_p, c_int64, c_int, c_int64, c_void_p, c_void_p]),
    "dr_changed_bitmap": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_void_p]),
    "dr_bitmap_gather": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_void_p]),
    "dr_bitmap_clear_rows": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_void_p]),
    "dr_discretize": (c_int, [c_void_p, c_void_p, c_int64, c_double, c_double, c_int32, c_void_p, c_void_p]),
    "dr_pair_presence": (c_int, [c_void_p, _PP, POINTER(c_int32), c_int, POINTER(c_int32), POINTER(c_int32), c_int,
                                 POINTER(c_int64), c_int64, c_int64, c_int64, c_void_p, c_void_p]),
    "dr_cooc": (c_int, [c_void_p, _PP, POINTER(c_int32), c_int, POINTER(c_int32), POINTER(c_int32), c_int,
                        POINTER(c_int64), c_int64, c_void_p, c_void_p]),
    "dr_domain_score": (c_int, [c_void_p, c_void_p, c_int64, c_void_p, c_int32, _PP, POINTER(c_int32), _PP, c_int,
                                c_void_p, POINTER(c_int64), c_int64, c_double, c_void_p, c_void_p, c_void_p,
                                c_void_p]),
    "dr_domain_prune": (c_int, [c_void_p, POINTER(dr_domain_target), c_int, c_int64, c_int64, c_double, c_void_p,
                                c_void_p]),
    "dr_gather_rows_masked": (c_int, [c_void_p, _PP, _PP, c_int, c_void_p, c_int64, c_void_p, c_void_p]),
    "dr_gather_rows_masked_f64": (c_int, [c_void_p, _PP, _PP, c_int, c_void_p, c_int64, c_void_p, c_void_p]),
    "dr_gather_rows_masked_nulls": (c_int, [c_void_p, _PP, _PP, c_int, c_void_p, c_int64, c_void_p, c_void_p,
                                            c_int64, c_void_p]),
    "dr_tile_null_bitmap": (c_int, [c_void_p, c_void_p, c_int64, c_int, c_int, c_void_p, c_void_p]),
    "dr_tile_null_bitmap_f64": (c_int, [c_void_p, c_void_p, c_int64, c_int, c_int, c_void_p, c_void_p]),
    "dr_gather_i32": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_void_p]),
    "dr_gather_f64": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_void_p]),
    "dr_tile_gather_i32": (c_int, [c_void_p, c_void_p, c_int, c_int, c_void_p, c_int64, c_void_p, c_void_p]),
    "dr_tile_gather_f64": (c_int, [c_void_p, c_void_p, c_int, c_int, c_void_p, c_int64, c_void_p, c_void_p]),
    "dr_lookup_sorted": (c_int, [c_void_p, c_void_p, c_int64, c_void_p, c_int64, c_void_p, c_void_p]),
    "dr_forest_predict": (c_int, [c_void_p, POINTER(dr_forest), c_void_p, c_int, c_void_p, c_int, c_void_p, c_int64,
                                  c_int, c_void_p, c_void_p]),
    "dr_cooc_skip": (c_int, [c_void_p, _PP, POINTER(c_int32), c_int, POINTER(c_int32), POINTER(c_int32), c_int,
                             POINTER(c_int64), c_int64, c_void_p, POINTER(c_int64), c_void_p, c_void_p]),
    "dr_key_presence": (c_int, [c_void_p, _PP, POINTER(c_int64), c_int, c_int64, c_int64, c_void_p, c_void_p]),
    "dr_key_flag": (c_int, [c_void_p, _PP, POINTER(c_int64), c_int, c_int64, c_int64, c_void_p, c_void_p, c_void_p]),
    "dr_dc_exists": (c_int, [c_void_p, _PP, _PP, POINTER(c_int32), c_int, c_int64, c_void_p, c_void_p, c_void_p,
                             c_void_p]),
    "dr_combine_counts": (c_int, [c_void_p, c_void_p, c_int, c_int64, POINTER(c_int64), POINTER(c_int32), c_int,
                                  c_void_p, c_void_p]),
    "dr_forest_predict_ranked": (c_int, [c_void_p, POINTER(dr_forest_ranked), c_void_p, c_int, c_void_p, c_int64,
                                         c_int, c_void_p, c_void_p]),
    "dr_gbdt_workspace_bytes": (c_int64, [c_int32, c_int32]),
    "dr_gbdt_train": (c_int, [c_void_p, POINTER(dr_gbdt_params), c_void_p, POINTER(c_int32), c_void_p, c_void_p,
                              c_void_p, POINTER(c_double), c_void_p, c_int64, c_void_p, c_void_p, c_void_p]),
    "dr_tile_fill_i32": (c_int, [c_void_p, c_void_p, c_int, c_int, c_void_p, c_int64, c_int32, c_void_p]),
    "dr_scatter_i32": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_void_p]),
    "dr_scatter_f64": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_void_p]),
    "dr_fd_map_build": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int32, c_void_p,
                                c_void_p, c_void_p]),
    "dr_tile_lut_fill": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_int64, c_void_p, c_int32,
                                 c_void_p]),
}

EXPORTED_SYMBOLS = tuple(sorted(_SIGNATURES))

_lib = None


def load_library():
    """dlopen the in-tree shared library and bind every entry point; raises if it is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise NativeError(
            "{} not found next to {} -- build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(there is no CPU fallback)".format(LIB_NAME, __file__))
    lib = ctypes.CDLL(LIB_PATH)
    for name, (restype, argtypes) in _SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the symbol is not exported
        fn.restype = restype
        fn.argtypes = argtypes
    _lib = lib
    return lib


def _ptr_array(ptrs):
    arr = (c_void_p * max(len(ptrs), 1))()
    for i, p in enumerate(ptrs):
        arr[i] = p
    return ctypes.cast(arr, _PP), arr


def _i32_array(vals):
    return (c_int32 * max(len(vals), 1))(*[int(v) for v in vals])


def _i64_array(vals):
    return (c_int64 * max(len(vals), 1))(*[int(v) for v in vals])


def _dp(t):
    """device pointer of a torch tensor (None -> NULL)."""
    return None if t is None else c_void_p(t.data_ptr())


class Context:
    """One ``dr_ctx`` (one GPU).  Methods take torch CUDA tensors purely as device-buffer carriers."""

    def __init__(self, device_index):
        import torch
        self.profile = None  # set to [] to collect (name, start_event, end_event) per C-ABI call
        if not torch.cuda.is_available():
            raise NativeError("no CUDA device is available; the repair engine has no CPU fallback")
        self.lib = load_library()
        self.device_index = int(device_index)
        self._h = c_void_p()
        rc = self.lib.dr_ctx_create(self.device_index, byref(self._h))
        if rc != 0:
            msg = self.lib.dr_last_error(self._h).decode() if self._h else "dr_ctx_create failed"
            raise NativeError(msg)

    def close(self):
        if getattr(self, "_h", None):
            self.lib.dr_ctx_destroy(self._h)
            self._h = None

    # One pooled context per device for the public API: a RepairModel.run() borrows it instead of creating
    # (cudaMallocHost + cudaMalloc) and destroying (cudaFree: a device synchronisation) its own, and the scratch
    # buffer it has grown stays grown for the next run.  A dr_ctx is not thread-safe: one run at a time per device.
    _pool = {}

    @classmethod
    def acquire(cls, device_index):
        ctx = cls._pool.pop(int(device_index), None)
        if ctx is None or not getattr(ctx, "_h", None):
            ctx = cls(device_index)
        ctx.profile = None
        ctx.launches_at_acquire = ctx.launch_count
        return ctx

    @classmethod
    def release(cls, ctx):
        if ctx is None or not getattr(ctx, "_h", None):
            return
        if int(ctx.device_index) in cls._pool:
            ctx.close()
        else:
            cls._pool[int(ctx.device_index)] = ctx

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc):
        if rc != 0:
            raise NativeError("libb200repair: " + self.lib.dr_last_error(self._h).decode())

    @staticmethod
    def _stream():
        import torch
        return c_void_p(torch.cuda.current_stream().cuda_stream)

    @property
    def launch_count(self):
        return int(self.lib.dr_launch_count(self._h))

    def widen_u8(self, src, n, dst):
        self._check(self.lib.dr_widen_u8(self._h, _dp(src), n, _dp(dst), self._stream()))

    # ---- Arrow ingest / egress ---------------------------------------------------------------------
    def h2d_copy(self, host_ptrs, dev_tensors_or_ptrs, nbytes, threads=0):
        """Pageable host buffers (addresses) -> device (tensors or addresses); blocks until complete."""
        sp, _k1 = _ptr_array(host_ptrs)
        dp, _k2 = _ptr_array([d if isinstance(d, int) else d.data_ptr() for d in dev_tensors_or_ptrs])
        self._check(self.lib.dr_h2d_copy(self._h, sp, dp, _i64_array(nbytes), len(host_ptrs), threads, self._stream()))

    def d2h_copy(self, dev_tensors_or_ptrs, host_ptrs, nbytes, threads=0):
        sp, _k1 = _ptr_array([d if isinstance(d, int) else d.data_ptr() for d in dev_tensors_or_ptrs])
        dp, _k2 = _ptr_array(host_ptrs)
        self._check(self.lib.dr_d2h_copy(self._h, sp, dp, _i64_array(nbytes), len(host_ptrs), threads, self._stream()))

    def index_presence(self, idx_ptr, width, validity_ptr, bit_offset, n_rows, dict_size, used):
        self._check(self.lib.dr_index_presence(self._h, c_void_p(idx_ptr), width, c_void_p(validity_ptr or 0),
                                               bit_offset, n_rows, dict_size, _dp(used), self._stream()))

    def index_remap(self, idx_ptr, width, validity_ptr, bit_offset, n_rows, lut_ptr, dict_size, dst_ptr):
        self._check(self.lib.dr_index_remap(self._h, c_void_p(idx_ptr), width, c_void_p(validity_ptr or 0), bit_offset,
                                            n_rows, c_void_p(lut_ptr), dict_size, c_void_p(dst_ptr), self._stream()))

    def ids_unique(self, ids, n):
        out = c_int()
        self._check(self.lib.dr_ids_unique_i64(self._h, _dp(ids), n, byref(out), self._stream()))
        return bool(out.value)

    def gather_i64(self, col, rows, n, out):
        self._check(self.lib.dr_gather_i64(self._h, _dp(col), _dp(rows), n, _dp(out), self._stream()))

    def valid_bits(self, codes, n, bits):
        self._check(self.lib.dr_valid_bits(self._h, _dp(codes), n, _dp(bits), self._stream()))

    # ---- detectors -------------------------------------------------------------------------------
    def scan_hist(self, cols, dom, n_rows, bitmaps, hist):
        cp, _k1 = _ptr_array([c.data_ptr() for c in cols])
        bp, _k2 = _ptr_array([0 if b is None else b.data_ptr() for b in bitmaps])
        self._check(self.lib.dr_scan_hist(self._h, cp, _i32_array(dom), len(cols), n_rows, bp, _dp(hist),
                                          self._stream()))

    def lut_scan(self, col, n_rows, lut, dict_size, bitmap):
        self._check(self.lib.dr_lut_scan(self._h, _dp(col), n_rows, _dp(lut), dict_size, _dp(bitmap), self._stream()))

    def quartiles(self, col, n_rows):
        q = (c_double * 2)()
        n = c_int64()
        self._check(self.lib.dr_quartiles(self._h, _dp(col), n_rows, q, byref(n), self._stream()))
        return float(q[0]), float(q[1]), int(n.value)

    def range_flag(self, col, n_rows, lower, upper, bitmap):
        self._check(self.lib.dr_range_flag(self._h, _dp(col), n_rows, lower, upper, _dp(bitmap), self._stream()))

    def lof_workspace_bytes(self, n):
        nbytes = int(self.lib.dr_lof_workspace_bytes(n))
        if nbytes < 0:
            raise NativeError("libb200repair: dr_lof_workspace_bytes({}) failed".format(n))
        return nbytes

    def lof_flag(self, col, n, k, row_begin, row_count, bitmap, workspace, out_lof=None, count=False):
        """Exact 1-D LOF of col[:n] (the whole column); rows in [row_begin, row_begin + row_count) with
        lof > 1.5 set bit (row - row_begin) of `bitmap`.  workspace: device uint8 tensor of at least
        lof_workspace_bytes(n) bytes.  With count=True, returns the number of flagged rows (synchronises)."""
        flagged = c_int64()
        self._check(self.lib.dr_lof_flag(self._h, _dp(col), n, k, row_begin, row_count, _dp(bitmap), _dp(out_lof),
                                         byref(flagged) if count else None, _dp(workspace), workspace.numel(),
                                         self._stream()))
        return int(flagged.value) if count else None

    def dc_const(self, cols, ops, args, n_rows, row_bitmap):
        cp, _k = _ptr_array([c.data_ptr() for c in cols])
        self._check(self.lib.dr_dc_const(self._h, cp, _i32_array(ops), _i32_array(args), len(cols), n_rows,
                                         _dp(row_bitmap), self._stream()))

    def dc_fd_build(self, key_cols, strides, b_col, n_rows, key_space, lo, hi):
        cp, _k = _ptr_array([c.data_ptr() for c in key_cols])
        self._check(self.lib.dr_dc_fd_build(self._h, cp, _i64_array(strides), len(key_cols), _dp(b_col), n_rows,
                                            key_space, _dp(lo), _dp(hi), self._stream()))

    def dc_fd_flag(self, key_cols, strides, n_rows, key_space, lo, hi, row_bitmap):
        cp, _k = _ptr_array([c.data_ptr() for c in key_cols])
        self._check(self.lib.dr_dc_fd_flag(self._h, cp, _i64_array(strides), len(key_cols), n_rows, key_space,
                                           _dp(lo), _dp(hi), _dp(row_bitmap), self._stream()))

    def dc_hash_build(self, key_cols, strides, b_col, n_rows, capacity, table_keys, lo, hi):
        cp, _k = _ptr_array([c.data_ptr() for c in key_cols])
        self._check(self.lib.dr_dc_hash_build(self._h, cp, _i64_array(strides), len(key_cols), _dp(b_col), n_rows,
                                              capacity, _dp(table_keys), _dp(lo), _dp(hi), self._stream()))

    def dc_hash_flag(self, key_cols, strides, x_col, mode, n_rows, capacity, table_keys, lo, hi, row_bitmap):
        cp, _k = _ptr_array([c.data_ptr() for c in key_cols])
        self._check(self.lib.dr_dc_hash_flag(self._h, cp, _i64_array(strides), len(key_cols), _dp(x_col), mode, n_rows,
                                             capacity, _dp(table_keys), _dp(lo), _dp(hi), _dp(row_bitmap),
                                             self._stream()))

    def dc_lt_flag(self, key_cols, strides, x_col, n_rows, key_space, hi, row_bitmap):
        cp, _k = _ptr_array([c.data_ptr() for c in key_cols])
        self._check(self.lib.dr_dc_lt_flag(self._h, cp, _i64_array(strides), len(key_cols), _dp(x_col), n_rows,
                                           key_space, _dp(hi), _dp(row_bitmap), self._stream()))

    # ---- bitmaps ---------------------------------------------------------------------------------
    def bitmap_or(self, dst, src, n_rows):
        self._check(self.lib.dr_bitmap_or(self._h, _dp(dst), _dp(src), n_rows, self._stream()))

    def bitmap_andnot(self, dst, src, n_rows):
        self._check(self.lib.dr_bitmap_andnot(self._h, _dp(dst), _dp(src), n_rows, self._stream()))

    def bitmap_count(self, bitmap, n_rows):
        n = c_int64()
        self._check(self.lib.dr_bitmap_count(self._h, _dp(bitmap), n_rows, byref(n), self._stream()))
        return int(n.value)

    def bitmap_count_many(self, bitmaps, n_rows):
        """Popcounts of several bitmaps with one host synchronisation."""
        out = []
        for i in range(0, len(bitmaps), 128):
            part = bitmaps[i:i + 128]
            bp, _keep = _ptr_array([b.data_ptr() for b in part])
            counts = (c_int64 * len(part))()
            self._check(self.lib.dr_bitmap_count_many(self._h, bp, len(part), n_rows, counts, self._stream()))
            out += [int(c) for c in counts]
        return out

    def bitmap_to_rows_async(self, bitmap, n_rows, out_rows, count):
        """Ordered compaction of a bitmap whose popcount is known: no host synchronisation."""
        self._check(self.lib.dr_bitmap_to_rows_async(self._h, _dp(bitmap), n_rows, _dp(out_rows), count,
                                                     self._stream()))

    def bitmaps_to_rows_many(self, bitmaps, n_rows, outs, counts):
        """Ordered compaction of several bitmaps with known popcounts (three launches per 128 bitmaps)."""
        for i in range(0, len(bitmaps), 128):
            bp, _k1 = _ptr_array([b.data_ptr() for b in bitmaps[i:i + 128]])
            op, _k2 = _ptr_array([o.data_ptr() if c else 0 for o, c in zip(outs[i:i + 128], counts[i:i + 128])])
            self._check(self.lib.dr_bitmaps_to_rows_many(self._h, bp, len(bitmaps[i:i + 128]), n_rows, op,
                                                         _i64_array(counts[i:i + 128]), self._stream()))

    def bitmap_to_rows(self, bitmap, n_rows, out_rows, capacity):
        n = c_int64()
        self._check(self.lib.dr_bitmap_to_rows(self._h, _dp(bitmap), n_rows, _dp(out_rows), capacity, byref(n),
                                               self._stream()))
        return int(n.value)

    def bitmap_rows_after_count(self, bitmap, n_rows, out_rows, capacity):
        self._check(self.lib.dr_bitmap_rows_after_count(self._h, _dp(bitmap), n_rows, _dp(out_rows), capacity,
                                                        self._stream()))

    def tile_null_bitmaps(self, tile, n, n_cols, words_per_col, out):
        self._check(self.lib.dr_tile_null_bitmaps(self._h, _dp(tile), n, n_cols, words_per_col, _dp(out),
                                                  self._stream()))

    def changed_bitmap(self, current, repaired, n, out):
        self._check(self.lib.dr_changed_bitmap(self._h, _dp(current), _dp(repaired), n, _dp(out), self._stream()))

    def bitmap_gather(self, src, rows, n, out):
        self._check(self.lib.dr_bitmap_gather(self._h, _dp(src), _dp(rows), n, _dp(out), self._stream()))

    def bitmap_clear_rows(self, bitmap, rows, flags, n):
        self._check(self.lib.dr_bitmap_clear_rows(self._h, _dp(bitmap), _dp(rows), _dp(flags), n, self._stream()))

    # ---- statistics ------------------------------------------------------------------------------
    def discretize(self, vals, n_rows, vmin, denom, thres, out):
        self._check(self.lib.dr_discretize(self._h, _dp(vals), n_rows, vmin, denom, thres, _dp(out), self._stream()))

    def pair_presence(self, cols, dom, px, py, bit_off, n_rows, block_rows, n_blocks, bits):
        cp, _k = _ptr_array([c.data_ptr() for c in cols])
        self._check(self.lib.dr_pair_presence(self._h, cp, _i32_array(dom), len(cols), _i32_array(px), _i32_array(py),
                                              len(px), _i64_array(bit_off), n_rows, block_rows, n_blocks, _dp(bits),
                                              self._stream()))

    def cooc(self, cols, dom, px, py, tab_off, n_rows, out):
        cp, _k = _ptr_array([c.data_ptr() for c in cols])
        self._check(self.lib.dr_cooc(self._h, cp, _i32_array(dom), len(cols), _i32_array(px), _i32_array(py), len(px),
                                     _i64_array(tab_off), n_rows, _dp(out), self._stream()))

    def cooc_skip(self, cols, dom, px, py, tab_off, n_rows, skip, skip_off, out):
        """dr_cooc with one uncounted entry per x value (skip: device int32 or None)."""
        cp, _k = _ptr_array([c.data_ptr() for c in cols])
        self._check(self.lib.dr_cooc_skip(self._h, cp, _i32_array(dom), len(cols), _i32_array(px), _i32_array(py),
                                          len(px), _i64_array(tab_off), n_rows, _dp(skip),
                                          _i64_array(skip_off) if skip is not None else None, _dp(out),
                                          self._stream()))

    def key_presence(self, cols, strides, n_rows, space, bits):
        cp, _k = _ptr_array([c.data_ptr() for c in cols])
        self._check(self.lib.dr_key_presence(self._h, cp, _i64_array(strides), len(cols), n_rows, space, _dp(bits),
                                             self._stream()))

    def key_flag(self, cols, strides, n_rows, space, viol_bits, row_bitmap):
        cp, _k = _ptr_array([c.data_ptr() for c in cols])
        self._check(self.lib.dr_key_flag(self._h, cp, _i64_array(strides), len(cols), n_rows, space, _dp(viol_bits),
                                         _dp(row_bitmap), self._stream()))

    def dc_exists(self, left, right, signs, n, group_begin, group_end, out):
        lp, _k1 = _ptr_array([c.data_ptr() for c in left])
        rp, _k2 = _ptr_array([c.data_ptr() for c in right])
        self._check(self.lib.dr_dc_exists(self._h, lp, rp, _i32_array(signs), len(signs), n, _dp(group_begin),
                                          _dp(group_end), _dp(out), self._stream()))

    def combine_counts(self, gathered, world, n, seg_off, seg_op, out):
        self._check(self.lib.dr_combine_counts(self._h, _dp(gathered), world, n, _i64_array(seg_off),
                                               _i32_array(seg_op), len(seg_op), _dp(out), self._stream()))

    def domain_score(self, rows, n_cells, target, dom_t, corr, dom_c, cooc, hist_t, tau, n_total, beta, out_top1,
                     out_prob, out_weak):
        cp, _k1 = _ptr_array([c.data_ptr() for c in corr])
        tp, _k2 = _ptr_array([c.data_ptr() for c in cooc])
        self._check(self.lib.dr_domain_score(self._h, _dp(rows), n_cells, _dp(target), dom_t, cp, _i32_array(dom_c),
                                             tp, len(corr), _dp(hist_t), _i64_array(tau), n_total, beta,
                                             _dp(out_top1), _dp(out_prob), _dp(out_weak), self._stream()))

    def domain_prune(self, targets, n_rows, n_total, beta, removed):
        """targets: [(target col, bitmap, hist_t ptr, dom_t, [(corr col, cooc ptr, dom_c, tau)])] -- pointers
        are device addresses (ints) or tensors; removed: device int64[len(targets)], accumulated."""
        arr = (dr_domain_target * max(len(targets), 1))()
        ptr = lambda x: x if isinstance(x, int) else x.data_ptr()  # noqa: E731
        for i, (tcol, bitmap, hist, dom_t, corr) in enumerate(targets):
            d = arr[i]
            d.target, d.bitmap, d.hist_t, d.dom_t, d.n_corr = ptr(tcol), ptr(bitmap), ptr(hist), dom_t, len(corr)
            for j, (ccol, cooc, dom_c, tau) in enumerate(corr):
                d.corr[j], d.cooc[j], d.dom_c[j], d.tau[j] = ptr(ccol), ptr(cooc), dom_c, tau
        self._check(self.lib.dr_domain_prune(self._h, arr, len(targets), n_rows, n_total, beta, _dp(removed),
                                             self._stream()))

    # ---- repair base / tile ----------------------------------------------------------------------
    def gather_rows_masked(self, cols, bitmaps, rows, n, out, f64=False, null_out=None):
        """null_out (int32 codes only): int32 [K][words] that receives the NULL bitmap of every tile column."""
        cp, _k1 = _ptr_array([c.data_ptr() for c in cols])
        bp, _k2 = _ptr_array([0 if b is None else b.data_ptr() for b in bitmaps])
        if null_out is not None:
            assert not f64
            self._check(self.lib.dr_gather_rows_masked_nulls(self._h, cp, bp, len(cols), _dp(rows), n, _dp(out),
                                                             _dp(null_out), int(null_out.shape[1]), self._stream()))
            return
        fn = self.lib.dr_gather_rows_masked_f64 if f64 else self.lib.dr_gather_rows_masked
        self._check(fn(self._h, cp, bp, len(cols), _dp(rows), n, _dp(out), self._stream()))

    def tile_null_bitmap(self, tile, n, n_cols, col, out, f64=False):
        fn = self.lib.dr_tile_null_bitmap_f64 if f64 else self.lib.dr_tile_null_bitmap
        self._check(fn(self._h, _dp(tile), n, n_cols, col, _dp(out), self._stream()))

    def gather(self, col, rows, n, out, f64=False):
        fn = self.lib.dr_gather_f64 if f64 else self.lib.dr_gather_i32
        self._check(fn(self._h, _dp(col), _dp(rows), n, _dp(out), self._stream()))

    def tile_gather(self, tile, n_cols, col, drows, n, out, f64=False):
        fn = self.lib.dr_tile_gather_f64 if f64 else self.lib.dr_tile_gather_i32
        self._check(fn(self._h, _dp(tile), n_cols, col, _dp(drows), n, _dp(out), self._stream()))

    def lookup_sorted(self, sorted_rows, n_sorted, keys, n, out):
        self._check(self.lib.dr_lookup_sorted(self._h, _dp(sorted_rows), n_sorted, _dp(keys), n, _dp(out),
                                              self._stream()))

    def forest_predict(self, forest_struct, tile, n_cols, ctile, n_ccols, cells, n_cells, target_col, out_margin=None):
        self._check(self.lib.dr_forest_predict(self._h, byref(forest_struct), _dp(tile), n_cols, _dp(ctile), n_ccols,
                                               _dp(cells), n_cells, target_col, _dp(out_margin), self._stream()))

    def forest_predict_ranked(self, forest_struct, tile, n_cols, cells, n_cells, target_col, out_margin=None):
        self._check(self.lib.dr_forest_predict_ranked(self._h, byref(forest_struct), _dp(tile), n_cols, _dp(cells),
                                                      n_cells, target_col, _dp(out_margin), self._stream()))

    def gbdt_train(self, params, bins, n_bins, y_class, y_value, weight, init, workspace, out_nodes, out_counts):
        self._check(self.lib.dr_gbdt_train(
            self._h, byref(params), _dp(bins), _i32_array(n_bins), _dp(y_class), _dp(y_value), _dp(weight),
            (c_double * len(init))(*[float(v) for v in init]), _dp(workspace), workspace.numel(), _dp(out_nodes),
            _dp(out_counts), self._stream()))

    def gbdt_workspace_bytes(self, n_rows, n_seq):
        return int(self.lib.dr_gbdt_workspace_bytes(n_rows, n_seq))

    def tile_fill(self, tile, n_cols, col, cells, n_cells, value):
        self._check(self.lib.dr_tile_fill_i32(self._h, _dp(tile), n_cols, col, _dp(cells), n_cells, value,
                                              self._stream()))

    def scatter(self, col, rows, vals, n, f64=False):
        fn = self.lib.dr_scatter_f64 if f64 else self.lib.dr_scatter_i32
        self._check(fn(self._h, _dp(col), _dp(rows), _dp(vals), n, self._stream()))

    def fd_map_build(self, x_col, x_mask, y_col, y_mask, n_rows, dom_x, lo, hi):
        self._check(self.lib.dr_fd_map_build(self._h, _dp(x_col), _dp(x_mask), _dp(y_col), _dp(y_mask), n_rows,
                                             dom_x, _dp(lo), _dp(hi), self._stream()))

    def tile_lut_fill(self, tile, n_cols, x_col, y_col, cells, n_cells, lut, lut_size):
        self._check(self.lib.dr_tile_lut_fill(self._h, _dp(tile), n_cols, x_col, y_col, _dp(cells), n_cells,
                                              _dp(lut), lut_size, self._stream()))


def _profiled(name, fn):
    def wrapper(self, *args, **kwargs):
        if self.profile is None:
            return fn(self, *args, **kwargs)
        import torch
        start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        start.record()
        try:
            return fn(self, *args, **kwargs)
        finally:
            end.record()
            self.profile.append((name, start, end))
    wrapper.__name__ = name
    return wrapper


for _name in ("widen_u8", "h2d_copy", "d2h_copy", "index_presence", "index_remap", "ids_unique", "gather_i64", "valid_bits",
              "scan_hist", "lut_scan", "quartiles", "range_flag", "lof_flag", "dc_const", "dc_fd_build", "dc_fd_flag", "bitmap_or",
              "bitmap_andnot", "bitmap_count", "bitmap_count_many", "bitmap_to_rows_async", "bitmaps_to_rows_many", "bitmap_to_rows", "bitmap_rows_after_count", "tile_null_bitmaps", "changed_bitmap", "bitmap_gather", "bitmap_clear_rows", "discretize",
              "pair_presence", "cooc", "cooc_skip", "key_presence", "key_flag", "dc_exists", "combine_counts", "dc_lt_flag",
              "dc_hash_build", "dc_hash_flag", "domain_score", "domain_prune", "gather_rows_masked", "tile_null_bitmap", "gather",
              "tile_gather", "lookup_sorted", "forest_predict", "forest_predict_ranked", "tile_fill", "gbdt_train"):
    setattr(Context, _name, _profiled(_name, getattr(Context, _name)))


def profile_summary(ctx):
    """{call name: (count, total milliseconds)} of the calls recorded while ctx.profile was a list
    (CUDA events on the launching stream)."""
    import torch
    torch.cuda.synchronize()
    out = {}
    for name, start, end in ctx.profile or []:
        c, t = out.get(name, (0, 0.0))
        out[name] = (c + 1, t + start.elapsed_time(end))
    return out
