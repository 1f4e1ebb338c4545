"""ctypes binding of libgnm.so (the C ABI declared in include/gnm.h).

The library is built in-tree (`graph_neural_mapping_b200/csrc/libgnm.so`, see
`__graft_entry__.build()` / `csrc/Makefile`). There is no CPU fallback: if the shared
object is missing or lacks a symbol, loading raises.
"""
import ctypes
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(_HERE, "csrc")
LIB_PATH = os.path.join(CSRC, "libgnm.so")
ABI_VERSION = 27

_c_i32 = ctypes.c_int
_c_i64 = ctypes.c_int64
_c_f32 = ctypes.c_float
_c_f64 = ctypes.c_double
_p = ctypes.c_void_p

# name -> argument ctypes, in the order of include/gnm.h
SIGNATURES = {
    "gnm_abi_version": [],
    "gnm_set_device": [_c_i32],
    "gnm_device_info": [_p, _p, _p, _p],
    "gnm_launch_counts": [_p, _c_i32],
    "gnm_set_pdl": [_c_i32],
    "gnm_stream_capture_status": [_p, _p],
    "gnm_csr_build": [_p, _c_i64, _p, _p, _c_i32, _c_i32, _c_i32, _c_i32, _p, _p, _p, _p],
    "gnm_csr_batch_gather": [_p, _p, _p, _p, _p, _c_i32, _p, _p, _p, _p],
    "gnm_aggregate": [_p, _p, _c_i32, _p, _c_i64, _p, _p, _c_i64, _c_i32, _c_i32, _p, _p, _p],
    "gnm_bitmap_build": [_p, _p, _p, _p, _c_i32, _p, _p, _p],
    "gnm_aggregate_dense": [_p, _p, _p, _c_i32, _c_i32, _p, _c_i64, _p, _p, _c_i64, _c_i32, _c_i32, _p, _p, _c_i32, _p, _p,
                            _p, _c_i64, _p, _p],
    "gnm_aggregate_dense_table": [_p, _p, _p, _c_i32, _c_i32, _p, _c_i64, _p, _p, _c_i64, _c_i32, _c_i32, _p, _p, _p, _p, _p],
    "gnm_aggregate_tc_status": [_p],
    "gnm_aggregate_tc_set_debug": [_p],
    "gnm_dot_rows": [_p, _c_i64, _p, _c_i64, _p, _c_i32, _c_i32, _p, _p],
    "gnm_scatter_rows_add": [_p, _c_i64, _p, _c_i32, _c_i32, _p, _c_i64, _c_i32, _p, _c_i64, _p],
    "gnm_scatter_rows_workspace": [_c_i32, _c_i32, _c_i32],
    "gnm_rows_period_sum": [_p, _c_i64, _c_i32, _c_i32, _c_i32, _p, _p, _c_i64, _c_i32, _p, _c_i64, _p],
    "gnm_rows_period_workspace": [_c_i32, _c_i32, _c_i32],
    "gnm_linear": [_p, _c_i64, _c_i32, _c_i32, _p, _c_i64, _c_i32, _p, _p, _p, _p, _c_i64, _c_i32, _p, _p, _p],
    "gnm_set_linear_impl": [_c_i32],
    "gnm_linear_wgrad": [_p, _c_i64, _p, _c_i64, _c_i32, _c_i32, _c_i32, _p, _p, _p, _c_i64, _p, _p],
    "gnm_bn_bwd_coeffs": [_p, _c_f64, _p, _p, _p, _p, _c_i32, _p, _p],
    "gnm_linear_bwd": [_p, _c_i64, _p, _c_i64, _p, _p, _c_i64, _p, _p, _p, _p, _p, _c_i64, _p, _c_i64, _p, _p, _c_i64,
                       _p, _c_i32, _c_i32, _c_i32, _p, _p],
    "gnm_col_stats": [_p, _c_i64, _c_i32, _c_i32, _p, _p],
    "gnm_bn_finalize": [_p, _c_f64, _p, _p, _c_f32, _c_f32, _p, _p, _p, _p, _p, _p, _p, _c_i32, _p, _p],
    "gnm_aggregate_dense_affine": [_p, _p, _p, _c_i32, _c_i32, _p, _c_i64, _p, _c_i64, _p, _p, _c_i64, _c_i32, _c_i32, _p],
    "gnm_aggregate_dense_relu_bn_bwd": [_p, _p, _p, _c_i32, _c_i32, _p, _c_i64, _c_i32, _c_i32, _p, _p, _c_i64, _p, _p, _p, _p,
                                        _p, _c_i64, _p, _p, _p, _c_i64, _p, _c_i64, _c_i32, _p, _c_i64, _p, _p, _p],
    "gnm_col_min": [_p, _c_i64, _c_i32, _c_i32, _p, _p],
    "gnm_aggregate_max": [_p, _p, _c_i32, _p, _c_i64, _c_i32, _p, _p, _p, _c_i64, _p, _p],
    "gnm_aggregate_max_bwd": [_p, _p, _c_i32, _p, _c_i64, _c_i32, _p, _p, _p, _p, _c_i64, _p],
    "gnm_p2p_buffer_bytes": [],
    "gnm_p2p_alloc": [_p, _p],
    "gnm_p2p_alloc_bytes": [_p, _p, _c_i64],
    "gnm_p2p_push": [_p, _c_i64, _p, _c_i32, _c_i64, _p],
    "gnm_sum_slots": [_p, _c_i32, _c_i64, _c_i64, _c_f32, _p, _p],
    "gnm_scatter_scaled_rows": [_p, _p, _p, _c_i64, _c_i32, _c_i32, _p, _c_i64, _c_i32, _p],
    "gnm_p2p_open": [_p, _p],
    "gnm_p2p_close": [_p, _c_i32],
    "gnm_p2p_allreduce": [_p, _c_i32, _p, _p],
    "gnm_p2p_status": [_p],
    "gnm_bn_eval_affine": [_p, _p, _p, _p, _c_f32, _p, _p, _p, _p, _c_i32, _p],
    "gnm_bn_relu_readout": [_p, _c_i64, _c_i32, _c_i32, _p, _p, _p, _c_i64, _p, _c_i32, _p, _p, _c_i64, _p],
    "gnm_relu_bn_bwd_reduce": [_p, _c_i64, _c_i32, _c_i32, _p, _p, _p, _p, _p, _c_i64, _p, _c_i64, _p, _p, _p,
                               _c_i64, _p, _c_i64, _c_i32, _p, _c_i32, _p, _c_i64, _p, _p, _p],
    "gnm_bn_bwd_apply": [_p, _c_i64, _c_i32, _c_i32, _p, _p, _p, _p, _c_f64, _p, _c_i64, _p],
    "gnm_gather_nf_rows": [_p, _c_i64, _c_i32, _c_i32, _c_i64, _c_i32, _p, _c_i64, _p, _p],
    "gnm_dgi_score_fwd": [_p, _c_i64, _c_i32, _c_i32, _c_i64, _c_i32, _p, _p, _p, _p, _c_i32, _p, _p, _c_i64, _p, _p],
    "gnm_dgi_score_bwd": [_p, _c_i64, _c_i32, _c_i32, _c_i64, _c_i32, _p, _p, _p, _p, _c_i32, _p, _c_i64, _p, _p, _p, _p],
    "gnm_dgi_score_train": [_p, _c_i64, _c_i32, _c_i32, _c_i64, _c_i32, _p, _p, _p, _p, _c_i32, _p, _p, _c_i64, _c_f32, _c_f64,
                            _p, _p, _p, _p, _p, _p, _p],
    "gnm_heads_ce_workspace": [_c_i32, _c_i32, _c_i32, _c_i32],
    "gnm_heads_ce": [_p, _c_i64, _c_i32, _c_i32, _c_i32, _c_i32, _p, _p, _p, _p, _c_f32, _p, _p, _p, _c_i64, _p, _p, _p,
                     _c_i64, _p, _p],
    "gnm_heads_fwd": [_p, _c_i64, _c_i32, _c_i32, _c_i32, _c_i32, _p, _p, _p, _p, _p],
    "gnm_heads_bwd": [_p, _c_i64, _c_i32, _c_i32, _c_i32, _c_i32, _p, _p, _p, _p, _c_i64, _p, _p, _p, _c_i64, _p, _p],
    "gnm_bce_logits": [_p, _c_i64, _c_i64, _c_f32, _c_f64, _p, _p, _p],
    "gnm_small_gemm": [_p, _c_i64, _c_i64, _p, _c_i64, _c_i64, _p, _c_i64, _c_i32, _c_i32, _c_i32, _c_i32, _p, _c_i64, _p,
                       _c_i64, _p, _c_i64, _p],
    "gnm_dgi_neg_grad": [_p, _p, _p, _c_i64, _c_i32, _c_i32, _p, _c_i64, _c_i32, _p],
    "gnm_adam_step": [_p, _p, _p, _p, _c_i32, _p, _p, _p, _p, _c_f64, _c_f64, _c_f32, _c_f32, _c_f32, _p, _c_i32, _p, _p],
    "gnm_rowdot_score": [_p, _c_i64, _c_i32, _c_i32, _p, _c_i64, _c_i32, _p, _p, _p, _p],
    "gnm_segment_weighted_colsum": [_p, _c_i64, _p, _c_i64, _p, _p, _c_i32, _c_i32, _p, _c_i32, _p, _p, _c_i64, _p],
    "gnm_ig_expand": [_p, _c_i64, _p, _p, _p, _c_i32, _c_i32, _c_i32, _c_i32, _p, _c_i64, _p],
    "gnm_ig_accumulate": [_p, _c_i64, _p, _p, _c_i32, _c_i32, _c_i32, _c_i32, _c_f32, _c_i32, _p, _c_i64, _p],
    "gnm_ig_attribute": [_p, _c_i64, _p, _c_i64, _c_i32, _p, _p, _c_i32, _c_i32, _p, _c_i64, _p],
    "gnm_occlusion_expand": [_p, _c_i64, _p, _p, _c_i64, _c_i32, _p, _p, _p, _p, _c_i32, _c_i32, _p, _p, _p, _c_i32,
                             _c_i32, _c_i32, _p, _p, _c_i64, _p],
}

_lib = None


def build(verbose=False):
    """Compile libgnm.so for sm_100a with nvcc (cross-compiles without a GPU)."""
    res = subprocess.run(["make", "-C", CSRC, "-j4"], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if verbose or res.returncode != 0:
        print(res.stdout)
    if res.returncode != 0:
        raise RuntimeError("building libgnm.so failed (make -C %s)" % CSRC)
    return LIB_PATH


def load():
    """Load libgnm.so and bind every entry point; raises if anything is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            "libgnm.so not found at %s: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "or `make -C graph_neural_mapping_b200/csrc`. There is no CPU fallback." % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    for name, argtypes in SIGNATURES.items():
        fn = getattr(lib, name)        # AttributeError if the symbol is missing
        fn.argtypes = argtypes
        fn.restype = ctypes.c_int
    lib.gnm_scatter_rows_workspace.restype = ctypes.c_int64
    lib.gnm_rows_period_workspace.restype = ctypes.c_int64
    lib.gnm_p2p_buffer_bytes.restype = ctypes.c_int64
    lib.gnm_error_string.argtypes = [ctypes.c_int]
    lib.gnm_error_string.restype = ctypes.c_char_p
    got = lib.gnm_abi_version()
    if got != ABI_VERSION:
        raise RuntimeError("libgnm.so ABI version %d, expected %d: rebuild it" % (got, ABI_VERSION))
    _lib = lib
    return lib


def check(code, what):
    if code != 0:
        msg = load().gnm_error_string(code).decode()
        raise RuntimeError("%s failed: %s (code %d)" % (what, msg, code))
