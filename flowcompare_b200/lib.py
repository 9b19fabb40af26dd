"""ctypes binding of `libflowcompare_b200.so` (the C ABI declared in include/flowcompare_b200.h).

No torch types cross this boundary: tensors are passed as raw device pointers + sizes, the stream as
the raw `cudaStream_t`.  If the library is missing the import fails loudly -- there is no fallback.
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# FLOWCOMPARE_B200_LIB: another build of the same library (kernel A/B experiments, scripts/build_variant.sh)
LIB_PATH = os.environ.get("FLOWCOMPARE_B200_LIB") or os.path.join(_HERE, "libflowcompare_b200.so")

FC_OK = 0
ERRORS = {0: "FC_OK", -1: "FC_ERR_INVALID_ARG", -2: "FC_ERR_CUDA", -3: "FC_ERR_LAUNCH",
          -4: "FC_ERR_WORKSPACE", -5: "FC_ERR_UNSUPPORTED", -6: "FC_ERR_MODEL"}

PREC_FP32 = 0
PREC_TENSOR = 1          # tcgen05 path; 3xTF32 or 3xFP16 according to the format of the packed weights
PREC_TF32X3 = 1
# engine precision name -> (precision argument of the C entry points, tensor-core weight format packed into the arena)
PRECISIONS = {"fp32": (PREC_FP32, "tf32"), "tf32x3": (PREC_TENSOR, "tf32"), "fp16x3": (PREC_TENSOR, "fp16")}

c_int, c_i64, c_f, c_vp = ctypes.c_int, ctypes.c_int64, ctypes.c_float, ctypes.c_void_p
c_u64 = ctypes.c_uint64

# name -> (restype, argtypes); must list every symbol include/flowcompare_b200.h declares
SIGNATURES = {
    "fc_version": (c_int, []),
    "fc_last_error": (ctypes.c_char_p, []),
    "fc_launch_count": (c_i64, []),
    "fc_knn_self": (c_int, [c_vp, c_int, c_int, c_int, c_int, c_int, c_vp, c_vp, c_vp]),
    "fc_knn_query": (c_int, [c_vp, c_vp, c_int, c_int, c_int, c_int, c_vp, c_vp]),
    "fc_knn_workspace_bytes": (c_i64, [c_int, c_int, c_int, c_int]),
    "fc_knn_self_ws": (c_int, [c_vp, c_int, c_int, c_int, c_int, c_int, c_vp, c_vp, c_vp, c_i64, c_vp]),
    "fc_knn_query_ws": (c_int, [c_vp, c_vp, c_int, c_int, c_int, c_int, c_vp, c_vp, c_i64, c_vp]),
    "fc_fps": (c_int, [c_vp, c_int, c_int, c_int, c_int, c_vp, c_vp, c_vp]),
    "fc_knn_heap": (c_int, [c_vp, c_vp, c_int, c_int, c_int, c_int, c_vp, c_vp, c_vp]),
    "fc_three_nn": (c_int, [c_vp, c_vp, c_int, c_int, c_int, c_vp, c_vp, c_vp]),
    "fc_three_interpolate": (c_int, [c_vp, c_int, c_int, c_vp, c_vp, c_int, c_int, c_int, c_vp, c_int, c_vp]),
    "fc_group_points": (c_int, [c_vp, c_int, c_int, c_vp, c_int, c_int, c_int, c_int, c_vp, c_int, c_vp]),
    "fc_gemm": (c_int, [c_vp, c_int, c_vp, c_int, c_vp, c_vp, c_int, c_int, c_int, c_int, c_int, c_int, c_vp]),
    "fc_gemm_tf32x3": (c_int, [c_vp, c_int, c_vp, c_vp, c_int, c_vp, c_vp, c_int, c_int, c_int, c_int, c_int, c_vp]),
    "fc_gemm_f16x3": (c_int, [c_vp, c_int, c_vp, c_vp, c_int, c_vp, c_vp, c_int, c_int, c_int, c_int, c_int, c_vp]),
    "fc_edgeconv_gather_max": (c_int, [c_vp, c_int, c_vp, c_int, c_int, c_int, c_int, c_vp, c_int, c_vp]),
    "fc_cross_attention": (c_int, [c_vp, c_int, c_vp, c_int, c_vp, c_int, c_int, c_int, c_int, c_int, c_f, c_vp]),
    "fc_cross_attention_tf32x3": (c_int, [c_vp, c_int, c_vp, c_int, c_vp, c_int, c_int, c_int, c_int, c_int, c_f, c_vp]),
    "fc_cross_attention_tc_scratch_bytes": (c_i64, [c_int, c_int]),
    "fc_cross_attention_tc": (c_int, [c_vp, c_int, c_vp, c_int, c_vp, c_int, c_int, c_int, c_int, c_int, c_f, c_vp, c_i64, c_vp]),
    "fc_cross_attention_tc_f16": (c_int, [c_vp, c_int, c_vp, c_int, c_vp, c_int, c_int, c_int, c_int, c_int, c_f, c_vp, c_i64, c_vp]),
    "fc_attention_maps": (c_int, [c_vp, c_int, c_vp, c_int, c_vp, c_int, c_vp, c_int, c_int, c_int, c_f, c_vp]),
    "fc_attention_score_grad": (c_int, [c_vp, c_int, c_vp, c_int, c_vp, c_int, c_vp, c_int, c_vp, c_int, c_vp, c_int, c_int, c_int,
                                        c_int, c_f, c_vp]),
    "fc_fps_points": (c_int, [c_vp, c_int, c_int, c_int, c_int, c_int, c_vp, c_vp, c_int, c_vp]),
    "fc_co_unit_sphere": (c_int, [c_vp, c_int, c_int, c_vp, c_int, c_int, c_int, c_vp, c_vp]),
    "fc_flow_create": (c_int, [c_vp, c_int, c_vp, c_int, c_vp, c_i64, ctypes.POINTER(c_vp)]),
    "fc_flow_destroy": (None, [c_vp]),
    "fc_flow_workspace_bytes": (c_i64, [c_vp, c_int, c_int, c_int]),
    "fc_flow_log_prob": (c_int, [c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_int, c_int, c_int, c_vp, c_i64, c_int, c_vp]),
    "fc_flow_log_prob_cif": (c_int, [c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_int, c_int, c_int, c_vp, c_i64, c_int, c_vp]),
    "fc_flow_cif_noise_dim": (c_int, [c_vp]),
    "fc_flow_log_prob_draws_workspace_bytes": (c_i64, [c_vp, c_int, c_int, c_int, c_int]),
    "fc_flow_log_prob_draws": (c_int, [c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_int, c_vp, c_int, c_int, c_int, c_vp, c_i64, c_int,
                                       c_vp]),
    "fc_logmeanexp": (c_int, [c_vp, c_int, c_i64, c_vp, c_vp]),
    "fc_rq_spline": (c_int, [c_vp, c_int, c_vp, c_int, c_int, c_int, c_int, c_vp, c_int, c_vp]),
    "fc_expm_action": (c_int, [c_vp, c_int, c_vp, c_int, c_int, c_vp, c_vp, c_int, c_int, c_vp]),
    "fc_flow_forward": (c_int, [c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_int, c_int, c_int, c_vp, c_i64, c_int, c_vp]),
    "fc_flow_attention_maps": (c_int, [c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_int, c_vp, c_int, c_vp, c_vp, c_int, c_int, c_int,
                                       c_vp, c_i64, c_int, c_vp]),
    "fc_flow_set_inverse": (c_int, [c_vp, c_vp, c_int, c_vp, c_int, c_vp, c_i64]),
    "fc_flow_sample": (c_int, [c_vp, c_vp, c_vp, c_vp, c_vp, c_int, c_int, c_int, c_vp, c_i64, c_int, c_vp]),
    "fc_flow_sample_cif": (c_int, [c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_int, c_int, c_int, c_vp, c_i64, c_int, c_vp]),
    "fc_flow_set_grad": (c_int, [c_vp, c_vp, c_int, c_vp, c_int, c_vp, c_i64]),
    "fc_flow_log_prob_grad_workspace_bytes": (c_i64, [c_vp, c_int, c_int, c_int]),
    "fc_flow_log_prob_grad": (c_int, [c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_int, c_int, c_int, c_vp, c_i64, c_int, c_vp]),
    "fc_flow_attention_score_grads": (c_int, [c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_int, c_vp, c_int, c_int, c_vp, c_vp, c_vp, c_int,
                                              c_int, c_int, c_vp, c_i64, c_int, c_vp]),
    "fc_embedder_create": (c_int, [c_vp, c_int, c_vp, c_int, c_vp, c_i64, ctypes.POINTER(c_vp)]),
    "fc_embedder_destroy": (None, [c_vp]),
    "fc_embedder_workspace_bytes": (c_i64, [c_vp, c_int, c_int]),
    "fc_embed": (c_int, [c_vp, c_vp, c_vp, c_int, c_int, c_vp, c_vp, c_i64, c_int, c_vp]),
    "fc_inner_loop_workspace_bytes": (c_i64, [c_vp, c_vp, c_int, c_int, c_int]),
    "fc_inner_loop": (c_int, [c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_int, c_int, c_int, c_vp, c_i64, c_int, c_vp]),
    "fc_inner_loop_host_workspace_bytes": (c_i64, [c_vp, c_vp, c_int, c_int, c_int]),
    "fc_inner_loop_host": (c_int, [c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_int, c_int, c_int, c_vp, c_i64, c_int, c_vp]),
    "fc_change_score": (c_int, [c_vp, c_vp, c_vp, c_int, c_int, c_f, c_int, c_f, c_vp]),
    "fc_profile_begin": (c_int, []),
    "fc_profile_end": (c_int, [c_vp, c_vp, c_vp, c_vp, c_int]),
    "fc_fill_normal": (c_int, [c_vp, c_i64, c_u64, c_u64, c_vp]),
}

_lib = None


class FlowCompareError(RuntimeError):
    pass


def load():
    """Loads the shared library (once) and declares every entry point's signature."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise FlowCompareError(
            f"{LIB_PATH} not found: build it with `make` (or `python -c 'import __graft_entry__ as g; g.build()'`). "
            "flowcompare_b200 has no CPU / PyTorch fallback.")
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the symbol is missing
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc, what=""):
    if rc != FC_OK:
        detail = load().fc_last_error().decode(errors="replace")
        raise FlowCompareError(f"{what} failed: {ERRORS.get(rc, rc)} {detail}")


def launch_count() -> int:
    return int(load().fc_launch_count())
