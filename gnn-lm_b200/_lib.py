"""ctypes binding of libgnnlm_sm100.so (include/gnnlm_sm100.h).  No fallback: if the library is
missing or a call fails, raise."""
import ctypes as C
import os

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libgnnlm_sm100.so")

F32, BF16, F16, F16X2, F24 = 0, 1, 2, 3, 4
MATH_FP32_SIMT, MATH_TF32X3, MATH_TF32, MATH_BF16, MATH_F16X3 = 0, 1, 2, 3, 4
# host-level mode: MATH_F16X3 everywhere, except that products whose activation operand carries an e4m3 companion (ops.Split.q8)
# run gnnlm_linear_f16f8 (fp16 main product + FP8 correction MMAs: two tensor-pass equivalents instead of three)
MATH_F16F8 = 5
MATH_NAMES = {"fp32": MATH_FP32_SIMT, "tf32x3": MATH_TF32X3, "tf32": MATH_TF32, "bf16": MATH_BF16, "f16x3": MATH_F16X3,
              "f16f8": MATH_F16F8}


def base_math(mode: int) -> int:
    """The `math` argument of the C ABI for a host-level mode."""
    return MATH_F16X3 if mode == MATH_F16F8 else mode

_p, _i64, _i32, _f32 = C.c_void_p, C.c_int64, C.c_int32, C.c_float

# name -> (restype, argtypes): must list every symbol include/gnnlm_sm100.h declares
SIGNATURES = {
    "gnnlm_version": (_i32, []),
    "gnnlm_last_error": (C.c_char_p, []),
    "gnnlm_has_tcgen05": (_i32, []),
    "gnnlm_host_copy": (_i32, [_p, _p, _i64, _i32, _i64, _i64, _i32, _p]),
    "gnnlm_graph_workspace_bytes": (_i64, [_i64]),
    "gnnlm_graph_count": (_i32, [_p, _p, _i64, _i64, _i64, _i32, _i32, _i64, _p, _p, _p, _i64, _p]),
    "gnnlm_graph_fill": (_i32, [_p, _p, _i64, _i64, _i64, _i32, _i32, _i64, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p]),
    "gnnlm_graph_tt_num_edges": (_i64, [_i64, _i64, _i64]),
    "gnnlm_graph_tt_csr": (_i32, [_i64, _i64, _i64, _p, _p, _p]),
    "gnnlm_graph_dedup_workspace_bytes": (_i64, [_i64, _i64, _i32]),
    "gnnlm_graph_dedup": (_i32, [_p, _p, _i64, _i64, _i64, _i64, _i32, _i32, _i64, _p, _p, _p, _p, _p, _p, _p, _p, _i64, _p]),
    "gnnlm_unique_workspace_bytes": (_i64, [_i64]),
    "gnnlm_unique_centres": (_i32, [_p, _p, _i64, _p, _p, _p, _p, _i64, _p]),
    "gnnlm_pq_gather_decode": (_i32, [_p, _i64, _i32, _p, _i32, _p, _p, _p, _i64, _p, _p, _i32, _i64, _p, _i32, _p, _p, _p]),
    "gnnlm_pq_gather_decode_presplit": (_i32, [_p, _i64, _i32, _p, _p, _i32, _p, _p, _i64, _p, _p, _i64, _p]),
    "gnnlm_pq_gather_decode_presplit_q8": (_i32, [_p, _i64, _i32, _p, _p, _i32, _p, _p, _i64, _p, _p, _i64, _p, _i64, _p]),
    "gnnlm_pq_gather_decode_hiq8": (_i32, [_p, _i64, _i32, _p, _p, _i32, _p, _p, _i64, _p, _p, _i64, _p, _i64, _p]),
    "gnnlm_pq_encode": (_i32, [_p, _i64, _i64, _i32, _i32, _p, _p, _p, _p]),
    "gnnlm_split_tf32": (_i32, [_p, _p, _p, _i64, _p]),
    "gnnlm_split_f16": (_i32, [_p, _f32, _p, _p, _i64, _p]),
    "gnnlm_linear": (_i32, [_p, _i32, _i64, _p, _p, _f32, _i64, _p, _p, _i32, _i64, _p, _i32, _i64, _i64, _p, _i64, _i64, _i32, _p]),
    "gnnlm_linear_batched_f16x3": (_i32, [_p, _i64, _i64, _p, _p, _i64, _i64, _f32, _p, _i64, _i64, _p, _i64, _i64, _i64, _i64,
                                          _i64, _i64, _i32, _p]),
    "gnnlm_split_to_q8": (_i32, [_p, _i64, _p, _i64, _i64, _p, _i64, _p]),
    "gnnlm_quant_w8": (_i32, [_p, _p, _i64, _p, _i64, _i64, _i64, _p]),
    "gnnlm_linear_f16f8": (_i32, [_p, _p, _i64, _i64, _i64, _p, _p, _i64, _i64, _i64, _p, _p, _f32, _i64, _i64, _p, _p, _i32, _i64,
                                  _i64, _p, _i64, _p, _p]),
    "gnnlm_lse_num_tiles": (_i64, [_i64, _i32]),
    "gnnlm_linear_lse": (_i32, [_p, _i32, _i64, _p, _p, _f32, _i64, _p, _p, _p, _p, _i64, _p, _i64, _i64, _i32, _p]),
    "gnnlm_lse_finish": (_i32, [_p, _p, _p, _i64, _p, _p, _i32, _i64, _p, _p]),
    "gnnlm_gather_rows": (_i32, [_p, _i64, _p, _p, _i64, _i64, _p, _i64, _i32, _p]),
    "gnnlm_embed_gather": (_i32, [_p, _i64, _i64, _p, _i32, _i64, _p, _p, _p, _i64, _i64, _p, _i64, _p, _p, _p]),
    "gnnlm_layernorm": (_i32, [_p, _i64, _p, _i32, _i64, _p, _p, _f32, _p, _i32, _i64, _i64, _p, _i64, _p]),
    "gnnlm_layernorm_q8": (_i32, [_p, _i64, _p, _i32, _i64, _p, _p, _f32, _p, _i32, _i64, _p, _i64, _i64, _p, _i64, _p]),
    "gnnlm_convert": (_i32, [_p, _i32, _p, _i32, _i64, _p]),
    "gnnlm_gelu": (_i32, [_p, _i64, _p, _i32, _i64, _i64, _p, _i64, _p]),
    "gnnlm_to_split_f16": (_i32, [_p, _i32, _i64, _p, _i64, _i64, _p, _i64, _p]),
    "gnnlm_hgt_edge_attn": (_i32, [_p, _i64, _p, _i64, _p, _i64, _i32, _p, _p, _p, _i64, _p, _i32, _i32, _p, _i64, _f32, _i32, _p]),
    "gnnlm_hgt_cluster_attn": (_i32, [_p, _i64, _p, _i64, _p, _i64, _i32, _p, _p, _p, _i64, _i32, _i32, _i32, _i32, _p, _i32, _i64, _p]),
    "gnnlm_hgt_cluster_attn_q8": (_i32, [_p, _i64, _p, _i64, _p, _i64, _i32, _p, _p, _p, _i64, _i32, _i32, _i32, _i32, _p, _i32, _i64,
                                         _p, _i64, _i32, _p]),
    "gnnlm_hgt_cluster_attn_hq": (_i32, [_p, _p, _i64, _p, _p, _i64, _p, _p, _i64, _p, _p, _p, _i64, _i32, _i32, _i32, _i32, _p, _i64, _p, _i64,
                                         _i32, _p, _p, _p, _p, _p, _p]),
    "gnnlm_rowstats_q8": (_i32, [_p, _i64, _p, _i64, _p, _i64, _p, _f32, _p, _i64, _p, _i64, _p, _i64, _p, _i64, _p]),
    "gnnlm_hgt_causal_attn": (_i32, [_p, _i64, _p, _i64, _p, _i64, _i32, _i64, _i64, _i64, _i32, _i32, _p, _i64, _f32, _i32, _p]),
    "gnnlm_hgt_causal_flash": (_i32, [_p, _i64, _p, _p, _i64, _i64, _i64, _i64, _i64, _i32, _i32, _p, _i64, _p, _i64, _i64, _f32, _i32, _p]),
    "gnnlm_hgt_causal_flash_tc": (_i32, [_p, _i64, _i64, _p, _i64, _i64, _i64, _i64, _i32, _i32, _p, _i64, _p, _i64, _i64, _f32, _i32, _p]),
    "gnnlm_hgt_inter_fused": (_i32, [_p, _i64, _p, _i32, _i64, _p, _i64, _i64, _i32, _i64, _p, _i64, _i64, _p, _f32, _p, _i64, _p]),
    "gnnlm_heads_split_f16": (_i32, [_p, _i64, _i64, _i32, _i32, _i32, _p, _p, _p]),
    "gnnlm_heads_transpose_split_f16": (_i32, [_p, _i64, _i64, _i32, _i32, _p, _p, _p]),
    "gnnlm_causal_softmax_split": (_i32, [_p, _i64, _i64, _i32, _i64, _p, _p]),
    "gnnlm_adapt_target": (_i32, [_p, _i64, _p, _i32, _p, _p, _p, _p, _p]),
    "gnnlm_knn_mix_nll": (_i32, [_p, _p, _f32, _p, _p, _i64, _p, _i32, _i64, _p, _f32, _f32, _f32, _p, _i64, _p, _i64, _p, _p, _p,
                                 _p, _i64, _p]),
    "gnnlm_knn_full_prob": (_i32, [_p, _p, _i64, _p, _i32, _i64, _f32, _f32, _p, _i64, _i64, _p]),
    "gnnlm_knn_sims_keys": (_i32, [_p, _i64, _p, _i32, _i64, _i32, _p, _i64, _i32, _i32, _p, _i64, _p]),
    "gnnlm_hgt_edge_attn_bwd": (_i32, [_p, _i64, _p, _i64, _p, _i64, _p, _i64, _p, _p, _p, _i64, _p, _i64, _i64, _i32, _i32, _f32, _p, _i64,
                                       _p, _i64, _p, _i64, _f32, C.c_uint64, _p]),
    "gnnlm_hgt_edge_attn_train_fwd": (_i32, [_p, _i64, _p, _i64, _p, _i64, _p, _p, _i64, _i64, _i64, _i32, _i32, _f32, _i32, _p, _i64, _f32,
                                             C.c_uint64, _p]),
    "gnnlm_dropout_f32": (_i32, [_p, _i64, _p, _i64, _i64, _i64, _f32, C.c_uint64, _p]),
    "gnnlm_hgt_causal_attn_bwd": (_i32, [_p, _i64, _p, _i64, _p, _i64, _p, _i64, _i64, _i64, _i64, _i32, _i32, _f32, _p, _i64, _p, _i64, _p, _i64,
                                         _p, _f32, C.c_uint64, _p]),
    "gnnlm_hgt_edge_attn_bwd_sym": (_i32, [_p, _i64, _p, _i64, _p, _i64, _p, _i64, _p, _p, _i64, _i32, _i32, _f32, _p, _i64, _p, _i64, _p, _i64, _p,
                                           _f32, C.c_uint64, _p]),
    "gnnlm_hgt_cluster_attn_bwd": (_i32, [_p, _i64, _p, _i64, _p, _i64, _p, _i64, _p, _p, _i64, _i32, _i32, _f32, _p, _i64, _p, _i64, _p, _i64,
                                          _f32, C.c_uint64, _p]),
    "gnnlm_scale_split_f16": (_i32, [_p, _i64, _f32, _p, _i64, _i64, _p, _i64, _p]),
    "gnnlm_transpose_split_f16": (_i32, [_p, _i64, _i64, _i64, _f32, _i64, _i32, _p, _p, _p]),
    "gnnlm_causal_softmax_drop_split": (_i32, [_p, _i64, _i64, _i32, _i64, _i64, _f32, C.c_uint64, _p, _p]),
    "gnnlm_hgt_cluster_attn_train_fwd": (_i32, [_p, _i64, _p, _i64, _p, _i64, _p, _p, _i64, _i32, _i32, _f32, _p, _i64, _f32, C.c_uint64, _p]),
    "gnnlm_causal_softmax_bwd_split": (_i32, [_p, _p, _i64, _i64, _i32, _i64, _f32, _f32, C.c_uint64, _p, _p, _p, _p, _p]),
    "gnnlm_layernorm_bwd": (_i32, [_p, _i64, _p, _i64, _p, _f32, _p, _i64, _i64, _p, _i64, _p, _i64, _p, _p, _p]),
    "gnnlm_xent_fwd_bwd": (_i32, [_p, _i64, _p, _i64, _i64, _f32, _p, _p]),
    "gnnlm_transpose_f32": (_i32, [_p, _i64, _i64, _p, _i64, _p, _i64, _i64, _p]),
    "gnnlm_colsum_f32": (_i32, [_p, _i64, _i64, _p, _i64, _p, _p]),
    "gnnlm_axpy_f32": (_i32, [_p, _i64, _p, _i64, _i64, _p, _i64, _f32, _p]),
    "gnnlm_scatter_add_rows": (_i32, [_p, _i64, _p, _i64, _p, _i64, _p, _i64, _p]),
    "gnnlm_knn_sims_pq": (_i32, [_p, _i64, _i32, _p, _i64, _p, _i64, _i32, _i32, _p, _p, _p, _i64, _i32, _p, _i32, _p, _i64, _p]),
    "gnnlm_knn_filter_f16x3": (_i32, [_p, _i64, _i64, _i64, _p, _p, _i64, _i64, _i64, _p, _p, _p, _p, _p, _i64, _p]),
    "gnnlm_topk_merge": (_i32, [_p, _p, _i64, _i32, _p, _p, _p, _i64, _p, _p]),
    "gnnlm_knn_key_bias": (_i32, [_p, _i32, _i64, _i64, _i64, _p, _p]),
    "gnnlm_knn_key_bias_pq": (_i32, [_p, _i64, _i32, _p, _p, _p]),
}

_lib = None
launches = 0          # number of CUDA kernels launched through the C ABI (bench.py's gpu_launches)
KERNELS_PER_CALL = {"gnnlm_graph_count": 3, "gnnlm_unique_centres": 2, "gnnlm_hgt_causal_attn_bwd": 2, "gnnlm_causal_softmax_bwd_split": 2, "gnnlm_hgt_edge_attn_bwd_sym": 2, "gnnlm_knn_full_prob": 2, "gnnlm_graph_dedup": 12,   # everything else launches exactly one
                    "gnnlm_host_copy": 0}
TIMING = None         # when a list: (name, tag, start_event, end_event, work) per call (bench.py per-kernel pass)


class GnnlmError(RuntimeError):
    pass


def load():
    """Load the shared library; raises if it is absent (there is no CPU fallback)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise GnnlmError(f"{LIB_PATH} not found: run `python -c 'import __graft_entry__ as g; g.build()'` "
                         "(nvcc, sm_100a). There is no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError if the header and the library disagree
        fn.restype, fn.argtypes = res, args
    _lib = lib
    return lib


def ptr(t):
    if t is None:
        return None
    assert t.is_cuda, "device tensor required"
    return t.data_ptr()


def dtype_code(dt):
    return {torch.float32: F32, torch.bfloat16: BF16, torch.float16: F16}[dt]


def stream_ptr():
    return torch.cuda.current_stream().cuda_stream


def call(name, *args, tag=None, work=None):
    """`work`: (M_cap, N, K) of a GEMM call, recorded with its timing for the roofline of bench.py."""
    global launches
    lib = load()
    if TIMING is not None:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
    rc = getattr(lib, name)(*args)
    if rc != 0:
        raise GnnlmError(f"{name} failed ({rc}): {lib.gnnlm_last_error().decode()}")
    if TIMING is not None:
        e1.record()
        TIMING.append((name, tag, e0, e1, work))
    launches += KERNELS_PER_CALL.get(name, 1)
    return rc
