"""ctypes binding of libogl_b200.so (the C ABI declared in include/ogl_b200.h).

No torch types cross the boundary: tensors are passed as raw device pointers and the
current CUDA stream as a void*.  There is no CPU fallback: if the library is missing the
import fails loudly, and every entry point fails without an sm_100 device.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libogl_b200.so")

OGL_F32, OGL_BF16, OGL_TF32, OGL_FP16 = 0, 1, 2, 3


class OglError(RuntimeError):
    pass


class PlanConfig(C.Structure):
    _fields_ = [("n_layers", C.c_int), ("dims", C.c_int * 8), ("fanouts", C.c_int * 8), ("max_seeds", C.c_int),
                ("v_cap", C.c_int64), ("mode", C.c_int), ("gemm_impl", C.c_int), ("seed", C.c_uint64),
                ("lr", C.c_float), ("beta1", C.c_float), ("beta2", C.c_float), ("eps", C.c_float), ("feat_drop", C.c_float)]


def _load():
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            "ogl_b200: %s is missing. Build it with `python online-gnn-learning_b200/build.py` "
            "(nvcc, sm_100a). This package has no CPU or eager-PyTorch fallback." % LIB_PATH)
    return C.CDLL(LIB_PATH)


lib = _load()

_vp, _i, _i64, _u32, _u64, _f, _d = C.c_void_p, C.c_int, C.c_int64, C.c_uint32, C.c_uint64, C.c_float, C.c_double
_pp = C.POINTER(C.c_void_p)

# name -> (restype, argtypes); must list every symbol of include/ogl_b200.h (tests check this)
SIGNATURES = {
    "ogl_last_error": (C.c_char_p, []),
    "ogl_version": (_i, []),
    "ogl_kernel_launches": (_i64, []),
    "ogl_graph_create": (_i, [_pp, _i64, _i64]),
    "ogl_graph_destroy": (_i, [_vp]),
    "ogl_graph_insert_vertices": (_i, [_vp, _i64, _vp]),
    "ogl_graph_insert_edges": (_i, [_vp, _vp, _vp, _i64, _i, _vp]),
    "ogl_graph_set_source_bound": (_i, [_vp, _i64]),
    "ogl_graph_insert_edges_host": (_i, [_vp, _vp, _vp, _i64, _i, _vp]),
    "ogl_graph_load_parent": (_i, [_vp, _vp, _vp, _vp, _i64, _vp]),
    "ogl_graph_set_active_prefix": (_i, [_vp, _i64, _vp]),
    "ogl_graph_num_vertices": (_i, [_vp, C.POINTER(_i64)]),
    "ogl_graph_num_edges": (_i, [_vp, C.POINTER(_i64)]),
    "ogl_graph_degrees": (_i, [_vp, _vp, _vp]),
    "ogl_graph_export_csr": (_i, [_vp, _vp, _vp, _vp, _vp]),
    "ogl_graph_compact": (_i, [_vp, _vp]),
    "ogl_graph_stats": (_i, [_vp, C.POINTER(_i64 * 4)]),
    "ogl_features_create": (_i, [_pp, _i64, _i, _i]),
    "ogl_features_destroy": (_i, [_vp]),
    "ogl_features_write": (_i, [_vp, _i64, _i64, _vp, _vp, _i, _vp]),
    "ogl_features_write_permuted": (_i, [_vp, _i64, _vp, _vp, _vp, _vp]),
    "ogl_plan_create": (_i, [_pp, C.POINTER(PlanConfig)]),
    "ogl_plan_destroy": (_i, [_vp]),
    "ogl_plan_param_count": (_i64, [_vp]),
    "ogl_plan_bind_params": (_i, [_vp, _vp, _vp, _vp]),
    "ogl_plan_refresh_params": (_i, [_vp, _vp]),
    "ogl_plan_set_step": (_i, [_vp, _u32, _vp]),
    "ogl_plan_error_flags": (_i, [_vp, C.POINTER(_u32)]),
    "ogl_plan_reset_optimizer": (_i, [_vp, _u32, _vp]),
    "ogl_plan_sample": (_i, [_vp, _vp, _vp, _i, _vp]),
    "ogl_plan_forward": (_i, [_vp, _vp, _vp, _vp]),
    "ogl_plan_loss_backward": (_i, [_vp, _vp, _f, _vp, _vp, _vp]),
    "ogl_plan_set_input": (_i, [_vp, _vp, _i, _vp]),
    "ogl_plan_backward": (_i, [_vp, _vp, _f, _vp]),
    "ogl_plan_adam_step": (_i, [_vp, _vp]),
    "ogl_plan_train_step": (_i, [_vp, _vp, _vp, _vp, _i, _i, _f, _i, _vp, _vp, _vp]),
    "ogl_plan_train_steps": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _f, _i, _vp, _vp, _vp]),
    "ogl_plan_step_begin": (_i, [_vp, _vp, _vp, _vp, _i, _i, _vp]),
    "ogl_plan_step_finish": (_i, [_vp, _vp, _f, _i, _vp, _vp, _vp]),
    "ogl_plan_step_finish_head": (_i, [_vp, _vp, _f, _vp, _vp, _vp]),
    "ogl_plan_step_finish_tail": (_i, [_vp, _vp, _vp]),
    "ogl_plan_step_finish_dp": (_i, [_vp, _vp, _vp, _f, _vp, _vp, _vp]),
    "ogl_plan_prefetch": (_i, [_vp, _vp, _vp, _vp, _i, _i, _vp]),
    "ogl_plan_prefetch_pending": (_i, [_vp]),
    "ogl_graph_row_degrees": (_i, [_vp, _vp, _i64, _vp, _vp]),
    "ogl_graph_gather_rows": (_i, [_vp, _vp, _i64, _vp, _vp, _vp]),
    "ogl_infer_rows_linear": (_i, [_vp, _i, _vp, _vp, _i, _vp, _vp, _i, _vp, _vp, _i, _vp, _i, _vp, _i, _vp, _i64, _i, _vp]),
    "ogl_infer_query": (_i, [_vp, _vp, _i, _i64, _i, _i, _i, _vp, _vp]),
    "ogl_infer_induced_mean": (_i, [_vp, _vp, _vp, _i64, _vp, _i, _i, _vp, _i, _vp]),
    "ogl_peer_create": (_i, [C.POINTER(_vp), _i, _i, _i64]),
    "ogl_peer_destroy": (_i, [_vp]),
    "ogl_peer_handle": (_i, [_vp, _vp]),
    "ogl_peer_connect": (_i, [_vp, _vp]),
    "ogl_peer_connect_local": (_i, [_vp, C.POINTER(_vp)]),
    "ogl_peer_buffer": (_i, [_vp, C.POINTER(_vp)]),
    "ogl_peer_wait_readers": (_i, [_vp, _vp]),
    "ogl_plan_peer_adam": (_i, [_vp, _vp, _i64, _i64, _i, _vp, _vp]),
    "ogl_plan_set_option": (_i, [_vp, C.c_char_p, _i]),
    "ogl_plan_graph_stats": (_i, [_vp, C.POINTER(_i64 * 2)]),
    "ogl_plan_eval_step": (_i, [_vp, _vp, _vp, _vp, _i, _i, _vp, _vp, _vp]),
    "ogl_plan_infer_full": (_i, [_vp, _vp, _vp, _vp, _i64, _vp, _vp]),
    "ogl_plan_infer_full_layer": (_i, [_vp, _vp, _vp, _i, _vp, _i, _vp, _i64, _i64, _vp, _i, _vp]),
    "ogl_plan_infer_full_loss": (_i, [_vp, _vp, _vp, _vp, _i64, _vp, _vp, _vp]),
    "ogl_plan_full_xent": (_i, [_vp, _vp, _vp, _i, _vp, _i64, _i64, _vp, _vp]),
    "ogl_graph_segment_max": (_i, [_vp, _i, _vp, _i, _i, _vp, _i64, _vp, _i, _vp]),
    "ogl_graph_in_frontier": (_i, [_vp, _vp, _i64, _vp, C.POINTER(_i64), C.POINTER(_i64), _vp]),
    "ogl_plan_profile": (_i, [_vp, _i]),
    "ogl_plan_profile_read": (_i, [_vp, C.c_char_p, _i, _vp, _vp, _i, C.POINTER(_i), _vp, C.POINTER(_i)]),
    "ogl_plan_level_nodes": (_i, [_vp, _i, _pp, _pp, C.POINTER(_i)]),
    "ogl_plan_block_edges": (_i, [_vp, _i, _pp, _pp, _pp, C.POINTER(_i)]),
    "ogl_plan_tensor": (_i, [_vp, C.c_char_p, _pp, C.POINTER(_i), C.POINTER(_i), C.POINTER(_i)]),
    "ogl_sample_neighbors": (_i, [_vp, _vp, _i64, _i, _u64, _u32, _u32, _vp, _vp, _vp]),
    "ogl_draw_uniform": (_i, [_i64, _i64, _u64, _u32, _vp, _vp]),
    "ogl_sumtree_create": (_i, [_pp, _i64]),
    "ogl_sumtree_destroy": (_i, [_vp]),
    "ogl_sumtree_set": (_i, [_vp, _vp, _vp, _i64, _vp]),
    "ogl_sumtree_set_from_loss": (_i, [_vp, _vp, _vp, _i64, _d, _d, _d, _d, _vp, _vp]),
    "ogl_sumtree_sum": (_i, [_vp, _i64, _i64, _vp, _vp]),
    "ogl_sumtree_find": (_i, [_vp, _vp, _i64, _vp, _vp]),
    "ogl_sumtree_sample_stratified": (_i, [_vp, _vp, _i64, _i64, _vp, _vp]),
    "ogl_sumtree_values": (_i, [_vp, _pp, C.POINTER(_i64)]),
    "ogl_eval_confusion": (_i, [_vp, _i, _i64, _i, _vp, _vp, _vp]),
    "ogl_gemm_bf16_nt": (_i, [_vp, _i, _vp, _i, _vp, _i, _i, _i, _i, _vp]),
    "ogl_gemm_bf16_nt_ex": (_i, [_vp, _i, _vp, _i, _vp, _i, _i, _i, _i, _i, _vp, _i, _i, _vp]),
    "ogl_gemm_bf16_tn": (_i, [_vp, _i, _vp, _i, _vp, _i, _i, _i, _i, _vp, _i64, _vp]),
    "ogl_gemm_tf32_nt_ex": (_i, [_vp, _i, _vp, _i, _vp, _i, _i, _i, _i, _i, _vp, _i, _vp, _i, _i, _vp]),
    "ogl_gemm_tf32_tn": (_i, [_vp, _i, _vp, _i, _vp, _i, _i, _i, _i, _vp, _i64, _vp]),
    "ogl_fp16_grad_scale": (_f, [_f]),
    "ogl_gemm_f16_nt_ex": (_i, [_vp, _i, _vp, _i, _vp, _i, _i, _i, _i, _i, _vp, _i, _vp, _i, _i, _vp]),
    "ogl_gemm_f16_tn": (_i, [_vp, _i, _vp, _i, _vp, _i, _i, _i, _i, _f, _vp, _i64, _vp]),
}

for _name, (_res, _args) in SIGNATURES.items():
    _fn = getattr(lib, _name)          # AttributeError here = the .so is stale: rebuild
    _fn.restype = _res
    _fn.argtypes = _args


def check(rc):
    if rc != 0:
        raise OglError("ogl_b200 error %d: %s" % (rc, lib.ogl_last_error().decode("utf-8", "replace")))


def kernel_launches():
    return int(lib.ogl_kernel_launches())
