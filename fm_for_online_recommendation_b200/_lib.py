"""ctypes loader for lib/libfmb200.so (the C-ABI boundary declared in include/fmb200.h).

There is NO CPU fallback: `require_cuda()` raises if the extension is missing or no B200 is visible,
and every wrapper raises `FmbError` on a non-zero status.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
SO_PATH = os.path.join(_HERE, "lib", "libfmb200.so")

c_i32p = C.POINTER(C.c_int32)
c_f32p = C.POINTER(C.c_float)
vp = C.c_void_p


class FmbError(RuntimeError):
    pass


_SIGS = {
    "fmb_version": (C.c_int, []),
    "fmb_last_error": (C.c_char_p, []),
    "fmb_device_count": (C.c_int, []),
    "fmb_rowp": (C.c_int, [C.c_int]),
    "fmb_kp4": (C.c_int, [C.c_int]),
    "fmb_fm_forward": (C.c_int, [vp, vp, vp, vp, C.c_int, C.c_int, C.c_int, vp, vp, vp, vp, vp, vp, C.c_int, vp, vp,
                                 vp]),
    "fmb_loss_delta": (C.c_int, [C.c_int, vp, vp, C.c_int, vp, vp, vp]),
    "fmb_sum_aten": (C.c_int, [vp, C.c_int64, vp, vp]),
    "fmb_afm_dense_floats": (C.c_size_t, [C.c_int, C.c_int]),
    "fmb_afm_step": (C.c_int, [vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, vp,
                               vp, vp, vp, vp, C.c_size_t, vp]),
    "fmb_afm_dense_update": (C.c_int, [vp, C.c_int, C.c_int, C.c_int, vp, vp, vp, vp, C.c_float, C.c_int, vp, vp]),
    "fmb_fm_backward_runs_all": (C.c_int, [vp, C.c_int64, vp, C.c_int, C.c_int, C.c_float, C.c_int, vp, C.c_size_t, vp]),
    "fmb_rrf_run": (C.c_int, [vp, vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_double, C.c_double, vp, vp, vp, vp, vp, vp]),
    "fmb_dataset_encode_ids": (C.c_int, [vp, C.c_int64, C.c_int, vp, vp, vp, vp]),
    "fmb_dataset_take": (C.c_int, [vp, vp, vp, C.c_int, C.c_int64, vp, C.c_int64, vp, vp, vp, vp, vp, vp]),
    "fmb_dict_encode_workspace_bytes": (C.c_size_t, [C.c_int64, C.c_int]),
    "fmb_dict_encode_first_seen": (C.c_int, [vp, C.c_int64, C.c_int, vp, vp, vp, vp, C.c_size_t, vp]),
    "fmb_metric_regression": (C.c_int, [vp, vp, C.c_int64, vp, vp]),
    "fmb_metric_classification": (C.c_int, [vp, vp, C.c_int64, vp, vp, vp]),
    "fmb_confusion": (C.c_int, [vp, vp, C.c_int64, vp, vp]),
    "fmb_auc_pairs": (C.c_int, [vp, vp, C.c_int64, vp, vp]),
    "fmb_sigmoid": (C.c_int, [vp, C.c_int, vp, vp]),
    "fmb_math_eval": (C.c_int, [C.c_int, vp, vp, C.c_int64, vp]),
    "fmb_update_dense": (C.c_int, [vp, vp, C.c_int64, C.c_float, C.c_int, vp]),
    "fmb_finish_step": (C.c_int, [vp, vp, C.c_int, vp, C.c_float, C.c_int, vp, vp]),
    "fmb_update_dense_ex": (C.c_int, [vp, vp, C.c_int64, C.c_float, C.c_int, vp, C.c_float, vp]),
    "fmb_sort_workspace_bytes": (C.c_size_t, [C.c_int64]),
    "fmb_sort_segment": (C.c_int, [vp, C.c_int64, C.c_int, vp, C.c_size_t, vp, vp, vp, vp, vp]),
    "fmb_bwd_workspace_bytes": (C.c_size_t, [C.c_int64, C.c_int]),
    "fmb_fm_backward_update": (C.c_int, [vp, vp, C.c_int64, vp, vp, C.c_int, C.c_int, vp, vp, C.c_int, vp, C.c_float,
                                         C.c_int, vp, C.c_size_t, vp]),
    "fmb_mlp_numel": (C.c_int64, [C.c_int, C.c_int, C.c_int]),
    "fmb_mlp_forward": (C.c_int, [vp, C.c_int, vp, C.c_int, C.c_int, C.c_int, C.c_int, vp, vp, vp]),
    "fmb_mlp_bwd_workspace_bytes": (C.c_size_t, [C.c_int, C.c_int]),
    "fmb_mlp_backward": (C.c_int, [vp, C.c_int, vp, vp, vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, vp, vp,
                                   C.c_int, vp, C.c_size_t, vp]),
    "fmb_set_tensor_cores": (None, [C.c_int]),
    "fmb_tensor_cores_enabled": (C.c_int, []),
    "fmb_tensor_core_threshold_log2": (C.c_int, []),
    "fmb_gemm_tc_nt": (C.c_int, [vp, vp, vp, C.c_int, C.c_int, C.c_int, vp]),
    "fmb_gemm_tc_strided": (C.c_int, [vp, C.c_int64, C.c_int64, vp, C.c_int64, C.c_int64, vp, C.c_int64, C.c_int,
                                      C.c_int, C.c_int, C.c_int, vp, vp, C.c_int64, vp, vp]),
    "fmb_gemm_tc_error": (C.c_int, []),
    "fmb_combine_logit": (C.c_int, [C.c_int, vp, vp, vp, vp, C.c_int, vp, vp]),
    "fmb_onn_heads": (C.c_int, [C.c_int, vp, vp, vp, vp, C.c_int, C.c_int, vp, vp]),
    "fmb_predict": (C.c_int, [vp, C.c_int, vp, vp]),
    "fmb_hedge_head_grad": (C.c_int, [vp, vp, C.c_int, vp, vp, vp]),
    "fmb_hedge_accumulate": (C.c_int, [vp, vp, vp, C.c_int, C.c_int, C.c_int, C.c_int, vp]),
    "fmb_hedge_apply": (C.c_int, [vp, vp, C.c_float, vp, vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_float,
                                  C.c_float, vp]),
    "fmb_mlp_backward_hedge": (C.c_int, [vp, C.c_int, vp, vp, vp, vp, C.c_int, C.c_int, C.c_int, C.c_int, vp, vp, C.c_size_t,
                                         vp]),
    "fmb_ftrl_fm_run": (C.c_int, [vp, vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_double, vp, vp, vp, vp, vp, vp, vp]),
    "fmb_sftrl_workspace_bytes": (C.c_size_t, [C.c_int, C.c_int]),
    "fmb_sftrl_run": (C.c_int, [vp, vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_double, vp, vp, vp, vp, vp,
                                vp, vp, vp, C.c_size_t, vp]),
    "fmb_fm_backward_update_ex": (C.c_int, [vp, vp, C.c_int64, C.c_int64, vp, vp, C.c_int, C.c_int, vp, C.c_int, vp,
                                            C.c_int, C.c_int, vp, C.c_int32, C.c_float, C.c_int, vp, C.c_size_t, vp]),
    "fmb_fm_backward_update_rl": (C.c_int, [vp, vp, C.c_int64, C.c_int64, vp, vp, C.c_int, C.c_int, vp, C.c_int, vp,
                                            C.c_int, C.c_int, vp, C.c_int32, C.c_float, C.c_int, vp, vp, C.c_size_t, vp]),
    "fmb_fm_backward_update_rl_ex": (C.c_int, [vp, vp, C.c_int64, C.c_int64, vp, vp, C.c_int, C.c_int, vp, C.c_int, vp,
                                               C.c_int, C.c_int, vp, C.c_int32, C.c_float, C.c_int, vp, vp, vp, C.c_size_t,
                                               vp]),
    "fmb_shard_pw": (C.c_int, [C.c_int]),
    "fmb_shard_cw": (C.c_int, [C.c_int]),
    "fmb_shard_sort_max_cap": (C.c_int, []),
    "fmb_transpose_ids": (C.c_int, [vp, C.c_int, C.c_int, vp, vp]),
    "fmb_shard_partial_forward": (C.c_int, [vp, vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, vp, vp]),
    "fmb_shard2_slot_floats": (C.c_int, []),
    "fmb_shard2_fused": (C.c_int, [vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, C.c_int, C.c_int, C.c_int, C.c_int,
                                   C.c_int, C.c_int, vp, C.c_size_t, vp, vp, C.c_int, vp, vp]),
    "fmb_shard2_push_rows": (C.c_int, [vp, vp, vp, vp, vp, vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, vp]),
    "fmb_shard2_push_hot": (C.c_int, [vp, vp, vp, vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, vp]),
    "fmb_shard2_runs": (C.c_int, [vp, C.c_int64, C.c_int, C.c_int, vp, C.c_size_t, vp, C.c_int, C.c_int, vp]),
    "fmb_shard2_push_keys": (C.c_int, [vp, C.c_int64, C.c_int, C.c_int, vp, vp]),
    "fmb_shard2_owner_apply": (C.c_int, [vp, vp, vp, vp, vp, vp, C.c_int, vp, vp, vp, C.c_int, C.c_int, C.c_int, C.c_int,
                                         C.c_int, C.c_float, C.c_int, vp, vp, C.c_int, vp, vp]),
    "fmb_shard_combine": (C.c_int, [vp, vp, vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, vp, vp, vp]),
    "fmb_shard_unpack_ctx": (C.c_int, [vp, C.c_int64, C.c_int, vp, vp, vp]),
    "fmb_shard_sort_fields": (C.c_int, [vp, C.c_int, C.c_int, C.c_int, C.c_int, vp, C.c_int, vp, vp, vp, vp, vp]),
    "fmb_shard_sort_fields_rl": (C.c_int, [vp, C.c_int, C.c_int, C.c_int, C.c_int, vp, C.c_int, vp, vp, vp, vp, vp, vp]),
    "fmb_shard_transpose_ids_peers": (C.c_int, [vp, C.c_int, C.c_int, C.c_int, C.c_int, vp, vp, vp, vp, vp, C.c_int, vp]),
    "fmb_shard_partial_forward_peers": (C.c_int, [vp, vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, vp, vp, vp, vp, vp,
                                                  C.c_int, vp]),
    "fmb_shard_combine_peers": (C.c_int, [vp, vp, vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, vp, vp, vp, vp, vp, vp,
                                          C.c_int, C.c_int, vp]),
    "fmb_shard3_tiles": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int]),
    "fmb_shard_sort_fields_pf": (C.c_int, [vp, C.c_int, C.c_int, C.c_int, C.c_int, vp, C.c_int, vp, vp, vp, vp, vp, vp, vp]),
    "fmb_shard3_step": (C.c_int, [vp, vp, vp, vp, vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_float,
                                  C.c_int, vp, C.c_size_t, vp, vp, vp, vp, vp, vp, vp, vp, vp]),
    "fmb_shard3_bump": (C.c_int, [vp, vp]),
    "fmb_shard_signal": (C.c_int, [vp, vp, vp, C.c_int, C.c_int, C.c_int, C.c_int, vp, vp]),
    "fmb_online_deep_run": (C.c_int, [C.c_int, vp, vp, vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, vp, vp, vp, vp,
                                      vp, C.c_float, C.c_float, C.c_float, C.c_int, vp, vp, vp]),
    "fmb_online_deep_run_ex": (C.c_int, [C.c_int, vp, vp, vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, vp, vp, vp,
                                         vp, vp, C.c_float, C.c_float, C.c_float, C.c_int, vp, vp, vp, vp]),
    "fmb_session_create": (C.c_int, [C.POINTER(vp), C.c_int, C.c_int, C.c_int64, vp]),
    "fmb_sort_fields_max_batch": (C.c_int, []),
    "fmb_sort_fields": (C.c_int, [vp, C.c_int, C.c_int, vp, vp, vp, vp]),
    "fmb_runlist_shape": (None, [C.c_int, C.c_int, vp, vp]),
    "fmb_sort_fields_sparse_min_rows": (C.c_int64, [C.c_int]),
    "fmb_sort_fields_ex": (C.c_int, [vp, C.c_int, C.c_int, vp, vp, vp, vp, vp, C.c_int, vp]),
    "fmb_session_destroy": (None, [vp]),
    "fmb_session_launches": (C.c_int64, [vp]),
    "fmb_session_graph_count": (C.c_int, [vp]),
    "fmb_session_fm_step": (C.c_int, [vp, vp, vp, vp, C.c_int, vp, vp, C.c_int, C.c_int, C.c_float, C.c_int, vp, vp]),
    "fmb_session_fm_step_host_async": (C.c_int, [vp, C.c_int, vp, vp, vp, C.c_int, vp, vp, C.c_int, C.c_int, C.c_float,
                                                 C.c_int, vp]),
    "fmb_session_presort": (C.c_int, [vp, vp, C.c_int, C.c_int]),
    "fmb_session_presort_invalidate": (None, [vp]),
    "fmb_session_set_ftrl": (C.c_int, [vp, vp, vp, C.c_float, C.c_float, C.c_float]),
    "fmb_session_set_adagrad": (C.c_int, [vp, vp, vp, C.c_float]),
    "fmb_session_set_sparse_adam": (C.c_int, [vp, vp]),
    "fmb_adam_scalars": (None, [C.c_float, C.c_double, C.c_double, C.c_int64, vp]),
    "fmb_sparse_adam_advance": (C.c_int, [vp, C.c_float, C.c_int]),
    "fmb_sparse_adam_online_steps": (C.c_int, [vp, C.c_float, C.c_int, C.c_int, vp]),
    "fmb_update_dense_adam": (C.c_int, [vp, vp, C.c_int64, vp, vp]),
    "fmb_fm_step_fused_ex": (C.c_int, [vp, vp, vp, vp, vp, vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_float, C.c_int, vp,
                                       vp, vp, vp, C.c_size_t, vp]),
    "fmb_fm_backward_runs_ex": (C.c_int, [vp, C.c_int64, vp, C.c_int, C.c_int, C.c_float, C.c_int, vp, vp, C.c_size_t,
                                          vp]),
    "fmb_finish_step_ex": (C.c_int, [vp, vp, C.c_int, vp, C.c_float, C.c_int, vp, vp, vp]),
    "fmb_session_fm_step_next": (C.c_int, [vp, vp, vp, vp, C.c_int, vp, vp, C.c_int, C.c_int, C.c_float, C.c_int, vp, vp,
                                           vp]),
    "fmb_pos_flags": (C.c_int, [vp, vp, C.c_int64, vp, vp]),
    "fmb_pos_flags_ex": (C.c_int, [vp, vp, C.c_int64, vp, vp, vp]),
    "fmb_fm_backward_runs_list": (C.c_int, [vp, C.c_int64, vp, C.c_int, C.c_int, C.c_float, C.c_int, vp, vp, vp,
                                            C.c_size_t, vp]),
    "fmb_fm_step_fused": (C.c_int, [vp, vp, vp, vp, vp, vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_float, C.c_int, vp, vp,
                                    vp, C.c_size_t, vp]),
    "fmb_fm_backward_runs": (C.c_int, [vp, C.c_int64, vp, C.c_int, C.c_int, C.c_float, C.c_int, vp, C.c_size_t, vp]),
    "fmb_session_wait_loss": (C.c_int, [vp, C.c_int, C.POINTER(C.c_float)]),
    "fmb_session_host_slots": (C.c_int, []),
    "fmb_session_fm_step_host": (C.c_int, [vp, vp, vp, vp, C.c_int, vp, vp, C.c_int, C.c_int, C.c_float, C.c_int,
                                           C.POINTER(C.c_float), vp]),
}

_lib = None


class RunList(C.Structure):
    """fmb_runlist_t (include/fmb200.h): the runs of >= 2 equal sorted keys, one segment per producer CTA."""
    _fields_ = [("entries", C.c_void_p), ("seg_count", C.c_void_p), ("nseg", C.c_int), ("seg_cap", C.c_int)]


class AdagradState(C.Structure):
    """fmb_adagrad_t (include/fmb200.h): update mode 3's sums of the table, the bias and the tower, and eps."""
    _fields_ = [("sums", C.c_void_p), ("bias_sum", C.c_void_p), ("mlp_sums", C.c_void_p), ("eps", C.c_float)]


class AdamStep(C.Structure):
    _fields_ = [("emb_step", C.c_float), ("bias_step", C.c_float), ("bias_bc2s", C.c_float), ("mlp_step", C.c_float),
                ("mlp_bc2s", C.c_float)]


class SparseAdamState(C.Structure):
    """fmb_sparse_adam_t (include/fmb200.h): update mode 4's moments, hyperparameters, step counters and the scalars of
    the step being run."""
    _fields_ = [("mv", C.c_void_p), ("bias_mv", C.c_void_p), ("mlp_mv", C.c_void_p), ("beta1", C.c_double),
                ("beta2", C.c_double), ("eps", C.c_float), ("step", C.c_int64), ("mlp_step", C.c_int64),
                ("cur", AdamStep), ("steps_dev", C.c_void_p)]


def load():
    """Load the shared library (works without a GPU: symbols only)."""
    global _lib
    if _lib is None:
        if not os.path.exists(SO_PATH):
            raise FmbError(f"{SO_PATH} is missing: run `python -m fm_for_online_recommendation_b200.build` "
                           "(there is no CPU fallback)")
        lib = C.CDLL(SO_PATH)
        for name, (res, args) in _SIGS.items():
            fn = getattr(lib, name)
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


def require_cuda():
    lib = load()
    if lib.fmb_device_count() < 1:
        raise FmbError("no CUDA device visible: fm_for_online_recommendation_b200 has no CPU fallback")
    return lib


def check(rc, what=""):
    if rc != 0:
        raise FmbError(f"{what} failed (status {rc}): {load().fmb_last_error().decode()}")


def ptr(t):
    """device/host pointer of a torch tensor (or None)."""
    return None if t is None else C.c_void_p(t.data_ptr())
