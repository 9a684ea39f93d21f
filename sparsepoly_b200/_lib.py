"""ctypes binding of libsparsepoly_b200.so (declared in include/sparsepoly_b200.h).

There is no CPU fallback: if the shared library cannot be loaded (or built), importing the
solvers fails loudly.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("SPARSEPOLY_B200_LIB") or os.path.join(_HERE, "libsparsepoly_b200.so")   # (override: A/B builds)

LOSS_IDS = {"squared": 0, "logistic": 1, "squared_hinge": 2}
REG_IDS = {"l1": 0, "l21": 1, "squaredl12": 2, "squaredl21": 3, "omegati": 4, "omegacs": 5}
LEARNING_RATE = {"constant": 0, "optimal": 1, "pegasos": 2, "invscaling": 3}

SP_OK, SP_ERR_INVALID, SP_ERR_UNSUPPORTED, SP_ERR_CUDA = 0, 1, 2, 3

_vp = C.c_void_p
_i = C.c_int
_d = C.c_double


class SpDataset(C.Structure):
    """struct sp_dataset (include/sparsepoly_b200.h)."""
    _fields_ = [("n_samples", C.c_int32), ("n_features", C.c_int32), ("nnz", C.c_int64),
                ("csr_indptr", _vp), ("csr_indices", _vp), ("csr_data", _vp),
                ("csc_indptr", _vp), ("csc_indices", _vp), ("csc_data", _vp),
                ("feat_hot", _vp), ("hot_feat", _vp), ("n_hot_feat", C.c_int32)]


class SpWPlan(C.Structure):
    """struct sp_wplan (include/sparsepoly_b200.h)."""
    _fields_ = [("window", C.c_int32), ("horizon", C.c_int32), ("n_windows", C.c_int32),
                ("slot_cap", C.c_int32), ("near", C.c_int32), ("flags", C.c_int32), ("cflag", _vp),
                ("ht_ptr", _vp), ("ht_cls", _vp), ("h_sd", _vp), ("h_x", _vp), ("n_slots", _vp),
                ("slot_row", _vp), ("sync", _vp), ("res", _vp), ("base", _vp)]


class SpPlan(C.Structure):
    """struct sp_plan (include/sparsepoly_b200.h)."""
    _fields_ = [("n_cta", C.c_int32), ("threads", C.c_int32), ("pos_ptr", _vp), ("flag_idx", _vp),
                ("idx_feat", _vp), ("pos_conf", _vp), ("win", C.POINTER(SpWPlan))]


MAX_RANKS = 8


class SpPsgdPlan(C.Structure):
    """struct sp_psgd_plan (include/sparsepoly_b200.h)."""
    _fields_ = [("n_minibatches", C.c_int32), ("batch_local", C.c_int32), ("n_local", C.c_int32),
                ("chunk", C.c_int32), ("short_max", C.c_int32),
                ("mb_eptr_host", _vp), ("mb_uptr_host", _vp), ("mb_sgptr_host", _vp), ("mb_shptr_host", _vp),
                ("mb_lcptr_host", _vp), ("mb_mlptr_host", _vp),
                ("e_pos", _vp), ("e_x", _vp), ("u_feat", _vp), ("u_ptr", _vp),
                ("sg_u", _vp), ("sg_feat", _vp), ("sg_pos", _vp), ("sg_x", _vp),
                ("sc_ptr", _vp), ("sc_u", _vp), ("sc_feat", _vp), ("sc_pos", _vp), ("sc_x", _vp), ("lc_u", _vp), ("lc_feat", _vp), ("lc_cnt", _vp),
                ("lc_e0", _vp), ("ml_u", _vp), ("ml_c0", _vp),
                ("max_chunks", C.c_int64), ("max_cols", C.c_int64),
                ("csr_slot", _vp), ("mb_owner_start_host", _vp), ("mb_optr_host", _vp), ("own_q", _vp), ("own_src", _vp)]


class SpPsgdCtx(C.Structure):
    """struct sp_psgd_ctx (include/sparsepoly_b200.h)."""
    _fields_ = [("P", _vp), ("w", _vp), ("lams", _vp), ("thr", _vp),
                ("n_orders", C.c_int32), ("k", C.c_int32), ("d_rows", C.c_int32), ("degree", C.c_int32),
                ("reg", C.c_int32), ("loss", C.c_int32), ("fit_linear", C.c_int32),
                ("world", C.c_int32), ("rank", C.c_int32),
                ("bufA", _vp), ("bufdL", _vp), ("sample_loss", _vp), ("part_g", _vp), ("part_w", _vp),
                ("work", _vp), ("xwork", _vp), ("C", C.c_double), ("Cw", C.c_double),
                ("seq", C.c_uint64), ("seq_generic", C.c_uint64),
                ("stage", _vp), ("stage_w", _vp), ("inbox_g", _vp), ("inbox_w", _vp), ("inbox_cap", C.c_int64),
                ("err", _vp),
                ("peer_P", _vp * MAX_RANKS), ("peer_w", _vp * MAX_RANKS),
                ("peer_inbox_g", _vp * MAX_RANKS), ("peer_inbox_w", _vp * MAX_RANKS),
                ("peer_xwork", _vp * MAX_RANKS), ("peer_flags", _vp * MAX_RANKS),
                ("seq_pull", C.c_uint64), ("aux_stream", _vp), ("aux_event", _vp * 2)]


class SpPcdModel(C.Structure):
    """struct sp_pcd_model (include/sparsepoly_b200.h): one model of sp_pcd_epoch_multi / sp_cd_linear_epoch_multi."""
    _fields_ = [("pos_ptr", _vp), ("flag_idx", _vp), ("idx_feat", _vp), ("pos_conf", _vp), ("P", _vp),
                ("lams", _vp), ("ab", C.c_double), ("gamma", C.c_double), ("eta", C.c_double), ("reg", C.c_int32),
                ("rec", _vp), ("regstate", _vp), ("viol", _vp), ("idx_comp_host", C.POINTER(C.c_int32))]


class SpPbcdModel(C.Structure):
    """struct sp_pbcd_model (include/sparsepoly_b200.h): one model of sp_pbcd_epoch_multi."""
    _fields_ = [("pos_ptr", _vp), ("flag_idx", _vp), ("idx_feat", _vp), ("P", _vp), ("lams", _vp),
                ("beta", C.c_double), ("gamma", C.c_double), ("eta", C.c_double), ("reg", C.c_int32),
                ("yrec", _vp), ("A", _vp), ("reg_norms", _vp), ("regstate", _vp), ("viol", _vp)]


PREDICT_MAX_MODELS = 256           # SP_PREDICT_MAX_MODELS
OBJECTIVE_MAX_ENTRIES = 256        # SP_OBJECTIVE_MAX_ENTRIES
CSR_REPORT_LEN = 8                 # SP_CSR_REPORT_LEN: sp_csr_prepare's report (its entries: dataset.check_X)


class SpPredictModel(C.Structure):
    """struct sp_predict_model (include/sparsepoly_b200.h): one model of sp_predict_multi."""
    _fields_ = [("P_dk", _vp), ("lams", _vp), ("w", _vp), ("out", _vp)]


class SpLossEntry(C.Structure):
    """struct sp_loss_entry (include/sparsepoly_b200.h): one sum of sp_loss_sum_multi."""
    _fields_ = [("y_pred", _vp), ("y", _vp), ("loss", C.c_int32), ("out", _vp)]


class SpSqnormEntry(C.Structure):
    """struct sp_sqnorm_entry (include/sparsepoly_b200.h): one sum of sp_sqnorm_multi."""
    _fields_ = [("v", _vp), ("out", _vp)]


class SpRegEntry(C.Structure):
    """struct sp_reg_entry (include/sparsepoly_b200.h): one Omega of sp_reg_eval_multi."""
    _fields_ = [("P_dk", _vp), ("reg", C.c_int32), ("out", _vp)]


_DSP = C.POINTER(SpDataset)
_PPP = C.POINTER(SpPsgdPlan)
_PCP = C.POINTER(SpPsgdCtx)
_PLP = C.POINTER(SpPlan)

# name -> (restype, argtypes); every symbol the header declares
SIGNATURES = {
    "sp_abi_version": (_i, []),
    "sp_last_error": (C.c_char_p, []),
    "sp_device_count": (_i, [C.POINTER(C.c_int)]),
    "sp_set_device": (_i, [_i]),
    "sp_profile_enable": (_i, [_i]),
    "sp_profile_collect": (_i, [C.POINTER(_d), C.POINTER(C.c_longlong)]),
    "sp_col_norm_sq": (_i, [_DSP, _vp, _vp]),
    "sp_plan_partition": (_i, [_DSP, _i, _vp, _vp]),
    "sp_plan_order": (_i, [_DSP, _i, _vp, _vp, _vp, _vp, _vp, _vp]),
    "sp_wplan_flag": (_i, [_DSP, _vp, _i, _i, _vp, _vp, _vp, _vp]),
    "sp_wplan_fill": (_i, [_DSP, _vp, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "sp_wplan_slot_cap": (_i, [_i]),
    "sp_pbcd_wplan_slot_cap": (_i, [_i, _i]),
    "sp_pbcd_wplan_base_doubles": (C.c_size_t, []),
    "sp_wprof_read": (_i, [C.POINTER(C.c_ulonglong)]),
    "sp_wtrace_read": (_i, [C.POINTER(C.c_longlong)]),
    "sp_wspec_read": (_i, [C.POINTER(C.c_ulonglong)]),
    "sp_transpose_f64": (_i, [_vp, _vp, _i, _i, _vp]),
    "sp_transpose_f64_batch": (_i, [_vp, _vp, _i, _i, _i, _vp]),
    "sp_rec_stride": (_i, [_i]),
    "sp_predict": (_i, [_DSP, _vp, _i, _vp, _i, _vp, _vp, _i, _i, _vp]),
    "sp_predict_multi": (_i, [_DSP, C.POINTER(SpPredictModel), _i, _i, _i, _i, _i, _vp]),
    "sp_kernel_matrix": (_i, [_DSP, _vp, _i, _i, _vp, _vp]),
    "sp_cd_linear_epoch": (_i, [_DSP, _PLP, _vp, _vp, _d, _i, _vp, _i, _vp, _vp]),
    "sp_pcd_epoch": (_i, [_DSP, _PLP, _vp, _i, _vp, _i, _d, _d, _d, _i, _i, _vp, _i, _vp, _vp,
                          C.POINTER(C.c_int32), _vp]),
    "sp_cd_linear_epoch_multi": (_i, [_DSP, _i, _i, _vp, C.POINTER(SpPcdModel), _i, _i, _i, _vp]),
    "sp_pcd_epoch_multi": (_i, [_DSP, _i, _i, C.POINTER(SpPcdModel), _i, _i, _i, _i, _i, _vp]),
    "sp_pbcd_epoch": (_i, [_DSP, _PLP, _vp, _i, _vp, _i, _d, _d, _d, _i, _i, _vp, _vp, _vp, _vp, _vp,
                           _vp]),
    "sp_pbcd_epoch_multi": (_i, [_DSP, _i, _i, C.POINTER(SpPbcdModel), _i, _i, _i, _i, _vp]),
    "sp_get_eta": (_i, [_i, _d, _d, _d, _d, C.c_int64, C.POINTER(_d), C.POINTER(_d)]),
    "sp_psgd_grad": (_i, [_DSP, _vp, _vp, _i, _i, _vp, _vp, _i, _i, _i, _vp, _i, _i, _vp, _vp, _vp, _vp]),
    "sp_psgd_step": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _d, _d, _d, _d, _i, _i, _vp]),
    "sp_prox_work_doubles": (C.c_size_t, [_i, _i]),
    "sp_prox": (_i, [_vp, _i, _i, _i, _d, _vp, _vp]),
    "sp_psgd_epoch": (_i, [_DSP, _vp, _vp, _i, _i, _vp, _vp, _i, _d, _d, _d, _i, _i, _vp, _vp, _vp,
                           _i, _d, _i, _d, _i, C.POINTER(C.c_int64), _vp, _vp, _vp]),
    "sp_psgd_plan_work_doubles": (C.c_size_t, [_i, _i]),
    "sp_psgd_plan_xwork_doubles": (C.c_size_t, [_i, _i, _i]),
    "sp_psgd_plan_begin": (_i, [_PCP, _vp]),
    "sp_psgd_plan_run": (_i, [_PCP, _DSP, _PPP, _vp, _vp, _d, _d, _d, _d, _i, _d, _i, _i, C.POINTER(C.c_int64), _vp]),
    "sp_psgd_plan_end": (_i, [_PCP, _i, _vp, _i, _vp]),
    "sp_psgd_plan_read": (_i, [_PCP, _vp, _vp, _vp]),
    "sp_psgd_plan_release": (_i, [_PCP]),
    "sp_psgd_plan_solver_stats": (_i, [_PCP, C.POINTER(_d), _vp]),
    "sp_shm_alloc": (_i, [C.c_size_t, C.POINTER(_vp)]),
    "sp_shm_free": (_i, [_vp]),
    "sp_ipc_export": (_i, [_vp, C.POINTER(C.c_ubyte)]),
    "sp_ipc_open": (_i, [C.POINTER(C.c_ubyte), C.POINTER(_vp)]),
    "sp_ipc_close": (_i, [_vp]),
    "sp_memcpy": (_i, [_vp, _vp, C.c_size_t, _i, _vp]),
    "sp_loss_sum": (_i, [_vp, _i, _vp, _i, _i, _i, _vp, _vp, _vp]),
    "sp_sqnorm": (_i, [_vp, C.c_int64, _vp, _vp, _vp]),
    "sp_sum_work_doubles": (C.c_size_t, []),
    "sp_reg_eval": (_i, [_vp, _i, _i, _i, _i, _vp, _vp, _vp]),
    "sp_reg_eval_work_doubles": (C.c_size_t, [_i, _i]),
    "sp_loss_sum_multi": (_i, [C.POINTER(SpLossEntry), _i, _i, _i, _i, _vp, _vp]),
    "sp_sqnorm_multi": (_i, [C.POINTER(SpSqnormEntry), _i, C.c_int64, _vp, _vp]),
    "sp_reg_eval_multi": (_i, [C.POINTER(SpRegEntry), _i, _i, _i, _i, _vp, _vp]),
    "sp_csr_prepare": (_i, [C.c_int64, C.c_int64, C.c_int64, _vp, _i, _vp, _i, _vp, _i, C.c_int64, C.c_int64, _i,
                            _vp, _vp, _vp, _vp, _vp]),
    "sp_csr_sum_runs": (_i, [C.c_int64, _vp, _vp, _vp, _vp, C.c_int64, _vp, _vp, _vp]),
}

_LIB = None


def load():
    """Load (building first if the .so is missing and nvcc is available)."""
    global _LIB
    if _LIB is not None:
        return _LIB
    if LIB_PATH == os.path.join(_HERE, "libsparsepoly_b200.so"):
        from . import build as _build
        try:
            _build.build()                       # no-op when the library is newer than every source
        except RuntimeError:
            if not os.path.exists(LIB_PATH):     # (a box without nvcc can still use a prebuilt library)
                raise
    try:
        import torch  # noqa: F401  (makes torch's libcudart.so.12 the shared runtime instance)
    except Exception:
        pass
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError if a declared symbol is missing
        fn.restype = res
        fn.argtypes = args
    if lib.sp_abi_version() != 4:
        raise ImportError("libsparsepoly_b200.so ABI version mismatch")
    _LIB = lib
    return lib


def check(rc):
    """Map a C status to the exception type the reference raises at the same spot."""
    if rc == SP_OK:
        return
    msg = load().sp_last_error().decode("utf-8", "replace")
    if rc in (SP_ERR_INVALID, SP_ERR_UNSUPPORTED):
        raise ValueError(msg)
    raise RuntimeError(msg)
