"""ctypes binding of libbfm.so (include/bfm.h).  There is NO fallback: if the CUDA library is missing
or fails to load, importing a compute entry point raises."""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("BFM_LIB") or os.path.join(_HERE, "libbfm.so")

BFM_OK, BFM_E_INVALID, BFM_E_UNSUPPORTED, BFM_E_CUDA = 0, -1, -2, -3
ABI_VERSION = 8

c_f = C.c_float
c_i = C.c_int
c_p = C.c_void_p
c_i64 = C.c_int64
c_u64 = C.c_uint64


class ZoomTab(C.Structure):
    _fields_ = [("lo", c_p * 3), ("hi", c_p * 3), ("wl", c_p * 3), ("wh", c_p * 3)]


class Deform(C.Structure):
    _fields_ = [("size", c_i * 3), ("src", c_i * 3), ("A", c_f * 9), ("c2", c_f * 3), ("ctr", c_f * 3),
                ("fsmall", c_p), ("fs", c_i * 3), ("photo", c_i), ("ftab", ZoomTab), ("F_full", c_p),
                ("cand", c_p * 3), ("ncand", c_i * 3)]


class Band(C.Structure):
    _fields_ = [("start", c_p), ("w", c_p), ("T", c_i), ("n_in", c_i), ("n_out", c_i), ("axis", c_i),
                ("build", c_i), ("sigma", C.c_double)]


MAX_AUX = 3


class GenSample(C.Structure):
    _fields_ = [("d", Deform),
                ("labels", c_p), ("label_is_u8", c_i), ("mu", c_p), ("sigma", c_p), ("eps_gmm", c_p),
                ("seed", c_u64), ("syn", c_p), ("bbox", c_p),
                ("mix", c_p * 3), ("mixw", c_f * 4),
                ("gamma", c_f), ("bfsmall", c_p), ("bs", c_i * 3), ("btab", ZoomTab),
                ("i_bf", c_p), ("bflog_out", c_p), ("flip", c_i),
                ("band", Band * 3), ("n_band", c_i), ("zero_first", c_i * 3),
                ("noise_std", c_f), ("eps_noise", c_p), ("tmp", c_p * 2), ("lowres", c_p), ("new_size", c_i * 3),
                ("utab", ZoomTab), ("maxval", c_p), ("out", c_p), ("residual", c_p),
                ("n_aux", c_i), ("aux_src", c_p * MAX_AUX), ("aux_raw", c_p * MAX_AUX), ("aux_out", c_p * MAX_AUX),
                ("aux_mm", c_p), ("x_begin", c_i), ("x_count", c_i),
                ("gen_small", c_i), ("fs_std", c_f), ("bf_std", c_f), ("real_input", c_i), ("syn_pair_ok", c_i),
                ("zoom_order", c_i), ("gmm_xr", c_p)]


class GenSeg(C.Structure):
    _fields_ = [("sample", c_i), ("cls", c_p), ("out", c_p)]


# ---- native host planner (bfm_plan_batch) ----------------------------------------------------------------
PLAN_MAX_SAMPLES = 16
c_d = C.c_double


class ZoomAxis(C.Structure):
    _fields_ = [("lo", c_p), ("hi", c_p), ("wl", c_p), ("wh", c_p), ("cand", c_p), ("ncand", c_i), ("valid", c_i)]


class PlanAug(C.Structure):
    _fields_ = [("gamma_std", c_d), ("bf_scale_min", c_d), ("bf_scale_max", c_d), ("bf_std_min", c_d),
                ("bf_std_max", c_d), ("noise_std_min", c_d), ("noise_std_max", c_d)]


class PlanCfg(C.Structure):
    _fields_ = [("size", c_i * 3), ("res", c_d * 3), ("low_res_only", c_i), ("nonlinear_transform", c_i),
                ("photo_prob", c_d), ("pathology_prob", c_d), ("random_shape_prob", c_d), ("flip_prob", c_d),
                ("max_rotation", c_d), ("max_shear", c_d), ("max_scaling", c_d),
                ("nonlin_scale_min", c_d), ("nonlin_scale_max", c_d), ("nonlin_std_max", c_d),
                ("ct_prob", c_d), ("mix_synth_prob", c_d), ("ct_group", C.c_int8 * 256), ("n_samples", c_i),
                ("bspline_zooming", c_i),
                ("aug", PlanAug * PLAN_MAX_SAMPLES), ("aug_real", PlanAug * PLAN_MAX_SAMPLES),
                ("fwd", c_p * 3), ("inv", c_p * 3), ("ends", c_p * 3), ("ident_start", c_p), ("ident_w", c_p)]


class PlanItem(C.Structure):
    _fields_ = [("labels", c_p), ("label_is_u8", c_i), ("src", c_i * 3), ("n_aux", c_i),
                ("aux_src", c_p * MAX_AUX), ("aux_out", c_p * MAX_AUX), ("aux_raw", c_p * MAX_AUX),
                ("eps_gmm", c_p * PLAN_MAX_SAMPLES), ("eps_noise", c_p * PLAN_MAX_SAMPLES),
                ("input_prob", c_d * 4), ("real_vol", c_p * 3), ("ct_vol", c_p)]


class PlanOut(C.Structure):
    _fields_ = [("out", c_p), ("bflog_out", c_p), ("residual", c_p), ("syn", c_p), ("i_bf", c_p), ("tmp", c_p * 2),
                ("lowres", c_p), ("syn_pair_ok", c_i64)]


class StepBufs(C.Structure):
    _fields_ = [("out", c_p), ("bflog_out", c_p), ("residual", c_p), ("syn", c_p), ("syn_stride", c_i64),
                ("i_bf", c_p), ("tmp", c_p), ("lowres", c_p), ("aux_out", c_p), ("aux_raw", c_p), ("pair_ok", c_i64)]


class PlanInfo(C.Structure):
    _fields_ = [("input_mode", c_i), ("photo_mode", c_i), ("flip", c_i), ("spac", c_d), ("resolution", c_d * 3), ("thickness", c_d * 3),
                ("scaling_factor_distances", c_d), ("A", c_f * 9), ("c2", c_f * 3), ("fs", c_i * 3),
                ("new_size", (c_i * 3) * PLAN_MAX_SAMPLES)]


class BfmError(RuntimeError):
    pass


_lib = None

_PROTOS = {
    "bfm_abi_version": (c_i, []),
    "bfm_last_error": (C.c_char_p, []),
    "bfm_launch_count": (c_u64, []),
    "bfm_trilerp_pull": (c_i, [c_p, c_i, c_i, c_i, c_i, c_p, c_p, c_p, c_i64, c_f, c_p, c_p, c_p]),
    "bfm_nearest_pull": (c_i, [c_p, c_i, c_i, c_i, c_i, c_i, c_p, c_p, c_p, c_i64, c_p, c_p]),
    "bfm_zoom_linear": (c_i, [c_p, c_i, c_i, c_i, c_i] + [c_p, c_p, c_p, c_p, c_i] * 3 + [c_p, c_p]),
    "bfm_blur_axis": (c_i, [c_p, c_p, c_i, c_i, c_i, c_i, c_p, c_i, c_p]),
    "bfm_band_axis": (c_i, [c_p, c_p, C.POINTER(c_i), c_i, c_i, c_p, c_p, c_i, c_f, c_p, c_u64, c_p]),
    "bfm_upload_pinned": (c_i, [c_p, c_p, c_i64, c_p]),
    "bfm_sanitize_f32": (c_i, [c_p, c_i64, c_p]),
    "bfm_ingest_volume": (c_i, [c_p, c_p, c_i, c_i64, c_f, c_f, c_p]),
    "bfm_add_noise_at": (c_i, [c_p, c_i64, c_f, c_u64, C.c_uint32, c_i64, c_p]),
    "bfm_philox_normal": (c_i, [c_p, c_i64, c_u64, C.c_uint32, c_u64, c_p]),
    "bfm_band_build": (c_i, [c_i, c_i, C.c_double, c_i, c_p, c_p, c_p]),
    "bfm_minmax": (c_i, [c_p, c_i64, c_p, c_p]),
    "bfm_shift_scale_flip": (c_i, [c_p, c_p, c_i, c_i64, c_p, c_p, c_f, c_i, c_p]),
    "bfm_deform_grid": (c_i, [C.POINTER(Deform), c_p, c_p, c_p]),
    "bfm_warp_volume": (c_i, [C.POINTER(Deform), c_p, c_p, c_f, c_f, c_i, c_p, c_p, c_p, c_p]),
    "bfm_label_warp_onehot": (c_i, [C.POINTER(Deform), c_p, c_p, c_p, c_i, c_i, c_p, c_i, c_p, c_p, c_p]),
    "bfm_svf_step": (c_i, [c_p, c_p, c_i, c_i, c_i, c_p]),
    "bfm_svf_integrate": (c_i, [c_p, c_p, c_i, c_i, c_i, c_i, c_f, c_p, c_p]),
    "bfm_gen_plan": (c_i, [c_p, c_p, c_i, c_p]),
    "bfm_gen_bbox": (c_i, [c_p, c_p, c_i, c_p]),
    "bfm_gen_gmm": (c_i, [c_p, c_p, c_i, c_p]),
    "bfm_gen_warp": (c_i, [c_p, c_p, c_i, c_p]),
    "bfm_gen_resample": (c_i, [c_p, c_p, c_i, c_p]),
    "bfm_gen_finish": (c_i, [c_p, c_p, c_i, c_p]),
    "bfm_gen_zoom_coords": (c_i, [c_i, c_i, c_p, c_p]),
    "bfm_gen_run": (c_i, [c_p, c_p, c_i, c_p]),
    "bfm_gen_segmentation": (c_i, [c_p, c_p, c_i, c_p, c_i, c_i, c_p, c_p]),
    "bfm_plan_batch": (c_i, [c_p, c_i, c_p, c_p, c_u64, c_u64, c_p, c_p, c_i64, C.POINTER(c_i64), C.POINTER(c_i64),
                             c_p, C.POINTER(c_p), c_p, c_p, c_i64, C.POINTER(c_i64)]),
    "bfm_plan_layout": (c_i, [c_p, c_i, c_p, c_p, c_p]),
    "bfm_plan_run": (c_i, [c_p, c_i, c_p, c_p, c_u64, c_u64, c_p, c_p, c_i64, c_i64, C.POINTER(c_i64), c_p,
                           C.POINTER(c_p), c_p, c_p]),
    "bfm_interpol": (c_i, [c_i, c_i, c_p, c_p, c_p, C.POINTER(c_i), C.POINTER(c_i), C.POINTER(c_i), c_i, c_i, c_i,
                           c_i, c_i, c_i, c_i64, c_p]),
    "bfm_interpol_grad_backward": (c_i, [c_i, c_p, c_p, c_p, c_p, c_p, C.POINTER(c_i), C.POINTER(c_i), C.POINTER(c_i),
                                         c_i, c_i, c_i, c_i, c_i64, c_p]),
    "bfm_interpol_pull_fast": (c_i, [c_p, C.POINTER(c_i64), c_p, c_i64, c_p, c_i, C.POINTER(c_i), c_i, C.POINTER(c_i),
                                     c_i, c_i, c_i, c_i64, c_p]),
    "bfm_compose_step": (c_i, [c_p, c_p, c_i, c_i, c_i, c_i, C.POINTER(c_i), c_i, c_p]),
    "bfm_exp_velocity": (c_i, [c_p, c_p, c_i, c_i, c_i, c_i, c_i, C.POINTER(c_i), c_i, c_p, c_p]),
    "bfm_add_identity_grid": (c_i, [c_p, c_p, c_i, c_i, c_i, c_i, c_p]),
    "bfm_spline_filter": (c_i, [c_p, c_i, c_i64, c_i, c_i64, c_i, C.POINTER(C.c_double), c_i, c_p]),
    "bfm_perlin3d": (c_i, [c_p, C.POINTER(c_i), C.POINTER(c_i), c_p, c_p]),
    "bfm_threshold_mask": (c_i, [c_p, c_p, c_i64, C.c_double, c_p]),
    "bfm_gradient3d": (c_i, [c_p, c_i, C.POINTER(c_i), c_i, C.POINTER(c_f), c_p, c_p]),
    "bfm_curl3d": (c_i, [c_p, c_p, c_p, c_i, C.POINTER(c_i), c_f, c_p, c_p, c_p, c_p]),
    "bfm_advect_rhs": (c_i, [c_p, c_i, c_p, c_p, c_p, C.POINTER(c_i), c_i, C.POINTER(c_f), c_p, c_p]),
    "bfm_diffuse_rhs": (c_i, [c_p, c_i, c_p, c_f, C.POINTER(c_i), c_i, C.POINTER(c_f), c_i, c_p, c_p]),
    "bfm_gmm_crop": (c_i, [c_p, c_i, C.POINTER(c_i), C.POINTER(c_i), c_p, c_p, c_p, c_u64, c_p, c_p]),
    "bfm_pathol_cerebral": (c_i, [c_p, c_p, c_i, C.POINTER(c_i), C.POINTER(c_i), c_p, c_p, c_p]),
    "bfm_zero_where_zero": (c_i, [c_p, c_i, c_p, c_i64, c_p]),
    "bfm_masked_mean": (c_i, [c_p, c_p, c_i, c_i64, c_p, c_p]),
    "bfm_encode_pathology": (c_i, [c_p, c_p, c_p, c_i, c_p, c_p, c_i, c_p, c_u64, c_i64, c_p]),
    "bfm_rk_combine": (c_i, [c_p, c_i, C.POINTER(c_p), C.POINTER(c_f), c_i, c_i64, c_p, c_i, c_p]),
    "bfm_rk_error_fused": (c_i, [C.POINTER(c_p), C.POINTER(c_f), c_i, c_p, c_p, c_i, c_i64, C.c_double, C.c_double, c_p,
                                 c_p, c_p]),
    "bfm_rk_error_sum": (c_i, [c_p, c_p, c_p, c_i, c_i64, C.c_double, C.c_double, c_p, c_p]),
    "bfm_dopri5_interp": (c_i, [c_p, c_p, c_p, c_p, c_p, C.c_double, C.c_double, c_i64, c_p, c_p]),
}


def exported_symbols():
    return sorted(_PROTOS)


def lib():
    """The loaded library; raises BfmError when it has not been built (python -m brainfm_b200.build)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise BfmError("libbfm.so not found at %s -- build it with `python -m brainfm_b200.build`; "
                           "there is no CPU fallback" % LIB_PATH)
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in _PROTOS.items():
            fn = getattr(L, name)
            fn.restype = res
            fn.argtypes = args
        if L.bfm_abi_version() != ABI_VERSION:
            raise BfmError("libbfm.so ABI mismatch")
        _lib = L
    return _lib


def check(rc):
    if rc == BFM_OK:
        return
    msg = lib().bfm_last_error().decode("utf-8", "replace")
    if rc == BFM_E_INVALID:
        raise ValueError(msg)
    if rc == BFM_E_UNSUPPORTED:
        raise NotImplementedError(msg)
    raise BfmError("libbfm: %s (code %d)" % (msg, rc))


def launch_count():
    return int(lib().bfm_launch_count())
