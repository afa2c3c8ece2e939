"""ctypes binding of the C-ABI library (libmmnn_b200.so).  No CPU fallback: a missing library is a hard error."""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libmmnn_b200.so")

_lib = None


class MMNNLibraryError(RuntimeError):
    pass


def lib():
    global _lib
    if _lib is None:
        if not os.path.isfile(LIB_PATH):
            raise MMNNLibraryError(
                f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(nvcc -gencode arch=compute_100a,code=sm_100a). There is no CPU fallback.")
        _lib = C.CDLL(LIB_PATH)
        _declare(_lib)
    return _lib


class BnSrc(C.Structure):
    _fields_ = [("sum", C.c_void_p), ("sumsq", C.c_void_p), ("gamma", C.c_void_p), ("beta", C.c_void_p),
                ("rmean", C.c_void_p), ("rvar", C.c_void_p), ("inv_count", C.c_float), ("eps", C.c_float),
                ("use_batch", C.c_int)]


class RowsParams(C.Structure):
    _fields_ = [("M", C.c_int), ("NT", C.c_int), ("Ncols", C.c_int), ("Cin", C.c_int), ("kbw", C.c_int),
                ("ntaps", C.c_int), ("tap_sign", C.c_int), ("Dz", C.c_int), ("Dy", C.c_int), ("Dx", C.c_int),
                ("Sz", C.c_int), ("Sy", C.c_int), ("Sx", C.c_int),
                ("a_src", C.c_void_p), ("a_pitch", C.c_longlong), ("bnA", BnSrc),
                ("b_packed", C.c_void_p), ("out", C.c_void_p), ("out_pitch", C.c_longlong),
                ("colscale", C.c_void_p), ("st_sum", C.c_void_p), ("st_sq", C.c_void_p),
                ("e_src", C.c_void_p), ("e_pitch", C.c_longlong), ("bnE", BnSrc), ("stages", C.c_int), ("acc_rstd", C.c_int), ("early_ch", C.c_int),
                ("t_src", C.c_void_p), ("t_pitch", C.c_longlong), ("t_gsum", C.c_void_p), ("t_gdot", C.c_void_p),
                ("t_inv_count", C.c_float), ("t_out", C.c_void_p), ("t_out_pitch", C.c_longlong), ("tma_a", C.c_int)]


class BrickParams(C.Structure):
    _fields_ = [("B", C.c_int), ("Dz", C.c_int), ("Dy", C.c_int), ("Dx", C.c_int), ("CH", C.c_int), ("NT", C.c_int),
                ("tap_sign", C.c_int), ("a_src", C.c_void_p), ("a_pitch", C.c_longlong), ("bnA", BnSrc),
                ("b_packed", C.c_void_p), ("out", C.c_void_p), ("out_pitch", C.c_longlong), ("colscale", C.c_void_p),
                ("st_sum", C.c_void_p), ("st_sq", C.c_void_p), ("e_src", C.c_void_p), ("e_pitch", C.c_longlong),
                ("bnE", BnSrc)]


class StemBrickParams(C.Structure):
    _fields_ = [("B", C.c_int), ("D0", C.c_int), ("H0", C.c_int), ("W0", C.c_int), ("Sz", C.c_int), ("Sy", C.c_int),
                ("Sx", C.c_int), ("xs2d", C.c_void_p), ("w_packed", C.c_void_p), ("out", C.c_void_p),
                ("out_pitch", C.c_longlong), ("st_sum", C.c_void_p), ("st_sq", C.c_void_p)]


class WgradParams(C.Structure):
    _fields_ = [("M", C.c_int), ("CB", C.c_int), ("NB", C.c_int), ("na_total", C.c_int), ("nb_total", C.c_int),
                ("Dz", C.c_int), ("Dy", C.c_int), ("Dx", C.c_int), ("Sz", C.c_int), ("Sy", C.c_int), ("Sx", C.c_int),
                ("a_src", C.c_void_p), ("a_pitch", C.c_longlong), ("bnA", BnSrc),
                ("b_src", C.c_void_p), ("b_pitch", C.c_longlong), ("bnB", BnSrc),
                ("dw", C.c_void_p), ("so_a", C.c_longlong), ("so_b", C.c_longlong), ("so_j", C.c_longlong),
                ("cin_real", C.c_int), ("stages", C.c_int), ("NP", C.c_int), ("slot_stride", C.c_longlong),
                ("tma_b", C.c_int), ("bx", C.c_int), ("by", C.c_int), ("bz", C.c_int), ("bn", C.c_int),
                ("a_bf16", C.c_int), ("tma_a", C.c_int)]


_P6 = C.c_void_p * 6


class MlpArgs(C.Structure):
    _fields_ = [("W", _P6), ("b", _P6), ("gamma", _P6), ("beta", _P6), ("rmean", _P6), ("rvar", _P6), ("nbt", _P6),
                ("Wo", C.c_void_p), ("bo", C.c_void_p), ("Wi", C.c_void_p), ("bi", C.c_void_p), ("Wc", C.c_void_p),
                ("bc", C.c_void_p), ("width", C.c_int * 7), ("B", C.c_int), ("C", C.c_int), ("blend", C.c_int),
                ("training", C.c_int), ("x", C.c_void_p), ("img_f", C.c_void_p), ("mask", C.c_void_p),
                ("z", C.c_void_p), ("a", C.c_void_p), ("stat", C.c_void_p), ("preds", C.c_void_p),
                ("dpreds", C.c_void_p), ("dW", _P6), ("db", _P6), ("dgamma", _P6), ("dbeta", _P6),
                ("dWo", C.c_void_p), ("dbo", C.c_void_p), ("dWi", C.c_void_p), ("dbi", C.c_void_p),
                ("dWc", C.c_void_p), ("dbc", C.c_void_p), ("d_img_f", C.c_void_p), ("scratch", C.c_void_p)]


class CoxArgs(C.Structure):
    _fields_ = [("h", C.c_void_p), ("h_seg_stride", C.c_longlong), ("h_stride", C.c_longlong),
                ("key", C.c_void_p), ("key_seg_stride", C.c_longlong), ("key_stride", C.c_longlong),
                ("w", C.c_void_p), ("w_seg_stride", C.c_longlong), ("w_stride", C.c_longlong),
                ("perm", C.c_void_p), ("N", C.c_int), ("S", C.c_int), ("eps", C.c_float),
                ("loss", C.c_void_p), ("grad", C.c_void_p)]


class CindexArgs(C.Structure):
    _fields_ = [("rank", C.c_void_p), ("is_death", C.c_void_p), ("group_end", C.c_void_p), ("orig", C.c_void_p),
                ("resample", C.c_void_p), ("N", C.c_int), ("R", C.c_int), ("nranks", C.c_int), ("counts", C.c_void_p)]


class GradcamArgs(C.Structure):      # csrc/heads.cu
    _fields_ = [("act", C.c_void_p), ("y", C.c_void_p), ("gamma5", C.c_void_p), ("rvar5", C.c_void_p), ("Wf", C.c_void_p),
                ("Wo", C.c_void_p), ("maps", C.c_void_p), ("eps", C.c_float)] + \
               [(n, C.c_int) for n in ("Ctot", "coff", "B", "C", "F", "d", "h", "w", "X", "Y", "Z")]


class PackDesc(C.Structure):
    _fields_ = [("src", C.c_void_p), ("dst", C.c_void_p), ("N", C.c_int), ("NT", C.c_int), ("Cin", C.c_int),
                ("kbw", C.c_int), ("ntaps", C.c_int), ("mode", C.c_int), ("cin_real", C.c_int), ("f16", C.c_int),
                ("sn", C.c_longlong), ("sc", C.c_longlong), ("st", C.c_longlong)]


class RnConvGeom(C.Structure):
    """csrc/resnet.cu RnConvGeom: channels-last conv geometry (input N,Di,Hi,Wi,Cin -> output Do,Ho,Wo,Cout; kernel, stride, pad)."""
    _fields_ = [(n, C.c_int) for n in ("N", "Di", "Hi", "Wi", "Cin", "Do", "Ho", "Wo", "Cout", "kd", "kh", "kw", "sd", "sh",
                                       "sw", "pd", "ph", "pw")]


A_LINEAR_CONV, A_STEM = 0, 1
T_NONE, T_BNRELU, T_BNBWD = 0, 1, 2
EP_STORE, EP_STORE_STATS, EP_MASK_STATS, EP_MASK_STATS_ACC = 0, 1, 2, 3
PACK_GENERIC, PACK_STEM, PACK_STEM_SW32 = 0, 1, 2


AUG_HIST_POINTS = 10


class AugSpatial(C.Structure):        # csrc/augment.cu
    _fields_ = [("a", C.c_float * 9), ("t", C.c_float * 3)]


class AugIntensity(C.Structure):      # csrc/augment.cu
    _fields_ = [("shift", C.c_float), ("gamma", C.c_float), ("noise_std", C.c_float), ("hist_on", C.c_int),
                ("hist_ref", C.c_float * AUG_HIST_POINTS), ("hist_flt", C.c_float * AUG_HIST_POINTS), ("seed", C.c_ulonglong)]


def _declare(l):
    l.mmnn_conv_rows.argtypes = [C.POINTER(RowsParams), C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]
    l.mmnn_act_is_fp16.restype = C.c_int
    l.mmnn_conv_rows.restype = C.c_int
    l.mmnn_pack_weights.argtypes = [C.POINTER(PackDesc), C.c_int, C.c_void_p, C.c_void_p]
    l.mmnn_pack_weights.restype = C.c_int
    l.mmnn_conv3_brick.argtypes = [C.POINTER(BrickParams), C.c_int, C.c_void_p]
    l.mmnn_conv3_brick.restype = C.c_int
    assert l.mmnn_sizeof_brick_params() == C.sizeof(BrickParams), (l.mmnn_sizeof_brick_params(), C.sizeof(BrickParams))
    l.mmnn_stem_brick.argtypes = [C.POINTER(StemBrickParams), C.c_void_p]
    l.mmnn_stem_brick.restype = C.c_int
    assert l.mmnn_sizeof_stem_brick_params() == C.sizeof(StemBrickParams), (l.mmnn_sizeof_stem_brick_params(), C.sizeof(StemBrickParams))
    l.mmnn_conv_wgrad.argtypes = [C.POINTER(WgradParams), C.c_int, C.c_int, C.c_void_p]
    l.mmnn_conv_wgrad.restype = C.c_int
    assert l.mmnn_sizeof_wgrad_params() == C.sizeof(WgradParams), (l.mmnn_sizeof_wgrad_params(), C.sizeof(WgradParams))
    VP, I, LL = C.c_void_p, C.c_int, C.c_longlong
    l.mmnn_encoder_create.argtypes = [I, C.POINTER(I), I, I, I, I]
    l.mmnn_encoder_create.restype = VP
    l.mmnn_encoder_destroy.argtypes = [VP]
    l.mmnn_encoder_destroy.restype = None
    for name in ("mmnn_encoder_num_params", "mmnn_encoder_num_buffers", "mmnn_encoder_num_layers", "mmnn_encoder_out_channels"):
        getattr(l, name).argtypes = [VP]
        getattr(l, name).restype = I
    l.mmnn_encoder_param_numel.argtypes = [VP, I]
    l.mmnn_encoder_param_numel.restype = LL
    l.mmnn_encoder_workspace_bytes.argtypes = [VP, I, I, I, I]
    l.mmnn_encoder_workspace_bytes.restype = LL
    l.mmnn_encoder_out_dims.argtypes = [VP, I, I, I, I, C.POINTER(I)]
    l.mmnn_encoder_out_dims.restype = I
    l.mmnn_encoder_forward.argtypes = [VP, I, I, I, I, VP, C.POINTER(VP), C.POINTER(VP), VP, VP, VP, I, VP]
    l.mmnn_encoder_forward.restype = I
    l.mmnn_encoder_forward_f16.argtypes = [VP, I, I, I, I, VP, C.POINTER(VP), C.POINTER(VP), VP, VP, VP, I, VP]
    l.mmnn_encoder_forward_f16.restype = I
    l.mmnn_encoder_backward.argtypes = [VP, I, I, I, I, C.POINTER(VP), C.POINTER(VP), C.POINTER(VP), VP, VP, VP, I, VP]
    l.mmnn_encoder_backward.restype = I
    l.mmnn_encoder_num_grad_groups.argtypes = [VP]
    l.mmnn_encoder_num_grad_groups.restype = I
    l.mmnn_encoder_grad_group_range.argtypes = [VP, I, C.POINTER(LL), C.POINTER(LL)]
    l.mmnn_encoder_grad_group_range.restype = I
    l.mmnn_encoder_wait_grad_group.argtypes = [VP, I, VP]
    l.mmnn_encoder_wait_grad_group.restype = I
    l.mmnn_encoder_debug_offsets.argtypes = [VP, I, I, I, I, C.POINTER(LL), C.POINTER(LL)]
    l.mmnn_encoder_debug_offsets.restype = I
    l.mmnn_mlp_heads.argtypes = [C.POINTER(MlpArgs), I, VP]
    l.mmnn_mlp_heads.restype = I
    l.mmnn_cox_nll.argtypes = [C.POINTER(CoxArgs), VP]
    l.mmnn_cox_nll.restype = I
    l.mmnn_cindex_bootstrap.argtypes = [C.POINTER(CindexArgs), VP]
    l.mmnn_cindex_bootstrap.restype = I
    l.mmnn_gradcam_maps.argtypes = [C.POINTER(GradcamArgs), VP]
    l.mmnn_gradcam_maps.restype = I
    l.mmnn_gradcam_ctas.argtypes = [C.POINTER(GradcamArgs)]
    l.mmnn_gradcam_ctas.restype = LL
    for nm, st in (("mmnn_sizeof_mlp_args", MlpArgs), ("mmnn_sizeof_cox_args", CoxArgs), ("mmnn_sizeof_cindex_args", CindexArgs),
                   ("mmnn_sizeof_gradcam_args", GradcamArgs)):
        getattr(l, nm).restype = I
        assert getattr(l, nm)() == C.sizeof(st), (nm, getattr(l, nm)(), C.sizeof(st))
    l.mmnn_sgd_step.argtypes = [C.POINTER(VP), C.POINTER(VP), C.POINTER(VP), C.POINTER(LL), I, C.c_float, C.c_float, C.c_float, I, VP]
    l.mmnn_sgd_step.restype = I
    l.mmnn_sgd_step_dev.argtypes = [C.POINTER(VP), C.POINTER(VP), C.POINTER(VP), C.POINTER(LL), I, VP, I, VP]
    l.mmnn_sgd_step_dev.restype = I
    l.mmnn_sgd_chunk_elems.restype = I
    l.mmnn_sgd_max_tensors.restype = I
    l.mmnn_bce_logits.argtypes = [VP, VP, VP, LL, I, LL, VP, VP, C.c_float, LL, VP, VP]
    l.mmnn_bce_logits.restype = I
    l.mmnn_preprocess_volumes.argtypes = [VP, VP, VP, I, I, I, I, I, I, I, I, C.c_float, C.c_float, VP]
    l.mmnn_preprocess_volumes.restype = I
    l.mmnn_augment_resample.argtypes = [VP, VP, VP, VP, I, I, I, I, I, I, I, I, C.c_float, C.c_float, VP]
    l.mmnn_augment_resample.restype = I
    l.mmnn_augment_intensity.argtypes = [VP, VP, VP, VP, VP, VP, I, I, I, I, I, I, I, VP]
    l.mmnn_augment_intensity.restype = I
    l.mmnn_sizeof_aug_spatial.restype = I
    l.mmnn_sizeof_aug_intensity.restype = I
    D, F, ULL, GP = C.c_double, C.c_float, C.c_ulonglong, C.POINTER(RnConvGeom)
    l.mmnn_sizeof_rn_conv_geom.restype = I
    assert l.mmnn_sizeof_rn_conv_geom() == C.sizeof(RnConvGeom), (l.mmnn_sizeof_rn_conv_geom(), C.sizeof(RnConvGeom))
    l.mmnn_rn_conv.argtypes = [GP, I, I, VP, VP, VP, VP, VP, VP]
    l.mmnn_rn_conv_wgrad.argtypes = [GP, I, VP, VP, VP, VP]
    l.mmnn_rn_conv_fwd_ds.argtypes = [GP, VP, VP, VP, VP, VP, VP, VP, VP]
    l.mmnn_rn_conv_dgrad_ds.argtypes = [GP, VP, VP, VP, VP, VP, VP]
    l.mmnn_rn_conv_fwd_ds.restype = I
    l.mmnn_rn_conv_dgrad_ds.restype = I
    l.mmnn_rn_bn_coeffs.argtypes = [VP, D, VP, VP, VP, VP, VP, F, F, I, I, VP, VP]
    l.mmnn_rn_bn_act.argtypes = [VP, VP, I, VP, VP, VP, LL, I, I, F, ULL, VP, VP]
    l.mmnn_rn_act_bwd_reduce.argtypes = [VP, VP, F, VP, VP, VP, VP, VP, LL, I, VP]
    l.mmnn_rn_bn_bwd_apply.argtypes = [VP, VP, F, VP, VP, VP, VP, VP, D, I, VP, VP, VP, VP, VP, VP, VP, LL, I, VP]
    l.mmnn_rn_head_fwd.argtypes = [VP, I, I, I, VP, VP, I, VP, VP, VP]
    l.mmnn_rn_head_bwd.argtypes = [VP, VP, VP, VP, I, I, I, I, VP, VP, VP, VP]
    for nm in ("mmnn_rn_conv", "mmnn_rn_conv_wgrad", "mmnn_rn_bn_coeffs", "mmnn_rn_bn_act", "mmnn_rn_act_bwd_reduce",
               "mmnn_rn_bn_bwd_apply", "mmnn_rn_head_fwd", "mmnn_rn_head_bwd"):
        getattr(l, nm).restype = I
    l.mmnn_profile_enable.argtypes = [I]
    l.mmnn_profile_enable.restype = None
    l.mmnn_launch_count.restype = LL
    l.mmnn_profile_collect.argtypes = [C.POINTER(C.c_float), C.POINTER(I)]
    l.mmnn_profile_collect.restype = I
    F32P = VP
    l.mmnn_gap_linear_fwd.argtypes = [F32P, I, I, I, F32P, F32P, F32P, I, F32P, F32P, VP]
    l.mmnn_gap_linear_fwd.restype = I
    l.mmnn_gap_linear_bwd.argtypes = [F32P, F32P, I, I, I, F32P, F32P, F32P, I, F32P, F32P, F32P, VP]
    l.mmnn_gap_linear_bwd.restype = I
    l.mmnn_sizeof_rows_params.restype = C.c_int
    l.mmnn_sizeof_pack_desc.restype = C.c_int
    assert l.mmnn_sizeof_rows_params() == C.sizeof(RowsParams), (l.mmnn_sizeof_rows_params(), C.sizeof(RowsParams))
    assert l.mmnn_sizeof_pack_desc() == C.sizeof(PackDesc), (l.mmnn_sizeof_pack_desc(), C.sizeof(PackDesc))


def check(code, what):
    if code != 0:
        raise MMNNLibraryError(f"{what} failed with status {code}")


def packed_elems(N, NT, Cin, kbw, ntaps):
    kb_per_tap = (Cin + kbw - 1) // kbw
    ntile = (N + NT - 1) // NT
    return ntile * ntaps * kb_per_tap * (kbw // 8) * NT * 8


PROF_CLASSES = ["pack", "s2d", "stem_fprop", "maxpool", "conv1_fprop", "conv2_fprop", "trans_pool", "trans_fprop", "norm5",
                "bn_running", "norm5_bwd", "extract", "conv2_wgrad", "conv2_dgrad", "bn_apply", "conv1_wgrad", "conv1_dgrad",
                "trans_wgrad", "trans_dgrad", "avgpool_bwd", "maxpool_bwd", "stem_wgrad", "tails", "heads", "sgd", "preprocess",
                "rn_fprop", "rn_dgrad", "rn_wgrad", "rn_eltwise", "rn_head"]


def profile_timeline(cap=4096):
    """[(class name, start ms, end ms)] of the launches recorded since mmnn_profile_enable(2)."""
    cls = (C.c_int * cap)(); t0 = (C.c_float * cap)(); t1 = (C.c_float * cap)()
    f = lib().mmnn_profile_timeline
    f.argtypes = [C.POINTER(C.c_int), C.POINTER(C.c_float), C.POINTER(C.c_float), C.c_int]
    f.restype = C.c_int
    n = f(cls, t0, t1, cap)
    return [(PROF_CLASSES[cls[i]], float(t0[i]), float(t1[i])) for i in range(n)]


def profile_collect():
    n = len(PROF_CLASSES)
    ms = (C.c_float * n)()
    cnt = (C.c_int * n)()
    got = lib().mmnn_profile_collect(ms, cnt)
    assert got == n, (got, n)
    return {PROF_CLASSES[i]: (float(ms[i]), int(cnt[i])) for i in range(n)}
