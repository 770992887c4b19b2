"""ctypes binding of libmrn_b200.so (include/mrn_b200.h).  No fallback: a missing library or a failing
call raises -- the product path never routes around the CUDA kernels."""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libmrn_b200.so")

MAX_EXPERTS = 8
PREC_FP32, PREC_BF16 = 0, 1
P_POS_EMBED, P_CONV0_W, P_CONV0_B, P_BN0_W, P_BN0_B, P_BN0_MEAN, P_BN0_VAR = range(7)
P_CONV1_W, P_CONV1_B, P_BN1_W, P_BN1_B, P_BN1_MEAN, P_BN1_VAR = range(7, 13)
P_BLOCK0 = 13
PB_COUNT = 12
(PB_NORM1_W, PB_NORM1_B, PB_QKV_W, PB_QKV_B, PB_PROJ_W, PB_PROJ_B, PB_NORM2_W, PB_NORM2_B, PB_FC1_W, PB_FC1_B,
 PB_FC2_W, PB_FC2_B) = range(12)
P_SUB0 = 13 + 12 * 12
PS_COUNT = 4
PS_CONV_W, PS_CONV_B, PS_NORM_W, PS_NORM_B = range(4)
P_SEQ_W = P_SUB0 + 3 * 4
P_SEQ_B = P_SEQ_W + 1
P_COUNT = P_SEQ_B + 1
ROUTER_NPARAMS = 20
# CRNN pack slots (include/mrn_b200.h MRNB_C_*)
(C_CONV0_W, C_CONV0_B, C_CONV1_W, C_CONV1_B, C_CONV2_W, C_CONV2_B, C_CONV3_W, C_CONV3_B, C_CONV4_W, C_BN4_W, C_BN4_B,
 C_BN4_MEAN, C_BN4_VAR, C_CONV5_W, C_BN5_W, C_BN5_B, C_BN5_MEAN, C_BN5_VAR, C_CONV6_W, C_CONV6_B) = range(20)
C_LSTM0 = 20
CL_COUNT = 5
CL_WIH, CL_WHH, CL_BIAS, CL_LIN_W, CL_LIN_B = range(5)
C_COUNT = C_LSTM0 + 2 * CL_COUNT


class MrnbSvtrPack(C.Structure):
    _fields_ = [("n_experts", C.c_int),
                ("p", C.c_void_p * P_COUNT),
                ("h", C.c_void_p * P_COUNT),
                ("fc_w", C.c_void_p * MAX_EXPERTS),
                ("fc_w16", C.c_void_p * MAX_EXPERTS),
                ("fc_b", C.c_void_p * MAX_EXPERTS),
                ("n_class", C.c_int * MAX_EXPERTS)]


class MrnbCrnnPack(C.Structure):
    _fields_ = [("n_experts", C.c_int),
                ("p", C.c_void_p * C_COUNT),
                ("h", C.c_void_p * C_COUNT),
                ("fc_w", C.c_void_p * MAX_EXPERTS),
                ("fc_w16", C.c_void_p * MAX_EXPERTS),
                ("fc_b", C.c_void_p * MAX_EXPERTS),
                ("n_class", C.c_int * MAX_EXPERTS)]


# CRNN training pack slots (include/mrn_b200.h MRNB_T_*)
(T_CONV0_W, T_CONV0_B, T_CONV1_W, T_CONV1_B, T_CONV2_W, T_CONV2_B, T_CONV3_W, T_CONV3_B, T_CONV4_W, T_BN4_W, T_BN4_B,
 T_CONV5_W, T_BN5_W, T_BN5_B, T_CONV6_W, T_CONV6_B) = range(16)
T_LSTM0 = 16
TL_COUNT = 6
TL_WIH, TL_WHH, TL_BIH, TL_BHH, TL_LIN_W, TL_LIN_B = range(6)
T_FC_W = T_LSTM0 + 2 * TL_COUNT
T_FC_B = T_FC_W + 1
T_COUNT = T_FC_B + 1


class MrnbCrnnTrainPack(C.Structure):
    _fields_ = [("p", C.c_void_p * T_COUNT),
                ("h", C.c_void_p * T_COUNT),
                ("bn_mean", C.c_void_p * 2),
                ("bn_var", C.c_void_p * 2),
                ("n_class", C.c_int)]


_vp, _i, _l, _f, _sz = C.c_void_p, C.c_int, C.c_long, C.c_float, C.c_size_t

_SIGNATURES = {
    "mrnb_version": (C.c_int, []),
    "mrnb_last_error": (C.c_char_p, []),
    "mrnb_launch_count": (C.c_long, []),
    "mrnb_reset_launch_count": (None, []),
    "mrnb_profile_enable": (None, [_i]),
    "mrnb_profile_reset": (None, []),
    "mrnb_profile_read": (_i, [_i, C.POINTER(C.c_double), C.POINTER(C.c_long), C.POINTER(C.c_double), C.POINTER(C.c_double)]),
    "mrnb_svtr_workspace_bytes": (_sz, [_i, _i, _i, _i]),
    "mrnb_svtr_heads": (_i, [C.POINTER(MrnbSvtrPack), _i, _i, _vp, C.POINTER(_vp), C.POINTER(_l), _vp, _sz, _vp]),
    "mrnb_svtr_experts_forward": (_i, [C.POINTER(MrnbSvtrPack), _vp, _i, _i, _i, _i, _i, _vp, _vp, C.POINTER(_vp),
                                       C.POINTER(_l), _vp, _sz, _vp]),
    "mrnb_svtr_train_workspace_bytes": (_sz, [_i, _i, _i]),
    "mrnb_svtr_train_forward": (_i, [C.POINTER(MrnbSvtrPack), _vp, _i, _i, _i, _i, _vp, _vp, _l, _vp, _sz, _vp]),
    "mrnb_svtr_train_backward": (_i, [C.POINTER(MrnbSvtrPack), C.POINTER(MrnbSvtrPack), _vp, _vp, _l, _i, _i, _i, _vp,
                                      _vp, _l, _vp, _sz, _vp]),
    "mrnb_svtr_train_forward_features": (_i, [C.POINTER(MrnbSvtrPack), _vp, _i, _i, _i, _i, _vp, _vp, _l, _vp, _vp, _sz, _vp]),
    "mrnb_svtr_train_backward_features": (_i, [C.POINTER(MrnbSvtrPack), C.POINTER(MrnbSvtrPack), _vp, _vp, _l, _vp, _i, _i,
                                               _i, _vp, _vp, _l, _vp, _sz, _vp]),
    "mrnb_crnn_train_workspace_bytes": (_sz, [_i, _i, _i]),
    "mrnb_crnn_train_forward": (_i, [C.POINTER(MrnbCrnnTrainPack), _vp, _i, _i, _i, _i, _vp, _l, _vp, _sz, _vp]),
    "mrnb_crnn_train_backward": (_i, [C.POINTER(MrnbCrnnTrainPack), C.POINTER(MrnbCrnnTrainPack), _vp, _l, _i, _i, _i, _vp,
                                      _l, _vp, _sz, _vp]),
    "mrnb_crnn_train_forward_features": (_i, [C.POINTER(MrnbCrnnTrainPack), _vp, _i, _i, _i, _i, _vp, _l, _vp, _vp, _sz, _vp]),
    "mrnb_crnn_train_backward_features": (_i, [C.POINTER(MrnbCrnnTrainPack), C.POINTER(MrnbCrnnTrainPack), _vp, _l, _vp, _i,
                                               _i, _i, _vp, _l, _vp, _sz, _vp]),
    "mrnb_svtr_train_backward_input": (_i, [C.POINTER(MrnbSvtrPack), C.POINTER(MrnbSvtrPack), _vp, _vp, _l, _vp, _i, _i,
                                            _i, _vp, _vp, _l, _vp, _vp, _sz, _vp]),
    "mrnb_crnn_train_backward_input": (_i, [C.POINTER(MrnbCrnnTrainPack), C.POINTER(MrnbCrnnTrainPack), _vp, _l, _vp, _i,
                                            _i, _i, _vp, _l, _vp, _vp, _sz, _vp]),
    "mrnb_svtr_conv0_dimage": (_i, [_vp, _vp, _vp, _i, _vp]),
    "mrnb_crnn_conv0_dimage": (_i, [_vp, _vp, _vp, _i, _vp]),
    "mrnb_crnn_workspace_bytes": (_sz, [_i, _i, _i]),
    "mrnb_crnn_experts_forward": (_i, [C.POINTER(MrnbCrnnPack), _vp, _i, _i, _i, _i, _vp, C.POINTER(_vp), C.POINTER(_l),
                                       _vp, _sz, _vp]),
    "mrnb_router_param_offsets": (_l, [_i, _i, _i, C.POINTER(_l)]),
    "mrnb_router_workspace_bytes": (_sz, [_i, _i, _i, _i, _i]),
    "mrnb_router_forward": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "mrnb_router_backward": (_i, [_vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _vp, _vp, _vp, _sz, _vp]),
    "mrnb_router_backward_dx": (_i, [_vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _sz, _vp]),
    "mrnb_dm_router_backward": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _i, _vp, _vp, _vp, _sz, _vp]),
    "mrnb_gate_combine": (_i, [C.POINTER(_vp), C.POINTER(_l), C.POINTER(_i), _i, _vp, _i, _i, _vp, _l, _vp, _vp, _vp,
                               _vp, _vp, _vp, _i, _vp, _vp, _vp]),
    "mrnb_gate_combine_backward_workspace_bytes": (_sz, [_i, _i, _i]),
    "mrnb_gate_combine_backward": (_i, [C.POINTER(_vp), C.POINTER(_l), C.POINTER(_i), _i, _i, _i, _vp, _l, _vp, _vp, _sz,
                                        _vp]),
    "mrnb_gate_combine_backward_experts": (_i, [C.POINTER(_vp), C.POINTER(_l), C.POINTER(_i), _i, _i, _i, _vp, _l, _vp,
                                                C.POINTER(_vp), C.POINTER(_l), _vp, _vp, _sz, _vp]),
    "mrnb_ctc_lattice": (_i, [_vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _f, _vp, _vp, _vp, _vp, _vp]),
    "mrnb_ctc_dense_grad": (_i, [_vp, _l, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _f, _vp, _l, _vp]),
    "mrnb_greedy_decode": (_i, [_vp, _vp, _i, _i, _vp, _vp, _vp, _vp]),
    "mrnb_ctc_topk": (_i, [C.POINTER(_vp), C.POINTER(_l), C.POINTER(_i), _i, _vp, _vp, _i, _i, _i, _vp, _vp, _vp, _vp]),
    "mrnb_ctc_beam_search": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _i, _vp, _vp, _vp, _vp]),
    "mrnb_resize_workspace_bytes": (_sz, [_i, _i, _i]),
    "mrnb_resize_normalize_rgba": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _vp, _vp, _sz, _vp]),
    "mrnb_clip_adam": (_i, [_vp, _vp, _vp, _vp, _l, _f, _f, _f, _f, _f, _i, _vp, _vp, _vp]),
    "mrnb_linear_f32": (_i, [_vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _vp]),
    "mrnb_linear_bf16": (_i, [_vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _vp]),
    "mrnb_tc_gemm_general": (_i, [_vp, _i, _vp, _i, _vp, _i, _i, _i, _i, _vp]),
    "mrnb_mlp_bf16": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _vp, _vp, _vp, _f, _i, _i, _vp]),
    "mrnb_mixer_bf16": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _f, _i, _i, _i, _vp]),
    "mrnb_layernorm_f32": (_i, [_vp, _vp, _vp, _vp, _l, _i, _f, _vp]),
    "mrnb_svtr_attention_f32": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _i, _i, _vp]),
    "mrnb_svtr_attention_bf16": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _i, _i, _vp]),
    "mrnb_attn_tc_train_forward": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _vp]),
    "mrnb_attn_tc_train_backward": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _vp]),
    "mrnb_cast_f32_to_bf16": (_i, [_vp, _vp, _l, _vp]),
    "mrnb_cast_f32_to_f16": (_i, [_vp, _vp, _l, _vp]),
}

EXPORTED_SYMBOLS = tuple(_SIGNATURES)
_lib = None


def load():
    """Load the shared library (once).  Raises if it has not been built: there is no fallback."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError("libmrn_b200.so is missing (%s): run `python -m mrn_b200.build` or "
                               "__graft_entry__.build(); mrn_b200 has no CPU / PyTorch fallback" % LIB_PATH)
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(lib, name)
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


def check(rc, what=""):
    if rc != 0:
        raise RuntimeError("mrn_b200 %s failed (%d): %s" % (what, rc, load().mrnb_last_error().decode()))
