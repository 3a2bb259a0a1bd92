"""ctypes binding of libavc_b200.so (C ABI in include/avc_b200.h).  Fails loudly when the library is missing."""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libavc_b200.so")

ERR_NOT_RESIDENT = -4
DTYPE_TF32 = 0
DTYPE_BF16 = 1
DTYPE_F16 = 3
ACT_NONE, ACT_RELU, ACT_TANH, ACT_LRELU, ACT_GELU, ACT_LOG10_CLAMP = 0, 1, 2, 3, 4, 5
ACTS = {"none": ACT_NONE, "relu": ACT_RELU, "tanh": ACT_TANH, "lrelu": ACT_LRELU, "gelu": ACT_GELU,
        "log10_clamp": ACT_LOG10_CLAMP}

EXPORTS = ["avc_version", "avc_last_error", "avc_launch_count", "avc_conv_gemm", "avc_lstm_seq", "avc_lstm_seq2", "avc_lstm_seq_ws", "avc_lstm_stack_ws",
           "avc_bilstm_small", "avc_concat_bcast", "avc_linear_l2norm", "avc_linear_rows", "avc_transpose_pad",
           "avc_conv_to_mono_tanh", "avc_gn_stats", "avc_gn_pool_residual", "avc_gn_apply", "avc_patchify",
           "avc_ln_transpose", "avc_meta_decoder_input", "avc_gather_codes", "avc_global_stats", "avc_adain", "avc_audio_frames",
           "avc_complex_mag", "avc_resblock", "avc_resblock2", "avc_reflect_halo", "avc_bn_batch_stats", "avc_bn_apply",
           "avc_zero_tail", "avc_segment_stats", "avc_adain_segmented"]


MAX_SOURCES = 4


class GemmDesc(ctypes.Structure):
    """struct avc_gemm_desc"""
    _fields_ = [
        ("a_ptr", ctypes.c_void_p * MAX_SOURCES),
        ("a_channels", ctypes.c_int * MAX_SOURCES),
        ("a_ld", ctypes.c_longlong * MAX_SOURCES),
        ("a_rows_per_utt", ctypes.c_int * MAX_SOURCES),
        ("a_taps", ctypes.c_int * MAX_SOURCES),
        ("a_tap_t0", ctypes.c_int * MAX_SOURCES),
        ("a_tap_dt", ctypes.c_int * MAX_SOURCES),
        ("w_ptr", ctypes.c_void_p),
        ("n_pad", ctypes.c_int),
        ("k_pad", ctypes.c_int),
        ("dtype", ctypes.c_int),
        ("B", ctypes.c_int),
        ("T", ctypes.c_int),
        ("N", ctypes.c_int),
        ("bias", ctypes.c_void_p),
        ("act", ctypes.c_int),
        ("out_phases", ctypes.c_int),
        ("out", ctypes.c_void_p),
        ("out_ld", ctypes.c_longlong),
        ("out_rows_per_utt", ctypes.c_int),
        ("out_row0", ctypes.c_int),
        ("out_dtype", ctypes.c_int),
        ("out_round_tf32", ctypes.c_int),
        ("out_reflect", ctypes.c_int),
        ("out_raw", ctypes.c_void_p),
        ("out_raw_ld", ctypes.c_longlong),
        ("out2", ctypes.c_void_p),
        ("out2_ld", ctypes.c_longlong),
        ("residual", ctypes.c_void_p),
        ("res_ld", ctypes.c_longlong),
        ("res_after_act", ctypes.c_int),
        ("block_n", ctypes.c_int),
        ("cta_group", ctypes.c_int),
        ("debug_clk", ctypes.c_void_p),
        ("out_raw_dtype", ctypes.c_int),
        ("out_phase0", ctypes.c_int),
        ("out_phase_count", ctypes.c_int),
    ]


class LstmDesc(ctypes.Structure):
    """struct avc_lstm_desc"""
    _fields_ = [
        ("xproj", ctypes.c_void_p),
        ("w_hh", ctypes.c_void_p),
        ("hseq", ctypes.c_void_p),
        ("hseq_f32", ctypes.c_void_p),
        ("h_last", ctypes.c_void_p),
        ("c_state", ctypes.c_void_p),
        ("B", ctypes.c_int),
        ("T", ctypes.c_int),
        ("H", ctypes.c_int),
        ("dtype", ctypes.c_int),
        ("gate_group", ctypes.c_int),
        ("persistent", ctypes.c_int),
        ("grid_barrier", ctypes.c_void_p),
        ("debug_clk", ctypes.c_void_p),
        ("xin", ctypes.c_void_p),
        ("xin_channels", ctypes.c_int),
        ("xin_ld", ctypes.c_longlong),
        ("w_ih", ctypes.c_void_p),
        ("bias", ctypes.c_void_p),
        ("lengths", ctypes.c_void_p),
    ]


class LstmWsDesc(ctypes.Structure):
    """struct avc_lstm_ws_desc"""
    _fields_ = [
        ("xproj", ctypes.c_void_p),
        ("w_hh", ctypes.c_void_p),
        ("hseq", ctypes.c_void_p),
        ("hseq_f32", ctypes.c_void_p),
        ("h_last", ctypes.c_void_p),
        ("grid_barrier", ctypes.c_void_p),
        ("B", ctypes.c_int),
        ("T", ctypes.c_int),
        ("H", ctypes.c_int),
        ("debug_clk", ctypes.c_void_p),
        ("dtype", ctypes.c_int),
        ("lengths", ctypes.c_void_p),
    ]


STACK_MAX_LAYERS = 4


class LstmStackDesc(ctypes.Structure):
    """struct avc_lstm_stack_desc"""
    _fields_ = [
        ("xproj0", ctypes.c_void_p),
        ("w_ih", ctypes.c_void_p * STACK_MAX_LAYERS),
        ("w_hh", ctypes.c_void_p * STACK_MAX_LAYERS),
        ("bias", ctypes.c_void_p * STACK_MAX_LAYERS),
        ("hs", ctypes.c_void_p),
        ("h_last", ctypes.c_void_p),
        ("grid_barrier", ctypes.c_void_p),
        ("B", ctypes.c_int),
        ("T", ctypes.c_int),
        ("H", ctypes.c_int),
        ("L", ctypes.c_int),
        ("debug_clk", ctypes.c_void_p),
        ("lengths", ctypes.c_void_p),
    ]


class ResblockDesc(ctypes.Structure):
    """struct avc_resblock_desc"""
    _fields_ = [
        ("xa", ctypes.c_void_p),
        ("xa_ld", ctypes.c_longlong),
        ("x", ctypes.c_void_p),
        ("x_ld", ctypes.c_longlong),
        ("w", ctypes.c_void_p),
        ("bias3", ctypes.c_void_p),
        ("bias1", ctypes.c_void_p),
        ("B", ctypes.c_int),
        ("L", ctypes.c_int),
        ("C", ctypes.c_int),
        ("dilation", ctypes.c_int),
        ("out", ctypes.c_void_p),
        ("out_ld", ctypes.c_longlong),
        ("out_rows_per_utt", ctypes.c_int),
        ("out_row0", ctypes.c_int),
        ("out_reflect", ctypes.c_int),
        ("out_raw", ctypes.c_void_p),
        ("out_raw_ld", ctypes.c_longlong),
        ("out2", ctypes.c_void_p),
        ("out2_ld", ctypes.c_longlong),
    ]


class Resblock2Desc(ctypes.Structure):
    """struct avc_resblock2_desc"""
    _fields_ = [
        ("x", ctypes.c_void_p),
        ("x_ld", ctypes.c_longlong),
        ("w", ctypes.c_void_p),
        ("bias3", ctypes.c_void_p),
        ("bias1", ctypes.c_void_p),
        ("B", ctypes.c_int),
        ("L", ctypes.c_int),
        ("C", ctypes.c_int),
        ("dilation", ctypes.c_int),
        ("y", ctypes.c_void_p),
        ("y_ld", ctypes.c_longlong),
        ("y_rows_per_utt", ctypes.c_int),
        ("y_row0", ctypes.c_int),
        ("y_reflect", ctypes.c_int),
        ("y_act", ctypes.c_int),
        ("out2", ctypes.c_void_p),
        ("out2_ld", ctypes.c_longlong),
        ("debug_clk", ctypes.c_void_p),
        ("wav", ctypes.c_void_p),
        ("mono_w", ctypes.c_void_p),
        ("mono_bias", ctypes.c_float),
        ("mono_taps", ctypes.c_int),
        ("lengths", ctypes.c_void_p),
        ("tile_start", ctypes.c_void_p),
        ("n_tiles", ctypes.c_int),
    ]


SEGMENT_CHUNK = 4096    # AVC_SEGMENT_CHUNK: avc_segment_stats needs 2 * B * ceil(T * C / SEGMENT_CHUNK) doubles
BN_MAX_PARTS = 256      # AVC_BN_MAX_PARTS: avc_bn_batch_stats needs 2 + 2 * BN_MAX_PARTS * C doubles of scratch


class BnApplyDesc(ctypes.Structure):
    """struct avc_bn_apply_desc"""
    _fields_ = [
        ("v", ctypes.c_void_p),
        ("v_ld", ctypes.c_longlong),
        ("scale_shift", ctypes.c_void_p),
        ("B", ctypes.c_int),
        ("T", ctypes.c_int),
        ("C", ctypes.c_int),
        ("act", ctypes.c_int),
        ("residual", ctypes.c_void_p),
        ("res_ld", ctypes.c_longlong),
        ("res_after_act", ctypes.c_int),
        ("out", ctypes.c_void_p),
        ("out_ld", ctypes.c_longlong),
        ("out_rows_per_utt", ctypes.c_int),
        ("out_row0", ctypes.c_int),
        ("out_dtype", ctypes.c_int),
        ("out_round_tf32", ctypes.c_int),
        ("out2", ctypes.c_void_p),
        ("out2_ld", ctypes.c_longlong),
    ]


_lib = None


def load():
    """Load the library once; raise (never fall back) when it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(there is no CPU / PyTorch fallback for the conversion path)")
    lib = ctypes.CDLL(LIB_PATH)
    lib.avc_version.restype = ctypes.c_int
    lib.avc_last_error.restype = ctypes.c_char_p
    lib.avc_launch_count.restype = ctypes.c_longlong
    lib.avc_conv_gemm.argtypes = [ctypes.POINTER(GemmDesc), ctypes.c_void_p]
    lib.avc_conv_gemm.restype = ctypes.c_int
    lib.avc_lstm_seq.argtypes = [ctypes.POINTER(LstmDesc), ctypes.c_void_p]
    lib.avc_lstm_seq.restype = ctypes.c_int
    lib.avc_lstm_seq2.argtypes = [ctypes.POINTER(LstmDesc), ctypes.POINTER(LstmDesc), ctypes.c_void_p]
    lib.avc_lstm_seq2.restype = ctypes.c_int
    lib.avc_lstm_seq_ws.argtypes = [ctypes.POINTER(LstmWsDesc), ctypes.c_void_p]
    lib.avc_lstm_seq_ws.restype = ctypes.c_int
    lib.avc_lstm_stack_ws.argtypes = [ctypes.POINTER(LstmStackDesc), ctypes.c_void_p]
    lib.avc_lstm_stack_ws.restype = ctypes.c_int
    lib.avc_resblock.argtypes = [ctypes.POINTER(ResblockDesc), ctypes.c_void_p]
    lib.avc_resblock.restype = ctypes.c_int
    lib.avc_reflect_halo.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_longlong, ctypes.c_int,
                                     ctypes.c_int, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p]
    lib.avc_reflect_halo.restype = ctypes.c_int
    lib.avc_zero_tail.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_longlong, ctypes.c_int,
                                  ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p]
    lib.avc_zero_tail.restype = ctypes.c_int
    lib.avc_resblock2.argtypes = [ctypes.POINTER(Resblock2Desc), ctypes.c_void_p]
    lib.avc_resblock2.restype = ctypes.c_int
    lib.avc_bilstm_small.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_int,
                                     ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                     ctypes.c_void_p, ctypes.c_void_p]
    lib.avc_bilstm_small.restype = ctypes.c_int
    lib.avc_concat_bcast.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_int,
                                     ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                     ctypes.c_void_p]
    lib.avc_concat_bcast.restype = ctypes.c_int
    lib.avc_linear_l2norm.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p,
                                      ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_void_p]
    lib.avc_linear_l2norm.restype = ctypes.c_int
    lib.avc_linear_rows.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p,
                                    ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_void_p]
    lib.avc_linear_rows.restype = ctypes.c_int
    lib.avc_transpose_pad.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                      ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_void_p]
    lib.avc_transpose_pad.restype = ctypes.c_int
    lib.avc_conv_to_mono_tanh.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_float, ctypes.c_void_p,
                                          ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_void_p,
                                          ctypes.c_void_p]
    lib.avc_conv_to_mono_tanh.restype = ctypes.c_int
    vp, ci = ctypes.c_void_p, ctypes.c_int
    lib.avc_gn_stats.argtypes = [vp, vp, ci, ctypes.c_longlong, ctypes.c_float, vp]
    lib.avc_gn_pool_residual.argtypes = [vp, vp, vp, vp, vp, ci, ci, ci, ci, ci, vp]
    lib.avc_gn_apply.argtypes = [vp, vp, vp, vp, vp, ci, ci, ci, ci, ci, vp]
    lib.avc_patchify.argtypes = [vp, vp, vp, vp, vp, ci, ci, ci, ci, ci, vp]
    lib.avc_ln_transpose.argtypes = [vp, vp, vp, ci, vp, ci, ci, vp, vp, ci, ci, ci, vp]
    lib.avc_meta_decoder_input.argtypes = [vp, vp, vp, ci, ci, ci, ci, ci, ci, ci, vp]
    lib.avc_gather_codes.argtypes = [vp, vp, ci, ci, ci, ci, vp]
    lib.avc_global_stats.argtypes = [vp, ctypes.c_longlong, vp, vp, vp]
    lib.avc_adain.argtypes = [vp, vp, vp, vp, vp, ci, ci, ctypes.c_longlong, ci, vp]
    lib.avc_global_stats.restype = lib.avc_adain.restype = ctypes.c_int
    lib.avc_segment_stats.argtypes = [vp, ci, ci, ci, vp, vp, vp, vp]
    lib.avc_adain_segmented.argtypes = [vp, vp, vp, ci, vp, vp, vp, ci, ci, ci, ci, ci, vp]
    lib.avc_segment_stats.restype = lib.avc_adain_segmented.restype = ctypes.c_int
    lib.avc_audio_frames.argtypes = [vp, vp, ci, ctypes.c_longlong, ci, ci, ci, ci, ci, vp]
    lib.avc_complex_mag.argtypes = [vp, vp, ctypes.c_longlong, ci, ci, ci, ci, vp]
    lib.avc_audio_frames.restype = lib.avc_complex_mag.restype = ctypes.c_int
    lib.avc_bn_batch_stats.argtypes = [vp, ctypes.c_longlong, ci, ctypes.c_longlong, vp, vp, ctypes.c_float,
                                       ctypes.c_float, ci, vp, vp, vp, vp, vp, vp]
    lib.avc_bn_apply.argtypes = [ctypes.POINTER(BnApplyDesc), vp]
    lib.avc_bn_batch_stats.restype = lib.avc_bn_apply.restype = ctypes.c_int
    for fn in (lib.avc_gn_stats, lib.avc_gn_pool_residual, lib.avc_gn_apply, lib.avc_patchify, lib.avc_ln_transpose,
               lib.avc_meta_decoder_input, lib.avc_gather_codes):
        fn.restype = ctypes.c_int
    _lib = lib
    return lib


def check(rc, what):
    if rc != 0:
        msg = load().avc_last_error().decode("utf-8", "replace")
        raise RuntimeError(f"{what} failed ({rc}): {msg}")


def launch_count():
    return int(load().avc_launch_count())
