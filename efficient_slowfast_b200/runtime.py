"""ctypes binding of libesf_b200.so (C ABI: include/esf.h).  There is no fallback: if the library is missing or a
call fails this module raises."""
import ctypes
import os

import torch

_LIB = None
_LIB_PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "csrc", "libesf_b200.so")

ACT_NONE, ACT_RELU, ACT_RELU6 = 0, 1, 2
BF16, F32, F16 = 0, 1, 2
_DTYPE_CODE = {torch.bfloat16: BF16, torch.float32: F32, torch.float16: F16}
TORCH_DTYPE = {"bf16": torch.bfloat16, "fp16": torch.float16, "fp32": torch.float16}   # "fp32": FP16 hi/lo operand pairs
HEAD_NONE, HEAD_SOFTMAX, HEAD_RELU, HEAD_SIGMOID, HEAD_HARD_SIGMOID = 0, 1, 2, 3, 4


class EsfView(ctypes.Structure):
    _fields_ = [("ptr", ctypes.c_void_p), ("B", ctypes.c_int32), ("T", ctypes.c_int32), ("H", ctypes.c_int32),
                ("W", ctypes.c_int32), ("C", ctypes.c_int32), ("sB", ctypes.c_int64), ("sT", ctypes.c_int64),
                ("sH", ctypes.c_int64), ("sW", ctypes.c_int64), ("dtype", ctypes.c_int32)]


class EsfConvDesc(ctypes.Structure):
    _fields_ = [("x", EsfView), ("y", EsfView), ("res", EsfView), ("w", ctypes.c_void_p), ("bias", ctypes.c_void_p),
                ("kT", ctypes.c_int32), ("kH", ctypes.c_int32), ("kW", ctypes.c_int32),
                ("sT", ctypes.c_int32), ("sH", ctypes.c_int32), ("sW", ctypes.c_int32),
                ("pT", ctypes.c_int32), ("pH", ctypes.c_int32), ("pW", ctypes.c_int32),
                ("dT", ctypes.c_int32), ("dH", ctypes.c_int32), ("dW", ctypes.c_int32),
                ("groups", ctypes.c_int32), ("act", ctypes.c_int32), ("out_dtype", ctypes.c_int32)]


class EsfError(RuntimeError):
    pass


def lib_path():
    return _LIB_PATH


def lib():
    """Load the shared library once; raises EsfError when it has not been built (python -m
    efficient_slowfast_b200._build, or __graft_entry__.build())."""
    global _LIB
    if _LIB is not None:
        return _LIB
    if not os.path.exists(_LIB_PATH):
        raise EsfError("libesf_b200.so not found at %s -- build it with `python -m efficient_slowfast_b200._build` "
                       "(there is no CPU or PyTorch fallback for the forward path)" % _LIB_PATH)
    # a library older than its sources must not be used silently: the stamp written by _build holds the digest of the
    # sources + flags it was compiled from
    from . import _build
    stamp = _LIB_PATH + ".stamp"
    if not os.path.exists(stamp) or open(stamp).read().strip() != _build._digest():
        try:
            _build.build()
        except Exception as e:  # noqa: BLE001
            raise EsfError("libesf_b200.so is older than csrc/ (digest mismatch) and the rebuild failed: %s" % e)
    L = ctypes.CDLL(_LIB_PATH)
    vp, i32, i64, f32 = ctypes.c_void_p, ctypes.c_int32, ctypes.c_int64, ctypes.c_float
    P = ctypes.POINTER
    L.esf_last_error.restype = ctypes.c_char_p
    L.esf_last_error.argtypes = []
    L.esf_launch_count.restype = i64
    L.esf_igemm_geometry.argtypes = [i32, i32, P(i32), P(i32), P(i32), P(i32)]
    L.esf_conv_igemm_create.argtypes = [P(EsfConvDesc), P(vp)]
    L.esf_gemm_clip_weights_create.argtypes = [P(EsfConvDesc), P(vp)]
    L.esf_conv_wfold_create.argtypes = [P(EsfConvDesc), ctypes.c_int32, P(vp)]
    L.esf_op_launch.argtypes = [vp, vp]
    L.esf_op_destroy.argtypes = [vp]
    L.esf_op_destroy.restype = None
    L.esf_conv_direct.argtypes = [P(EsfConvDesc), vp]
    L.esf_stem_conv.argtypes = [vp, i32, i32, i32, i32, i32, vp, vp, i32, i32, i32, i32, i32, i32, i32, i32, i32, i32,
                                i32, P(EsfView), vp]
    L.esf_stem_geometry.argtypes = [i32, i32, i32, i32, i32, P(i32), P(i32), P(i32)]
    L.esf_stem_pack.argtypes = [vp, i32, i32, i32, i32, i32, i32, i32, i32, vp, vp]
    L.esf_stem_pack_gather.argtypes = [vp, i32, i32, i32, i32, i32, vp, i32, i32, i32, i32, vp, vp]
    L.esf_row_softmax.argtypes = [vp, i64, i32, i64, f32, i32, i32, vp, i64, vp]
    L.esf_transpose16.argtypes = [vp, i32, i32, i32, i64, i64, vp, i64, i64, vp]
    L.esf_global_mean_scratch_floats.argtypes = [i32, i32]
    L.esf_global_mean_scratch_floats.restype = ctypes.c_int64
    L.esf_global_mean.argtypes = [P(EsfView), vp, vp, i32, i32, vp]
    L.esf_dwconv_padded.argtypes = [P(EsfConvDesc), i32, vp]
    L.esf_pointwise_padded.argtypes = [P(EsfConvDesc), i32, vp]
    L.esf_group_mean.argtypes = [vp, i32, i32, i32, vp, vp]
    L.esf_stem_pack_u8.argtypes = [vp, i32, i32, i32, i32, i32, vp, i32, P(i32), vp, i32, i32, vp, vp]
    L.esf_frames_to_clip.argtypes = [vp, i32, i32, i32, i32, i32, vp, i32, P(i32), vp, vp, vp]
    L.esf_stem_pack_u8_rings.argtypes = [vp, i32, i32, i32, i32, i32, vp, P(i32), i32, vp, P(i32), i32, P(i32), vp, i32,
                                         i32, vp, vp]
    L.esf_frames_to_clip_rings.argtypes = [vp, i32, i32, i32, i32, i32, vp, P(i32), i32, vp, P(i32), i32, P(i32), vp,
                                           vp, vp]
    L.esf_stem_pack_u8_crop.argtypes = [vp, i32, i32, i32, i32, i32, vp, i32, P(i32), vp, vp, vp, i32, vp, vp, i32,
                                        P(i32), i32, i32, i32, i32, i32, vp, vp]
    L.esf_frames_to_clip_crop.argtypes = [vp, i32, i32, i32, i32, i32, vp, i32, P(i32), vp, vp, vp, i32, vp, vp, i32,
                                          P(i32), i32, i32, vp, vp]
    L.esf_stem_pack_u8_crop_ragged.argtypes = [vp, i32, i32, i32, vp, i32, P(i32), vp, P(i32), vp, P(i32), i32, i32, i32,
                                               i32, i32, vp, vp]
    L.esf_frames_to_clip_crop_ragged.argtypes = [vp, i32, i32, i32, vp, i32, P(i32), vp, P(i32), vp, P(i32), i32, i32,
                                                 vp, vp]
    L.esf_stem_pack_u8_crop_videos.argtypes = [vp, i32, i32, vp, i32, P(i32), vp, P(i32), vp, P(i32), i32, i32, i32, i32,
                                               i32, vp, vp]
    L.esf_frames_to_clip_crop_videos.argtypes = [vp, i32, i32, vp, i32, P(i32), vp, P(i32), vp, P(i32), i32, i32, vp, vp]
    L.esf_stem_pack_u8_ava.argtypes = [vp, i32, i32, i32, i32, i32, vp, i32, P(i32), vp, vp, vp, vp, vp, i32, vp, vp, i32,
                                       i32, i32, i32, vp, vp]
    L.esf_frames_to_clip_ava.argtypes = [vp, i32, i32, i32, i32, i32, vp, i32, P(i32), vp, vp, vp, vp, vp, i32, vp, vp,
                                         i32, vp, vp]
    L.esf_ava_boxes.argtypes = [vp, i32, i32, i32, i32, i32, i32, i32, vp, vp]
    L.esf_resize_u8_cv2.argtypes = [vp, vp, P(i32), vp, i32, i32, vp]
    L.esf_jpeg_scratch_bytes.argtypes = [vp, i32, i32, vp]
    L.esf_jpeg_decode.argtypes = [vp, i64, vp, i32, vp, i32, i32, i32, vp, i64, vp, i32, i32, i32, i32, vp, vp]
    L.esf_stem_igemm_create.argtypes = [vp, i32, i32, i32, i32, i32, i32, vp, vp, i32, i32, i32, i32, i32, i32, i32,
                                        i32, i32, i32, P(EsfView), P(vp)]
    L.esf_stem_tband_create.argtypes = L.esf_stem_igemm_create.argtypes
    L.esf_stem_tband_wb.argtypes = [i32] * 8
    L.esf_pool3d.argtypes = [P(EsfView), P(EsfView), i32, i32, i32, i32, i32, i32, i32, i32, i32, i32, i32, vp]
    L.esf_shuffle_concat.argtypes = [P(EsfView), P(EsfView), i32, P(EsfView), vp]
    L.esf_eltwise_add.argtypes = [P(EsfView), P(EsfView), P(EsfView), i32, vp]
    L.esf_channel_scale.argtypes = [P(EsfView), vp, P(EsfView), vp]
    L.esf_eca_scratch_floats.argtypes = [i32, i32]
    L.esf_eca_scratch_floats.restype = i64
    L.esf_eca_fuse.argtypes = [P(EsfView), i32, vp, i32, vp, vp, vp, P(EsfView), vp]
    L.esf_attn_tc_pack_bytes.argtypes = [i32, i32, i32]
    L.esf_attn_tc_pack_bytes.restype = i64
    L.esf_attn_tc_pack.argtypes = [vp, i32, i32, i32, i32, vp, vp]
    L.esf_attn_tc_create.argtypes = [vp, i32, i32, i32, i32, i32, f32, vp, vp, i32, P(EsfView), P(vp)]
    L.esf_attn_tc_vlo_bytes.argtypes = [i32, i32, i32]
    L.esf_attn_tc_vlo_bytes.restype = i64
    L.esf_attn_tc_pack_vlo.argtypes = [vp, i32, i32, i32, vp, vp]
    L.esf_attn_tc_create_split.argtypes = [vp, vp, i32, i32, i32, i32, i32, f32, vp, vp, i32, P(EsfView), P(vp)]
    L.esf_attn_generic.argtypes = [vp, i32, i32, i32, i32, i32, f32, vp, vp, i32, P(EsfView), vp]
    L.esf_head_pool.argtypes = [P(EsfView), P(EsfView), vp, vp]
    L.esf_head_fc.argtypes = [vp, i32, i32, i32, vp, vp, i32, i32, vp, i32, vp]
    L.esf_temporal_mean.argtypes = [P(EsfView), vp, vp]
    L.esf_roi_align_max.argtypes = [vp, i32, i32, i32, i32, vp, i32, f32, i32, i32, vp, i32, i32, vp]
    L.esf_p32_post.argtypes = [P(EsfView), vp, vp, P(EsfView), i32, P(EsfView), P(EsfView), i32, i32, vp]
    L.esf_p32_post3.argtypes = [P(EsfView), P(EsfView), P(EsfView), vp, vp, i32, P(EsfView), P(EsfView), i32, vp]
    L.esf_stem_pack_lo.argtypes = [vp, i32, i32, i32, i32, i32, i32, i32, i32, vp, vp]
    L.esf_p32_row_softmax.argtypes = [vp, i64, i32, i64, f32, i32, vp, i64, i32, vp]
    L.esf_p32_pool3d.argtypes = [P(EsfView), P(EsfView), i32, i32, i32, i32, i32, i32, i32, i32, i32, i32, vp]
    L.esf_p32_eca_scratch_floats.argtypes = [i32, i32]
    L.esf_p32_eca_scratch_floats.restype = i64
    L.esf_p32_eca_fuse.argtypes = [P(EsfView), i32, vp, i32, vp, vp, vp, P(EsfView), vp]
    L.esf_p32_head_pool.argtypes = [P(EsfView), vp, i32, i32, vp]
    L.esf_p32_attention.argtypes = [vp, i32, i32, i32, i32, i32, f32, vp, vp, i32, P(EsfView), vp]
    _LIB = L
    return L


def check(rc, what=""):
    if rc != 0:
        msg = lib().esf_last_error().decode("utf-8", "replace")
        raise EsfError("%s failed (%d): %s" % (what or "libesf_b200 call", rc, msg))


def launch_count():
    return int(lib().esf_launch_count())


def view(t):
    """esf_view of a channels-last activation tensor (B,T,H,W,C), possibly a channel slice of a wider buffer."""
    assert t.dim() == 5 and t.stride(4) == 1, "activation views are (B,T,H,W,C) with unit channel stride"
    B, T, H, W, C = t.shape
    sB, sT, sH, sW, _ = t.stride()
    return EsfView(t.data_ptr(), B, T, H, W, C, sB, sT, sH, sW, _DTYPE_CODE[t.dtype])


def null_view():
    return EsfView(None, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0)


def dtype_code(t):
    return _DTYPE_CODE[t.dtype if isinstance(t, torch.Tensor) else t]


def igemm_geometry(cin, cout):
    kc, kch, nt, npad = (ctypes.c_int32() for _ in range(4))
    check(lib().esf_igemm_geometry(cin, cout, ctypes.byref(kc), ctypes.byref(kch), ctypes.byref(nt),
                                   ctypes.byref(npad)), "esf_igemm_geometry")
    return kc.value, kch.value, nt.value, npad.value


def stem_geometry(W, cin, kW, sW, pW):
    """(pitch, lpad, window) of the packed stem rows, or None when the banded-GEMM stem does not apply."""
    pitch, lpad, win = (ctypes.c_int32() for _ in range(3))
    rc = lib().esf_stem_geometry(W, cin, kW, sW, pW, ctypes.byref(pitch), ctypes.byref(lpad), ctypes.byref(win))
    if rc != 0 or ((W + 2 * pW - kW) // sW + 1) % 8 != 0:
        return None
    return pitch.value, lpad.value, win.value


def stem_tband_wb(W, cin, cout, kT, kH, kW, sW, pW):
    """Output-column block of the temporal-band stem kernel (esf_stem_tband_create) for this geometry, 0 when it does not
    apply and the banded stem of esf_stem_igemm_create runs instead."""
    return int(lib().esf_stem_tband_wb(W, cin, cout, kT, kH, kW, sW, pW))


def current_stream_ptr():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
