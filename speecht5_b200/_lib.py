"""ctypes binding of libspeecht5_b200.so (declared in include/speecht5_b200.h).

The product path has NO CPU / PyTorch fallback: if the CUDA library is missing or an entry point fails, we raise.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libspeecht5_b200.so")

F32, BF16 = 0, 1
ACT_NONE, ACT_RELU, ACT_GELU, ACT_TANH, ACT_GELU_TANH = 0, 1, 2, 3, 4
ACT_GATE, ACT_GELU_TANH_GATE = 5, 6  # include/speecht5_b200.h ST5_ACT_GATE / ST5_ACT_GELU_TANH_GATE
ACT_IDS = {None: ACT_NONE, "none": ACT_NONE, "relu": ACT_RELU, "gelu": ACT_GELU, "tanh": ACT_TANH,
           "gelu_tanh": ACT_GELU_TANH, "gate": ACT_GATE, "gelu_tanh_gate": ACT_GELU_TANH_GATE}


class GemmArgs(C.Structure):
    _fields_ = [
        ("M", C.c_int32), ("N", C.c_int32), ("K", C.c_int32), ("nb1", C.c_int32), ("nb2", C.c_int32),
        ("a_mn", C.c_int32), ("b_mn", C.c_int32), ("c_fp32", C.c_int32), ("act", C.c_int32),
        ("accumulate", C.c_int32), ("bias2_rows", C.c_int32),
        ("a", C.c_void_p), ("a_ld", C.c_int64), ("a_bs1", C.c_int64), ("a_bs2", C.c_int64),
        ("b", C.c_void_p), ("b_ld", C.c_int64), ("b_bs1", C.c_int64), ("b_bs2", C.c_int64),
        ("c", C.c_void_p), ("c_ld", C.c_int64), ("c_bs1", C.c_int64), ("c_bs2", C.c_int64),
        ("c_pre", C.c_void_p), ("bias", C.c_void_p), ("bias2", C.c_void_p), ("residual", C.c_void_p),
        ("alpha", C.c_float), ("drop_p", C.c_float), ("drop_seed", C.c_uint64), ("drop_offset", C.c_uint64),
        ("actgrad_pre", C.c_void_p), ("actgrad_act", C.c_int32),
    ]


class AttnArgs(C.Structure):
    _fields_ = [
        ("B", C.c_int32), ("H", C.c_int32), ("Tq", C.c_int32), ("Tk", C.c_int32), ("dtype", C.c_int32),
        ("causal", C.c_int32), ("maxpos", C.c_int32), ("probs_dtype", C.c_int32),
        ("q", C.c_void_p), ("q_ld", C.c_int64), ("q_bs", C.c_int64),
        ("k", C.c_void_p), ("k_ld", C.c_int64), ("k_bs", C.c_int64),
        ("v", C.c_void_p), ("v_ld", C.c_int64), ("v_bs", C.c_int64),
        ("key_pad", C.c_void_p), ("pe_k", C.c_void_p),
        ("out", C.c_void_p), ("o_ld", C.c_int64), ("o_bs", C.c_int64),
        ("probs", C.c_void_p), ("p_ld", C.c_int64),
        ("scale", C.c_float), ("drop_p", C.c_float), ("seed", C.c_uint64), ("offset", C.c_uint64),
        ("dout", C.c_void_p), ("dprobs_ext", C.c_void_p), ("ds", C.c_void_p),
        ("dq", C.c_void_p), ("dk", C.c_void_p), ("dv", C.c_void_p), ("dpe_k", C.c_void_p),
        ("probs_heads", C.c_int32),
    ]


_vp, _i64, _i32, _f, _u64 = C.c_void_p, C.c_int64, C.c_int32, C.c_float, C.c_uint64
_PROTOS = {
    "st5_version": (C.c_int, []),
    "st5_last_error": (C.c_char_p, []),
    "st5_device_ok": (C.c_int, []),
    "st5_gemm_bf16": (C.c_int, [C.POINTER(GemmArgs), _vp]),
    "st5_cast_bf16": (C.c_int, [_vp, _i64, _vp, _vp, _i64, _i64, _i64, _vp]),
    "st5_posenc_fwd": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _i32, _i64, _i64, _i64, _f, _u64, _u64, _vp]),
    "st5_posenc_bwd": (C.c_int, [_vp, _vp, _i64, _vp, _vp, _vp, _vp, _i32, _i64, _i64, _i64, _f, _u64, _u64, _vp]),
    "st5_ln_fwd": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i32, _i64, _i64, _f, _f, _u64, _u64, _vp]),
    "st5_ln_fwd_stream": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i32, _i64, _i64, _f, _f, _u64,
                                    _u64, _vp]),
    "st5_ln_bwd_blocks": (C.c_int64, [_i64]),
    "st5_ln_bwd": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i32, _i64, _i64, _f, _u64, _u64, _vp]),
    "st5_lrelu_pad": (C.c_int, [_vp, _vp, _i64, _i64, _i64, _i64, _i32, _i32, _i32, _f, _vp]),
    "st5_dropout": (C.c_int, [_vp, _vp, _i32, _i64, _f, _u64, _u64, _vp]),
    "st5_act_bwd": (C.c_int, [_vp, _vp, _vp, _i32, _i32, _i64, _f, _u64, _u64, _vp]),
    "st5_colsum": (C.c_int, [_vp, _i64, _vp, _i32, _i64, _i64, _i64, _i32, _vp]),
    "st5_attn_fwd": (C.c_int, [C.POINTER(AttnArgs), _vp]),
    "st5_attn_bwd": (C.c_int, [C.POINTER(AttnArgs), _vp]),
    "st5_attn_fused_fwd": (C.c_int, [C.POINTER(AttnArgs), _vp, _vp, _vp, _vp, _vp]),
    "st5_attn_flash_fwd": (C.c_int, [C.POINTER(AttnArgs), _vp, _vp, _vp, _vp, _vp]),
    "st5_attn_fused_bwd": (C.c_int, [C.POINTER(AttnArgs), _vp, _vp, _vp, _vp, _vp, _i32, _vp]),
    "st5_attn_softmax_fwd": (C.c_int, [_vp, _vp, _i64, _vp, _vp, _vp, _vp, _i32, _i32, _i32, _i32, _i64, _i32, _i32, _f,
                                       _u64, _u64, _vp]),
    "st5_attn_ds": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _i32, _i32, _i32, _i32, _i64, _f, _u64, _u64, _vp]),
    "st5_attn_dqp_scatter": (C.c_int, [_vp, _vp, _i32, _i32, _i32, _i32, _i64, _i32, _i32, _vp]),
    "st5_bn_fwd": (C.c_int, [_vp, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _vp, _i32, _i64, _i64, _i32, _f, _f,
                             _i32, _f, _u64, _u64, _vp, _vp]),
    "st5_bn_bwd": (C.c_int, [_vp, _i64, _vp, _i64, _vp, _vp, _vp, _vp, _vp, _i64, _vp, _vp, _i32, _i64, _i64, _i32,
                             _f, _u64, _u64, _vp, _vp]),
    "st5_conv0_ws_floats": (C.c_int64, [_i32, _i64, _i32, _i32, _i32]),
    "st5_conv0_ln_ws_floats": (C.c_int64, [_i32, _i64, _i32, _i32, _i32]),
    "st5_conv0_ln_gelu_fwd": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _i32, _vp, _vp, _i32, _i64, _i32, _i32, _i32, _f, _i32,
                                        _vp]),
    "st5_conv0_ln_gelu_bwd": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i32, _i32, _i64, _i32,
                                        _i32, _i32, _i32, _vp]),
    "st5_act_fwd": (C.c_int, [_vp, _vp, _i32, _i32, _i64, _vp]),
    "st5_conv0_gn_gelu_fwd": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _i32, _vp, _vp, _vp, _i32, _i64, _i32, _i32, _i32, _f,
                                        _i32, _vp]),
    "st5_conv0_gn_gelu_bwd": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i32, _i32, _i64, _i32,
                                        _i32, _i32, _i32, _vp]),
    "st5_ctc_ws_floats": (C.c_int64, [_i32, _i32, _i32]),
    "st5_ctc_loss": (C.c_int, [_vp, _i64, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i32, _i32, _i32, _i32, _i32, _i32,
                               _vp]),
    "st5_tts_loss_ws_floats": (C.c_int64, [_i32, _i32]),
    "st5_guided_attn_ws_floats": (C.c_int64, [_i32, _i32, _i32, _i32]),
    "st5_tts_loss_fwd": (C.c_int, [_vp, _vp, _vp, _vp, _i64, _vp, _i64, _vp, _i32, _i32, _i32, _i32, _f, _vp, _vp, _vp]),
    "st5_tts_loss_bwd": (C.c_int, [_vp, _vp, _vp, _vp, _i64, _vp, _i64, _vp, _vp, _vp, _i32, _i32, _i32, _i32, _f, _vp,
                                   _vp, _vp, _vp]),
    "st5_guided_attn_fwd": (C.c_int, [_vp, _i32, _i32, _i32, _i32, _i32, _i32, _i64, _vp, _vp, _i32, _f, _f, _vp, _vp,
                                      _vp]),
    "st5_guided_attn_bwd": (C.c_int, [_vp, _i32, _i32, _i32, _i32, _i32, _i32, _i64, _vp, _vp, _i32, _f, _f, _vp, _vp,
                                      _i32, _vp]),
    "st5_ctc_prefix_init": (C.c_int, [_vp, _i64, _i64, _vp, _vp, _i32, _i32, _i32, _i32, _vp]),
    "st5_ctc_prefix_score": (C.c_int, [_vp, _i64, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i32, _i32, _i32, _i32,
                                       _i32, _i32, _vp]),
    "st5_beam_gather_rows": (C.c_int, [_vp, _vp, _vp, _i32, _i32, _i32, _i64, _i64, _i64, _vp]),
    "st5_sumsq": (C.c_int, [_vp, _i64, _vp, _vp]),
    "st5_adam_step": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _i64, _f, _f, _f, _f, _f, _i64, _vp, _f, _f, _vp, _vp, _vp]),
}
EXPORTS = tuple(_PROTOS.keys())

_lib = None


def load():
    """Load the shared library (building nothing: see speecht5_b200.build / __graft_entry__.build)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"speecht5_b200: CUDA library not found at {LIB_PATH}. Run `python -m speecht5_b200.build` "
            "(or __graft_entry__.build()). There is no CPU fallback for the product path.")
    # ST5_LIB: an alternative build of the same ABI (tools/build_variant.sh makes A/B builds for tuning runs)
    lib = C.CDLL(os.environ.get("ST5_LIB") or LIB_PATH)
    for name, (res, args) in _PROTOS.items():
        fn = getattr(lib, name)  # AttributeError if the symbol is missing: fail loudly
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc, what=""):
    if rc != 0:
        msg = load().st5_last_error().decode("utf-8", "replace")
        raise RuntimeError(f"speecht5_b200 {what} failed (code {rc}): {msg}")
