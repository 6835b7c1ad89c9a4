"""ctypes binding of libxlstm_b200.so (include/xlstm_b200.h). Thin: pointers and ints only.

There is NO CPU fallback: if the shared library is missing or the CUDA device is absent the product path
raises. (Loading the library and querying its symbols works without a GPU; compute calls do not.)
"""
from __future__ import annotations

import ctypes as C
import os
import re

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libxlstm_b200.so")
HEADER_PATH = os.path.join(os.path.dirname(HERE), "include", "xlstm_b200.h")

# status codes
XL_OK = 0
XL_ERR_INVALID_ARG, XL_ERR_UNSUPPORTED, XL_ERR_CUDA, XL_ERR_NOT_READY, XL_ERR_NO_DEVICE = -1, -2, -3, -4, -5

# modes / flags
XL_MODE_PER_TOKEN, XL_MODE_FUSED = 0, 1
XL_FLAG_DISCRETE, XL_FLAG_GRAPH, XL_FLAG_SIMPLE_GEMM, XL_FLAG_STATE_EMBEDS = 1, 2, 4, 8

# state parts
XL_STATE_C, XL_STATE_N, XL_STATE_M, XL_STATE_CONV, XL_STATE_SLSTM = 0, 1, 2, 3, 4
XL_ABI_VERSION = 3

# weight ids (xl_weight_id)
W = dict(
    XLSTM_NORM=0, PROJ_UP=1, Q_PROJ=2, K_PROJ=3, V_PROJ=4, CONV_W=5, CONV_B=6, IGATE_W=7, IGATE_B=8,
    FGATE_W=9, FGATE_B=10, OUTNORM=11, SKIP=12, PROJ_DOWN=13,
    S_GATE_I=14, S_GATE_F=15, S_GATE_Z=16, S_GATE_O=17, S_RECURRENT=18, S_BIAS=19, S_GROUP_NORM=20,
    FFN_NORM=21, FFN_UP=22, FFN_DOWN=23,
    POST_NORM=32, EMBED_STATE_W=33, EMBED_STATE_B=34, EMBED_RETURN_W=35, EMBED_RETURN_B=36,
    EMBED_REWARD_W=37, EMBED_REWARD_B=38, EMBED_LN_W=39, EMBED_LN_B=40, HEAD_W=41, HEAD_B=42,
)


class XLConfig(C.Structure):
    _fields_ = [
        ("embedding_dim", C.c_int32), ("num_blocks", C.c_int32), ("num_heads", C.c_int32),
        ("inner_dim", C.c_int32), ("conv_kernel", C.c_int32), ("qkv_blocksize", C.c_int32),
        ("state_dim", C.c_int32), ("act_dim", C.c_int32), ("action_channels", C.c_int32),
        ("discrete_actions", C.c_int32), ("tokens_per_step", C.c_int32), ("action_token_pos", C.c_int32),
        ("max_batch", C.c_int32),
        ("ln_eps", C.c_float), ("cell_eps", C.c_float), ("embed_ln_eps", C.c_float),
        ("tok_min_val", C.c_float), ("tok_max_val", C.c_float),
        ("slstm_mask_lo", C.c_uint32), ("slstm_mask_hi", C.c_uint32), ("ffn_dim", C.c_int32),
    ]


class XLSampling(C.Structure):
    """xl_sampling: parameters of the device sampler (xl_set_sampling)."""
    _fields_ = [("temperature", C.c_float), ("top_p", C.c_float), ("top_k", C.c_int32), ("env_id_base", C.c_int32),
                ("env_id_stride", C.c_int32), ("seed", C.c_uint64)]


class XLSeqOutputs(C.Structure):
    """xl_seq_outputs: device buffers of xl_policy_forward(_embeds) (each nullable)."""
    _fields_ = [("tokens", C.c_void_p), ("actions", C.c_void_p), ("logits", C.c_void_p), ("targets", C.c_void_p),
                ("logprobs", C.c_void_p)]


class XLError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"xlstm_b200 error {code}: {msg}")
        self.code = code


_lib = None


def declared_symbols():
    """Every function include/xlstm_b200.h declares (used by the CPU-only ABI test)."""
    with open(HEADER_PATH) as fh:
        src = fh.read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(xl_[a-z_0-9]+)\s*\(", src)))


def load():
    """Load the shared library (building it first if the .so is absent and nvcc is available)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        from . import build as _build
        _build.build()
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(f"{LIB_PATH} is missing and could not be built: the xlstm_b200 path has no "
                           f"CPU fallback")
    lib = C.CDLL(LIB_PATH)
    vp, i32, i64, u32, sz = C.c_void_p, C.c_int, C.c_int64, C.c_uint, C.c_size_t
    lib.xl_abi_version.restype = i32
    lib.xl_last_error.restype = C.c_char_p
    lib.xl_create.argtypes = [C.POINTER(XLConfig), C.POINTER(vp)]
    lib.xl_create.restype = i32
    lib.xl_destroy.argtypes = [vp]
    lib.xl_destroy.restype = None
    lib.xl_state_dim_padded.argtypes = [vp]
    lib.xl_state_dim_padded.restype = i32
    lib.xl_bind_weight.argtypes = [vp, i32, i32, vp, i32, i64]
    lib.xl_bind_weight.restype = i32
    lib.xl_weights_ready.argtypes = [vp]
    lib.xl_weights_ready.restype = i32
    lib.xl_encoder_weights_ready.argtypes = [vp]
    lib.xl_encoder_weights_ready.restype = i32
    lib.xl_state_bytes.argtypes = [vp, i32]
    lib.xl_state_bytes.restype = sz
    lib.xl_state_layout.argtypes = [vp, i32, i32, i32, C.POINTER(sz), C.POINTER(sz)]
    lib.xl_state_layout.restype = i32
    lib.xl_state_reset.argtypes = [vp, vp, vp, i32, vp]
    lib.xl_state_reset.restype = i32
    lib.xl_encoder_step.argtypes = [vp, vp, vp, vp, i32, i32, i32, u32, vp]
    lib.xl_encoder_step.restype = i32
    lib.xl_mlstm_cell_step.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, i32, i32, i32, i32, vp]
    lib.xl_mlstm_cell_step.restype = i32
    lib.xl_policy_step.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp, vp, i32, i32, u32, vp]
    lib.xl_policy_step.restype = i32
    lib.xl_policy_step_host.argtypes = [vp, vp, vp, vp, vp, vp, vp, i32, i32, u32, vp]
    lib.xl_policy_step_host.restype = i32
    lib.xl_prefill.argtypes = [vp, vp, vp, vp, i32, i32, u32, vp]
    lib.xl_prefill.restype = i32
    lib.xl_policy_prefill.argtypes = [vp, vp, vp, vp, vp, i32, i32, u32, vp]
    lib.xl_policy_prefill.restype = i32
    lib.xl_prefill_ragged.argtypes = [vp, vp, vp, vp, vp, i32, i32, u32, vp]
    lib.xl_prefill_ragged.restype = i32
    lib.xl_policy_prefill_ragged.argtypes = [vp, vp, vp, vp, vp, vp, i32, i32, u32, vp]
    lib.xl_policy_prefill_ragged.restype = i32
    lib.xl_policy_forward.argtypes = [vp, vp, vp, vp, vp, vp, i32, i32, C.POINTER(XLSeqOutputs), u32, vp]
    lib.xl_policy_forward.restype = i32
    lib.xl_policy_prefill_embeds.argtypes = [vp, vp, vp, vp, vp, vp, i32, i32, u32, vp]
    lib.xl_policy_prefill_embeds.restype = i32
    lib.xl_policy_forward_embeds.argtypes = [vp, vp, vp, vp, vp, vp, i32, i32, C.POINTER(XLSeqOutputs), u32, vp]
    lib.xl_policy_forward_embeds.restype = i32
    lib.xl_linear.argtypes = [vp, vp, vp, vp, vp, vp, i32, i32, i32, i32, vp]
    lib.xl_linear.restype = i32
    lib.xl_set_token_ring.argtypes = [vp, vp, i32, i32, vp]
    lib.xl_set_token_ring.restype = i32
    lib.xl_set_sampling.argtypes = [vp, C.POINTER(XLSampling), u32, vp]
    lib.xl_set_sampling.restype = i32
    lib.xl_sample_actions.argtypes = [vp, vp, i32, u32, C.POINTER(XLSampling), u32, vp, vp, vp]
    lib.xl_sample_actions.restype = i32
    lib.xl_set_option.argtypes = [vp, C.c_char_p, i32]
    lib.xl_set_option.restype = i32
    lib.xl_profile_begin.argtypes = [vp]
    lib.xl_profile_begin.restype = i32
    lib.xl_profile_end.argtypes = [vp, C.POINTER(C.c_double), C.POINTER(i64), C.POINTER(C.c_double)]
    lib.xl_profile_end.restype = i32
    lib.xl_launch_count.argtypes = [vp]
    lib.xl_launch_count.restype = i64
    _lib = lib
    return lib


def check(rc: int):
    if rc != XL_OK:
        raise XLError(rc, load().xl_last_error().decode("utf-8", "replace"))
