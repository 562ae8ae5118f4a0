"""ctypes binding of libard_b200.so (the C ABI declared in include/ard.h).

The library is the product: there is no CPU or PyTorch fallback. `load()` raises if the shared object is missing or
lacks a declared symbol, and every call maps a negative return code to the exception type the reference raises for the
same condition (SURVEY.md §8b "Error convention").
"""
import ctypes as C
import os
import re

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("ARD_LIB_PATH") or os.path.join(_HERE, "libard_b200.so")   # ARD_LIB_PATH: A/B builds of the same ABI (tools/)
HEADER = os.path.join(os.path.dirname(_HERE), "include", "ard.h")

ARD_OK, ARD_ERR_SHAPE, ARD_ERR_DTYPE, ARD_ERR_CUDA, ARD_ERR_STATE, ARD_ERR_KEY, ARD_ERR_NOTIMPL = 0, -1, -2, -3, -4, -5, -6
ACT_NONE, ACT_GELU, ACT_RELU, ACT_GELU_F16 = 0, 1, 2, 3

c_float_p = C.POINTER(C.c_float)
c_double_p = C.POINTER(C.c_double)


class ArdConfig(C.Structure):
    _fields_ = [("embed_dim", C.c_int), ("depths", C.c_int * 4), ("num_heads", C.c_int * 4), ("joint_dim", C.c_int),
                ("enable_fusion", C.c_int)]


class ArdForwardArgs(C.Structure):
    _fields_ = [("waveform", C.c_void_p), ("mel_fusion", C.c_void_p), ("B", C.c_int), ("quantize", C.c_int),
                ("embedding", C.c_void_p), ("audio_embed", C.c_void_p),
                ("layers_residuals", C.c_void_p * 4), ("layers_attention", C.c_void_p * 4),
                ("framewise_output", C.c_void_p), ("clipwise_output", C.c_void_p), ("fine_grained_embedding", C.c_void_p),
                ("save_for_backward", C.c_int), ("head_outputs", C.c_void_p * 4), ("precision", C.c_int)]


class ArdBackwardArgs(C.Structure):
    _fields_ = [("B", C.c_int), ("grad_audio_embed", C.c_void_p), ("grad_embedding", C.c_void_p), ("grad_lambda", C.c_void_p * 4),
                ("generation", C.c_longlong)]


class ArdOutputGrads(C.Structure):
    _fields_ = [("grad_framewise_output", C.c_void_p), ("grad_clipwise_output", C.c_void_p), ("grad_fine_grained_embedding", C.c_void_p),
                ("grad_layers_residuals", C.c_void_p * 4), ("grad_layers_attention", C.c_void_p * 4)]


_lib = None


def declared_symbols():
    """Every function name include/ard.h declares (used by build() and the CPU test-suite)."""
    text = open(HEADER).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(ard_[a-z0-9_]+)\s*\(", text)))


def load(check_symbols=False):
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(f"{LIB_PATH} is missing: run `python __graft_entry__.py` (nvcc, sm_100a). "
                               "audio_residual_b200 has no CPU / PyTorch fallback.")
        lib = C.CDLL(LIB_PATH)
        lib.ard_last_error.restype = C.c_char_p
        lib.ard_workspace_bytes.restype = C.c_longlong
        lib.ard_launch_counter_read.restype = C.c_longlong
        lib.ard_tape_generation.restype = C.c_longlong
        vp, ll, i, f = C.c_void_p, C.c_longlong, C.c_int, C.c_float
        lib.ard_create.argtypes = [C.POINTER(ArdConfig), C.POINTER(vp)]
        lib.ard_destroy.argtypes = [vp]
        lib.ard_set_weight.argtypes = [vp, C.c_char_p, vp, ll]
        lib.ard_finalize_weights.argtypes = [vp, vp]
        lib.ard_set_block_residual.argtypes = [vp, i, i, vp, vp, i, i]
        lib.ard_clear_block_residual.argtypes = [vp, i, i]
        lib.ard_set_block_lambda.argtypes = [vp, i, i, vp, vp]
        lib.ard_set_layer_lambda.argtypes = [vp, i, vp, vp]
        lib.ard_encoder_forward.argtypes = [vp, C.POINTER(ArdForwardArgs), vp]
        lib.ard_encoder_backward.argtypes = [vp, C.POINTER(ArdBackwardArgs), vp]
        lib.ard_encoder_backward_outputs.argtypes = [vp, C.POINTER(ArdBackwardArgs), C.POINTER(ArdOutputGrads), vp]
        lib.ard_window_attention_bwd_pgrad.argtypes = [vp, vp, vp, f, vp, vp, i, i, i, i, i, i, vp]
        lib.ard_window_attention_f32_bwd_pgrad.argtypes = [vp, vp, vp, f, vp, vp, i, i, i, i, i, i, vp]
        lib.ard_tail_backward.argtypes = [vp, vp, i, vp, vp, vp, vp, i, i, vp, vp]
        lib.ard_block_forward.argtypes = [vp, i, i, vp, i, vp, vp, vp, vp]
        lib.ard_attention_block.argtypes = [vp, i, i, vp, i, vp, vp]
        lib.ard_workspace_bytes.argtypes = [vp]
        lib.ard_last_launch_count.argtypes = [vp]
        lib.ard_gemm_bf16.argtypes = [vp, ll, vp, ll, vp, ll, i, i, i, i, vp, i, vp, ll, vp, ll, vp]
        lib.ard_gemm_dual.argtypes = [i, vp, ll, vp, ll, vp, ll, vp, ll, vp, ll, i, i, i, vp, vp, vp, i, vp]
        lib.ard_gemm_f16.argtypes = [vp, ll, vp, ll, vp, ll, i, i, i, i, vp, i, vp, ll, vp, ll, vp]
        lib.ard_layernorm_bf16.argtypes = [vp, vp, vp, vp, ll, i, vp]
        lib.ard_ffn_fused_96.argtypes = [vp, vp, vp, ll, vp, vp, vp, vp, vp, vp, vp]
        lib.ard_ffn_fused_wide.argtypes = [vp, vp, vp, ll, i, vp, vp, vp, vp, vp, vp, vp]
        lib.ard_ln_qkv_96.argtypes = [vp, vp, vp, vp, vp, vp, ll, vp]
        lib.ard_window_attention.argtypes = [vp, vp, vp, vp, f, i, i, i, i, i, i, i, vp]
        lib.ard_window_attention_bwd.argtypes = [vp, vp, vp, vp, i, i, i, i, i, i, vp]
        lib.ard_window_attention_f32_bwd.argtypes = [vp, vp, vp, vp, i, i, i, i, i, i, vp]
        lib.ard_layernorm_bwd.argtypes = [vp, vp, vp, vp, vp, ll, i, vp]
        lib.ard_f32_to_bf16.argtypes = [vp, vp, ll, f, vp]
        lib.ard_quantize_waveform.argtypes = [vp, vp, ll, vp]
        lib.ard_logmel.argtypes = [vp, vp, i, i, i, i, vp, vp]
        lib.ard_fusion_mel.argtypes = [vp, vp, i, i, i, vp, vp]
        lib.ard_patch_embed.argtypes = [vp, vp, i, vp, vp]
        lib.ard_stats_accumulate.argtypes = [vp, ll, i, vp, vp, vp]
        lib.ard_stats_accumulate_strided.argtypes = [vp, ll, ll, i, vp, vp, vp]
        lib.ard_sym_eigvals_workspace.restype = C.c_longlong
        lib.ard_sym_eigvals_workspace.argtypes = [i, i]
        lib.ard_sym_eigvals.argtypes = [vp, ll, i, i, vp, vp, ll, vp]
        lib.ard_sym_eigh_workspace.restype = C.c_longlong
        lib.ard_sym_eigh_workspace.argtypes = [i, i]
        lib.ard_sym_eigh.argtypes = [vp, ll, i, i, vp, vp, ll, vp, vp, ll, vp]
        lib.ard_tape_generation.argtypes = [vp]
        lib.ard_residual_forward.argtypes = [vp, vp, vp, vp, vp, ll, i, i, vp]
        lib.ard_residual_backward.argtypes = [vp, vp, vp, vp, vp, vp, vp, ll, i, i, vp]
        lib.ard_head_forward.argtypes = [vp, vp, vp, i, i, i, vp, vp]
        lib.ard_ce_forward.argtypes = [vp, vp, i, i, vp, vp, vp]
        lib.ard_head_backward.argtypes = [vp, vp, vp, i, i, i, vp, vp, vp, vp]
        lib.ard_eval_metrics.argtypes = [vp, vp, ll, i, i, vp, vp, vp, vp]
        lib.ard_fill_clips.argtypes = [vp, i, vp, vp, i, i, i, i, vp, vp]
        lib.ard_profile_enable.argtypes = [i]
        lib.ard_profile_read.argtypes = [c_double_p, c_double_p, c_double_p, C.POINTER(C.c_int), i]
        _lib = lib
    if check_symbols:
        missing = [s for s in declared_symbols() if not hasattr(_lib, s)]
        if missing:
            raise RuntimeError(f"libard_b200.so lacks symbols declared in include/ard.h: {missing}")
    return _lib


_EXC = {ARD_ERR_SHAPE: ValueError, ARD_ERR_DTYPE: TypeError, ARD_ERR_CUDA: RuntimeError, ARD_ERR_STATE: RuntimeError,
        ARD_ERR_KEY: KeyError, ARD_ERR_NOTIMPL: NotImplementedError}


def check(rc, exc=None):
    """Raise the Python exception matching a negative ARD_ERR_* code (exc overrides the type, e.g. AssertionError for
    the conditions the reference asserts on)."""
    if rc == 0:
        return
    msg = load().ard_last_error().decode("utf-8", "replace")
    raise (exc or _EXC.get(rc, RuntimeError))(msg)


def stream_ptr():
    import torch
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def ptr(t):
    """Device/host pointer of a contiguous tensor (or None)."""
    if t is None:
        return None
    assert t.is_contiguous(), "tensor handed to the C ABI must be contiguous"
    return C.c_void_p(t.data_ptr())


PROF_CLASSES = ("gemm_tc", "window_attention", "layernorm", "frontend", "heads", "other", "ffn_fused")


def profile_enable(on=True):
    check(load().ard_profile_enable(int(on)))


def profile_read():
    """{class: {"ms", "flops", "bytes", "launches"}} accumulated since the last read (synchronises the device)."""
    n = len(PROF_CLASSES)
    ms, fl, by, ln = (C.c_double * n)(), (C.c_double * n)(), (C.c_double * n)(), (C.c_int * n)()
    check(load().ard_profile_read(ms, fl, by, ln, n))
    return {PROF_CLASSES[i]: {"ms": ms[i], "flops": fl[i], "bytes": by[i], "launches": ln[i]} for i in range(n)}
