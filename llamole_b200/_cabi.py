"""ctypes binding of include/llamole_b200.h.

The library is the only compute path: if it is missing or the device is not sm_100 the calls raise, there
is no PyTorch/CPU fallback (by design; see DESIGN.md).
"""
from __future__ import annotations

import ctypes as C
import os
import threading

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libllamole_b200.so")

LLB_OK = 0
ACT_NONE, ACT_GELU, ACT_SILU, ACT_SOFTSIGN = 0, 1, 2, 3

_F = C.c_void_p       # const float*
_FF = C.POINTER(C.c_void_p)  # const float* const*


class DitConfig(C.Structure):
    _fields_ = [("hidden", C.c_int32), ("depth", C.c_int32), ("heads", C.c_int32), ("mlp_hidden", C.c_int32),
                ("max_nodes", C.c_int32), ("timesteps", C.c_int32), ("y_dim", C.c_int32), ("text_dim", C.c_int32),
                ("guide_scale", C.c_float)]


class DitWeights(C.Structure):
    _fields_ = [
        ("x_embed_w", _F), ("x_embed_ln_w", _F), ("x_embed_ln_b", _F),
        ("t_mlp0_w", _F), ("t_mlp0_b", _F), ("t_mlp2_w", _F), ("t_mlp2_b", _F),
        ("y_drop", _F), ("y_mlp0_w", _FF), ("y_mlp0_b", _FF), ("y_mlp2_w", _FF),
        ("txt_drop", _F), ("txt_w", _F), ("txt_b", _F),
        ("qkv_w", _FF), ("q_norm_w", _FF), ("q_norm_b", _FF), ("k_norm_w", _FF), ("k_norm_b", _FF),
        ("proj_w", _FF), ("proj_b", _FF), ("fc1_w", _FF), ("fc1_b", _FF), ("fc2_w", _FF), ("fc2_b", _FF),
        ("ada0_w", _FF), ("ada0_b", _FF), ("ada2_w", _FF), ("ada2_b", _FF),
        ("out_fc1_w", _F), ("out_fc1_b", _F), ("out_fc2_w", _F), ("out_fc2_b", _F),
        ("out_ada0_w", _F), ("out_ada0_b", _F), ("out_ada2_w", _F), ("out_ada2_b", _F),
        ("x_marg", _F), ("e_marg", _F), ("xe", _F), ("ex", _F), ("betas", _F), ("alphas_bar", _F),
    ]


class GinConfig(C.Structure):
    _fields_ = [("hidden", C.c_int32), ("layers", C.c_int32), ("predictor", C.c_int32), ("out_dim", C.c_int32),
                ("text_dim", C.c_int32)]


class GinWeights(C.Structure):
    _fields_ = [
        ("atom_emb", _F), ("vn_emb", _F),
        ("eps", _FF), ("mlp0_w", _FF), ("mlp0_b", _FF), ("mlp_ln_w", _FF), ("mlp_ln_b", _FF), ("mlp4_w", _FF),
        ("mlp4_b", _FF), ("bond_emb", _FF), ("norm_w", _FF), ("norm_b", _FF),
        ("vn0_w", _FF), ("vn0_b", _FF), ("vn_ln_w", _FF), ("vn_ln_b", _FF), ("vn4_w", _FF), ("vn4_b", _FF),
        ("adapter_w", _FF), ("adapter_b", _FF), ("text_dropping", _F),
        ("head0_w", _F), ("head0_b", _F), ("head_ln_w", _F), ("head_ln_b", _F), ("head4_w", _F), ("head4_b", _F),
    ]


# name -> (restype, argtypes); mirrors include/llamole_b200.h one to one
_P = C.c_void_p
_SZ = C.c_size_t
_I = C.c_int
SIGNATURES = {
    "llb_last_error": (C.c_char_p, []),
    "llb_version": (_I, []),
    "llb_arch_check": (_I, [_I]),
    "llb_profile_enable": (_I, [_I]),
    "llb_profile_read": (_I, [_I, C.POINTER(C.c_double), C.POINTER(C.c_int64)]),
    "llb_profile_slot_name": (C.c_char_p, [_I]),
    "llb_kernel_launches": (C.c_int64, [_I]),
    "llb_gemm_bf16": (_I, [_P, _I, _P, _I, _P, _P, _I, _I, _I, _I, _I, _I, _P]),
    "llb_gemm_ln_workspace_bytes": (_I, [C.POINTER(_SZ)]),
    "llb_gemm_ln_residual_ws": (_I, [_P, _I, _P, _I, _P, _P, _P, _P, _P, _I, _P, _I, _P, _I, _I, _I, _I, _P, _SZ, _P]),
    "llb_dit_packed_bytes": (_I, [C.POINTER(DitConfig), C.POINTER(_SZ)]),
    "llb_dit_pack_weights": (_I, [C.POINTER(DitConfig), C.POINTER(DitWeights), _P, _SZ, _P]),
    "llb_dit_create": (_I, [C.POINTER(DitConfig), _P, _SZ, C.POINTER(_P)]),
    "llb_dit_destroy": (None, [_P]),
    "llb_dit_workspace_bytes": (_I, [C.POINTER(DitConfig), _I, C.POINTER(_SZ)]),
    "llb_dit_begin": (_I, [_P, _P, _SZ, _I, C.POINTER(C.c_int32), _P, _P, C.c_int64, _P]),
    "llb_dit_set_state": (_I, [_P, _P, _P, _P]),
    "llb_dit_get_state": (_I, [_P, _P, _P, _P]),
    "llb_dit_init_state": (_I, [_P, C.c_uint64, _P, _P, _P]),
    "llb_dit_denoise": (_I, [_P, _I, _I, _P, _P, _P]),
    "llb_dit_step": (_I, [_P, _I, C.c_uint64, _P, _P, _P, _P, _P]),
    "llb_dit_sample": (_I, [_P, _I, _I, C.c_uint64, _P, _P, _P]),
    "llb_dit_launch_count": (C.c_int64, [_P]),
    "llb_dit_graph_state": (C.c_int, [_P]),
    "llb_dit_posterior_sample": (_I, [_P, _I, _P, _P, _P, _P, C.c_uint64, _P, _P, _P, _P, _P]),
    "llb_gin_packed_bytes": (_I, [C.POINTER(GinConfig), C.POINTER(_SZ)]),
    "llb_gin_pack_weights": (_I, [C.POINTER(GinConfig), C.POINTER(GinWeights), _P, _SZ, _P]),
    "llb_gin_create": (_I, [C.POINTER(GinConfig), _P, _SZ, C.POINTER(_P)]),
    "llb_gin_destroy": (None, [_P]),
    "llb_gin_workspace_bytes": (_I, [C.POINTER(GinConfig), _I, _I, _I, _I, C.POINTER(_SZ)]),
    "llb_gin_bind": (_I, [_P, _P, _SZ, _I, _I, _I, _P, _P, _P, _P, _P]),
    "llb_gin_input_flags": (_I, [_P, C.POINTER(C.c_int32), _P]),
    "llb_gin_encoder_forward": (_I, [_P, _P, _P, _P]),
    "llb_gin_predictor_forward": (_I, [_P, _P, _P, _P]),
    "llb_gin_predictor_topk": (_I, [_P, _P, _I, _P, _P, _P]),
    "llb_gin_grad_packed_bytes": (_I, [C.POINTER(GinConfig), C.POINTER(_SZ)]),
    "llb_gin_pack_grad_weights": (_I, [_P, _P, _SZ, _P]),
    "llb_gin_saved_bytes": (_I, [C.POINTER(GinConfig), _I, _I, _I, C.POINTER(_SZ)]),
    "llb_gin_predictor_forward_saved": (_I, [_P, _P, _P, _P, _SZ, _P]),
    "llb_gin_predictor_backward_c": (_I, [_P, _I, _I, _I, _P, _P, _P, _SZ, _P, _SZ, _P, _P]),
    "llb_gin_launch_count": (C.c_int64, [_P]),
    "llb_gin_stat": (C.c_int64, [_P, _I]),
    "llb_softmax_topk": (_I, [_P, _I, _I, _I, _I, _P, _P, _P, _P]),
    "llb_cost_mlp": (_I, [_P, _P, _P, _P, _P, _I, _I, _I, _P, _P]),
}

_lib = None
_lock = threading.Lock()


class LlamoleB200Error(RuntimeError):
    pass


def lib() -> C.CDLL:
    """The loaded C-ABI library.  Raises if it has not been built (python -m llamole_b200.build)."""
    global _lib
    if _lib is None:
        with _lock:
            if _lib is None:
                if not os.path.exists(LIB_PATH):
                    raise LlamoleB200Error(
                        f"{LIB_PATH} is missing: build it with `python -m llamole_b200.build` (needs nvcc). "
                        "llamole_b200 has no PyTorch/CPU fallback.")
                l = C.CDLL(LIB_PATH)
                for name, (res, args) in SIGNATURES.items():
                    fn = getattr(l, name)
                    fn.restype = res
                    fn.argtypes = args
                _lib = l
    return _lib


def check(status: int, what: str = "") -> None:
    if status != LLB_OK:
        msg = lib().llb_last_error()
        raise LlamoleB200Error(f"{what or 'llamole_b200'} failed ({status}): {msg.decode() if msg else '?'}")


def ptr(t) -> C.c_void_p:
    """Device (or host) pointer of a torch tensor, None -> NULL."""
    return C.c_void_p(None if t is None else t.data_ptr())


def ptr_array(tensors):
    arr = (C.c_void_p * len(tensors))(*[t.data_ptr() for t in tensors])
    return arr


def stream_ptr() -> C.c_void_p:
    import torch

    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def params_fingerprint(module) -> tuple:
    """Identity + version of every parameter of `module`: changes when a parameter is replaced, moved, cast or written in
    place (torch bumps `_version` on every in-place write), which is when a packed-weight blob made from it is stale."""
    return tuple((p.data_ptr(), p._version, p.dtype) for p in module.parameters())


def require_cuda(t, name: str):
    if not t.is_cuda:
        raise LlamoleB200Error(f"{name} must live on a CUDA (sm_100) device; llamole_b200 has no CPU path")


KERN_GEMM_1CTA, KERN_GEMM_2CTA, KERN_GEMM_LN_PAIR, KERN_GEMM_LN_CLUSTER, KERN_GIN_FUSED_MLP, KERN_HEAD_TOPK = range(6)


def kernel_launches(family: int) -> int:
    """Launches of a kernel family since the library was loaded (include/llamole_b200.h: LLB_KERN_*)."""
    return int(lib().llb_kernel_launches(int(family)))


PROF_SLOTS = 19


def profile_enable(on: bool) -> None:
    check(lib().llb_profile_enable(int(on)), "llb_profile_enable")


def profile_read() -> dict:
    """{slot name: (total_ms, launches)} since the last read; synchronises on the recorded events."""
    out = {}
    for i in range(PROF_SLOTS):
        ms, n = C.c_double(), C.c_int64()
        check(lib().llb_profile_read(i, C.byref(ms), C.byref(n)), "llb_profile_read")
        if n.value:
            out[lib().llb_profile_slot_name(i).decode()] = (ms.value, n.value)
    return out
