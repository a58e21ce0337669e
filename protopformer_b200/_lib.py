"""ctypes binding of libprotohead_b200.so (the C ABI declared in include/protohead.h).

There is no fallback of any kind: if the shared library is missing this module raises at first use, and every
compute entry point needs a CUDA device (sm_100a).  The library is built in-tree by ``protopformer_b200.build``.
"""
from __future__ import annotations

import ctypes as C
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libprotohead_b200.so")

MODE_FP32_FMA, MODE_BF16X3, MODE_BF16 = 0, 1, 2
MODES = {"fp32_fma": MODE_FP32_FMA, "fp32": MODE_BF16X3, "bf16x3": MODE_BF16X3, "bf16": MODE_BF16}
ACT_LOG, ACT_LINEAR = 0, 1
ACTS = {"log": ACT_LOG, "linear": ACT_LINEAR}

_p, _i, _f = C.c_void_p, C.c_int, C.c_float

# name -> argtypes (restype is always int unless listed in _RESTYPES); mirrors include/protohead.h one to one
SIGNATURES = {
    "pph_version": [],
    "pph_last_error_string": [],
    "pph_sm_count": [],
    "pph_set_option": [C.c_char_p, _i],
    "pph_select_topk": [_p, _i, _i, _i, _i, _p, _p, _p],
    "pph_addon_fwd": [_p, _p, _p, _p, _i, _i, _i, _i, _i, _p, _p, _p, _p, _f, _p, _p, _p, _p, _p, _p, _p, _p, _p],
    "pph_split_rows": [_p, _i, _i, _f, _p, _p, _p, _p, _p, _p],
    "pph_similarity_fwd": [_i, _i, _f, _i, _i, _i, _i, _i] + [_p] * 24,
    "pph_similarity_plan": [_i, _i, _i, _i, _i, _i, _i, C.POINTER(C.c_int), C.POINTER(C.c_int)],
    "pph_logits_fwd": [_p, _p, _p, _p, _i, _i, _i, _i, _f, _p, _p, _p, _p],
    "pph_ppc_fwd": [_p, _p, _p, _p, _p, _p, _i, _i, _i, _i, _i, _i, _i, _f, _f, _f, _p, _p, _p, _p, _p, _p],
    "pph_ppc_bwd": [_p, _p, _p, _p, _p, _p, _p, _f, _f, _i, _i, _i, _i, _i, _i, _i, _f, _f, _f, _i, _p, _p, _p],
    "pph_logits_bwd": [_p, _p, _p, _p, _p, _p, _p, _i, _i, _i, _i, _f, _i, _f, _p, _p, _p],
    "pph_last_layer_wgrad": [_p] * 5 + [_i] * 4 + [_f] + [_p] * 3,
    "pph_similarity_bwd_ws_bytes": [_i, _i, _i, _i, _i, C.POINTER(C.c_longlong)],
    "pph_similarity_bwd": [_p, _p, _p, _p, _p, _p, _p, _i, _i, _i, _i, _i, _p, _i, _p, _p, _p, _p, _p, _p, _p],
    "pph_loss_tail": [_p, _p, _p, _f, _f, _f, _i, _i, _p, _p, _p, _p, _p],
    "pph_loss_combine": [_p, _p, _f, _f, _p, _p],
    "pph_rollout_ws_bytes": [_i, _i, _i, _i, C.POINTER(C.c_longlong)],
    "pph_rollout_scores": [_p, _i, _i, _i, _i, _i, _i, _f, _p, _i, _p, _p, _i, _p, _p, _p],
    "pph_adamw_step": [_i, _p, _p, _p, _p, _p, _p, _p, C.c_double, C.c_double, _f, _f, _p, _p],
    "pph_rollout_cls_rows": [_p, _i, _i, _i, _i, _i, _i, _f, _p, _p],
    "pph_class_maps": [_p, _p, _p, _p, _p, _p, _i, _i, _i, _i, _i, _i, _i, _f, _p, _p],
    "pph_addon_bwd_ws_bytes": [_i, _i, _i, _i, _i, C.POINTER(C.c_longlong)],
    "pph_addon_bwd": [_p, _p, _p, _p, _p, _p, _p, _i, _i, _i, _i, _i, _p, _i, _p, _p, _p, _p],
    # fused step (round 2)
    "pph_head_prep_supported": [_i, _i, _i, _i, _i],
    "pph_head_prep": [_p, _p, _p, _p, _i, _i, _i, _i, _i, _i, _f] + [_p] * 14 + [_p, _i, _p, _p, _p, _p, _p] * 2 + [_p],
    "pph_head_mid_ws_bytes": [_i, _i, _i, _i, _i, _i, _i, C.POINTER(C.c_longlong)],
    "pph_head_mid": [_p] * 8 + [_i] * 8 + [_f, _i, _f, _f, _i, _i] + [_p] * 5 + [_f] * 4 + [_p] * 14,
    "pph_last_layer_pattern": [_p, _i, _p, _i, _i, _p, _p],
    "pph_similarity_bwd2_supported": [_i, _i, _i, _i, _i],
    "pph_similarity_bwd2_ws_bytes": [_i, _i, _i, _i, C.POINTER(C.c_longlong)],
    "pph_similarity_bwd2": [_i] + [_p] * 8 + [_i] * 6 + [_p, _p, _i] + [_p] * 5,
    "pph_addon_bwd2_supported": [_i, _i, _i, _i, _i],
    "pph_addon_bwd2_ws_bytes": [_i, _i, _i, _i, _i, C.POINTER(C.c_longlong)],
    "pph_addon_bwd2": [_i] + [_p] * 5 + [_i] * 5 + [_p] * 5,
    "pph_similarity_bwd_fused": [_i] + [_p] * 7 + [_i] * 6 + [_p, _p, _p, _p, _i] + [_p] * 5,
    "pph_addon_tc2_supported": [_i, _i, _i, _i, _i],
    "pph_addon_tc2_ws_bytes": [_i, _i, _i, _i, _i, C.POINTER(C.c_longlong)],
    "pph_addon_fwd2": [_p, _p, _p, _p, _i, _i, _i, _i, _i, _p, _p, _p, _p, _f] + [_p] * 10,
    "pph_addon_bwd3": [_i] + [_p] * 6 + [_i] * 5 + [_p] * 5,
    "pph_select_addon_fwd": [_p, _i, _p, _p, _p, _i, _i, _i, _i, _i, _p, _p, _p, _p, _p, _f] + [_p] * 10,
    "pph_ppc_dense_fwd": [_p, _p, _p, _i, _i, _i, _i, _i, _f, _f, _p, _p, _p, _p, _p],
    "pph_ppc_dense_bwd": [_p, _p, _p, _p, _p, _p, _i, _i, _i, _i, _i, _f, _p, _p],
    "pph_gather_rows_host": [_p, _p, _i, _i, _i, _i, _p, _i, _p],
    # gradient exchange over peer memory
    "pph_peer_flag_bytes": [C.POINTER(C.c_longlong)],
    "pph_peer_allreduce": [_p, C.c_ulonglong, C.c_longlong, _i, _i, C.c_longlong, C.c_longlong, _i, _i, _p],
}
_RESTYPES = {"pph_last_error_string": C.c_char_p}

# kernels launched per entry-point call (memset nodes are not counted); used for the bench's `gpu_launches` claim
KERNELS_PER_CALL = {
    "pph_select_topk": 1, "pph_addon_fwd": 1, "pph_split_rows": 1, "pph_logits_fwd": 1, "pph_ppc_fwd": 1,
    "pph_ppc_bwd": 1, "pph_logits_bwd": 1, "pph_last_layer_wgrad": 1, "pph_similarity_bwd": 2, "pph_addon_bwd": 3, "pph_loss_tail": 1, "pph_loss_combine": 1, "pph_rollout_scores": 2, "pph_adamw_step": 1, "pph_class_maps": 1, "pph_rollout_cls_rows": 1,
    "pph_head_prep": 1, "pph_head_mid": 1, "pph_last_layer_pattern": 1, "pph_similarity_bwd_fused": 1, "pph_addon_bwd2": 1, "pph_addon_fwd2": 1,
    "pph_peer_allreduce": 1, "pph_gather_rows_host": 1,
    "pph_ppc_dense_fwd": 1, "pph_ppc_dense_bwd": 1, "pph_select_addon_fwd": 1,
}

_ENV_OPTIONS = {"PPH_PDL": "pdl", "PPH_SIM_LANES": "sim_lanes", "PPH_SIM_SHARED": "sim_shared", "PPH_SIM_EPI": "sim_epi",
                "PPH_ROLLOUT": "rollout", "PPH_CLASSMAP": "classmap", "PPH_DEBUG": "debug",
                "PPH_LOGITS_BWD": "logits_bwd", "PPH_GATHER": "gather"}

_lib = None
_launches = 0


def launch_count() -> int:
    """Number of protohead kernels launched (or recorded into a CUDA graph) by this process so far."""
    return _launches


def load() -> C.CDLL:
    """Load the shared library (once).  Raises if it has not been built -- never falls back to another path."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} is missing: build it with `python -m protopformer_b200.build` "
                "(needs nvcc; there is no CPU or PyTorch fallback for the prototype head)")
        lib = C.CDLL(LIB_PATH)
        for name, args in SIGNATURES.items():
            fn = getattr(lib, name)      # AttributeError here = header / library mismatch
            fn.argtypes = args
            fn.restype = _RESTYPES.get(name, C.c_int)
        # variant switches are resolved HERE, once, from the environment (the C side never calls getenv)
        for env, opt in _ENV_OPTIONS.items():
            v = os.environ.get(env)
            if v is not None and v.strip() != "":
                if lib.pph_set_option(opt.encode(), int(v)) != 0:
                    raise RuntimeError(f"{env}: {lib.pph_last_error_string().decode()}")
        _lib = lib
    return _lib


_DTYPES = (torch.float32, torch.int32, torch.int64, torch.bfloat16, torch.uint8, torch.int8, torch.uint16, torch.int16)


def _ptr(t):
    if t is None:
        return None
    assert t.is_cuda, "prototype-head tensors must live on a CUDA device (no CPU path exists)"
    assert t.is_contiguous(), "prototype-head tensors must be contiguous"
    # the C ABI takes float / int32 / int64 data, bf16 operand copies and byte workspaces: a half or double tensor
    # (e.g. after model.half()) would be reinterpreted silently -- refuse it here
    assert t.dtype in _DTYPES, f"prototype-head entry points do not take {t.dtype} tensors (cast to float32 first)"
    return t.data_ptr()


def _stream():
    return torch.cuda.current_stream().cuda_stream


def call(name: str, *args):
    """Invoke an entry point on the current CUDA stream; tensors are passed as device pointers."""
    lib = load()
    conv = [(_ptr(a) if (a is None or isinstance(a, torch.Tensor)) else a) for a in args]
    conv = [(C.cast(a, C.c_void_p) if isinstance(a, C.Array) else a) for a in conv]      # host pointer tables
    rc = getattr(lib, name)(*conv, _stream())
    global _launches
    if name == "pph_similarity_fwd":
        _launches += 2 if conv[0] == MODE_FP32_FMA else 1      # local + global kernels vs one fused tcgen05 kernel
    elif name == "pph_similarity_bwd":
        _launches += (1 if conv[13] & 1 else 0) + (1 if conv[13] & 2 else 0)
    elif name == "pph_similarity_bwd2":
        _launches += bin(conv[0] & 7).count("1")
    elif name == "pph_addon_bwd3":
        _launches += bin(conv[0] & 3).count("1")
    elif name == "pph_addon_bwd":
        _launches += (2 if conv[13] & 1 else 0) + (1 if conv[13] & 2 else 0)
    else:
        _launches += KERNELS_PER_CALL.get(name, 0)
    if rc != 0:
        msg = lib.pph_last_error_string()
        raise RuntimeError(f"{name} failed (rc={rc}): {msg.decode() if msg else ''}")
