"""Host-side operators of the prototype head: thin autograd wrappers over the C ABI (include/protohead.h).

Every function launches sm_100a kernels on the current CUDA stream through ``_lib.call``; nothing here computes
on the CPU or through PyTorch math (torch is used to allocate device buffers and to carry autograd edges).
Reference lines are those of /root/reference/protopformer.py.
"""
from __future__ import annotations

import dataclasses
import math

import torch

from . import _lib


@dataclasses.dataclass(frozen=True)
class HeadConfig:
    """Scalars of one prototype head (PPNet ctor arguments that reach the kernels, protopformer.py:14-44)."""

    K: int                        # reserve_token_nums[-1]
    global_coe: float = 0.5
    act_fn: str = "log"           # prototype_activation_function: 'log' | 'linear'
    eps: float = 1e-4             # PPNet.epsilon
    mode: str = "fp32"            # 'fp32' (= bf16x3 on tcgen05) | 'bf16' | 'fp32_fma'
    ppc_cov_thresh: float = 1.0
    ppc_mean_thresh: float = 2.0
    center: float = 0.5           # tensor-core operands are taken from (z - center), (p - center); see protohead.h

    @property
    def mode_id(self) -> int:
        return _lib.MODES[self.mode]

    @property
    def act_id(self) -> int:
        return _lib.ACTS[self.act_fn]


def _empty(shape, dtype, like):
    return torch.empty(shape, dtype=dtype, device=like.device)


TOKEN_DTYPES = (torch.float32, torch.bfloat16)


def token_entry(name: str, dtype) -> str:
    """The entry point that reads backbone tokens of `dtype`: `name` itself for float32, its bf16 twin (`name` + "_bf16tok",
    include/protohead.h) for bfloat16.  Any other dtype raises TypeError here, before anything is launched."""
    if dtype == torch.float32:
        return name
    if dtype == torch.bfloat16:
        return name + _lib.BF16TOK
    raise TypeError(f"backbone tokens must be torch.float32 or torch.bfloat16, got {dtype} "
                    "(fp16 tokens are taken only inside an autocast region, which casts them to float32)")


def _autocast_casts() -> bool:
    """Inside a CUDA autocast region the head's autograd functions cast their floating inputs to float32 (custom_fwd)."""
    return torch.is_autocast_enabled("cuda")


def check_head_dtypes(tokens, *params):
    """Refuse, before any launch, what the kernels cannot read: tokens other than float32 / bfloat16 and head parameters
    other than float32.  Inside an autocast region nothing is refused: the float32 cast policy applies there as before."""
    if _autocast_casts():
        return
    token_entry("", tokens.dtype)
    for p in params:
        if p is not None and p.dtype != torch.float32:
            raise TypeError(f"prototype-head parameters must be torch.float32, got {p.dtype} of shape {tuple(p.shape)} "
                            "(bf16 backbone tokens are supported; bf16 head parameters are not)")


def tc_supported(D: int, K: int) -> bool:
    """Shapes the tcgen05 similarity kernel was built for (include/protohead.h, pph_similarity_fwd)."""
    return D % 64 == 0 and 64 <= D <= 512 and 1 <= K <= 256


# ------------------------------------------------------------------------------------------------------------------
# (a1) selection -- protopformer.py:157-158
# ------------------------------------------------------------------------------------------------------------------
def select_topk(scores: torch.Tensor, K: int, want_int64: bool = False):
    """scores (B,N) or (B,H,N) fp32 -> ascending int32 index list (B,K) [and its int64 twin]."""
    s = scores.detach()
    if s.dtype != torch.float32:
        s = s.float()
    s = s.contiguous()
    if s.dim() == 2:
        B, N = s.shape
        H = 1
    else:
        B, H, N = s.shape
    idx32 = _empty((B, K), torch.int32, s)
    idx64 = _empty((B, K), torch.int64, s) if want_int64 else None
    _lib.call("pph_select_topk", s, B, H, N, K, idx32, idx64)
    return (idx32, idx64) if want_int64 else idx32


# ------------------------------------------------------------------------------------------------------------------
# (next #1) attention rollout -> CLS-row score -- tools/deit_models_attn.py:99-124, :226
# ------------------------------------------------------------------------------------------------------------------
FUSIONS = {"mean": 0, "max": 1, "min": 2}
_rollout_ws: dict = {}


def rollout_workspace(L: int, B: int, T: int, k_discard: int, device) -> torch.Tensor:
    import ctypes
    n = ctypes.c_longlong(0)
    if _lib.load().pph_rollout_ws_bytes(L, B, T, k_discard, ctypes.byref(n)) != 0:
        raise RuntimeError("pph_rollout_ws_bytes failed")
    return torch.empty(max(int(n.value), 256), dtype=torch.uint8, device=device)


def _attn_tables(maps, entry: str):
    """The entry point and layer list for one set of attention maps: bf16 or fp16 maps, all of one of those dtypes, go
    to the half-precision twin of `entry` as they are (no fp32 copy); any other list is widened to an fp32 copy."""
    maps = [m.detach() for m in maps]
    dt = maps[0].dtype
    if dt in _lib.ATTN_TWINS and all(m.dtype == dt for m in maps):
        return entry + _lib.ATTN_TWINS[dt], [m.contiguous() for m in maps]
    return entry, [m.float().contiguous() for m in maps]


def rollout_scores(all_attn, discard_ratio: float = 0.9, head_fusion: str = "mean", identity_w: float = 0.2,
                   v0: torch.Tensor | None = None, drop_first: bool = True, workspace: torch.Tensor | None = None,
                   topk: int = 0, want_int64: bool = False):
    """``attn_rollout(all_attn)[:, 0, 1:]`` of the reference (deit_models_attn.py:99-124, :226) without the (T,T)
    products.  all_attn: list of L CUDA tensors (B,H,T,T) (the attention maps of the first L blocks): fp32, or all
    bf16 / all fp16, read as they are with the result of their fp32 widening bit for bit (other lists are widened to
    fp32 first); returns the detached score (B, T-1) [(B,T) when drop_first is False].  ``v0`` (B,T): start row instead of e_0
    (CaiT, cait_models_attn.py:255-259).  The result is not differentiable -- the reference detaches it (:225).
    ``topk`` = K > 0: the same launch also selects the K highest-scoring tokens of every image (ascending int32 index
    list, deit_models_attn.py:229-230 / protopformer.py:157-158) and ``(scores, idx32[, idx64])`` is returned."""
    import ctypes
    L = len(all_attn)
    assert L >= 1
    entry, layers = _attn_tables(all_attn, "pph_rollout_scores")
    B, H, T, T2 = layers[0].shape
    assert T == T2 and all(a.shape == layers[0].shape for a in layers), "square (B,H,T,T) maps of one shape expected"
    k = int(T * T * discard_ratio)                    # deit_models_attn.py:110
    dev = layers[0].device
    if workspace is None:
        key = (L, B, T, k, dev)
        workspace = _rollout_ws.get(key)
        if workspace is None:
            workspace = _rollout_ws[key] = rollout_workspace(L, B, T, k, dev)
    scores = _empty((B, T - int(drop_first)), torch.float32, layers[0])
    table = (ctypes.c_void_p * L)(*[_ptr_of(a) for a in layers])
    if v0 is not None:
        v0 = v0.detach().float().contiguous()
    idx32 = _empty((B, topk), torch.int32, layers[0]) if topk > 0 else None
    idx64 = _empty((B, topk), torch.int64, layers[0]) if (topk > 0 and want_int64) else None
    _lib.call(entry, table, L, B, H, T, k, FUSIONS[head_fusion], float(identity_w), v0,
              int(drop_first), workspace, scores, int(topk), idx32, idx64)
    if topk > 0:
        return (scores, idx32, idx64) if want_int64 else (scores, idx32)
    return scores


def rollout_scores_cait(all_attn, pre_layer_num: int, discard_ratio: float = 0.9, head_fusion: str = "mean",
                        identity_w: float = 0.2):
    """``attn_rollout_cait(all_attn, discard_ratio, head_fusion, layer_nums=[pre_layer_num, i])[1][:, 0]`` of the
    reference (tools/cait_models_attn.py:223-261, :328-330): all_attn = pre_layer_num patch-layer maps (B,H,T,T)
    followed by i >= 1 class-attention maps (B,H,1,T+1).  Returns the detached token score (B,T).  The dtype rule of
    ``rollout_scores`` applies to the patch maps and to the class-attention maps separately."""
    import ctypes
    patch, cls = list(all_attn[:pre_layer_num]), list(all_attn[pre_layer_num:])
    assert patch and cls, "CaiT rollout needs patch layers and at least one class-attention layer"
    entry, cls = _attn_tables(cls, "pph_rollout_cls_rows")
    B, H, R, Tc = cls[0].shape
    assert R == 1 and all(c.shape == cls[0].shape for c in cls)
    v0 = _empty((B, Tc - 1), torch.float32, cls[0])
    table = (ctypes.c_void_p * len(cls))(*[_ptr_of(c) for c in cls])
    _lib.call(entry, table, len(cls), B, H, Tc, int(Tc * discard_ratio), FUSIONS[head_fusion],
              float(identity_w), v0)
    return rollout_scores(patch, discard_ratio, head_fusion, identity_w, v0=v0, drop_first=False)


def _ptr_of(t: torch.Tensor) -> int:
    assert t.is_cuda and t.is_contiguous()
    return t.data_ptr()


# ------------------------------------------------------------------------------------------------------------------
# (a2) gather + add-on layer -- protopformer.py:159-172
# ------------------------------------------------------------------------------------------------------------------
class _Addon(torch.autograd.Function):
    @staticmethod
    @torch.amp.custom_fwd(device_type="cuda", cast_inputs=torch.float32)
    def forward(ctx, tokens, idx32, Wa, ba, want_split, center):
        ctx.set_materialize_grads(False)
        tokens, Wa, ba = tokens.contiguous(), Wa.contiguous(), ba.contiguous()
        B, n1, Din = tokens.shape
        N, K, D = n1 - 1, idx32.shape[1], Wa.shape[0]
        f32, bf = torch.float32, torch.bfloat16
        check_head_dtypes(tokens, Wa, ba)
        Zs, Zc = _empty((B, K, D), f32, tokens), _empty((B, D), f32, tokens)
        z2s, z2c = _empty((B, K), f32, tokens), _empty((B,), f32, tokens)
        if want_split:
            z2s_ctr, z2c_ctr = _empty((B, K), f32, tokens), _empty((B,), f32, tokens)
            z2s_hi, z2c_hi = _empty((B, K), f32, tokens), _empty((B,), f32, tokens)
            Zs_hi, Zs_lo = _empty((B * K, D), bf, tokens), _empty((B * K, D), bf, tokens)
            Zc_hi, Zc_lo = _empty((B, D), bf, tokens), _empty((B, D), bf, tokens)
        else:
            z2s_ctr = z2c_ctr = z2s_hi = z2c_hi = Zs_hi = Zs_lo = Zc_hi = Zc_lo = None
        _lib.call(token_entry("pph_addon_fwd", tokens.dtype), tokens, idx32, Wa, ba, B, N, Din, D, K, Zs, Zc, z2s, z2c, float(center),
                  z2s_ctr, z2c_ctr, z2s_hi, z2c_hi, Zs_hi, Zs_lo, Zc_hi, Zc_lo)
        ctx.save_for_backward(tokens, idx32, Wa, Zs, Zc)
        ctx.dims = (B, N, Din, D, K)
        aux = [z2s, z2c, z2s_ctr, z2c_ctr, z2s_hi, z2c_hi, Zs_hi, Zs_lo, Zc_hi, Zc_lo]
        aux = [a if a is not None else _empty((0,), f32, tokens) for a in aux]
        ctx.mark_non_differentiable(*aux)
        return (Zs, Zc, *aux)

    @staticmethod
    @torch.amp.custom_bwd(device_type="cuda")
    def backward(ctx, dZs, dZc, *_unused):
        tokens, idx32, Wa, Zs, Zc = ctx.saved_tensors
        B, N, Din, D, K = ctx.dims
        dZs = torch.zeros_like(Zs) if dZs is None else dZs.contiguous()
        dZc = torch.zeros_like(Zc) if dZc is None else dZc.contiguous()
        dWa, dba = torch.empty_like(Wa), _empty((D,), torch.float32, Wa)
        want_dtok = ctx.needs_input_grad[0]
        bits = _lib.load().pph_addon_tc2_supported(B, N, Din, D, K)
        if (bits & 4) and (not want_dtok or (bits & 2)):
            # single-shot tcgen05 kernels (the fused step's): 2e-5 of float64 on dtokens where the pipelined round-1 kernel
            # measured 3e-4 (scripts/measure_tolerances.py); they take the pre-activation gradient
            dpre_s, dpre_c = dZs * Zs * (1.0 - Zs), dZc * Zc * (1.0 - Zc)
            ws = _cached_zero_ws("pph_addon_tc2_ws_bytes", (B, N, Din, D, K), tokens.device)
            dtok = torch.zeros_like(tokens) if want_dtok else None       # a bf16 leaf gets a bf16 gradient
            _lib.call(token_entry("pph_addon_bwd3", tokens.dtype), 1 | (2 if want_dtok else 0), tokens, idx32, Wa, dpre_s, dpre_c, None, B, N, Din, D, K,
                      ws, dWa, dba, dtok)
            return dtok, None, dWa, dba, None, None
        dtok = torch.empty_like(tokens) if want_dtok else None
        ws = addon_bwd_workspace(B, N, Din, D, K, tokens.device)
        _lib.call(token_entry("pph_addon_bwd", tokens.dtype), tokens, idx32, Wa, Zs, Zc, dZs, dZc, B, N, Din, D, K, ws,
                  1 | (2 if dtok is not None else 0), dWa, dba, dtok)
        return dtok, None, dWa, dba, None, None


_zero_ws_cache = {}


def _cached_zero_ws(fn: str, dims, device):
    """Workspace of `fn(*dims)` bytes, zero-filled ONCE per (entry point, shape, device, stream): the kernels' counters reset
    themselves, and launches on one stream are serial."""
    key = (fn, tuple(dims), str(device), torch.cuda.current_stream(device).cuda_stream)
    ws = _zero_ws_cache.get(key)
    if ws is None:
        ws = _zero_ws_cache[key] = _ws(fn, *dims, zero=True, device=device)
    return ws


@dataclasses.dataclass
class TokenFeatures:
    """Output of the add-on stage: fp32 features (autograd-tracked) + the operands the tensor-core kernel reads."""

    Zs: torch.Tensor            # (B,K,D)
    Zc: torch.Tensor            # (B,D)
    z2s: torch.Tensor           # (B,K)  |z|^2
    z2c: torch.Tensor           # (B,)
    z2s_ctr: torch.Tensor | None   # |z - center|^2            (BF16X3 mode)
    z2c_ctr: torch.Tensor | None
    z2s_hi: torch.Tensor | None    # |bf16(z - center)|^2      (BF16 mode)
    z2c_hi: torch.Tensor | None
    Zs_hi: torch.Tensor | None  # (B*K,D) bf16
    Zs_lo: torch.Tensor | None
    Zc_hi: torch.Tensor | None
    Zc_lo: torch.Tensor | None
    idx32: torch.Tensor         # (B,K)


def addon(tokens, idx32, Wa, ba, want_split: bool, center: float = 0.5) -> TokenFeatures:
    """tokens (B,1+N,Din) float32 or bfloat16, idx32 (B,K), Wa (D,Din) or (D,Din,1,1), ba (D)."""
    check_head_dtypes(tokens, Wa, ba)
    Wa2 = Wa.reshape(Wa.shape[0], -1)
    out = _Addon.apply(tokens, idx32, Wa2, ba, want_split, center)
    Zs, Zc, z2s, z2c, z2s_ctr, z2c_ctr, z2s_hi, z2c_hi, Zs_hi, Zs_lo, Zc_hi, Zc_lo = out
    if not want_split:
        z2s_ctr = z2c_ctr = z2s_hi = z2c_hi = Zs_hi = Zs_lo = Zc_hi = Zc_lo = None
    return TokenFeatures(Zs, Zc, z2s, z2c, z2s_ctr, z2c_ctr, z2s_hi, z2c_hi, Zs_hi, Zs_lo, Zc_hi, Zc_lo, idx32)


# ------------------------------------------------------------------------------------------------------------------
# operand preparation for prototypes -- the p2 term of protopformer.py:207-208 (+ bf16 split for tcgen05)
# ------------------------------------------------------------------------------------------------------------------
@dataclasses.dataclass
class ProtoOperands:
    P: torch.Tensor                 # (R,D) fp32 (detached, contiguous)
    p2: torch.Tensor                # (R,)  |p|^2
    p2_ctr: torch.Tensor | None     # |p - center|^2
    p2_hi: torch.Tensor | None      # |bf16(p - center)|^2
    hi: torch.Tensor | None         # (R,D) bf16
    lo: torch.Tensor | None


def prepare_prototypes(P2d: torch.Tensor, want_split: bool, center: float = 0.5) -> ProtoOperands:
    P = P2d.detach()
    if P.dtype != torch.float32:
        P = P.float()
    P = P.contiguous()
    R, D = P.shape
    p2 = _empty((R,), torch.float32, P)
    if want_split:
        hi, lo = _empty((R, D), torch.bfloat16, P), _empty((R, D), torch.bfloat16, P)
        p2_ctr, p2_hi = _empty((R,), torch.float32, P), _empty((R,), torch.float32, P)
    else:
        hi = lo = p2_ctr = p2_hi = None
    _lib.call("pph_split_rows", P, R, D, float(center), hi, lo, p2, p2_ctr, p2_hi)
    return ProtoOperands(P, p2, p2_ctr, p2_hi, hi, lo)


# ------------------------------------------------------------------------------------------------------------------
# (a3-a6) similarity + pooling + last layers -- protopformer.py:201-247, 297-300
# ------------------------------------------------------------------------------------------------------------------
def _similarity_raw(cfg: HeadConfig, tf: TokenFeatures, pl: ProtoOperands, pg: ProtoOperands,
                    want_maps: bool = False, mode_id: int | None = None):
    """Launch pph_similarity_fwd; returns dmin_l, argmin, act_l, dmin_g, act_g (+ dist_map, act_map)."""
    Zs = tf.Zs.detach()
    B, K, D = Zs.shape
    P, Pg = pl.P.shape[0], pg.P.shape[0]
    mode = cfg.mode_id if mode_id is None else mode_id
    f32 = torch.float32
    dmin_l, act_l = _empty((B, P), f32, Zs), _empty((B, P), f32, Zs)
    argmin = _empty((B, P), torch.int32, Zs)
    dmin_g, act_g = _empty((B, Pg), f32, Zs), _empty((B, Pg), f32, Zs)
    dist_map = act_map = None
    if want_maps:
        assert mode == _lib.MODE_FP32_FMA
        dist_map, act_map = _empty((B, P, K), f32, Zs), _empty((B, P, K), f32, Zs)
    # norms must match the operands the mode contracts: plain (FP32_FMA), centred fp32 (BF16X3), centred rounded (BF16)
    sel = {_lib.MODE_FP32_FMA: lambda a, b, c: a, _lib.MODE_BF16X3: lambda a, b, c: b, _lib.MODE_BF16: lambda a, b, c: c}[mode]
    _lib.call("pph_similarity_fwd", mode, cfg.act_id, float(cfg.eps), B, K, D, P, Pg,
              Zs, tf.Zc.detach(), sel(tf.z2s, tf.z2s_ctr, tf.z2s_hi), sel(tf.z2c, tf.z2c_ctr, tf.z2c_hi),
              tf.Zs_hi, tf.Zs_lo, tf.Zc_hi, tf.Zc_lo,
              pl.P, pg.P, sel(pl.p2, pl.p2_ctr, pl.p2_hi), sel(pg.p2, pg.p2_ctr, pg.p2_hi),
              pl.hi, pl.lo, pg.hi, pg.lo,
              dmin_l, argmin, act_l, dmin_g, act_g, dist_map, act_map)
    return dmin_l, argmin, act_l, dmin_g, act_g, dist_map, act_map


class _SimilarityLogits(torch.autograd.Function):
    """(Zs, Zc, P, Pg, Wl, Wg) -> logits.  Wl / Wg are frozen in the reference (protopformer.py:130-131); one that requires
    grad gets its weight gradient from pph_last_layer_wgrad (the frozen default saves nothing extra and launches nothing)."""

    @staticmethod
    @torch.amp.custom_fwd(device_type="cuda", cast_inputs=torch.float32)
    def forward(ctx, Zs, Zc, P2d, Pg2d, Wl, Wg, tf, cfg):
        ctx.set_materialize_grads(False)
        want_split = cfg.mode_id != _lib.MODE_FP32_FMA
        pl = prepare_prototypes(P2d, want_split, cfg.center)
        pg = prepare_prototypes(Pg2d, want_split, cfg.center)
        dmin_l, argmin, act_l, dmin_g, act_g, _, _ = _similarity_raw(cfg, tf, pl, pg)
        B, P = act_l.shape
        Pg, C = act_g.shape[1], Wl.shape[0]
        Wl, Wg = Wl.detach().contiguous(), Wg.detach().contiguous()
        logits = _empty((B, C), torch.float32, Zs)
        logits_g, logits_l = torch.empty_like(logits), torch.empty_like(logits)
        _lib.call("pph_logits_fwd", act_l, act_g, Wl, Wg, B, P, Pg, C, float(cfg.global_coe), logits, logits_g, logits_l)
        want_w = ctx.needs_input_grad[4] or ctx.needs_input_grad[5]
        ctx.save_for_backward(Zs, Zc, pl.P, pg.P, Wl, Wg, dmin_l, dmin_g, argmin, *((act_l, act_g) if want_w else ()))
        ctx.cfg = cfg
        ctx.mark_non_differentiable(act_l, act_g, dmin_l, dmin_g, argmin, pl.p2)
        return logits, logits_g, logits_l, act_l, act_g, dmin_l, dmin_g, argmin, pl.p2

    @staticmethod
    @torch.amp.custom_bwd(device_type="cuda")
    def backward(ctx, dlogits, dlogits_g, dlogits_l, *_unused):
        Zs, Zc, Pl, Pgl, Wl, Wg, dmin_l, dmin_g, argmin, *acts = ctx.saved_tensors
        cfg = ctx.cfg
        B, K, D = Zs.shape
        P, Pg, C = Pl.shape[0], Pgl.shape[0], Wl.shape[0]
        f32 = torch.float32
        if dlogits is None:
            dlogits = torch.zeros((B, C), dtype=f32, device=Zs.device)
        dlogits = dlogits.contiguous()
        dlogits_g = None if dlogits_g is None else dlogits_g.contiguous()
        dlogits_l = None if dlogits_l is None else dlogits_l.contiguous()
        g_l, g_g = _empty((B, P), f32, Zs), _empty((B, Pg), f32, Zs)
        _lib.call("pph_logits_bwd", dlogits, dlogits_g, dlogits_l, Wl, Wg, dmin_l, dmin_g, B, P, Pg, C,
                  float(cfg.global_coe), cfg.act_id, float(cfg.eps), g_l, g_g)
        dZs, dZc = torch.empty_like(Zs), torch.empty_like(Zc)
        dPl, dPg = torch.empty_like(Pl), torch.empty_like(Pgl)
        ws = bwd_workspace(B, K, D, P, Pg, Zs.device)
        _lib.call("pph_similarity_bwd", g_l, g_g, argmin, Zs, Zc, Pl, Pgl, B, K, D, P, Pg, ws, 3, None, None,
                  dZs, dZc, dPl, dPg)
        dWl = torch.empty_like(Wl) if ctx.needs_input_grad[4] else None
        dWg = torch.empty_like(Wg) if ctx.needs_input_grad[5] and Pg > 0 else None
        if dWl is not None or dWg is not None:
            act_l, act_g = acts
            _lib.call("pph_last_layer_wgrad", dlogits, dlogits_g, dlogits_l, act_l, act_g, B, P, Pg, C,
                      float(cfg.global_coe), dWl, dWg)
        return dZs, dZc, dPl, dPg, dWl, dWg, None, None


def addon_bwd_workspace(B, N, Din, D, K, device) -> torch.Tensor:
    """Scratch for pph_addon_bwd (split-K partials of the add-on weight gradient)."""
    import ctypes
    n = ctypes.c_longlong(0)
    if _lib.load().pph_addon_bwd_ws_bytes(B, N, Din, D, K, ctypes.byref(n)) != 0:
        raise RuntimeError("pph_addon_bwd_ws_bytes failed")
    return torch.empty(max(int(n.value), 256), dtype=torch.uint8, device=device)


def bwd_workspace(B, K, D, P, Pg, device) -> torch.Tensor:
    """Zero-filled scratch for pph_similarity_bwd (token bins + self-resetting counters)."""
    import ctypes
    n = ctypes.c_longlong(0)
    rc = _lib.load().pph_similarity_bwd_ws_bytes(B, K, D, P, Pg, ctypes.byref(n))
    if rc != 0:
        raise RuntimeError("pph_similarity_bwd_ws_bytes failed")
    return torch.zeros(max(int(n.value), 256), dtype=torch.uint8, device=device)


@dataclasses.dataclass
class HeadOutput:
    logits: torch.Tensor
    logits_global: torch.Tensor
    logits_local: torch.Tensor
    act_l: torch.Tensor         # (B,P) pooled local activations
    act_g: torch.Tensor         # (B,Pg)
    dmin_l: torch.Tensor        # (B,P) min distance over tokens
    dmin_g: torch.Tensor
    argmin: torch.Tensor        # (B,P) int32 token slot of the max activation
    p2l: torch.Tensor           # (P,) |prototype|^2 (reused by the PPC loss)
    tf: TokenFeatures


def head_forward(cfg: HeadConfig, tokens, scores, Wa, ba, P, Pg, Wl, Wg) -> HeadOutput:
    """The whole prototype head after the backbone: selection -> add-on -> similarity/pool -> logits.

    tokens (B,1+N,Din) float32 or bfloat16 (a bf16 backbone's output, read as it is), scores (B,N)|(B,H,N),
    Wa (D,Din[,1,1]), ba (D), P (P,D[,1,1]), Pg (Pg,D[,1,1]), Wl (C,P), Wg (C,Pg) float32.
    Replaces protopformer.py:156-172 + 311-316.
    """
    check_head_dtypes(tokens, Wa, ba, P, Pg, Wl, Wg)
    if tokens.shape[0] == 0:
        return _empty_head_output(cfg, tokens, Wa, P, Pg, Wl)
    idx32 = select_topk(scores, cfg.K)
    want_split = cfg.mode_id != _lib.MODE_FP32_FMA
    tf = addon(tokens, idx32, Wa, ba, want_split, cfg.center)
    P2d, Pg2d = P.reshape(P.shape[0], -1), Pg.reshape(Pg.shape[0], -1)
    out = _SimilarityLogits.apply(tf.Zs, tf.Zc, P2d, Pg2d, Wl, Wg, tf, cfg)
    logits, lg, ll, act_l, act_g, dmin_l, dmin_g, argmin, p2l = out
    return HeadOutput(logits, lg, ll, act_l, act_g, dmin_l, dmin_g, argmin, p2l, tf)


def _empty_head_output(cfg, tokens, Wa, P, Pg, Wl) -> HeadOutput:
    """B == 0 (e.g. an empty last shard): nothing to launch."""
    f32, dev = torch.float32, tokens.device
    D, Pn, Pgn, C = Wa.shape[0], P.shape[0], Pg.shape[0], Wl.shape[0]
    z = lambda *s, dt=f32: torch.zeros(s, dtype=dt, device=dev)  # noqa: E731
    tf = TokenFeatures(z(0, cfg.K, D), z(0, D), z(0, cfg.K), z(0), None, None, None, None, None, None, None, None,
                       z(0, cfg.K, dt=torch.int32))
    return HeadOutput(z(0, C), z(0, C), z(0, C), z(0, Pn), z(0, Pgn), z(0, Pn), z(0, Pgn), z(0, Pn, dt=torch.int32),
                      z(Pn), tf)


def materialize_maps(cfg: HeadConfig, tf: TokenFeatures, P, Pg):
    """Full (B,P,K) distance and activation maps (eval aux `distances` :301, push_forward `proto_acts` :344).
    Always computed by the FP32-FMA kernel; not part of the autograd graph."""
    pl = prepare_prototypes(P.reshape(P.shape[0], -1), False)
    pg = prepare_prototypes(Pg.reshape(Pg.shape[0], -1), False)
    _, _, _, _, _, dist_map, act_map = _similarity_raw(cfg, tf, pl, pg, want_maps=True, mode_id=_lib.MODE_FP32_FMA)
    return dist_map, act_map


def class_activation_maps(cfg: HeadConfig, tf: TokenFeatures, P, labels, m: int, N: int, p2l=None):
    """(B, m, side, side) activation maps of each image's label-class prototypes on the original token grid, zeros on
    pruned tokens -- eval_interpretability.py:195-225 (gather of the class rows of `proto_acts` + scatter from the
    h x w reserved tokens to the 14 x 14 grid) without materialising the (B,P,h,w) map.  Not differentiable."""
    side = int(round(math.sqrt(N)))
    assert side * side == N
    P2d = P.detach().reshape(P.shape[0], -1).float().contiguous()
    if p2l is None:
        p2l = prepare_prototypes(P2d, False).p2
    Zs = tf.Zs.detach()
    B, K, D = Zs.shape
    maps = _empty((B, m, N), torch.float32, Zs)
    _lib.call("pph_class_maps", Zs, tf.z2s, P2d, p2l, tf.idx32, labels.to(torch.int64).contiguous(), B, K, D,
              P2d.shape[0], m, N, cfg.act_id, float(cfg.eps), maps)
    return maps.view(B, m, side, side)


# ------------------------------------------------------------------------------------------------------------------
# (a7) PPC loss -- protopformer.py:249-288
# ------------------------------------------------------------------------------------------------------------------
class _PPC(torch.autograd.Function):
    @staticmethod
    @torch.amp.custom_fwd(device_type="cuda", cast_inputs=torch.float32)
    def forward(ctx, Zs, P2d, z2s, p2l, idx32, labels, m, N, cfg):
        ctx.set_materialize_grads(False)
        Zs, Pl = Zs.contiguous(), P2d.contiguous()
        B, K, D = Zs.shape
        P = Pl.shape[0]
        f32 = torch.float32
        labels = labels.to(torch.int64).contiguous()
        dslice, stats = _empty((B, m, K), f32, Zs), _empty((B, m, 8), f32, Zs)
        partial = _empty((B, 2), f32, Zs)
        counter = torch.zeros((1,), dtype=torch.int32, device=Zs.device)
        losses = _empty((2,), f32, Zs)
        _lib.call("pph_ppc_fwd", Zs, z2s, Pl, p2l, idx32, labels, B, K, D, P, m, N, cfg.act_id, float(cfg.eps),
                  float(cfg.ppc_cov_thresh), float(cfg.ppc_mean_thresh), dslice, stats, partial, counter, losses)
        ctx.save_for_backward(Zs, Pl, idx32, labels, dslice, stats)
        ctx.meta = (m, N, cfg)
        return losses[0], losses[1]

    @staticmethod
    @torch.amp.custom_bwd(device_type="cuda")
    def backward(ctx, g_cov, g_mean):
        Zs, Pl, idx32, labels, dslice, stats = ctx.saved_tensors
        m, N, cfg = ctx.meta
        B, K, D = Zs.shape
        P = Pl.shape[0]
        zero = torch.zeros((), dtype=torch.float32, device=Zs.device)
        g = torch.stack([zero if g_cov is None else g_cov.float(), zero if g_mean is None else g_mean.float()])
        dZs, dP = torch.empty_like(Zs), torch.zeros_like(Pl)
        _lib.call("pph_ppc_bwd", Zs, Pl, idx32, labels, dslice, stats, g, 1.0, 1.0, B, K, D, P, m, N, cfg.act_id,
                  float(cfg.eps), float(cfg.ppc_cov_thresh), float(cfg.ppc_mean_thresh), 0, dZs, dP)
        return dZs, dP, None, None, None, None, None, None, None


def ppc_loss(cfg: HeadConfig, tf: TokenFeatures, P, p2l, labels, m: int, N: int):
    """-> (ppc_cov_loss, ppc_mean_loss) 0-dim tensors; gradients reach Zs (hence the add-on and tokens) and P."""
    side = int(round(math.sqrt(N)))
    assert side * side == N, "original_fea_len must be a perfect square (protopformer.py:260)"
    P2d = P.reshape(P.shape[0], -1)
    if p2l is None:
        p2l = prepare_prototypes(P2d, False).p2
    return _PPC.apply(tf.Zs, P2d, tf.z2s, p2l, tf.idx32, labels, m, N, cfg)


class _PPCDense(torch.autograd.Function):
    """get_PPC_loss on a dense (B,P,K) activation tensor (protopformer.py:259-288); gradient w.r.t. the tensor."""

    @staticmethod
    def forward(ctx, act, idx32, labels, m, N, cov_thresh, mean_thresh):
        B, P, K = act.shape
        dev = act.device
        stats = torch.empty(B, m, 8, dtype=torch.float32, device=dev)
        partial = torch.empty(B, 2, dtype=torch.float32, device=dev)
        counter = torch.zeros(1, dtype=torch.int32, device=dev)
        losses = torch.empty(2, dtype=torch.float32, device=dev)
        _lib.call("pph_ppc_dense_fwd", act, idx32, labels, B, P, K, m, N, float(cov_thresh), float(mean_thresh), stats,
                  partial, counter, losses)
        ctx.save_for_backward(act, idx32, labels, stats)
        ctx.dims = (B, P, K, m, N, float(mean_thresh))
        return losses[0], losses[1]

    @staticmethod
    def backward(ctx, g_cov, g_mean):
        act, idx32, labels, stats = ctx.saved_tensors
        B, P, K, m, N, mean_thresh = ctx.dims
        zero = torch.zeros((), dtype=torch.float32, device=act.device)
        g_cov = zero if g_cov is None else g_cov.to(torch.float32).contiguous()
        g_mean = zero if g_mean is None else g_mean.to(torch.float32).contiguous()
        dact = torch.empty_like(act)
        _lib.call("pph_ppc_dense_bwd", act, idx32, labels, stats, g_cov, g_mean, B, P, K, m, N, mean_thresh, dact)
        return dact, None, None, None, None, None, None


def ppc_loss_dense(cfg: HeadConfig, total_proto_act: torch.Tensor, cls_attn_rollout: torch.Tensor, labels, m: int, N: int):
    """The reference's `get_PPC_loss` signature for a caller that holds the activation map as a (B,P,h,w) tensor:
    the selected-token list is recomputed from `cls_attn_rollout` exactly as protopformer.py:273-274 does (top-K with
    K = h*w, ascending), the label-class rows are gathered from the map.  -> (ppc_cov_loss, ppc_mean_loss)."""
    side = int(round(math.sqrt(N)))
    assert side * side == N, "original_fea_len must be a perfect square (protopformer.py:260)"
    assert total_proto_act.is_cuda and total_proto_act.dtype == torch.float32, "float32 CUDA tensor expected (no CPU path)"
    act = total_proto_act.flatten(2).contiguous()
    K = act.shape[-1]
    idx32 = select_topk(cls_attn_rollout.detach(), K)
    return _PPCDense.apply(act, idx32, labels.contiguous(), m, N, cfg.ppc_cov_thresh, cfg.ppc_mean_thresh)


# ------------------------------------------------------------------------------------------------------------------
# Fused training / inference step: the same entry points in a fixed sequence over pre-allocated buffers, no autograd
# graph and no PyTorch glue kernels in between (what tools/engine_proto.py:49-76 amounts to for the head).
# ------------------------------------------------------------------------------------------------------------------
def _last_layer_grad_targets(train: bool, Wl, Wg, grads):
    """(dWl, dWg) the training step writes, None for a frozen layer.  A last layer is trained iff its weight requires grad
    (the reference's switch, protopformer.py:130-131); its gradient is OVERWRITTEN in grads["Wl"] / grads["Wg"]."""
    if not train:
        return None, None
    out = []
    for k, W in (("Wl", Wl), ("Wg", Wg)):
        g = (grads or {}).get(k) if W.requires_grad else None
        if W.requires_grad and g is None:
            raise ValueError(f"the {k} last layer requires grad: pass grads[{k!r}] for the step to write its gradient into")
        out.append(g)
    return tuple(out)


def _step_token_entries(step, tokens, *params):
    """Host-side checks of a fused step's inputs (before any launch) -> name -> the entry point for the step's token type."""
    if tokens.dtype != step.token_dtype:
        token_entry("", tokens.dtype)
        raise TypeError(f"this step was built for {step.token_dtype} tokens, got {tokens.dtype} "
                        "(pass token_dtype= to the constructor)")
    check_head_dtypes(tokens, *params)
    return lambda name: token_entry(name, step.token_dtype)


class FusedHeadStepV1:
    """Round-1 launch sequence (16 launches over three streams), kept as the fallback for shapes the round-2 step (FusedHeadStep)
    was not built for and as an A/B arm.  forward (+ PPC + cross-entropy + backward) of the head for a fixed shape.

    step(tokens, scores, labels, Wa, ba, P, Pg, Wl, Wg, grads) launches, in order:
      select_topk, addon_fwd, split_rows x2, similarity_fwd, logits_fwd, [ppc_fwd,] loss_tail,
      [logits_bwd, similarity_bwd, ppc_bwd(accumulate), addon_bwd]
    Results live in attributes: losses (4,) = (total, ce, ppc_cov, ppc_mean), logits, logits_g, logits_l, act_l,
    dmin_l, argmin, idx32, dtokens; parameter gradients are OVERWRITTEN in the tensors of `grads`
    (keys Wa, ba, P, Pg -- e.g. views of one flat all-reduce buffer -- and Wl / Wg for a last layer whose weight requires
    grad: pph_last_layer_wgrad right after the loss tail)."""

    def __init__(self, cfg: HeadConfig, B, N, Din, D, P, Pg, C, m, device, heads: int = 0, ppc_cov_coe: float = 0.1,
                 ppc_mean_coe: float = 0.5, train: bool = True, use_ppc: bool = True, token_dtype=torch.float32):
        token_entry("", token_dtype)
        self.cfg, self.train, self.use_ppc, self.token_dtype = cfg, train, use_ppc, token_dtype
        self.dims = (B, N, Din, D, P, Pg, C, m, heads)
        self.cov_coe, self.mean_coe = float(ppc_cov_coe), float(ppc_mean_coe)
        K = cfg.K
        f32, bf, i32 = torch.float32, torch.bfloat16, torch.int32
        e = lambda *s, dt=f32: torch.empty(s, dtype=dt, device=device)  # noqa: E731
        z = lambda *s, dt=f32: torch.zeros(s, dtype=dt, device=device)  # noqa: E731
        self.split = cfg.mode_id != _lib.MODE_FP32_FMA
        self.idx32 = e(B, K, dt=i32)
        self.Zs, self.Zc, self.z2s, self.z2c = e(B, K, D), e(B, D), e(B, K), e(B)
        if self.split:
            self.z2s_ctr, self.z2c_ctr, self.z2s_hi, self.z2c_hi = e(B, K), e(B), e(B, K), e(B)
            self.Zs_hi, self.Zs_lo, self.Zc_hi, self.Zc_lo = e(B * K, D, dt=bf), e(B * K, D, dt=bf), e(B, D, dt=bf), e(B, D, dt=bf)
            self.P_hi, self.P_lo, self.Pg_hi, self.Pg_lo = e(P, D, dt=bf), e(P, D, dt=bf), e(Pg, D, dt=bf), e(Pg, D, dt=bf)
            self.p2_ctr, self.p2_hi, self.pg2_ctr, self.pg2_hi = e(P), e(P), e(Pg), e(Pg)
        else:
            for n in ("z2s_ctr", "z2c_ctr", "z2s_hi", "z2c_hi", "Zs_hi", "Zs_lo", "Zc_hi", "Zc_lo", "P_hi", "P_lo",
                      "Pg_hi", "Pg_lo", "p2_ctr", "p2_hi", "pg2_ctr", "pg2_hi"):
                setattr(self, n, None)
        self.p2, self.pg2 = e(P), e(Pg)
        self.dmin_l, self.act_l, self.argmin = e(B, P), e(B, P), e(B, P, dt=i32)
        self.dmin_g, self.act_g = e(B, Pg), e(B, Pg)
        self.logits, self.logits_g, self.logits_l = e(B, C), e(B, C), e(B, C)
        self.dslice, self.stats, self.ppc_partial = e(B, m, K), e(B, m, 8), e(B, 2)
        self.ppc_counter, self.ppc_losses = z(1, dt=i32), z(2)
        self.ce_partial, self.ce_counter, self.losses = e(B), z(1, dt=i32), z(4)
        self.losses_ce = z(4)
        if train:
            self.dlogits, self.g_l, self.g_g = e(B, C), e(B, P), e(B, Pg)
            self.dZs, self.dZc = e(B, K, D), e(B, D)
            self.dZs_ppc, self.dP_ppc = e(B, K, D), z(P, D)
            self.dtokens = e(B, 1 + N, Din, dt=token_dtype)
            self.ws = bwd_workspace(B, K, D, P, Pg, device)
            self.ws_addon = addon_bwd_workspace(B, N, Din, D, K, device)
        # independent kernels run on a forked stream (under CUDA-graph capture this becomes a parallel branch)
        self.side = torch.cuda.Stream(device=device)
        self.side2 = torch.cuda.Stream(device=device)
        self.ev = [torch.cuda.Event() for _ in range(10)]

    def step(self, tokens, scores, labels, Wa, ba, P, Pg, Wl, Wg, grads=None, upstream: float = 1.0):
        B, N, Din, D, Pn, Pgn, C, m, H = self.dims
        cfg, K = self.cfg, self.cfg.K
        c = _lib.call
        tok = _step_token_entries(self, tokens, Wa, ba, P, Pg, Wl, Wg)
        main, side, ev = torch.cuda.current_stream(), self.side, self.ev
        # Three streams while training with the PPC loss: the token bins run on their own branch, and the cross-entropy
        # tail does not wait for the PPC loss (their weighted sum is a separate 1-thread kernel on the side branch).
        # Measured against a two-stream order (profiles/r1b_ab_variants.txt): 187.6 -> 171.8 us per step at the CUB
        # shape, B = 64.
        ppc = self.use_ppc and self.train
        # branch: prototype operand preparation || selection + add-on
        ev[0].record(main)
        side.wait_event(ev[0])
        with torch.cuda.stream(side):
            if ppc:
                self.dP_ppc.zero_()
            c("pph_split_rows", P, Pn, D, float(cfg.center), self.P_hi, self.P_lo, self.p2, self.p2_ctr, self.p2_hi)
            c("pph_split_rows", Pg, Pgn, D, float(cfg.center), self.Pg_hi, self.Pg_lo, self.pg2, self.pg2_ctr, self.pg2_hi)
            ev[1].record(side)
        c("pph_select_topk", scores, B, max(H, 1), N, K, self.idx32, None)
        c(tok("pph_addon_fwd"), tokens, self.idx32, Wa, ba, B, N, Din, D, K, self.Zs, self.Zc, self.z2s, self.z2c,
          float(cfg.center), self.z2s_ctr, self.z2c_ctr, self.z2s_hi, self.z2c_hi, self.Zs_hi, self.Zs_lo,
          self.Zc_hi, self.Zc_lo)
        main.wait_event(ev[1])
        mode = cfg.mode_id
        sel = {_lib.MODE_FP32_FMA: 0, _lib.MODE_BF16X3: 1, _lib.MODE_BF16: 2}[mode]
        c("pph_similarity_fwd", mode, cfg.act_id, float(cfg.eps), B, K, D, Pn, Pgn, self.Zs, self.Zc,
          (self.z2s, self.z2s_ctr, self.z2s_hi)[sel], (self.z2c, self.z2c_ctr, self.z2c_hi)[sel],
          self.Zs_hi, self.Zs_lo, self.Zc_hi, self.Zc_lo, P, Pg,
          (self.p2, self.p2_ctr, self.p2_hi)[sel], (self.pg2, self.pg2_ctr, self.pg2_hi)[sel],
          self.P_hi, self.P_lo, self.Pg_hi, self.Pg_lo,
          self.dmin_l, self.argmin, self.act_l, self.dmin_g, self.act_g, None, None)

        if ppc:   # branch: PPC loss || last layers (forked after the persistent similarity kernel so it cannot delay it)
            ev[2].record(main)
            side.wait_event(ev[2])
            with torch.cuda.stream(side):
                c("pph_ppc_fwd", self.Zs, self.z2s, P, self.p2, self.idx32, labels, B, K, D, Pn, m, N, cfg.act_id,
                  float(cfg.eps), float(cfg.ppc_cov_thresh), float(cfg.ppc_mean_thresh), self.dslice, self.stats,
                  self.ppc_partial, self.ppc_counter, self.ppc_losses)
                # the PPC backward only needs the PPC forward: its contributions go to side buffers that the gradient
                # kernel adds while it writes dZs / dP
                c("pph_ppc_bwd", self.Zs, P, self.idx32, labels, self.dslice, self.stats, None,
                  self.cov_coe * float(upstream), self.mean_coe * float(upstream), B, K, D, Pn, m, N, cfg.act_id,
                  float(cfg.eps), float(cfg.ppc_cov_thresh), float(cfg.ppc_mean_thresh), 0, self.dZs_ppc,
                  self.dP_ppc)
            # the token bins of the backward only need argmin: off the critical path, on a third branch
            self.side2.wait_event(ev[2])
            with torch.cuda.stream(self.side2):
                c("pph_similarity_bwd", None, None, self.argmin, None, None, None, None, B, K, D, Pn, Pgn, self.ws,
                  1, None, None, None, None, None, None)
                ev[7].record(self.side2)
        c("pph_logits_fwd", self.act_l, self.act_g, Wl, Wg, B, Pn, Pgn, C, float(cfg.global_coe), self.logits,
          self.logits_g, self.logits_l)
        c("pph_loss_tail", self.logits, labels, None, self.cov_coe, self.mean_coe, float(upstream), B, C,
          self.ce_partial, self.ce_counter, self.losses_ce if ppc else self.losses, self.dlogits if self.train else None)
        if ppc:
            ev[8].record(main)
            side.wait_event(ev[8])
            with torch.cuda.stream(side):
                c("pph_loss_combine", self.losses_ce, self.ppc_losses, self.cov_coe, self.mean_coe, self.losses)
                ev[4].record(side)
        if not self.train:
            return self.losses
        dWl, dWg = _last_layer_grad_targets(self.train, Wl, Wg, grads)
        if dWl is not None or dWg is not None:
            c("pph_last_layer_wgrad", self.dlogits, None, None, self.act_l, self.act_g, B, Pn, Pgn, C,
              float(cfg.global_coe), dWl, dWg)
        c("pph_logits_bwd", self.dlogits, None, None, Wl, Wg, self.dmin_l, self.dmin_g, B, Pn, Pgn, C,
          float(cfg.global_coe), cfg.act_id, float(cfg.eps), self.g_l, self.g_g)
        if ppc:                                        # bins were produced on a side branch next to the PPC loss
            main.wait_event(ev[4])
            main.wait_event(ev[7])
        c("pph_similarity_bwd", self.g_l, self.g_g, self.argmin, self.Zs, self.Zc, P, Pg, B, K, D, Pn, Pgn, self.ws,
          2 if ppc else 3, self.dZs_ppc if ppc else None, self.dP_ppc if ppc else None,
          self.dZs, self.dZc, grads["P"], grads["Pg"])
        # weight gradient || token gradient (independent GEMMs, 82 + 41 CTAs: they share the machine)
        ev[5].record(main)
        side.wait_event(ev[5])
        with torch.cuda.stream(side):
            c(tok("pph_addon_bwd"), tokens, self.idx32, Wa, self.Zs, self.Zc, self.dZs, self.dZc, B, N, Din, D, K,
              self.ws_addon, 2, None, None, self.dtokens)
            ev[6].record(side)
        c(tok("pph_addon_bwd"), tokens, self.idx32, Wa, self.Zs, self.Zc, self.dZs, self.dZc, B, N, Din, D, K,
          self.ws_addon, 1, grads["Wa"], grads["ba"], None)
        main.wait_event(ev[6])
        return self.losses


# ------------------------------------------------------------------------------------------------------------------
# Five-launch step (round 2): head_prep -> similarity_fwd -> head_mid -> similarity_bwd2 -> addon_bwd2 on ONE stream
# ------------------------------------------------------------------------------------------------------------------
def _ws(fn: str, *dims, zero: bool, device) -> torch.Tensor:
    import ctypes
    n = ctypes.c_longlong(0)
    if getattr(_lib.load(), fn)(*dims, ctypes.byref(n)) != 0:
        raise RuntimeError(f"{fn} failed: {_lib.load().pph_last_error_string().decode()}")
    alloc = torch.zeros if zero else torch.empty
    return alloc(max(int(n.value), 256), dtype=torch.uint8, device=device)


def fused_step_supported(B, N, Din, D, K, P, Pg, C, m, token_dtype=torch.float32) -> bool:
    """Host-side check (no device needed): can FusedHeadStep (the round-2 launch sequence) run this shape?"""
    lib = _lib.load()
    if C > 256 or B < 1 or B > 64 * 74 or (token_dtype == torch.bfloat16 and Din % 8 != 0):
        return False
    ppc_smem = 4 * (m * D + K * (D + 4) + 2 * m * K + 8 * m + 32)
    return bool(lib.pph_head_prep_supported(B, N, Din, D, K) and lib.pph_addon_bwd2_supported(B, N, Din, D, K)
                and ppc_smem <= 200 * 1024 and D % 4 == 0 and D <= 512)


class FusedHeadStep:
    """forward (+ PPC + cross-entropy + backward) of the head for a fixed shape: 11 launches over the current stream and two
    side branches (default variants; DESIGN.md section 4.0):

      pph_select_addon_fwd      selection + gather + add-on + sigmoid + bf16 operands (tcgen05, single shot)
        || pph_split_rows x2    bf16 operands / norms of both prototype tensors, memset of dtokens           (side branch)
        || pph_last_layer_pattern  do Wl, Wg still hold the class-connection pattern? (verdict for pph_head_mid)
      pph_similarity_fwd        tcgen05 distances, log similarity, min / argmin over tokens (the (B,P,K) map stays in TMEM)
      pph_head_mid (LL)         last layers (class-sum form when the verdict allows) + cross-entropy + last-layer backward,
                                token bins, class lists
        || pph_head_mid (PPC)   PPC loss forward + backward                                        [training, side branch]
        || pph_last_layer_wgrad dWl, dWg (+ their exchange)        [training with an unfrozen last layer, own branch]
      pph_similarity_bwd_fused  argmin-routed gradients: dP, dPg, pre-activation gradients of the tokens      [training]
        || ppc rows add         PPC prototype rows onto dP                                          [training, side branch]
      pph_addon_bwd3 x2         dtokens, then dWa | dba (tcgen05, single shot)                                [training]

    `variants` selects alternative kernels per stage (exact-FP32 CUDA-core add-on kernels, the staged sparse backward, the
    stand-alone selection launch, PPC inline) -- every combination is covered by tests/test_step2_gpu.py.

    Same results interface as FusedHeadStepV1: losses (4,) = (total, ce, ppc_cov, ppc_mean), logits, logits_g, logits_l,
    act_l, dmin_l, argmin, idx32, dtokens; parameter gradients are OVERWRITTEN in the tensors of `grads`
    (keys Wa, ba, P, Pg -- e.g. views of one flat all-reduce buffer -- and Wl / Wg for a last layer whose weight requires
    grad; with both frozen, the default, the step is exactly the 11 launches above).  Reference: tools/engine_proto.py:49-76."""

    def __init__(self, cfg: HeadConfig, B, N, Din, D, P, Pg, C, m, device, heads: int = 0, ppc_cov_coe: float = 0.1,
                 ppc_mean_coe: float = 0.5, train: bool = True, use_ppc: bool = True, variants=None,
                 token_dtype=torch.float32):
        token_entry("", token_dtype)
        if not fused_step_supported(B, N, Din, D, cfg.K, P, Pg, C, m, token_dtype):
            raise ValueError("shape outside FusedHeadStep's kernels: use FusedHeadStepV1")
        self.cfg, self.train, self.use_ppc, self.token_dtype = cfg, train, use_ppc, token_dtype
        # kernel choice per stage: "tc" = single-shot tcgen05 kernels (pph_addon_fwd2 / pph_addon_bwd3) where the shape
        # allows, "simt" = the exact-FP32 CUDA-core kernels (pph_head_prep / pph_addon_bwd2)
        tc_bits = _lib.load().pph_addon_tc2_supported(B, N, Din, D, cfg.K)
        # "bwd": "gather" = round-1 argmin-routed L2 gather kernel fed by pph_head_mid's bins, "staged" = the three
        # shared-memory-staged kinds of pph_similarity_bwd2;  "ppc": "inline" = PPC role inside the pph_head_mid launch,
        # "split" = its own concurrent launch joined before the backward, "late" = concurrent launch that overlaps the
        # last layers AND the token-side gradients (its token gradient enters through the add-on backward's operand,
        # its prototype rows through the prototype-row launch on the same side branch)
        # "prep": "tc" = single-shot tcgen05 add-on forward (k range resident: Din <= 192), "tc1" = the pipelined tcgen05 kernel
        # of round 1 (any Din % 8 == 0: DeiT-S / Dogs, Din = 384), "simt" = exact-FP32 CUDA-core kernel
        tc1_ok = Din % 8 == 0 and D % 8 == 0 and cfg.mode_id != _lib.MODE_FP32_FMA
        v = {"prep": "tc" if (tc_bits & 1) else ("tc1" if tc1_ok else "simt"),
             "addon_bwd": "tc" if (tc_bits & 6) == 6 else "simt", "bwd": "gather", "ppc": "late",
             "select": "fused" if (tc_bits & 8) else "kernel"}
        v.update(variants or {})
        if v["select"] == "fused" and not (tc_bits & 8):
            v["select"] = "kernel"
        if v["prep"] == "tc" and not (tc_bits & 1):
            v["prep"] = "tc1" if tc1_ok else "simt"
        if v["prep"] == "tc1" and not tc1_ok:
            v["prep"] = "simt"
        if v["addon_bwd"] == "tc" and (tc_bits & 6) != 6:
            v["addon_bwd"] = "simt"
        if v["bwd"] == "staged" and not _lib.load().pph_similarity_bwd2_supported(B, cfg.K, D, P, Pg):
            v["bwd"] = "gather"
        self.variants = v
        self.stop_after = 0             # measurement aid (scripts/step_times.py): truncate the step after stage n
        self.dims = (B, N, Din, D, P, Pg, C, m, heads)
        self.cov_coe, self.mean_coe = float(ppc_cov_coe), float(ppc_mean_coe)
        K = cfg.K
        f32, bf, i32 = torch.float32, torch.bfloat16, torch.int32
        e = lambda *s, dt=f32: torch.empty(s, dtype=dt, device=device)  # noqa: E731
        self.split = cfg.mode_id != _lib.MODE_FP32_FMA
        self.idx32 = e(B, K, dt=i32)
        self.Zs, self.Zc, self.z2s, self.z2c = e(B, K, D), e(B, D), e(B, K), e(B)
        names = ("z2s_ctr", "z2c_ctr", "z2s_hi", "z2c_hi", "Zs_hi", "Zs_lo", "Zc_hi", "Zc_lo", "P_hi", "P_lo", "Pg_hi",
                 "Pg_lo", "p2_ctr", "p2_hi", "pg2_ctr", "pg2_hi")
        if self.split:
            shapes = ((B, K), (B,), (B, K), (B,), (B * K, D), (B * K, D), (B, D), (B, D), (P, D), (P, D), (Pg, D), (Pg, D),
                      (P,), (P,), (Pg,), (Pg,))
            for n, sh in zip(names, shapes):
                setattr(self, n, e(*sh, dt=bf if ("_hi" in n or "_lo" in n) and n[0] in "ZP" else f32))
        else:
            for n in names:
                setattr(self, n, None)
        self.p2, self.pg2 = e(P), e(Pg)
        self.dmin_l, self.act_l, self.argmin = e(B, P), e(B, P), e(B, P, dt=i32)
        self.dmin_g, self.act_g = e(B, Pg), e(B, Pg)
        self.logits, self.logits_g, self.logits_l = e(B, C), e(B, C), e(B, C)
        self.losses = torch.zeros(4, dtype=f32, device=device)
        self.ws_mid = _ws("pph_head_mid_ws_bytes", B, K, D, P, Pg, C, m, zero=True, device=device)
        self.ws_tc = _ws("pph_addon_tc2_ws_bytes", B, N, Din, D, K, zero=True, device=device)
        self.side = torch.cuda.Stream(device=device)
        self.side2 = torch.cuda.Stream(device=device)
        self.ev = [torch.cuda.Event() for _ in range(9)]
        self.side_ll = torch.cuda.Stream(device=device)         # last-layer weight gradients (unfrozen last layers only)
        self.ev_ll = [torch.cuda.Event() for _ in range(2)]
        self.dlogits = self.g_l = self.g_g = self.pairT = self.ws_bins = None
        self.dZs_ppc = self.dP_img = None
        if train:
            Bp = (B + 63) // 64 * 64
            self.dlogits, self.g_l, self.g_g = e(B, C), e(B, P), e(B, Pg)
            self.pairT = e(P + Pg, Bp, 2)
            self.ws_bins = _ws("pph_similarity_bwd2_ws_bytes", B, K, D, P, zero=True, device=device)
            self.ws_gather = bwd_workspace(B, K, D, P, Pg, device)
            if use_ppc:
                self.dZs_ppc, self.dP_img = e(B, K, D), e(B, m, D)
            self.dZs, self.dZc = e(B, K, D), e(B, D)
            self.dtokens = e(B, 1 + N, Din, dt=token_dtype)
            self.ws_addon = _ws("pph_addon_bwd2_ws_bytes", B, N, Din, D, K, zero=True, device=device)
            if self.variants["addon_bwd"] == "tc":
                self.dtokens.zero_()


    def step(self, tokens, scores, labels, Wa, ba, P, Pg, Wl, Wg, grads=None, upstream: float = 1.0, reduce_hook=None,
             idx32=None, loss_mirror=None):
        """reduce_hook(which): called once with "protos" when grads["P"], grads["Pg"] are final (on the stream that
        produced them) and once with "addon" after grads["Wa"], grads["ba"]: the data-parallel caller issues its
        asynchronous all-reduces there so that the first one overlaps the add-on backward.  With an unfrozen last layer
        also once with "last", on the last-layer branch right after grads["Wl"] / grads["Wg"] are written.
        idx32: the ascending selected-token list (B,K) if the caller already ranked this batch's scores (the
        selection-first host transfer does): the step then skips its own selection launch and `self.idx32` is not
        updated.  loss_mirror: address of 4 floats (16-byte aligned, e.g. mapped pinned host memory) that receive
        (total, ce, ppc_cov, ppc_mean) straight from the kernel that completes the loss."""
        own_idx = self.idx32  # noqa: F841
        sel_idx = own_idx if idx32 is None else idx32
        B, N, Din, D, Pn, Pgn, C, m, H = self.dims
        cfg, K = self.cfg, self.cfg.K
        c = _lib.call
        tok = _step_token_entries(self, tokens, Wa, ba, P, Pg, Wl, Wg)
        main, side, side2, ev = torch.cuda.current_stream(), self.side, self.side2, self.ev
        hook = reduce_hook or (lambda which: None)

        def last_layer_pattern():
            # do both last layers still hold the class-connection pattern?  Decided on the device every step (a weight
            # copy through .data leaves no trace on the host); pph_head_mid reads the verdict (joined through ev[8])
            c("pph_last_layer_pattern", Wl, Pn, Wg, Pgn, C, self.ws_mid)
            ev[8].record(side)

        if self.variants["prep"] in ("tc", "tc1"):
            # selection -> tcgen05 add-on || operand split of both prototype tensors (side branch)
            ev[3].record(main)
            side.wait_event(ev[3])
            with torch.cuda.stream(side):
                c("pph_split_rows", P, Pn, D, float(cfg.center), self.P_hi, self.P_lo, self.p2, self.p2_ctr, self.p2_hi)
                c("pph_split_rows", Pg, Pgn, D, float(cfg.center), self.Pg_hi, self.Pg_lo, self.pg2, self.pg2_ctr, self.pg2_hi)
                if self.train and self.variants["addon_bwd"] == "tc":
                    self.dtokens.zero_()            # rows of unselected tokens: a memset node off the critical path
                ev[4].record(side)
                last_layer_pattern()
            if self.variants["prep"] == "tc1":
                if idx32 is None:
                    c("pph_select_topk", scores, B, max(H, 1), N, K, sel_idx, None)
                c(tok("pph_addon_fwd"), tokens, sel_idx, Wa, ba, B, N, Din, D, K, self.Zs, self.Zc, self.z2s, self.z2c,
                  float(cfg.center), self.z2s_ctr, self.z2c_ctr, self.z2s_hi, self.z2c_hi, self.Zs_hi, self.Zs_lo,
                  self.Zc_hi, self.Zc_lo)
            elif idx32 is None and self.variants["select"] == "fused":
                # the ranking runs in the add-on kernel's prologue: one launch for protopformer.py:157-172
                c(tok("pph_select_addon_fwd"), scores, max(H, 1), tokens, Wa, ba, B, N, Din, D, K, sel_idx, self.Zs, self.Zc,
                  self.z2s, self.z2c, float(cfg.center), self.z2s_ctr, self.z2c_ctr, self.z2s_hi, self.z2c_hi, self.Zs_hi,
                  self.Zs_lo, self.Zc_hi, self.Zc_lo, self.ws_tc)
            else:
                if idx32 is None:
                    c("pph_select_topk", scores, B, max(H, 1), N, K, sel_idx, None)
                c(tok("pph_addon_fwd2"), tokens, sel_idx, Wa, ba, B, N, Din, D, K, self.Zs, self.Zc, self.z2s, self.z2c,
                  float(cfg.center), self.z2s_ctr, self.z2c_ctr, self.z2s_hi, self.z2c_hi, self.Zs_hi, self.Zs_lo,
                  self.Zc_hi, self.Zc_lo, self.ws_tc)
            main.wait_event(ev[4])
        else:
            ev[3].record(main)
            side.wait_event(ev[3])
            with torch.cuda.stream(side):
                if self.train and self.variants["addon_bwd"] == "tc":
                    self.dtokens.zero_()
                    ev[4].record(side)
                last_layer_pattern()
            c(tok("pph_head_prep"), scores, tokens, Wa, ba, B, max(H, 1), N, Din, D, K, float(cfg.center), sel_idx, None,
              self.Zs, self.Zc, self.z2s, self.z2c, self.z2s_ctr, self.z2c_ctr, self.z2s_hi, self.z2c_hi,
              self.Zs_hi, self.Zs_lo, self.Zc_hi, self.Zc_lo,
              P, Pn, self.P_hi, self.P_lo, self.p2, self.p2_ctr, self.p2_hi,
              Pg, Pgn, self.Pg_hi, self.Pg_lo, self.pg2, self.pg2_ctr, self.pg2_hi)
            if self.train and self.variants["addon_bwd"] == "tc":
                main.wait_event(ev[4])
        if self.stop_after == 1:
            main.wait_event(ev[8])
            return self.losses
        mode = cfg.mode_id
        sel = {_lib.MODE_FP32_FMA: 0, _lib.MODE_BF16X3: 1, _lib.MODE_BF16: 2}[mode]
        c("pph_similarity_fwd", mode, cfg.act_id, float(cfg.eps), B, K, D, Pn, Pgn, self.Zs, self.Zc,
          (self.z2s, self.z2s_ctr, self.z2s_hi)[sel], (self.z2c, self.z2c_ctr, self.z2c_hi)[sel],
          self.Zs_hi, self.Zs_lo, self.Zc_hi, self.Zc_lo, P, Pg,
          (self.p2, self.p2_ctr, self.p2_hi)[sel], (self.pg2, self.pg2_ctr, self.pg2_hi)[sel],
          self.P_hi, self.P_lo, self.Pg_hi, self.Pg_lo,
          self.dmin_l, self.argmin, self.act_l, self.dmin_g, self.act_g, None, None)
        main.wait_event(ev[8])
        if self.stop_after == 2:
            return self.losses
        ppc = self.use_ppc and self.train
        vr = self.variants
        late = ppc and vr["ppc"] == "late" and vr["bwd"] == "gather" and vr["addon_bwd"] == "tc"
        split_ppc = ppc and (vr["ppc"] == "split" or late)

        def mid(use_ppc):
            c("pph_head_mid", self.act_l, self.act_g, self.dmin_l, self.dmin_g, self.argmin, Wl, Wg, labels,
              B, K, D, Pn, Pgn, C, m, N, float(cfg.global_coe), cfg.act_id, float(cfg.eps), float(upstream),
              1 if self.train else 0, use_ppc, self.Zs, self.z2s, P, self.p2, sel_idx,
              float(cfg.ppc_cov_thresh), float(cfg.ppc_mean_thresh), self.cov_coe, self.mean_coe,
              self.ws_mid, self.ws_bins, self.logits, self.logits_g, self.logits_l, self.losses, self.dlogits,
              self.g_l, self.g_g, self.pairT if vr["bwd"] == "staged" else None, self.dZs_ppc if ppc else None,
              self.dP_img if ppc else None, loss_mirror)

        if split_ppc:        # PPC loss forward + backward as a concurrent branch beside the last layers
            ev[0].record(main)
            side.wait_event(ev[0])
            with torch.cuda.stream(side):
                mid(3 + (4 if late else 0))     # late: dZs_ppc leaves as dpre, consumed by the add-on backward
                ev[6 if late else 1].record(side)
            mid(2)
            if not late:
                main.wait_event(ev[1])
        else:
            mid(1 if ppc else 0)
        dWl, dWg = _last_layer_grad_targets(self.train, Wl, Wg, grads)
        train_ll = dWl is not None or dWg is not None
        if train_ll:
            # last-layer weight gradients need only dlogits (final after the LL role above) and act_l / act_g: their own
            # branch beside the similarity backward, joined at the end -- the critical path never waits for it
            self.ev_ll[0].record(main)
            self.side_ll.wait_event(self.ev_ll[0])
            with torch.cuda.stream(self.side_ll):
                c("pph_last_layer_wgrad", self.dlogits, None, None, self.act_l, self.act_g, B, Pn, Pgn, C,
                  float(cfg.global_coe), dWl, dWg)
                hook("last")
                self.ev_ll[1].record(self.side_ll)

        def join_ll():
            if train_ll:
                main.wait_event(self.ev_ll[1])

        if not self.train or self.stop_after == 3:
            if late:
                main.wait_event(ev[6])
            join_ll()
            return self.losses

        def gather(parts, add, dpi):
            c("pph_similarity_bwd_fused", parts, self.g_l, self.g_g, self.argmin, self.Zs, self.Zc, P, Pg, B, K, D, Pn, Pgn,
              m, self.ws_gather, self.ws_bins, add, dpi, 1, self.dZs, self.dZc, grads["P"], grads["Pg"])

        dpre_add = None
        if late:
            # main: both gradient parts in one launch (as round 1) -> add-on backward.  The PPC branch (side) overlaps
            # the last layers and this launch; its token gradient joins inside the add-on backward's operand
            # (dpre_add_s), its prototype rows are added onto dP by a small launch beside the add-on backward.
            gather(3, None, None)                   # one launch for both parts: split in two they only slow each other
            ev[2].record(main)
            with torch.cuda.stream(side):           # after the PPC branch and this launch: the PPC prototype rows onto dP
                side.wait_event(ev[2])
                gather(4, None, self.dP_img)
                hook("protos")
                ev[1].record(side)
            dpre_add = self.dZs_ppc
        elif vr["bwd"] == "gather":
            gather(3, self.dZs_ppc if ppc else None, self.dP_img if ppc else None)
            hook("protos")
            ev[1].record(main)          # (joined at the end like the staged prototype branch)
        else:
            bwd = lambda parts: c("pph_similarity_bwd2", parts, self.g_l, self.g_g, self.pairT, self.ws_bins, self.Zs,  # noqa: E731
                                  self.Zc, P, Pg, B, K, D, Pn, Pgn, m, self.dZs_ppc if ppc else None,
                                  self.dP_img if ppc else None, 1, self.dZs, self.dZc, grads["P"], grads["Pg"])
            ev[0].record(main)
            side.wait_event(ev[0])
            side2.wait_event(ev[0])
            with torch.cuda.stream(side):
                bwd(2)                      # prototype rows: not needed by the add-on backward, joins at the end
                ev[1].record(side)
            with torch.cuda.stream(side2):
                bwd(4)                      # CLS rows
                ev[2].record(side2)
            bwd(1)                          # token rows
            main.wait_event(ev[2])
            if reduce_hook is not None:     # dP (side) and dPg (side2) are both needed: join first
                main.wait_event(ev[1])
                hook("protos")
        if self.stop_after == 4:
            main.wait_event(ev[1])
            join_ll()
            return self.losses
        if vr["addon_bwd"] == "tc":
            if late:
                main.wait_event(ev[6])              # dZs_ppc (as dpre) from the PPC branch
            # token gradient (82 CTAs) then weight gradient (112 CTAs behind a grid barrier): both want one CTA per SM, as
            # graph branches they only time-slice the machine (measured), so they run back to back
            def dgrad():
                c(tok("pph_addon_bwd3"), 2, tokens, sel_idx, Wa, self.dZs, self.dZc, dpre_add, B, N, Din, D, K, self.ws_tc,
                  None, None, self.dtokens)

            def wgrad():
                c(tok("pph_addon_bwd3"), 1, tokens, sel_idx, Wa, self.dZs, self.dZc, dpre_add, B, N, Din, D, K, self.ws_tc,
                  grads["Wa"], grads["ba"], None)

            if reduce_hook is not None:     # weight gradient first: its exchange then runs under the token gradient
                wgrad()
                ev[5].record(main)
                with torch.cuda.stream(side2):
                    side2.wait_event(ev[5])
                    hook("addon")
                    ev[7].record(side2)
                dgrad()
                main.wait_event(ev[7])
            else:
                dgrad()
                wgrad()
        else:
            c(tok("pph_addon_bwd2"), 3, tokens, sel_idx, Wa, self.dZs, self.dZc, B, N, Din, D, K,
              self.ws_addon, grads["Wa"], grads["ba"], self.dtokens)
            hook("addon")
        main.wait_event(ev[1])
        join_ll()
        return self.losses
