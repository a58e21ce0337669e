"""Caller of the score producer: the backbone-side loop that decides which tokens survive (SURVEY.md §8(f) next #1).

The reference's DeiT wrapper runs its transformer blocks, and at every reserve layer turns the attention maps seen so
far into the CLS-row rollout score, keeps the top-K tokens and masks the rest for the remaining blocks
(tools/deit_models_attn.py:205-241, ``MyVisionTransformer.forward_feature_mask_train_direct``).  This module is that
loop with the rollout + top-K done by ONE fused launch sequence (``ops.rollout_scores(..., topk=K)``: no (B,T,T)
product chain, no ATen topk over 38 809 entries per image and layer, no separate topk/sort for the selection).  The
transformer blocks themselves stay the backbone's own modules -- they are out of this path's scope.

    from protopformer_b200.backbone import patch_deit_features, patch_cait_features
    patch_deit_features(ppnet.features)        # binds the method below over the reference's one; same signature
    patch_cait_features(ppnet.features)        # ... the CaiT form (tools/cait_models_attn.py:310-343)

Not differentiable through the score, exactly like the reference (``attn_rollout.detach()``, :225).  The blocks' maps are
passed as they come: a bf16 or fp16 backbone's maps are read in that precision, without an fp32 copy.
"""
from __future__ import annotations

import types

import torch


def forward_feature_mask_train_direct(self, cls_embed, x_embed, token_attn=None, reserve_layer_nums=(), rollout=None):
    """Same arguments and return value as tools/deit_models_attn.py:205-241:
    cls_embed (B,1,dim), x_embed (B,N,dim), reserve_layer_nums = [(layer index, tokens to keep), ...] ->
    (tokens (B,1+N,dim) after ``self.norm``, (cls_token_attn (B,N), None)).

    ``self`` needs ``blocks`` (each ``blk(x, policy) -> (x, attn (B,H,1+N,1+N))``) and ``norm``.
    ``rollout(all_attn, topk=K, want_int64=True) -> (scores, idx32, idx64)`` defaults to the CUDA op."""
    if rollout is None:
        from . import ops
        rollout = ops.rollout_scores
    B, patch_num = x_embed.shape[0], x_embed.shape[1]
    layer_ids = [r[0] for r in reserve_layer_nums]
    dev = x_embed.device
    policy = torch.ones(B, 1 + patch_num, 1, device=dev)                                   # :214
    x = torch.cat([cls_embed, x_embed], dim=1)                                             # :215
    all_attn = []
    cls_token_attn = None
    for i, blk in enumerate(self.blocks):
        if i in layer_ids:
            keep = reserve_layer_nums[layer_ids.index(i)][1]
            # :219-231  rollout of the first i maps -> CLS row without its own column -> sorted top-K (+1: skip CLS)
            cls_token_attn, _, idx64 = rollout(all_attn[:i], topk=keep, want_int64=True)
            policy = torch.zeros(B, 1 + patch_num, device=dev)                             # :232-234
            policy[:, 0] = 1.0
            policy.scatter_(1, idx64 + 1, 1.0)
            policy = policy[:, :, None]
        x, attn = blk(x, policy)
        all_attn.append(attn)
    x = self.norm(x)
    return x, (cls_token_attn, None)


def forward_feature_mask_train_direct_cait(self, cls_embed, x_embed, token_attn=None, reserve_layer_nums=(),
                                           rollout_cait=None, select=None):
    """CaiT form of the loop, same arguments and return value as tools/cait_models_attn.py:310-343
    (``MyCait.forward_feature_mask_train_direct``): all patch blocks run first (``blk(x) -> (x, attn (B,H,N,N))``), then
    the token-only blocks (``blk(x, cls_tokens, policy) -> (cls_tokens, attn (B,H,1,1+N))``); at a reserve layer i >= 1 the
    score is the rolled-out mean class-attention row over the patch-layer product (:328-330).

    ``self`` needs ``blocks``, ``blocks_token_only``, ``norm`` and ``layer_nums`` (``layer_nums[0]`` = number of patch
    blocks).  ``rollout_cait(all_attn, pre_layer_num) -> scores (B,N)`` and ``select(scores, K, want_int64=True) ->
    (idx32, idx64)`` default to the CUDA ops."""
    if rollout_cait is None or select is None:
        from . import ops
        rollout_cait = rollout_cait or ops.rollout_scores_cait
        select = select or ops.select_topk
    B, patch_num = x_embed.shape[0], x_embed.shape[1]
    cls_tokens, x = cls_embed, x_embed
    dev = x_embed.device
    all_attn = []
    for blk in self.blocks:                                                                # :314-316
        x, attn = blk(x)
        all_attn.append(attn)
    layer_ids = [r[0] for r in reserve_layer_nums]
    policy = torch.ones(B, 1 + patch_num, 1, device=dev)                                   # :319
    cls_token_attn = None
    for i, blk in enumerate(self.blocks_token_only):
        if i in layer_ids:
            keep = reserve_layer_nums[layer_ids.index(i)][1]
            cls_token_attn = rollout_cait(all_attn, self.layer_nums[0])                    # :323-325
            _, idx64 = select(cls_token_attn, keep, want_int64=True)                       # :327-330
            policy = torch.zeros(B, 1 + patch_num, device=dev)                             # :331-333
            policy[:, 0] = 1.0
            policy.scatter_(1, idx64 + 1, 1.0)
            policy = policy[:, :, None]
        cls_tokens, attn = blk(x, cls_tokens, policy)
        all_attn.append(attn)
    x = torch.cat((cls_tokens, x), dim=1)
    x = self.norm(x)
    return x, (cls_token_attn, None)


def patch_cait_features(features):
    """Bind the CaiT loop over ``features.forward_feature_mask_train_direct``.  Returns ``features``."""
    features.forward_feature_mask_train_direct = types.MethodType(forward_feature_mask_train_direct_cait, features)
    return features


def patch_deit_features(features):
    """Bind the fused-rollout loop over ``features.forward_feature_mask_train_direct`` (the method PPNet calls,
    protopformer.py:155).  Returns ``features``."""
    features.forward_feature_mask_train_direct = types.MethodType(forward_feature_mask_train_direct, features)
    return features
