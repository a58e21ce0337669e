"""Fused AdamW for the head's parameter groups (SURVEY.md §8(f) next #3).

Mirrors what the reference builds for the head in tools/create_optimizer.py:31-39 + :92
(``optim.AdamW(split_weights(model, lrs), weight_decay=args.weight_decay, eps=args.opt_eps)``) and steps in
tools/engine_proto.py:76-78: same update rule, same ``param_groups`` / ``state_dict`` layout as ``torch.optim.AdamW``,
but ONE kernel launch (``pph_adamw_step``) for all tensors, with the step count and the per-group (lr, weight_decay)
in device memory so the launch can live inside the CUDA graph of the training step while a scheduler changes
``group['lr']`` between replays (call ``sync_hyper()`` after changing a group, as ``scheduler.step`` would).

There is no CPU path: parameters must be CUDA fp32 tensors.
"""
from __future__ import annotations

import ctypes

import torch

from . import _lib

MAX_TENSORS = 8


def head_param_groups(ppnet, lrs: dict, weight_decay: float):
    """The head's part of ``split_weights`` (tools/create_optimizer.py:31-39): add-on layers with their own lr and a
    fixed 1e-3 weight decay, the two prototype tensors with the prototype lr and the optimizer-level weight decay.
    Last layers whose weight requires grad (frozen by default, protopformer.py:130-131) form one more group with
    ``lrs["last_layer"]`` and no weight decay, as ProtoPNet's last-layer optimizer.
    (The ``features`` group -- the backbone -- is outside this path.)"""
    groups = [{"params": list(ppnet.add_on_layers.parameters()), "lr": lrs["add_on_layers"], "weight_decay": 1e-3}]
    if hasattr(ppnet, "prototype_vectors"):
        groups.append({"params": [ppnet.prototype_vectors], "lr": lrs["prototype_vectors"],
                       "weight_decay": weight_decay})
    if hasattr(ppnet, "prototype_vectors_global"):
        groups.append({"params": [ppnet.prototype_vectors_global], "lr": lrs["prototype_vectors"],
                       "weight_decay": weight_decay})
    last = [layer.weight for layer in (getattr(ppnet, "last_layer", None), getattr(ppnet, "last_layer_global", None))
            if layer is not None and layer.weight.requires_grad]
    if last:
        if "last_layer" not in lrs:
            raise KeyError("lrs['last_layer'] is missing: the last layers require grad, so they need a learning rate")
        groups.append({"params": last, "lr": lrs["last_layer"], "weight_decay": 0.0})
    return groups


class FusedHeadAdamW:
    """``torch.optim.AdamW`` semantics (decoupled weight decay, bias correction, no amsgrad) in one launch.

    params: iterable of tensors or of ``{'params': [...], 'lr': ..., 'weight_decay': ...}`` groups (<= 8 tensors,
    <= 8 groups).  ``grads``: optional list of gradient tensors to read instead of ``p.grad`` (e.g. the views of the
    flat all-reduce buffer, ``FlatGradReducer.views``), in parameter order.
    """

    def __init__(self, params, lr: float = 1e-3, betas=(0.9, 0.999), eps: float = 1e-8, weight_decay: float = 1e-2,
                 grads=None):
        params = list(params)
        if params and not isinstance(params[0], dict):
            params = [{"params": params}]
        self.defaults = dict(lr=lr, betas=tuple(betas), eps=eps, weight_decay=weight_decay)
        self.param_groups = []
        for g in params:
            g = dict(g)
            g["params"] = list(g["params"])
            for k, v in self.defaults.items():
                g.setdefault(k, v)
            self.param_groups.append(g)
        flat = [p for g in self.param_groups for p in g["params"]]
        if not 1 <= len(flat) <= MAX_TENSORS or len(self.param_groups) > MAX_TENSORS:
            raise ValueError(f"FusedHeadAdamW handles 1..{MAX_TENSORS} tensors in <= {MAX_TENSORS} groups")
        betas0 = self.param_groups[0]["betas"]
        eps0 = self.param_groups[0]["eps"]
        for g in self.param_groups:
            if tuple(g["betas"]) != tuple(betas0) or g["eps"] != eps0:
                raise ValueError("one (betas, eps) for all groups (as the reference configures AdamW)")
        for p in flat:
            if not (p.is_cuda and p.dtype == torch.float32 and p.is_contiguous()):
                raise ValueError("FusedHeadAdamW needs contiguous CUDA fp32 parameters (there is no CPU path)")
        self._flat = flat
        self._group_of = [gi for gi, g in enumerate(self.param_groups) for _ in g["params"]]
        self._grads = list(grads) if grads is not None else None
        dev = flat[0].device
        self.state = {p: {"exp_avg": torch.zeros_like(p), "exp_avg_sq": torch.zeros_like(p)} for p in flat}
        self._step_state = torch.zeros(2, dtype=torch.int32, device=dev)        # {t, ticket}
        self._hyper_host = torch.zeros(MAX_TENSORS, 2, dtype=torch.float32).pin_memory()
        self._hyper = torch.zeros(MAX_TENSORS, 2, dtype=torch.float32, device=dev)
        self.sync_hyper()

    # ------------------------------------------------------------------------------------------------------
    def sync_hyper(self):
        """Publish ``group['lr']`` / ``group['weight_decay']`` to the device table the kernel reads."""
        for gi, g in enumerate(self.param_groups):
            self._hyper_host[gi, 0] = float(g["lr"])
            self._hyper_host[gi, 1] = float(g["weight_decay"])
        self._hyper.copy_(self._hyper_host, non_blocking=True)

    @property
    def step_count(self) -> int:
        return int(self._step_state[0].item())

    def zero_grad(self, set_to_none: bool = True):
        """torch.optim semantics (set_to_none by default, as the reference's loop relies on), EXCEPT when the optimizer was
        built over external gradient buffers (`grads=`: e.g. the views of dist.FlatGradReducer's flat all-reduce buffer): those
        are zeroed in place and stay attached -- dropping them would make autograd accumulate into fresh tensors while the
        all-reduce and this optimizer keep reading the stale buffer (ADVICE round 1)."""
        if self._grads is not None:
            for gr, p in zip(self._grads, self._flat):
                gr.zero_()
                if p.grad is not None and p.grad.data_ptr() != gr.data_ptr():
                    p.grad = None
                if p.requires_grad and p.is_leaf and p.grad is None:
                    p.grad = gr
            return
        for p in self._flat:
            if p.grad is not None:
                if set_to_none:
                    p.grad = None
                else:
                    p.grad.zero_()

    @torch.no_grad()
    def step(self, grad_scale: float = 1.0):
        """One AdamW update of every tensor (launches on the current stream; CUDA-graph capturable)."""
        n = len(self._flat)
        grads = self._grads if self._grads is not None else [p.grad for p in self._flat]
        for gr, p in zip(grads, self._flat):
            if gr is None or gr.shape != p.shape or not gr.is_contiguous() or gr.dtype != torch.float32:
                raise RuntimeError("every head parameter needs a contiguous fp32 gradient of its own shape")
        vp = ctypes.c_void_p
        tbl = lambda ts: (vp * n)(*[t.data_ptr() for t in ts])  # noqa: E731
        numel = (ctypes.c_longlong * n)(*[p.numel() for p in self._flat])
        group = (ctypes.c_int * n)(*self._group_of)
        b1, b2 = self.param_groups[0]["betas"]
        _lib.call("pph_adamw_step", n, tbl(self._flat), tbl(grads), tbl([self.state[p]["exp_avg"] for p in self._flat]),
                  tbl([self.state[p]["exp_avg_sq"] for p in self._flat]), numel, group, self._hyper, float(b1),
                  float(b2), float(self.param_groups[0]["eps"]), float(grad_scale), self._step_state)

    # ------------------------------------------------------------------------------------------------------
    def state_dict(self):
        """Same layout as ``torch.optim.AdamW.state_dict()`` (what main.py:420-427 checkpoints)."""
        t = self.step_count
        state, groups, i = {}, [], 0
        for g in self.param_groups:
            ids = []
            for p in g["params"]:
                s = self.state[p]
                state[i] = {"step": torch.tensor(float(t)), "exp_avg": s["exp_avg"], "exp_avg_sq": s["exp_avg_sq"]}
                ids.append(i)
                i += 1
            gg = {k: v for k, v in g.items() if k != "params"}
            gg.update(amsgrad=False, maximize=False, foreach=None, capturable=False, differentiable=False, fused=None)
            gg["params"] = ids
            groups.append(gg)
        return {"state": state, "param_groups": groups}

    def load_state_dict(self, sd):
        i, t = 0, 0
        for g, sg in zip(self.param_groups, sd["param_groups"]):
            for k in ("lr", "weight_decay", "betas", "eps"):
                if k in sg:
                    g[k] = tuple(sg[k]) if k == "betas" else sg[k]
            for p in g["params"]:
                s = sd["state"].get(i)
                if s is not None:
                    self.state[p]["exp_avg"].copy_(s["exp_avg"])
                    self.state[p]["exp_avg_sq"].copy_(s["exp_avg_sq"])
                    t = int(float(s["step"]))
                i += 1
        self._step_state.copy_(torch.tensor([t, 0], dtype=torch.int32))
        self.sync_hyper()
