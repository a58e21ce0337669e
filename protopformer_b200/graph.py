"""Static-shape training / inference step of the prototype head captured in CUDA graphs.

At the CUB shape the whole head costs tens of microseconds on a B200, i.e. it is launch-bound from Python; the
idiomatic B200 answer is to record the step once (forward + PPC loss + cross-entropy + backward, 11 kernels) and
replay it.  The step goes through exactly the public operators of ``ops`` (nothing is bypassed), reads its inputs
from static device buffers ("slots") and leaves its results in static tensors:

    step = GraphedHeadStep(params, cfg, B=64, N=196, C=200, m=10, n_slots=2)
    step.load(slot, tokens, scores, labels)      # device or pinned-host tensors -> async copy into the slot
    step.run(slot)                               # replay
    step.loss[slot], step.logits[slot], step.dtokens[slot], param.grad (views of step.reducer.flat)

Slots hold INPUTS only.  The results (loss, logits, PPC terms, dtokens, parameter gradients) live in ONE set of buffers
shared by all slots -- replays are serial on one stream -- so `step.loss[a]` and `step.loss[b]` are the same tensor:
read (or copy out) the results of a replay before the next `run()`.  `use_ppc=False` leaves the PPC terms out of the
loss and the gradients, which is what the reference does before epoch 20 (tools/engine_proto.py:63).

Reference call sites this mirrors: tools/engine_proto.py:49-66 (forward, CE, get_PPC_loss, weighted sum) and :76
(backward).  The optimizer step and the backbone are outside this path.
"""
from __future__ import annotations

import torch
import torch.nn.functional as F

from . import ops
from .dist import FlatGradReducer, PeerGradReducer


class GraphedHeadStep:
    def __init__(self, params: dict, cfg: ops.HeadConfig, B: int, N: int, C: int, m: int, n_slots: int = 1,
                 heads: int = 0, ppc_cov_coe: float = 0.1, ppc_mean_coe: float = 0.5, train: bool = True,
                 process_group=None, device=None, fused: bool = True, allreduce_in_graph: bool = False,
                 schedule: int | None = None, use_ppc: bool = True, impl: str = "auto", variants=None,
                 exchange: str = "nccl"):
        """params: dict with Wa (D,Din), ba (D), P (P,D), Pg (Pg,D) [leaf tensors, requires_grad in training] and
        the last layers Wl (C,P), Wg (C,Pg), frozen as in the reference unless their requires_grad is set: a training step
        then also writes their gradients (appended to the flat buffer behind ba, Wl before Wg).  ppc_*_coe follow
        scripts/train_cub.sh:43-44."""
        self.p, self.cfg, self.B, self.N, self.C, self.m = params, cfg, B, N, C, m
        self.train = train
        self.cov_coe, self.mean_coe = ppc_cov_coe, ppc_mean_coe
        dev = device or params["P"].device
        Din = params["Wa"].shape[1]
        sshape = (B, heads, N) if heads > 0 else (B, N)
        self.tokens = [torch.zeros(B, 1 + N, Din, device=dev, requires_grad=train) for _ in range(n_slots)]
        self.scores = [torch.zeros(sshape, device=dev) for _ in range(n_slots)]
        self.labels = [torch.zeros(B, dtype=torch.int64, device=dev) for _ in range(n_slots)]
        self.loss = [None] * n_slots
        self.logits = [None] * n_slots
        self.ppc = [None] * n_slots
        self.dtokens = [None] * n_slots
        self.graphs = [None] * n_slots
        self.reducer = None
        if train:
            # unfrozen last layers go last: the existing segments keep their offsets and ("Wl", "Wg") is contiguous
            named = [(k, params[k]) for k in ("P", "Pg", "Wa", "ba")]
            named += [(k, params[k]) for k in ("Wl", "Wg") if params[k].requires_grad]
            # exchange: "nccl" = NCCL all-reduce of the flat buffer, "peer" / "peer_nomc" = the library's own one-kernel
            # all-reduce over peer-mapped memory (with / without the NVLS multicast mapping)
            self.exchange, self.exchange_note = exchange, ""
            if exchange in ("peer", "peer_nomc"):
                try:
                    self.reducer = PeerGradReducer(named, process_group, multicast=(exchange == "peer"))
                    if exchange == "peer" and not self.reducer.multicast_ptr:
                        self.exchange = "peer_nomc"
                except Exception as exc:      # no peer-mapped memory on this box (no P2P / symmetric memory): NCCL instead
                    self.exchange = "nccl"
                    self.exchange_note = f"peer memory unavailable ({type(exc).__name__}: {exc}); fell back to NCCL"
                    self.reducer = FlatGradReducer(named, process_group)
            else:
                self.reducer = FlatGradReducer(named, process_group)
        self.kernel_launches_per_step = 0
        self.allreduce_in_graph = allreduce_in_graph      # record the NCCL gradient all-reduce inside the CUDA graph
        self.fused = None
        if fused:
            # one set of intermediate buffers shared by all slots (replays are serial on one stream)
            D, P, Pg = params["Wa"].shape[0], params["P"].shape[0], params["Pg"].shape[0]
            # impl: "v2" = the round-2 launch sequence (11 launches), "v1" = the round-1 sequence (fallback / A-B arm), "auto" = v2 if the
            # shape is inside what those kernels were built for
            if impl == "auto":
                impl = "v2" if ops.fused_step_supported(B, N, Din, D, cfg.K, P, Pg, C, m) else "v1"
            self.impl = impl
            cls = ops.FusedHeadStep if impl == "v2" else ops.FusedHeadStepV1
            kw = dict(variants=variants) if impl == "v2" else {}
            self.fused = cls(cfg, B, N, Din, D, P, Pg, C, m, dev, heads=heads, ppc_cov_coe=ppc_cov_coe,
                             ppc_mean_coe=ppc_mean_coe, train=train, use_ppc=use_ppc, schedule=schedule, **kw)
            if train:
                self.grads = dict(zip((n for n, _ in self.reducer.named), self.reducer.views))

    # --------------------------------------------------------------------------------------------------------
    def _step_fused(self, slot: int, **extra):
        p, f = self.p, self.fused
        works = []
        hook = None
        last, aligned = False, True
        if self.train and self.allreduce_in_graph and self.impl == "v2":
            # overlapped exchange: the prototype gradients (95 % of the flat buffer) are final before the add-on backward
            # starts, so their all-reduce is issued there (on the step's side branch) and runs under those kernels on
            # NCCL's stream; the add-on part follows the weight-gradient kernel.  Both join the step's stream below.
            seg = {"protos": self.reducer.segment(("P", "Pg")), "addon": self.reducer.segment(("Wa", "ba"))}
            # unfrozen last layers: a third exchange ("last", peer slot 2) on their own branch, right behind their kernel
            last = any(n in ("Wl", "Wg") for n, _ in self.reducer.named)
            if last:
                seg["last"] = self.reducer.segment(("Wl", "Wg"))

            aligned = all(v % 4 == 0 for v in seg["protos"])
            if last:
                aligned = aligned and all(v % 4 == 0 for v in seg["addon"])

            def hook(which):
                lo, hi = seg[which]
                if not aligned:           # odd sizes: one exchange of the whole buffer after the last gradient
                    if which == "protos" or last:
                        return            # (with the last-layer branch: below, once the step has joined it)
                    lo, hi = 0, None
                peer_slot = {"protos": 0, "addon": 1, "last": 2}[which]
                w = self.reducer.allreduce(async_op=True, lo=lo, hi=hi, check=False, slot=peer_slot)
                if w is not None:
                    works.append(w)
        with torch.no_grad():
            kw = dict(reduce_hook=hook) if hook is not None else {}
            kw.update(extra)
            f.step(self.tokens[slot], self.scores[slot], self.labels[slot], p["Wa"], p["ba"], p["P"], p["Pg"],
                   p["Wl"], p["Wg"], self.grads if self.train else None, **kw)
        for w in works:
            w.wait()                      # the capturing / current stream waits for NCCL's stream
        if self.train and self.allreduce_in_graph and (hook is None or (last and not aligned)):
            self.reducer.allreduce(check=False)
        self.loss[slot] = f.losses[0]
        self.logits[slot] = f.logits
        self.ppc[slot] = (f.losses[2], f.losses[3])
        self.dtokens[slot] = f.dtokens if self.train else None

    def _step(self, slot: int):
        if self.fused is not None:
            return self._step_fused(slot)
        p, cfg = self.p, self.cfg
        tok = self.tokens[slot]
        if self.train:
            self.reducer.zero()
            tok.grad = None
        out = ops.head_forward(cfg, tok, self.scores[slot], p["Wa"], p["ba"], p["P"], p["Pg"], p["Wl"], p["Wg"])
        self.logits[slot] = out.logits
        if not self.train:
            self.loss[slot] = F.cross_entropy(out.logits, self.labels[slot])
            return
        cov, mean = ops.ppc_loss(cfg, out.tf, p["P"], out.p2l, self.labels[slot], self.m, self.N)
        loss = F.cross_entropy(out.logits, self.labels[slot]) + self.cov_coe * cov + self.mean_coe * mean
        loss.backward()
        self.loss[slot] = loss.detach()
        self.ppc[slot] = (cov.detach(), mean.detach())
        self.dtokens[slot] = tok.grad

    def capture(self, warmup: int = 3):
        from . import _lib
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        ctx = torch.enable_grad() if self.train else torch.no_grad()
        with ctx:
            with torch.cuda.stream(side):
                for _ in range(warmup):
                    self._step(0)
            torch.cuda.current_stream().wait_stream(side)
            torch.cuda.synchronize()
            pool = None
            for slot in range(len(self.tokens)):
                g = torch.cuda.CUDAGraph()
                n0 = _lib.launch_count()
                with torch.cuda.graph(g, pool=pool, capture_error_mode="thread_local"):
                    self._step(slot)
                self.kernel_launches_per_step = _lib.launch_count() - n0
                pool = g.pool()
                self.graphs[slot] = g
        return self

    # --------------------------------------------------------------------------------------------------------
    def load(self, slot: int, tokens, scores, labels):
        """Asynchronous copy of one batch into the slot (host tensors should be pinned)."""
        with torch.no_grad():
            self.tokens[slot].copy_(tokens, non_blocking=True)
            self.scores[slot].copy_(scores, non_blocking=True)
            self.labels[slot].copy_(labels, non_blocking=True)

    def capture_host_pipeline(self):
        """Second set of step graphs for callers that feed the slots through load_host(): the step takes the selected-token
        list the transfer already computed (no selection launch of its own) and the kernel that completes the loss also
        stores (total, ce, ppc_cov, ppc_mean) into `self.loss_host[slot]` (pinned host memory) -- the caller's device->host
        read of the result costs no copy node and no stream round trip.  Replay with run_host(slot)."""
        assert self.fused is not None and self.impl == "v2", "host pipeline graphs need the v2 step"
        dev = self.tokens[0].device
        if not hasattr(self, "_load_idx"):
            self._load_idx = [torch.empty(self.B, self.cfg.K, dtype=torch.int32, device=dev) for _ in self.tokens]
        self.loss_host = [torch.zeros(4).pin_memory() for _ in self.tokens]
        self.graphs_host = []
        ctx = torch.enable_grad() if self.train else torch.no_grad()
        with ctx:
            for slot in range(len(self.tokens)):
                extra = dict(idx32=self._load_idx[slot], loss_mirror=self.loss_host[slot].data_ptr())
                from . import _lib
                with torch.no_grad():                     # a valid index list for the eager warm-up below
                    _lib.call("pph_select_topk", self.scores[slot], self.B,
                              self.scores[slot].shape[1] if self.scores[slot].dim() == 3 else 1, self.N, self.cfg.K,
                              self._load_idx[slot], None)
                side = torch.cuda.Stream()
                side.wait_stream(torch.cuda.current_stream())
                with torch.cuda.stream(side):
                    self._step_fused(slot, **extra)
                torch.cuda.current_stream().wait_stream(side)
                torch.cuda.synchronize()
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g, capture_error_mode="thread_local"):
                    self._step_fused(slot, **extra)
                self.graphs_host.append(g)
        return self

    def capture_host_overlapped(self, slot: int, next_tokens, next_scores, next_labels, n_ctas: int = 48):
        """ONE graph for a whole end-to-end iteration: the step of `slot` (as run_host) on the capture's main branch and, on a
        forked branch, the selection-first transfer of the NEXT batch (pinned host tensors) into the other slot.  A caller that
        cycles through a ring of pinned staging buffers replays one of these per step -- one host call, no cross-stream
        events -- and alternates slots 0 and 1.  Needs capture_host_pipeline()."""
        assert len(self.tokens) >= 2 and slot in (0, 1) and hasattr(self, "graphs_host"), "slots 0 / 1, capture_host_pipeline() first"
        other = 1 - slot
        if not hasattr(self, "_xfer_stream"):
            self._xfer_stream = torch.cuda.Stream()
            self._xfer_ev = [torch.cuda.Event(), torch.cuda.Event()]
        self.load_host(other, next_tokens, next_scores, next_labels, n_ctas)      # warm-up outside the capture
        torch.cuda.synchronize()
        extra = dict(idx32=self._load_idx[slot], loss_mirror=self.loss_host[slot].data_ptr())
        g = torch.cuda.CUDAGraph()
        ctx = torch.enable_grad() if self.train else torch.no_grad()
        with ctx, torch.cuda.graph(g, capture_error_mode="thread_local"):
            main = torch.cuda.current_stream()
            self._xfer_ev[0].record(main)
            self._xfer_stream.wait_event(self._xfer_ev[0])
            with torch.cuda.stream(self._xfer_stream):
                self.load_host(other, next_tokens, next_scores, next_labels, n_ctas)
                self._xfer_ev[1].record(self._xfer_stream)
            self._step_fused(slot, **extra)
            main.wait_event(self._xfer_ev[1])
        return g

    def run_host(self, slot: int = 0):
        self.graphs_host[slot].replay()
        return self.loss_host[slot]

    def load_host(self, slot: int, tokens, scores, labels, n_ctas: int = 48):
        """Selection-first transfer of one batch from PINNED host tensors (current stream): scores and labels by copy,
        the top-K ranking on the device, then only the CLS row and the K selected rows of every image are read out of
        the host buffer by a gather kernel (pph_gather_rows_host).  The slot's other token rows keep stale values that
        neither the forward nor the backward reads.  Returns the bytes that crossed the bus."""
        from . import _lib
        assert tokens.is_pinned() and tokens.is_contiguous() and tokens.dtype == torch.float32
        if not hasattr(self, "_load_idx"):
            self._load_idx = [torch.empty(self.B, self.cfg.K, dtype=torch.int32, device=self.tokens[0].device)
                              for _ in self.tokens]
        B, N, K = self.B, self.N, self.cfg.K
        H = scores.shape[1] if scores.dim() == 3 else 1
        Din = tokens.shape[-1]
        with torch.no_grad():
            self.scores[slot].copy_(scores, non_blocking=True)
            self.labels[slot].copy_(labels, non_blocking=True)
            _lib.call("pph_select_topk", self.scores[slot], B, H, N, K, self._load_idx[slot], None)
            _lib.call("pph_gather_rows_host", tokens.data_ptr(), self._load_idx[slot], B, N, Din, K,
                      self.tokens[slot].detach(), n_ctas)
        return scores.numel() * 4 + labels.numel() * 8 + B * (K + 1) * Din * 4

    def capture_load_host(self, slot: int, tokens, scores, labels, n_ctas: int = 48):
        """load_host() of one fixed (slot, pinned staging buffer) pair recorded as a CUDA graph: a caller that cycles
        through a ring of staging buffers replays it (one host call) on its copy stream."""
        self.load_host(slot, tokens, scores, labels, n_ctas)          # allocates the index buffers outside the capture
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, capture_error_mode="thread_local"):
            self.load_host(slot, tokens, scores, labels, n_ctas)
        return g

    def run(self, slot: int = 0):
        self.graphs[slot].replay()
        return self.loss[slot]

    def allreduce_grads(self):
        """Gradient all-reduce of the step just run (no-op when it is already part of the captured graph)."""
        if self.reducer is not None and not self.allreduce_in_graph:
            self.reducer.allreduce()
