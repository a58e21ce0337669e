"""Data-parallel plumbing of the head: one process per GPU, batch sharded, head parameters replicated.

The only exchange step of the path is the gradient all-reduce of the trainable head parameters
(`prototype_vectors`, `prototype_vectors_global`, `add_on_layers.*`, and `last_layer.weight` /
`last_layer_global.weight` when the caller unfreezes them -- the reference freezes them, protopformer.py:130-131) --
what DDP does implicitly in the reference (main.py:370).  Here the gradients of those parameters are views into ONE flat
fp32 buffer (3.2 MB at the CUB shape, +3.2 MB with both last layers unfrozen), averaged over the ranks in segments
that the graphed step exchanges as soon as each is final (latency-bound over NVLink/NVSwitch).
"""
from __future__ import annotations

import torch
import torch.distributed as dist


def head_parameters(module):
    """Trainable head parameters in a fixed order (names follow tools/create_optimizer.py:31-39); the last layers follow
    the four others, and only when their weight requires grad (frozen by default, protopformer.py:130-131)."""
    names = ["prototype_vectors", "prototype_vectors_global", "add_on_layers.0.weight", "add_on_layers.0.bias",
             "last_layer.weight", "last_layer_global.weight"]
    params = dict(module.named_parameters())
    return [(n, params[n]) for n in names if n in params and params[n].requires_grad]


class FlatGradReducer:
    """Keeps `.grad` of the given parameters as views of one flat buffer and averages it across ranks."""

    in_stream = False        # True: allreduce() is a kernel on the current stream (nothing to wait for on the host)

    def __init__(self, named_params, process_group=None):
        self.named = list(named_params)
        self.group = process_group
        total = sum(p.numel() for _, p in self.named)
        ref = self.named[0][1]
        self.flat = self._allocate(total, ref.device)
        off = 0
        self.views = []
        for _, p in self.named:
            v = self.flat[off:off + p.numel()].view_as(p)
            p.grad = v
            self.views.append(v)
            off += p.numel()

    def _allocate(self, total, device):
        return torch.zeros(total, dtype=torch.float32, device=device)

    def zero(self):
        """Zero the flat buffer and re-attach the views (autograd then accumulates in place)."""
        self.flat.zero_()
        for (_, p), v in zip(self.named, self.views):
            if p.grad is None or p.grad.data_ptr() != v.data_ptr():
                p.grad = v

    def check_attached(self):
        """Raises if some parameter's .grad no longer aliases the flat buffer (e.g. after an optimizer's
        zero_grad(set_to_none=True)): reducing the flat buffer would then average stale values while autograd
        accumulates somewhere else."""
        for (n, p), v in zip(self.named, self.views):
            if p.grad is None or p.grad.data_ptr() != v.data_ptr():
                raise RuntimeError(f"gradient of {n} is detached from the flat all-reduce buffer: call "
                                   "FlatGradReducer.zero() (not optimizer.zero_grad(set_to_none=True)) between steps")

    def segment(self, names):
        """[lo, hi) of the flat buffer covered by the (contiguous, in construction order) parameters `names`."""
        off, lo, hi = 0, None, None
        for n, p in self.named:
            if n in names:
                lo = off if lo is None else lo
                hi = off + p.numel()
            off += p.numel()
        return lo, hi

    def allreduce(self, async_op: bool = False, lo: int = 0, hi: int | None = None, check: bool = True, slot: int = 0):
        """Average flat[lo:hi] (default: all of it) over the process group (no-op for a single process)."""
        if not (dist.is_available() and dist.is_initialized()):
            return None
        world = dist.get_world_size(self.group)
        if world == 1:
            return None
        if check:
            self.check_attached()
        buf = self.flat if (lo == 0 and hi is None) else self.flat[lo:hi]
        if dist.get_backend(self.group) == "nccl":
            return dist.all_reduce(buf, op=dist.ReduceOp.AVG, group=self.group, async_op=async_op)
        work = dist.all_reduce(buf, op=dist.ReduceOp.SUM, group=self.group, async_op=False)
        buf.div_(world)
        return work


class PeerGradReducer(FlatGradReducer):
    """FlatGradReducer whose buffer is a peer-mapped (symmetric) allocation and whose all-reduce is ONE kernel of
    libprotohead_b200 on the caller's stream (pph_peer_allreduce: flag barrier over NVLink, reduce chunk `rank` --
    in the switch through the multicast mapping when there is one -- write the average to every peer, flag barrier).
    No NCCL call on the data path, so the exchange can be a branch of the step's CUDA graph beside the add-on backward.
    The symmetric allocation and the address exchange come from torch.distributed._symmetric_memory (plumbing)."""

    in_stream = True

    def __init__(self, named_params, process_group=None, n_ctas: int = 32, multicast: bool = True):
        self.n_ctas, self.want_multicast = int(n_ctas), bool(multicast)
        super().__init__(named_params, process_group)

    def _allocate(self, total, device):
        import ctypes
        import torch.distributed._symmetric_memory as symm
        from . import _lib
        group = self.group if self.group is not None else dist.group.WORLD
        nb = ctypes.c_longlong(0)
        rc = _lib.load().pph_peer_flag_bytes(ctypes.byref(nb))
        assert rc == 0
        self.total = total
        self.padded = (total + 3) // 4 * 4
        self.flag_off = (self.padded * 4 + 15) // 16 * 16
        n_alloc = (self.flag_off + nb.value + 3) // 4
        buf = symm.empty(n_alloc, dtype=torch.float32, device=device)
        buf.zero_()
        torch.cuda.synchronize(device)
        h = symm.rendezvous(buf, group)
        self.handle, self.buf = h, buf
        self.rank, self.world = int(h.rank), int(h.world_size)
        local_off = buf.data_ptr() - int(h.buffer_ptrs[self.rank])
        self.ptr_table = (ctypes.c_ulonglong * self.world)(*[int(p) + local_off for p in h.buffer_ptrs])
        mc = int(h.multicast_ptr) if self.want_multicast else 0
        self.multicast_ptr = (mc + local_off) if mc else 0
        dist.barrier(group)               # every rank's flag block is zero before anyone's first exchange
        torch.cuda.synchronize(device)
        return buf[:total]

    def allreduce(self, async_op: bool = False, lo: int = 0, hi: int | None = None, check: bool = True, slot: int = 0):
        from . import _lib
        if self.world == 1:
            return None
        if check:
            self.check_attached()
        hi = self.total if hi is None else hi
        if (lo % 4) or ((hi - lo) % 4):
            if hi != self.total or lo % 4:
                raise ValueError("PeerGradReducer: segment bounds must be multiples of 4 floats")
            hi = self.padded              # the tail of the last segment: padding floats are zero on every rank
        _lib.call("pph_peer_allreduce", self.ptr_table, self.multicast_ptr, self.flag_off, self.rank, self.world,
                  lo, hi - lo, self.n_ctas, slot)
        return None


def shard_batch(n_items: int, rank: int, world: int):
    """Contiguous batch shard [lo, hi) of rank `rank` (images are independent: no data-path collective)."""
    per, rem = divmod(n_items, world)
    lo = rank * per + min(rank, rem)
    return lo, lo + per + (1 if rank < rem else 0)
