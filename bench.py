#!/usr/bin/env python
"""Benchmark of the prototype-head path (BASELINE.json metric: prototype-head images/sec fwd+bwd).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload W] [--mode fp32|bf16] [--impl ours|reference]

A step = one training pass of the head over one per-GPU batch of BASELINE.json configs[1] (CUB / DeiT-Ti shape,
batch 64 per GPU): selection -> add-on -> similarity/pool -> last layers -> PPC loss -> cross-entropy -> backward
(token, prototype and add-on gradients) [-> gradient all-reduce when N > 1, recorded inside the CUDA graph and
overlapped with the add-on backward].  Other workloads (--workload): dogs_b256_eval (configs[2], forward only),
cars_b64_bf16 (configs[3]), sweep:K=..,D=..,P=..,B=.. (one point of configs[4]).  Synthetic inputs, random-init
parameters (protopformer_b200/synth.py).  Prints ONE JSON line (rank 0).

  value        device-resident throughput: inputs already in HBM, CUDA-graph replays, CUDA events, max over ranks.
               The step rotates over NBUF distinct input batches whose total size exceeds L2 (config.l2).
  e2e          same metric through the public API with HOST (pinned) inputs, every step inside the timed region: the
               selection-first transfer of the step's batch (scores + labels by copy, then exactly the token rows the head
               consumes read from the mapped host batch by pph_gather_rows_host -- e2e.h2d_bytes_per_step) into the other
               of two slots while the current step runs (one CUDA graph per iteration), and the result (total, ce, ppc_cov,
               ppc_mean) stored to pinned host memory by the kernel that completes the loss (e2e.d2h_bytes_per_step = 16).
               Asserted bit-identical to the device-resident result of the same batch.  --e2e-load full copies whole batches.
  roofline     the kernel with the largest share of the step, timed alone with CUDA events on its launch stream,
               plus roofline.step = the whole step's algorithmic flops against the sustained bf16 peak.
  forward_only the eval path (no PPC / CE / backward) on the same inputs; dropin_module_path = PPNet.forward +
               get_PPC_loss + autograd backward launched eagerly from Python.
  cpu_baseline the oracle's ATen-call-faithful port of the reference head (oracle/protohead_oracle.RefStyleHead)
               timed on this box's host cores on a bounded sample (rank 0, N=1 only).
  --impl reference : that CPU port as its own arm (the reference is pure Python over ATen; /root/reference does not
               exist on the GPU box, so the port stands in: cpu_baseline.kind = "port").

  --dump-outputs DIR  after the timed device-resident steps, writes what the last of them returned to the caller as
               DIR/<name>.npy (float32): logits, and in training loss, ppc_cov, ppc_mean, dtokens and the parameter
               gradients grad_P, grad_Pg, grad_Wa, grad_ba (rank 0).  The inputs depend only on the arguments, so two
               builds run with the same arguments can be compared output for output.  Above DUMP_BYTES in all, the
               largest arrays are cut to a fixed seeded sample of their leading-dimension rows (the same rows every run).
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

METRIC = "prototype_head_train_images_per_sec"
METRIC_EVAL = "prototype_head_forward_images_per_sec"
UNIT = "images/s"
DEFAULT_WORKLOAD = "cub_b64"    # BASELINE.json configs[1]: deit_tiny CUB shape, training step, batch 64 per GPU
DUMP_BYTES = 60 * 2 ** 20       # --dump-outputs: data bytes written in all (headroom under 64 MB for the .npy headers)


def parse_workload(name: str, mode_flag: str | None):
    """-> (canonical name, HeadShape, mode, train).  Named workloads are BASELINE.json's configs[1], [2], [3]; a
    "sweep:" spec is one point of configs[4] (tokens 49-196, prototypes 1000-8000, dim 192/384, batch 32-1024):
        sweep:K=81,D=192,P=2000,B=1024[,Pg=2000][,C=200][,mode=bf16][,eval=1]"""
    from protopformer_b200 import synth
    if name == "cub_b64":
        return name, synth.SHAPES["cub_b64"], mode_flag or "fp32", True
    if name == "dogs_b256_eval":
        return name, synth.SHAPES["dogs_b256"], mode_flag or "fp32", False
    if name == "cars_b64_bf16":
        return name, synth.SHAPES["cars_b64"], "bf16", True
    if name.startswith("sweep:"):
        kv = dict(item.split("=") for item in name[6:].split(",") if item)
        K, D, P, B = int(kv.get("K", 81)), int(kv.get("D", 192)), int(kv.get("P", 2000)), int(kv.get("B", 64))
        C = int(kv.get("C", P // 10))
        Pg = int(kv.get("Pg", 10 * C))
        shape = synth.HeadShape(name, B, 196, D, D, K, P, Pg, C, 0.5, 1.0, 2.0)
        return name, shape, kv.get("mode", mode_flag or "fp32"), kv.get("eval", "0") in ("0", "", "false")
    raise SystemExit(f"unknown workload {name!r}: cub_b64 | dogs_b256_eval | cars_b64_bf16 | sweep:K=..,D=..,P=..,B=..")


def make_config(workload, shape, mode, train, world, nbuf, in_graph, exchange="peer"):
    """The `config` object of the JSON line: built by this one function for BOTH arms so that they are equal."""
    in_bytes = 4 * shape.B * ((1 + shape.N) * shape.Din + shape.N) + 8 * shape.B
    step = ("head fwd + PPC + CE + bwd (dtokens, dP, dPg, dWa, dba)" if train
            else "head forward (selection -> add-on -> similarity/pool -> last layers)")
    if world > 1 and train:
        how = "NCCL grad all-reduce" if exchange == "nccl" else "grad all-reduce kernel over NVLink peer memory"
        step += f" + {how} (" + ("in graph, overlapped with the add-on backward" if in_graph else "after each replay") + ")"
    return {"workload": workload, "per_gpu_batch": shape.B, "tokens": shape.K, "dim": shape.D,
            "prototypes": shape.P, "global_prototypes": shape.Pg, "classes": shape.C, "mode": mode, "step": step,
            "l2": f"inputs rotate over {nbuf} batches = {nbuf * in_bytes / 1e6:.0f} MB > 126 MB L2; parameters stay "
                  "L2-resident",
            "parallelism": f"dp{world}", "cuda_graph": True}


def step_flops(shape, train: bool) -> float:
    """Algorithmic flops of one step (SURVEY.md 8(d)): add-on, similarity, last layers; backward = 2x the two GEMMs of
    each forward GEMM that has a trainable / differentiated operand (the similarity backward is argmin-routed, i.e.
    sparse: B*(P+Pg) rows of D, not a GEMM)."""
    s = shape
    rows = s.B * (s.K + 1)
    f_addon = 2.0 * rows * s.Din * s.D
    f_sim = s.B * (2.0 * s.K * s.D * s.P + 2.0 * s.D * s.Pg)
    f_ll = 2.0 * s.B * s.C * (s.P + s.Pg)
    fwd = f_addon + f_sim + f_ll
    if not train:
        return fwd
    f_bwd = 2.0 * f_addon + f_ll + 6.0 * s.B * (s.P + s.Pg) * s.D
    return fwd + f_bwd


def bind_to_gpu_numa(index: int):
    """Pin this process to the CPUs of the NUMA node its GPU hangs off, BEFORE the pinned staging buffers are
    allocated (first touch then places them on that node): eight ranks each pushing ~10 MB per step over PCIe should
    not all read one socket's memory.  Best effort; returns a description for the JSON line."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        bus = pynvml.nvmlDeviceGetPciInfo(h).busId
        bus = (bus.decode() if isinstance(bus, bytes) else bus).lower()
        if len(bus.split(":")[0]) == 8:
            bus = bus[4:]
        node = int(open(f"/sys/bus/pci/devices/{bus}/numa_node").read())
        if node < 0:
            return "numa_node=-1 (single node): not bound"
        cpus = []
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            a, _, b = part.partition("-")
            cpus += list(range(int(a), int(b or a) + 1))
        allowed = sorted(set(cpus) & os.sched_getaffinity(0))
        if not allowed:
            return f"node {node}: none of its CPUs are in this process's affinity mask"
        os.sched_setaffinity(0, allowed)
        return f"bound to NUMA node {node} ({len(allowed)} CPUs) of GPU {index}"
    except Exception as exc:
        return f"not bound ({type(exc).__name__}: {exc})"


def _peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        d = json.load(open(path))
        return dict(hbm=float(d["hbm_gbs"]), tf_burst=float(d["bf16_tflops"]),
                    tf_sust=float(d.get("bf16_tflops_sustained", d["bf16_tflops"])), src="measured")
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sust=1400.0, src="fallback")


def _measured_traffic(workload, mode, kernel):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed ncu --set full capture of this
    workload (profiles/r2_kernel_traffic.json, written by scripts/ncu_traffic.py from the .ncu-rep) or None."""
    path = os.path.join(ROOT, "profiles", "r2_kernel_traffic.json")
    try:
        return json.load(open(path)).get(f"{workload}/{mode}", {}).get(kernel)
    except Exception:
        return None


def graph_time_us(fn, per_graph: int, replays: int = 10) -> float:
    """Average device time of one `fn()` call: `per_graph` calls recorded in a CUDA graph (no host launch gaps),
    replayed `replays` times between two events on the current stream."""
    for _ in range(3):
        fn(0)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for i in range(per_graph):
            fn(i)
    g.replay()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(replays):
        g.replay()
    b.record()
    torch.cuda.synchronize()
    return 1e3 * a.elapsed_time(b) / (replays * per_graph)


def step_outputs(step, slot: int, train: bool) -> dict:
    """Host copies of what a caller of the graphed step receives from the replay just run on `slot`."""
    out = {"logits": step.logits[slot]}
    if train:
        out.update(loss=step.loss[slot], ppc_cov=step.ppc[slot][0], ppc_mean=step.ppc[slot][1], dtokens=step.dtokens[slot])
        out.update({f"grad_{k}": g for k, g in step.grads.items()})
    return {k: v.detach().float().cpu() for k, v in out.items()}


def dump_outputs(out_dir: str, arrays: dict, budget: int = DUMP_BYTES):
    """Writes every array as out_dir/<name>.npy (float32), smallest first.  An array larger than an equal share of the
    budget left keeps a sample of its leading-dimension rows drawn from a fixed seed (sorted, so the same rows of the same
    shape in every run)."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    order = sorted(arrays, key=lambda k: arrays[k].numel())
    for i, name in enumerate(order):
        t = arrays[name]
        share = budget // (len(order) - i)
        if t.dim() > 0 and t.shape[0] > 1 and 4 * t.numel() > share:
            keep = max(1, share // (4 * (t.numel() // t.shape[0])))
            rows = torch.randperm(t.shape[0], generator=torch.Generator().manual_seed(0))[:keep].sort().values
            t = t[rows]
        np.save(os.path.join(out_dir, name + ".npy"), t.numpy())
        budget -= 4 * t.numel()


# ---------------------------------------------------------------------------------------------------------------
# clocks sampler (NVML from a thread: the timed region is short)
# ---------------------------------------------------------------------------------------------------------------
class ClockSampler:
    def __init__(self, index: int):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._t = None
        self.window = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def _loop(self):
        nv = self.nv
        names = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20,
                 "hw_power_brake": 0x80}
        while not self._stop.is_set():
            try:
                mhz = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                self.samples.append((time.perf_counter(), mhz, [k for k, b in names.items() if r & b]))
            except Exception:
                pass
            time.sleep(0.004)

    def start(self):
        if self.nv is not None:
            self._t = threading.Thread(target=self._loop, daemon=True)
            self._t.start()

    def stop(self):
        self._stop.set()
        if self._t:
            self._t.join(timeout=1)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": [], "samples": 0}
        t0, t1 = self.window or (0, float("inf"))
        inside = [s for s in self.samples if t0 <= s[0] <= t1] or self.samples
        reasons = sorted({r for s in inside for r in s[2]})
        return {"sm_mhz": statistics.median(s[1] for s in inside), "sm_max_mhz": self.max_mhz,
                "reasons": reasons, "samples": len(inside)}


# ---------------------------------------------------------------------------------------------------------------
# CPU arm: the reference head's ATen call sequence on the host cores
# ---------------------------------------------------------------------------------------------------------------
def _cpu_step_fn(shape, sample_B, train):
    from oracle import protohead_oracle as O
    from protopformer_b200 import synth
    s = shape.with_batch(sample_B)
    case = synth.make_case(s, seed=1)
    head = O.RefStyleHead(case, s)
    if train:
        return lambda: head.train_step(case["tokens"], case["scores"], case["labels"])

    def fwd():
        with torch.no_grad():
            return head.forward(case["tokens"], case["scores"])
    return fwd


def cpu_port_rate(shape, budget_s: float, sample_B: int, iters_min: int = 3, train: bool = True):
    """images/s of the port's training step (or forward) on a `sample_B`-image slice of the workload, ~budget_s."""
    fn = _cpu_step_fn(shape, sample_B, train)
    fn()                                                                      # warm-up
    times = []
    t_end = time.perf_counter() + budget_s
    while len(times) < iters_min or (time.perf_counter() < t_end and len(times) < 50):
        t = time.perf_counter()
        fn()
        times.append(time.perf_counter() - t)
    return sample_B / statistics.median(times), len(times)


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    world = int(os.environ.get("WORLD_SIZE", str(args.gpus)))
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    workload, shape, mode, train = parse_workload(args.workload, args.mode)
    # bounded sample: a per-step slice of the per-GPU batch sized so that (K + W) steps end within ~150 s
    probe, _ = cpu_port_rate(shape, 2.0, min(8, shape.B), train=train)
    per_step = 150.0 / max(1, args.steps + args.warmup)
    sample_B = max(1, min(shape.B, int(probe * per_step)))
    fn = _cpu_step_fn(shape, sample_B, train)
    for _ in range(args.warmup):
        fn()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        fn()
    dt = time.perf_counter() - t0
    value = sample_B * args.steps / dt
    sample = (f"{sample_B} of {shape.B} images per step ({workload}), fp32, torch {torch.__version__} CPU, ONE process "
              f"on rank 0's host cores" + (f" (the GPU arm at n_gpus={world} processes {world}x{shape.B} images per step: "
                                           "the driver's ratio is N GPUs vs this one CPU process)" if world > 1 else ""))
    line = {
        "impl": "reference", "metric": METRIC if train else METRIC_EVAL, "value": value, "unit": UNIT,
        "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": make_config(workload, shape, mode, train, world, args.nbuf, not args.eager_allreduce, args.exchange),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)
    return 0


def measure_next_rows(shape, params, dev, peaks):
    """Device time of the two HBM-bound rows next to the head, each against the measured HBM bandwidth:
    attention rollout -> CLS-row score (DeiT-Ti: 11 layers x 3 heads x 197^2 per image, read once) and the fused AdamW
    step over the head's parameter groups (28 B per element)."""
    from protopformer_b200 import ops
    from protopformer_b200.optim import FusedHeadAdamW
    out = {}
    with torch.no_grad():
        L, H, T, B = 11, 3, shape.N + 1, min(shape.B, 64)
        g = torch.Generator(device=dev).manual_seed(0)
        attn = [torch.softmax(2.0 * torch.randn(B, H, T, T, device=dev, generator=g), dim=-1) for _ in range(L)]
        us = graph_time_us(lambda i: ops.rollout_scores(attn), 4)
        nbytes = float(L * B * H * T * T * 4)
        out["rollout"] = {"kernel": "rollout_prepare2_kernel + rollout_chain2_kernel", "bound": "hbm",
                          "achieved": nbytes / us / 1e3, "peak": peaks["hbm"], "unit": "GB/s",
                          "frac": nbytes / us / 1e3 / peaks["hbm"], "us_per_call": us,
                          "algorithmic_bytes_per_call": nbytes,
                          "workload": f"L={L} H={H} T={T} B={B} fp32 maps ({nbytes / 1e6:.0f} MB > L2), read once"}
        del attn
        ps = [params[k].detach().clone() for k in ("Wa", "ba", "P", "Pg")]
        gs = [torch.randn_like(p) * 0.01 for p in ps]
        opt = FusedHeadAdamW([{"params": ps[:2], "lr": 3e-3, "weight_decay": 1e-3},
                              {"params": ps[2:], "lr": 3e-3, "weight_decay": 0.05}], grads=gs)
        us = graph_time_us(lambda i: opt.step(), 20)
        nbytes = 28.0 * sum(p.numel() for p in ps)
        out["adamw"] = {"kernel": "adamw_kernel (4 tensors, one launch)", "bound": "hbm",
                        "achieved": nbytes / us / 1e3, "peak": peaks["hbm"], "unit": "GB/s",
                        "frac": nbytes / us / 1e3 / peaks["hbm"], "us_per_call": us,
                        "algorithmic_bytes_per_call": nbytes,
                        "note": "22.5 MB working set is L2-resident between replays: an upper bound on the HBM rate"}
    return out


# ---------------------------------------------------------------------------------------------------------------
# the drop-in module path: PPNet.forward + get_PPC_loss + autograd backward, eager (what a user of the reference's
# training loop gets without adopting the graphed step), tools/engine_proto.py:49-76
# ---------------------------------------------------------------------------------------------------------------
class _TokenFeed(torch.nn.Module):
    """Stands in for the backbone (out of this path's scope): hands the preloaded tokens / CLS-attention scores to the
    head through the two backbone methods PPNet calls (protopformer.py:149, 155)."""

    def __init__(self, Din, N):
        super().__init__()
        self.proj = torch.nn.Linear(Din, Din)           # PPNet reads the last nn.Linear's out_features
        self.patch_embed = type("PE", (), {"num_patches": N})()
        self.cur = None

    def __repr__(self):
        return "MYVISIONTRANSFORMER(token feed)"

    def forward_feature_patch_embed_all(self, x):
        return None, None

    def forward_feature_mask_train_direct(self, cls_embed, x_embed, mask, reserve_layer_nums):
        tokens, scores = self.cur
        return tokens, (scores, None)


def measure_dropin(shape, mode, params, step, nbuf, steps):
    from protopformer_b200.head import PPNet
    dev = params["P"].device
    net = PPNet(_TokenFeed(shape.Din, shape.N), 224, (shape.P, shape.D, 1, 1), None, shape.C, reserve_layers=[11],
                reserve_token_nums=[shape.K], use_global=True, use_ppc_loss=True, ppc_cov_thresh=shape.ppc_cov_thresh,
                ppc_mean_thresh=shape.ppc_mean_thresh, global_coe=shape.global_coe,
                global_proto_per_class=shape.Pg // shape.C, add_on_layers_type="regular", precision=mode).to(dev)
    with torch.no_grad():
        net.add_on_layers[0].weight.copy_(params["Wa"].reshape(net.add_on_layers[0].weight.shape))
        net.add_on_layers[0].bias.copy_(params["ba"])
        net.prototype_vectors.copy_(params["P"].reshape(net.prototype_vectors.shape))
        net.prototype_vectors_global.copy_(params["Pg"].reshape(net.prototype_vectors_global.shape))
        net.last_layer.weight.copy_(params["Wl"])
        net.last_layer_global.weight.copy_(params["Wg"])
    net.train()
    feed = net.features
    ce = torch.nn.CrossEntropyLoss()

    def one(i):
        tok = step.tokens[i % nbuf].detach().requires_grad_(True)
        feed.cur = (tok, step.scores[i % nbuf])
        for p in net.parameters():
            p.grad = None
        logits, aux = net(None)
        cov, mean = net.get_PPC_loss(aux[2], aux[3], aux[4], step.labels[i % nbuf])
        loss = ce(logits, step.labels[i % nbuf]) + 0.1 * cov + 0.5 * mean
        loss.backward()
        return loss

    for i in range(5):
        one(i)
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for i in range(steps):
        loss = one(i)
    b.record()
    torch.cuda.synchronize()
    ms = a.elapsed_time(b) / steps
    return {"value": shape.B / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms, "loss": float(loss.item()),
            "path": "PPNet.forward + get_PPC_loss + CrossEntropyLoss + autograd backward, eager launches from Python "
                    "(device-resident inputs)"}


# ---------------------------------------------------------------------------------------------------------------
# our arm
# ---------------------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2000)
    ap.add_argument("--warmup", type=int, default=100)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=DEFAULT_WORKLOAD,
                    help="cub_b64 (default, BASELINE configs[1]) | dogs_b256_eval | cars_b64_bf16 | sweep:K=..,D=..,P=..,B=..")
    ap.add_argument("--mode", default=None, choices=["fp32", "bf16"],
                    help="similarity precision: fp32 = 3-term bf16 split (1e-4 parity), bf16 = single pass")
    ap.add_argument("--nbuf", type=int, default=16, help="distinct input batches the step rotates over")
    ap.add_argument("--e2e-load", default="selected", choices=["selected", "full"],
                    help="end-to-end leg: transfer only the token rows the head consumes (default) or the whole batch")
    ap.add_argument("--no-overlap-graph", action="store_true",
                    help="end-to-end leg: separate transfer / step graphs tied by events instead of one graph per iteration")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-extras", action="store_true", help="headline numbers only (no roofline / next rows / drop-in legs)")
    ap.add_argument("--exchange", default="peer", choices=["peer", "peer_nomc", "nccl"],
                    help="N>1 gradient exchange: the library's one-kernel all-reduce over peer memory (NVLS multicast when "
                         "available / plain peer pointers) or NCCL")
    ap.add_argument("--eager-allreduce", action="store_true",
                    help="N>1: issue the NCCL gradient all-reduce after each graph replay instead of inside the graph")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step returned as DIR/<name>.npy (float32, at most 64 MB in all)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the CUDA step: use it with --impl ours")
    if args.warmup < 3:
        args.warmup = 3
    if args.impl == "reference":
        return run_reference_arm(args)

    import torch.distributed as dist
    from protopformer_b200 import synth                       # synthetic input generator (bench infrastructure)
    from protopformer_b200 import _lib, ops
    from protopformer_b200.graph import GraphedHeadStep

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a CUDA device: the prototype head has no CPU path"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    numa = bind_to_gpu_numa(local) if world > 1 else "single process: not bound"
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    _lib.load()

    workload, shape, mode, train = parse_workload(args.workload, args.mode)
    in_graph = world > 1 and train and not args.eager_allreduce
    case = synth.make_case(shape, seed=1)
    params = {k: case[k].to(dev) for k in ("Wa", "ba", "P", "Pg", "Wl", "Wg")}
    if train:
        for k in ("Wa", "ba", "P", "Pg"):
            params[k].requires_grad_(True)
    cfg = ops.HeadConfig(K=shape.K, global_coe=shape.global_coe, mode=mode,
                         ppc_cov_thresh=shape.ppc_cov_thresh, ppc_mean_thresh=shape.ppc_mean_thresh)
    nbuf = args.nbuf
    step = GraphedHeadStep(params, cfg, B=shape.B, N=shape.N, C=shape.C, m=shape.m, n_slots=nbuf, train=train,
                           allreduce_in_graph=in_graph, exchange=args.exchange if (world > 1 and train) else "nccl")
    # distinct synthetic batches per slot and per rank (weak scaling: fixed per-GPU batch)
    host = []
    for i in range(nbuf):
        c = synth.make_case(shape, seed=100 + rank * nbuf + i) if i < 4 else None
        if c is None:       # cheaper variants of the first four: permute images (keeps every tensor distinct)
            b = host[i % 4]
            perm = torch.randperm(shape.B, generator=torch.Generator().manual_seed(i))
            c = dict(tokens=b["tokens"][perm].contiguous(), scores=b["scores"][perm].contiguous(),
                     labels=b["labels"][perm].contiguous())
        if i == 0:
            first = {k: c[k].clone() for k in ("tokens", "scores", "labels")}
        host.append({k: c[k].pin_memory() for k in ("tokens", "scores", "labels")})
        step.load(i, host[i]["tokens"], host[i]["scores"], host[i]["labels"])
    torch.cuda.synchronize()
    step.capture()
    in_bytes = sum(host[0][k].numel() * host[0][k].element_size() for k in host[0])

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def one(i):
        step.run(i % nbuf)
        if world > 1 and train:
            step.allreduce_grads()            # no-op when the all-reduce is part of the graph

    # ---- the result of slot 0 against the CPU oracle, once (rank 0 compares; every rank runs the step) -----------
    one(0)
    torch.cuda.synchronize()
    oracle_check = None
    if rank == 0 and not args.no_cpu and shape.B * shape.P * shape.K <= (1 if train else 2) * 64 * 2000 * 121:
        from oracle import protohead_oracle as O               # the checker, never the thing measured
        ocase = dict(case)
        ocase.update(first)
        tol = 1e-4 if mode == "fp32" else 5e-4
        if train and world == 1:
            ref = O.head_train_step(ocase, shape)
            got, want = float(step.loss[0].item()), float(ref["loss"].item())
        else:                                  # forward-only workloads (and N>1, whose graph averages gradients only)
            ref = O.head_forward(ocase, shape.K, shape.global_coe)
            got, want = float(step.logits[0].abs().sum().item()), float(ref["logits"].abs().sum().item())
        rel = abs(got - want) / abs(want)
        oracle_check = {"what": "loss of the first batch" if (train and world == 1) else "sum |logits| of the first batch",
                        "gpu": got, "oracle": want, "rel_err": rel, "tol": tol}
        assert rel <= tol, f"bench result differs from the CPU oracle: {oracle_check}"

    sampler = ClockSampler(local)
    sampler.start()

    # ---- device-resident timing ------------------------------------------------------------------------------
    for i in range(args.warmup):
        one(i)
    barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_w0 = time.perf_counter()
    ev0.record()
    for i in range(args.steps):
        one(i)
    ev1.record()
    barrier()
    t_w1 = time.perf_counter()
    sampler.window = (t_w0, t_w1)
    # copied out now: the legs below replay the step again
    outputs = step_outputs(step, (args.steps - 1) % nbuf, train) if args.dump_outputs and rank == 0 else None
    ms = ev0.elapsed_time(ev1)
    if world > 1:
        t = torch.tensor([ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    value = world * shape.B * args.steps / (ms * 1e-3)

    # ---- end to end through the public API with host buffers ---------------------------------------------------
    copy_stream = torch.cuda.Stream()
    # the result a caller reads back every step: the loss in training, the logits in inference
    result_of = (lambda s: step.loss[s].reshape(1)) if train else (lambda s: step.logits[s])
    out_host = torch.zeros(1 if train else shape.B * shape.C).reshape(-1 if train else shape.B, *(() if train else (shape.C,))).pin_memory()
    ready = [torch.cuda.Event() for _ in range(2)]
    done = [torch.cuda.Event() for _ in range(2)]

    selected = args.e2e_load == "selected"
    h2d_bytes = (4 * shape.B * shape.N + 8 * shape.B + 4 * shape.B * (shape.K + 1) * shape.Din) if selected else in_bytes
    # what the last e2e step must reproduce: the same batch through the device-resident path
    last_slot = (args.steps - 1) % nbuf
    step.run(last_slot)
    if world > 1 and train:
        step.allreduce_grads()
    torch.cuda.synchronize()
    want_last = float(result_of(last_slot).reshape(-1)[0].item())

    host_pipe = selected and train and step.impl == "v2" and (world == 1 or in_graph)
    if host_pipe:
        step.capture_host_pipeline()
    load_graphs = {}
    if selected:      # one recorded transfer per (slot, staging buffer) pair of the ring
        for s in range(2):
            for i in range(nbuf):
                if i % 2 == s or nbuf % 2:
                    b = host[i]
                    load_graphs[(s, i)] = step.capture_load_host(s, b["tokens"], b["scores"], b["labels"])
        step.run(last_slot)           # slots 0 / 1 were overwritten by the captures' warm-up transfers: harmless
        torch.cuda.synchronize()

    # host pipeline with two slots: one graph per iteration = the step of this slot || the transfer of the next batch into the
    # other slot (one host call per step, no cross-stream events)
    overlapped = host_pipe and not args.no_overlap_graph
    if overlapped:
        pair_graphs = {(s, j): step.capture_host_overlapped(s, host[j]["tokens"], host[j]["scores"], host[j]["labels"])
                       for s in range(2) for j in range(nbuf) if (j % 2 != s or nbuf % 2)}

    def e2e_loop_overlapped(n):
        b0 = host[0]
        step.load_host(0, b0["tokens"], b0["scores"], b0["labels"])          # the first batch; every later one rides in a graph
        for i in range(n):
            pair_graphs[(i % 2, (i + 1) % nbuf)].replay()
        torch.cuda.synchronize()
        return float(step.loss_host[(n - 1) % 2][0].item())

    def e2e_loop(n):
        if overlapped:
            return e2e_loop_overlapped(n)
        cur = torch.cuda.current_stream()
        for i in range(n):
            s = i % 2
            with torch.cuda.stream(copy_stream):
                copy_stream.wait_event(done[s])                 # slot s no longer read by step i-2
                b = host[i % nbuf]
                if selected:
                    load_graphs[(s, i % nbuf)].replay()
                else:
                    step.load(s, b["tokens"], b["scores"], b["labels"])
                ready[s].record(copy_stream)
            cur.wait_event(ready[s])
            if host_pipe:             # selection from the transfer, loss stored to pinned host memory by the kernel itself
                step.run_host(s)
            else:
                step.run(s)
                if world > 1 and train:
                    step.allreduce_grads()
                out_host.copy_(result_of(s), non_blocking=True)
            done[s].record(cur)
        torch.cuda.synchronize()
        return float(step.loss_host[(n - 1) % 2][0].item()) if host_pipe else float(out_host.reshape(-1)[0].item())

    for s in range(2):
        done[s].record(torch.cuda.current_stream())
    e2e_loop(max(3, args.warmup // 10))
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    last_loss = e2e_loop(args.steps)
    e1.record()
    assert last_loss == want_last, f"end-to-end result {last_loss} != device-resident result {want_last} of the same batch"
    barrier()
    ms_e2e = e0.elapsed_time(e1)
    if world > 1:
        t = torch.tensor([ms_e2e], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_e2e = float(t.item())
    e2e_value = world * shape.B * args.steps / (ms_e2e * 1e-3)
    sampler.stop()
    # restore the rotation the device-resident legs below read
    for i in range(2):
        step.load(i, host[i]["tokens"], host[i]["scores"], host[i]["labels"])
    torch.cuda.synchronize()

    peaks = _peaks()
    extras = rank == 0 and not args.no_extras
    us_step = 1e3 * ms / args.steps

    # ---- forward-only rate (eval path, tools/engine_proto.py:156-162 -> protopformer.py:292-301) ---------------------
    forward_only = None
    if extras and train:
        try:
            ev_params = {k: v.detach() for k, v in params.items()}
            fstep = GraphedHeadStep(ev_params, cfg, B=shape.B, N=shape.N, C=shape.C, m=shape.m, n_slots=nbuf, train=False)
            for i in range(nbuf):
                fstep.load(i, step.tokens[i].detach(), step.scores[i], step.labels[i])
            fstep.capture()
            for i in range(20):
                fstep.run(i % nbuf)
            torch.cuda.synchronize()
            f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            f0.record()
            for i in range(args.steps):
                fstep.run(i % nbuf)
            f1.record()
            torch.cuda.synchronize()
            fms = f0.elapsed_time(f1) / args.steps
            ff = step_flops(shape, False)
            forward_only = {"metric": METRIC_EVAL, "value": shape.B / (fms * 1e-3), "unit": UNIT, "ms_per_step": fms,
                            "gpu_launches_per_step": fstep.kernel_launches_per_step,
                            "tensor_frac_sustained": ff / (fms * 1e-3) / 1e12 / peaks["tf_sust"]}
            del fstep
        except Exception as exc:
            forward_only = {"error": str(exc)}

    # ---- roofline: the kernel with the largest share of the step + the step itself ---------------------------------
    roof = None
    if extras:
        roof = measure_roofline(step, shape, cfg, mode, params, train, peaks, us_step, workload, nbuf)

    next_rows = dropin = None
    if extras:
        try:
            next_rows = measure_next_rows(shape, params, dev, peaks)
        except Exception as exc:      # auxiliary: the headline line must print regardless
            next_rows = {"error": str(exc)}
        if train:
            try:
                dropin = measure_dropin(shape, mode, params, step, nbuf, args.steps)
            except Exception as exc:
                dropin = {"error": f"{type(exc).__name__}: {exc}"}

    # ---- CPU baseline (rank 0, N = 1 only) ---------------------------------------------------------------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        cores = os.cpu_count() or 1
        torch.set_num_threads(cores)
        sb = min(shape.B, 64)
        rate, n = cpu_port_rate(shape, 12.0, sb, train=train)
        cpu = {"value": rate, "unit": UNIT, "cores": cores, "kind": "port",
               "sample": f"{n} {'training steps' if train else 'forward passes'} of a {sb}-image batch ({workload}), "
                         "fp32, torch CPU"}
        try:                              # per-core figure (BASELINE.md section 3): same port on ONE thread, small sample
            torch.set_num_threads(1)
            rate1, n1 = cpu_port_rate(shape, 4.0, 8, iters_min=2, train=train)
            cpu["value_1_core"] = rate1
            cpu["sample_1_core"] = f"{n1} steps of an 8-image slice, 1 thread"
        except Exception as exc:
            cpu["value_1_core"] = None
            cpu["sample_1_core"] = f"failed: {exc}"
        finally:
            torch.set_num_threads(cores)

    if rank == 0:
        line = {
            "metric": METRIC if train else METRIC_EVAL, "value": value, "unit": UNIT, "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "bf16x3 split, fp32 accumulate (fp32-grade)" if mode == "fp32" else "bf16, fp32 accumulate",
            "data": "synthetic",
            "config": make_config(workload, shape, mode, train, world, nbuf, not args.eager_allreduce, args.exchange),
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d_bytes,
                    "h2d": ("selection first: scores + labels by copy, then the CLS row and the K selected token rows of every "
                            "image read from the pinned host batch by pph_gather_rows_host (the other rows are never read by "
                            f"the head; a full copy would be {in_bytes} bytes)") if selected else "full batch by cudaMemcpyAsync", "d2h_bytes_per_step": 16 if host_pipe else out_host.numel() * 4,
                    "d2h": ("(total, ce, ppc_cov, ppc_mean) stored into pinned host memory by the kernel that completes the loss"
                            if host_pipe else "cudaMemcpyAsync of the result on the step's stream"),
                    "ms_per_step": ms_e2e / args.steps, "last_loss" if train else "last_logit": last_loss, "host_buffers": numa},
            "gpu_launches": step.kernel_launches_per_step * args.steps,
            "gpu_launches_per_step": step.kernel_launches_per_step,
            "step_impl": step.impl,
            "exchange": getattr(step, "exchange", None) if world > 1 else None,
            "exchange_note": getattr(step, "exchange_note", "") if world > 1 else "",
            "clocks": sampler.summary(),
            "roofline": roof,
            "oracle_check": oracle_check,
            "forward_only": forward_only,
            "dropin_module_path": dropin,
            "next_rows": next_rows,
            "cpu_baseline": cpu,
        }
        if outputs is not None:
            dump_outputs(args.dump_outputs, outputs)
        print(json.dumps(line), flush=True)
    if world > 1:
        # graphs that recorded NCCL kernels keep the communicator busy: drop them first, and never let a stuck teardown
        # turn a finished measurement into a hang
        step.graphs.clear()
        import gc
        gc.collect()
        torch.cuda.synchronize()
        t = threading.Thread(target=dist.destroy_process_group, daemon=True)
        t.start()
        t.join(20)
        sys.stdout.flush()
        os._exit(0)
    return 0


def measure_roofline(step, shape, cfg, mode, params, train, peaks, us_step, workload, nbuf):
    """`roofline` of the JSON line: the kernel with the largest share of the step (timed alone, CUDA graph of back-to-back
    launches on the current stream, events around the replays), the tensor-core similarity kernel the same way, and the
    step-level fraction (algorithmic flops of the whole step / step time / sustained bf16 peak)."""
    from protopformer_b200 import _lib, ops
    f = step.fused
    B, K, D, P, Pg = shape.B, shape.K, shape.D, shape.P, shape.Pg
    cands = {}
    with torch.no_grad():
        try:
            tfs = []
            for i in range(min(nbuf, 4)):
                idx = ops.select_topk(step.scores[i], K)
                tfs.append(ops.addon(step.tokens[i].detach(), idx, params["Wa"].detach(), params["ba"].detach(), True))
            pl = ops.prepare_prototypes(params["P"].detach(), True)
            pg = ops.prepare_prototypes(params["Pg"].detach(), True)
            us = graph_time_us(lambda i: ops._similarity_raw(cfg, tfs[i % len(tfs)], pl, pg), 16)
            flops = B * (2.0 * K * D * P + 2.0 * D * Pg)                   # F_sim, SURVEY.md 8(d)
            ach = flops / (us * 1e-6) / 1e12
            cands["similarity"] = {
                "kernel": "similarity_tc2_kernel (tcgen05 + TMA, resident prototype tile, mode %s)" % mode,
                "bound": "tensor", "achieved": ach, "peak": peaks["tf_burst"], "unit": "TFLOP/s",
                "frac": ach / peaks["tf_burst"], "traffic": _measured_traffic(workload, mode, "similarity_tc2_kernel"),
                "us_per_launch": us, "algorithmic_flops_per_launch": flops,
                "note": ("fp32 mode issues 3 bf16 MMA passes per algorithmic flop: tensor-pipe work is 3x the "
                         "algorithmic figure" if mode == "fp32" else "")}
            del tfs
        except Exception as exc:
            cands["similarity"] = {"error": str(exc), "us_per_launch": 0.0}
        if train and step.impl == "v2":
            try:
                gP, gPg = torch.empty_like(params["P"]), torch.empty_like(params["Pg"])
                us = graph_time_us(lambda i: _lib.call(
                    "pph_similarity_bwd_fused", 3, f.g_l, f.g_g, f.argmin, f.Zs, f.Zc, params["P"].detach(),
                    params["Pg"].detach(), B, K, D, P, Pg, shape.m, f.ws_gather, f.ws_bins, None, None, 1, f.dZs, f.dZc,
                    gP, gPg), 16)
                # compulsory bytes: Zs, Zc, P, Pg, g_l, g_g, argmin, bins read once; dZs, dZc, dP, dPg written once
                byts = 4.0 * (2 * B * K * D + 2 * B * D + 2 * (P + Pg) * D + B * (P + Pg) + 2 * B * P)
                ach = byts / (us * 1e-6) / 1e9
                cands["sim_grads"] = {
                    "kernel": "sim_grads_kernel (argmin-routed sparse backward: dP, dPg, dZs as dpre, dZc)", "bound": "hbm",
                    "achieved": ach, "peak": peaks["hbm"], "unit": "GB/s", "frac": ach / peaks["hbm"],
                    "traffic": _measured_traffic(workload, mode, "sim_grads_kernel"), "us_per_launch": us,
                    "algorithmic_bytes_per_launch": byts,
                    "note": "gathers 2*B*P rows of D floats from L2-resident operands: L2-latency bound, far from the HBM "
                            "roofline by construction (its working set never leaves L2 at this shape)"}
            except Exception as exc:
                cands["sim_grads"] = {"error": str(exc), "us_per_launch": 0.0}
    key = max(cands, key=lambda k: cands[k].get("us_per_launch", 0.0))
    roof = dict(cands[key])
    roof["share_of_step"] = roof.get("us_per_launch", 0.0) / us_step
    roof["peak_source"] = peaks["src"] + (" bf16 burst" if roof.get("bound") == "tensor" else " HBM copy") + \
        " (kernel timed alone)"
    fl = step_flops(shape, train)
    tf = fl / (us_step * 1e-6) / 1e12
    roof["step"] = {"bound": "tensor", "algorithmic_flops_per_step": fl, "achieved": tf, "unit": "TFLOP/s",
                    "peak": peaks["tf_sust"], "frac": tf / peaks["tf_sust"],
                    "peak_source": peaks["src"] + " bf16 sustained (step timed in a long loop)", "us_per_step": us_step}
    roof["other_kernels"] = {k: v for k, v in cands.items() if k != key}
    return roof


if __name__ == "__main__":
    sys.exit(main())
