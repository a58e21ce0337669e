"""What unfreezing the last layers costs the graphed training step, and what pph_last_layer_wgrad achieves alone.

    python scripts/last_layer_grad_bench.py [--workloads cub_b64,cars_b64_bf16,cub_b1024] [--rounds 3] [--window 0.25]
                                            [--out FILE] [--timeline] [--dry-run]

Per workload, in ONE process: the graphed step with frozen last layers and the same step with trainable ones (Wl, Wg
requires_grad), alternated --rounds times; each arm is timed with CUDA events over a window of >= --window seconds of
replays after a warm-up.  The replays rotate over input slots whose token rows read by the step add up to more than the
126 MB L2 of a B200 (each slot is a distinct seeded batch; the weights and intermediate buffers are the same in both
arms and stay L2-resident either way).  Then pph_last_layer_wgrad alone: CUDA events around a CUDA graph of 100 launches
on the step's own dlogits / act_l / act_g (hot in L2, as inside the step), replayed for >= --window seconds; achieved
GB/s and GFLOP/s from the shapes:
    bytes = 4 (C (P+Pg) + B (C + P + Pg))      flops = 2 B C (P+Pg)
The GPU name and power limit are read in the same call.  --timeline adds a torch.profiler list of the kernels of one
trainable replay at cub_b64 (start, duration).  --dry-run prints the workloads and the shape arithmetic without a device.
"""
import argparse
import json
import math
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

from protopformer_b200 import synth  # noqa: E402

L2_BYTES = 126 * 2 ** 20
WORKLOADS = {          # name -> (shape, similarity mode); cars_b64_bf16 is the shape of bench.py's workload of that name
    "cub_b64": (synth.SHAPES["cub_b64"], "fp32"),
    "cars_b64_bf16": (synth.SHAPES["cars_b64"], "bf16"),
    "cub_b1024": (synth.SHAPES["cub_b64"].with_batch(1024), "fp32"),
}


def kernel_bytes_flops(s):
    return 4 * (s.C * (s.P + s.Pg) + s.B * (s.C + s.P + s.Pg)), 2 * s.B * s.C * (s.P + s.Pg)


def slot_read_bytes(s):
    """Input bytes one replay reads from its slot: the CLS row and the K selected token rows of every image, the scores."""
    return 4 * s.B * (s.K + 1) * s.Din + 4 * s.B * s.N + 8 * s.B


def n_slots(s, cap=64):
    return max(2, min(cap, math.ceil(1.5 * L2_BYTES / slot_read_bytes(s))))


def gpu_identity():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError) as exc:
        q = f"unknown ({type(exc).__name__})"
    return name, q


def make_step(s, mode, train_ll, inputs):
    from protopformer_b200 import ops
    from protopformer_b200.graph import GraphedHeadStep
    case = synth.make_case(s.with_batch(1), seed=1)            # weights only (they do not depend on B)
    cfg = ops.HeadConfig(K=s.K, global_coe=s.global_coe, mode=mode, ppc_cov_thresh=s.ppc_cov_thresh,
                         ppc_mean_thresh=s.ppc_mean_thresh)
    params = {k: case[k].cuda() for k in ("Wa", "ba", "P", "Pg", "Wl", "Wg")}
    for k in ("Wa", "ba", "P", "Pg") + (("Wl", "Wg") if train_ll else ()):
        params[k].requires_grad_(True)
    st = GraphedHeadStep(params, cfg, B=s.B, N=s.N, C=s.C, m=s.m, n_slots=len(inputs))
    for i, (t, sc, lb) in enumerate(inputs):
        st.load(i, t, sc, lb)
    torch.cuda.synchronize()
    st.capture()
    return st


def make_inputs(s, n):
    g = torch.Generator(device="cuda").manual_seed(7)
    out = []
    for _ in range(n):
        tokens = torch.randn(s.B, 1 + s.N, s.Din, device="cuda", generator=g)
        scores = (torch.argsort(torch.rand(s.B, s.N, device="cuda", generator=g), dim=1) + 1).float() / (s.N * (s.N + 1) // 2)
        labels = torch.randint(0, s.C, (s.B,), device="cuda", generator=g)
        out.append((tokens, scores, labels))
    return out


def time_replays(fn, window, warm=20):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    n = 50
    while True:
        e[0].record()
        for _ in range(n):
            fn()
        e[1].record()
        torch.cuda.synchronize()
        ms = e[0].elapsed_time(e[1])
        if ms >= 1e3 * window:
            return 1e3 * ms / n
        n = int(n * max(2.0, 1.2 * 1e3 * window / max(ms, 1e-3)))


def time_kernel(st, window, per_graph=100):
    from protopformer_b200 import _lib
    f, s = st.fused, st
    B, C = s.B, s.C
    P, Pg = s.p["P"].shape[0], s.p["Pg"].shape[0]
    gc = float(s.cfg.global_coe)

    def launch():
        _lib.call("pph_last_layer_wgrad", f.dlogits, None, None, f.act_l, f.act_g, B, P, Pg, C, gc, s.grads["Wl"], s.grads["Wg"])

    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(3):
            launch()
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, capture_error_mode="thread_local"):
        for _ in range(per_graph):
            launch()
    return time_replays(g.replay, window, warm=3) / per_graph


def timeline(st, reps=6):
    from torch.profiler import ProfilerActivity, profile
    for i in range(3):
        st.run(i % len(st.graphs))
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for i in range(reps):
            st.run(i % len(st.graphs))
        torch.cuda.synchronize()
    evs = sorted((e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA), key=lambda e: e.time_range.start)
    per = len(evs) // reps
    one = evs[(reps - 2) * per:(reps - 1) * per]
    t0 = one[0].time_range.start
    lines = [f"# {per} device activities per replay (trainable last layers)"]
    lines += [f"{e.time_range.start - t0:9.2f} us  +{e.time_range.end - e.time_range.start:8.2f} us  {e.name[:90]}" for e in one]
    lines.append(f"# next replay starts at {evs[(reps - 1) * per].time_range.start - t0:.2f} us")
    return lines


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--workloads", default=",".join(WORKLOADS))
    ap.add_argument("--rounds", type=int, default=3, help="frozen / trainable alternations (>= 3)")
    ap.add_argument("--window", type=float, default=0.25, help="seconds of replays per timed arm (>= 0.2)")
    ap.add_argument("--out", default=None, help="also write the report to this file")
    ap.add_argument("--timeline", action="store_true", help="torch.profiler kernel list of one trainable replay at cub_b64")
    ap.add_argument("--dry-run", action="store_true", help="workloads and shape arithmetic only (no device)")
    args = ap.parse_args()
    names = [w for w in args.workloads.split(",") if w]
    for w in names:
        if w not in WORKLOADS:
            ap.error(f"unknown workload {w!r} (known: {', '.join(WORKLOADS)})")
    if args.rounds < 3:
        ap.error("--rounds must be at least 3")
    if args.window < 0.2:
        ap.error("--window must be at least 0.2 s")
    report = []

    def emit(line):
        print(line, flush=True)
        report.append(line)

    if not args.dry_run:
        assert torch.cuda.is_available(), "last_layer_grad_bench.py measures on a CUDA device (use --dry-run without one)"
        name, power = gpu_identity()
        emit(f"# GPU: {name}; power.limit, clocks.max.sm: {power}")
    for w in names:
        s, mode = WORKLOADS[w]
        nbytes, flops = kernel_bytes_flops(s)
        ns = n_slots(s)
        foot = ns * slot_read_bytes(s)
        res = {"workload": w, "B": s.B, "C": s.C, "P": s.P, "Pg": s.Pg, "mode": mode, "kernel_bytes": nbytes,
               "kernel_flops": flops, "slots": ns, "slot_read_MB": round(foot / 2 ** 20, 1),
               "slots_exceed_L2": foot > L2_BYTES}
        if args.dry_run:
            emit(json.dumps(res))
            continue
        inputs = make_inputs(s, ns)
        arms = {"frozen": make_step(s, mode, False, inputs), "trainable": make_step(s, mode, True, inputs)}
        res["launches"] = {k: v.kernel_launches_per_step for k, v in arms.items()}
        t = {"frozen": [], "trainable": []}
        for _ in range(args.rounds):
            for arm, st in arms.items():
                k = [0]

                def one(st=st, k=k):
                    st.run(k[0] % ns)
                    k[0] += 1
                t[arm].append(time_replays(one, args.window))
        res["us_per_step"] = {a: [round(x, 2) for x in v] for a, v in t.items()}
        med = {a: sorted(v)[len(v) // 2] for a, v in t.items()}
        res["median_us"] = {a: round(v, 2) for a, v in med.items()}
        res["trainable_minus_frozen_us"] = round(med["trainable"] - med["frozen"], 2)
        kus = time_kernel(arms["trainable"], args.window)
        res["wgrad_kernel_us"] = round(kus, 3)
        res["wgrad_GBps"] = round(nbytes / (kus * 1e-6) / 1e9, 1)
        res["wgrad_GFLOPps"] = round(flops / (kus * 1e-6) / 1e9, 1)
        emit(f"{w}: frozen {med['frozen']:.2f} us/step, trainable {med['trainable']:.2f} us/step "
             f"(difference {res['trainable_minus_frozen_us']:+.2f} us; rounds {res['us_per_step']}); "
             f"pph_last_layer_wgrad alone {kus:.2f} us = {res['wgrad_GBps']} GB/s, {res['wgrad_GFLOPps']} GFLOP/s")
        emit(json.dumps(res))
        if args.timeline and w == "cub_b64":
            for line in timeline(arms["trainable"]):
                emit(line)
        del arms, inputs
        torch.cuda.empty_cache()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(report) + "\n")


if __name__ == "__main__":
    main()
