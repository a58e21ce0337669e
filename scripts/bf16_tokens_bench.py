"""fp32 against bf16 backbone tokens: the graphed step, device-resident and end to end from pinned host memory.

    python scripts/bf16_tokens_bench.py [--workloads cub_b64,cars_b64_bf16,dogs_b256_eval] [--rounds 3] [--window 0.3]
                                        [--e2e-steps 2000] [--out FILE] [--dry-run]

Both arms get the same values: the bf16 arm holds bf16 tokens, the fp32 arm the same tokens widened to fp32, so their
results are asserted bit-identical (dtokens: the fp32 arm's rounded to bf16) before anything is timed.

Device-resident: per workload, the two graphed steps (GraphedHeadStep(token_dtype=...)) are alternated --rounds times in
ONE process; each arm is timed with CUDA events over >= --window seconds of replays that rotate over input slots whose token
rows read by the step add up to more than the 126 MB L2 of a B200 in the fp32 arm.

End to end (cub_b64, training, one GPU): what bench.py's e2e leg does, once per token dtype, alternated --rounds times:
a ring of pinned host batches, one graph per iteration = the step of one slot || the selection-first transfer of the next
batch into the other slot (pph_gather_rows_host[_bf16tok]), loss stored to pinned host memory by the kernel that completes it.
Reported: images/s over --e2e-steps steps and the bytes that cross the bus per step.  Where eight GPUs exist the same loop
also runs as eight processes, one per GPU, started together for every timed arm (a barrier before each): the aggregate rate
of eight pipelines that share the host->device path -- the limit DESIGN.md section 6 names for the 8-GPU end-to-end figure.
These eight pipelines do not exchange gradients (bench.py's harness adds the in-graph exchange, ~10 us per step).

The GPU name and power limit are read in the same call.  --dry-run prints the workloads and byte counts without a device.
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
WORKLOADS = {          # name -> (shape, similarity mode, train): bench.py's workloads of these names
    "cub_b64": (synth.SHAPES["cub_b64"], "fp32", True),
    "cars_b64_bf16": (synth.SHAPES["cars_b64"], "bf16", True),
    "dogs_b256_eval": (synth.SHAPES["dogs_b256"], "fp32", False),
}
DTYPES = {"fp32": torch.float32, "bf16": torch.bfloat16}


def row_bytes(s, dt):
    """Input bytes one step reads (and load_host moves): CLS + K selected token rows per image, scores, labels."""
    return (2 if dt == torch.bfloat16 else 4) * s.B * (s.K + 1) * s.Din + 4 * s.B * s.N + 8 * s.B


def n_slots(s, cap=64):
    return max(2, min(cap, math.ceil(1.5 * L2_BYTES / row_bytes(s, torch.float32))))


def gpu_identity():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError) as exc:
        q = f"unknown ({type(exc).__name__})"
    return name, q


def make_batches(s, n, device):
    g = torch.Generator(device="cpu").manual_seed(11)
    out = []
    for _ in range(n):
        tokens = torch.randn(s.B, 1 + s.N, s.Din, generator=g).to(torch.bfloat16)     # bf16-exact values in both arms
        scores = (torch.argsort(torch.rand(s.B, s.N, generator=g), dim=1) + 1).float() / (s.N * (s.N + 1) // 2)
        labels = torch.randint(0, s.C, (s.B,), generator=g)
        out.append({"tokens_bf16": tokens.to(device), "scores": scores.to(device), "labels": labels.to(device)})
    return out


def make_step(s, mode, train, dt, n):
    from protopformer_b200 import ops
    from protopformer_b200.graph import GraphedHeadStep
    case = synth.make_case(s.with_batch(1), seed=1)            # weights only (they do not depend on B)
    cfg = ops.HeadConfig(K=s.K, global_coe=s.global_coe, mode=mode, ppc_cov_thresh=s.ppc_cov_thresh,
                         ppc_mean_thresh=s.ppc_mean_thresh)
    params = {k: case[k].cuda() for k in ("Wa", "ba", "P", "Pg", "Wl", "Wg")}
    for k in ("Wa", "ba", "P", "Pg"):
        params[k].requires_grad_(train)
    return GraphedHeadStep(params, cfg, B=s.B, N=s.N, C=s.C, m=s.m, n_slots=n, train=train, token_dtype=dt), params


def tokens_of(b, dt):
    return b["tokens_bf16"] if dt == torch.bfloat16 else b["tokens_bf16"].float()


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


def check_identical(arms, params, train):
    """Both arms on slot 0 (the same batch): every output bit-identical, dtokens up to the one bf16 rounding."""
    for st in arms.values():
        st.run(0)
    torch.cuda.synchronize()
    a, b = arms["bf16"].fused, arms["fp32"].fused
    assert torch.equal(a.losses, b.losses) and torch.equal(a.logits, b.logits)
    if train:
        assert torch.equal(a.dtokens, b.dtokens.to(torch.bfloat16))
        for k in ("P", "Pg", "Wa", "ba"):
            assert torch.equal(params["bf16"][k].grad, params["fp32"][k].grad), k


def device_resident(w, rounds, window):
    s, mode, train = WORKLOADS[w]
    ns = n_slots(s)
    batches = make_batches(s, ns, "cuda")
    arms, params = {}, {}
    for name, dt in DTYPES.items():
        st, p = make_step(s, mode, train, dt, ns)
        for i, b in enumerate(batches):
            st.load(i, tokens_of(b, dt), b["scores"], b["labels"])
        torch.cuda.synchronize()
        st.capture()
        arms[name], params[name] = st, p
    check_identical(arms, params, train)
    t = {k: [] for k in arms}
    for _ in range(rounds):
        for name, st in arms.items():
            k = [0]

            def one(st=st, k=k):
                st.run(k[0] % ns)
                k[0] += 1
            t[name].append(time_replays(one, window))
    med = {a: sorted(v)[len(v) // 2] for a, v in t.items()}
    res = {"workload": w, "leg": "device_resident", "B": s.B, "train": train, "mode": mode, "slots": ns,
           "launches": {k: v.kernel_launches_per_step for k, v in arms.items()},
           "us_per_step": {a: [round(x, 2) for x in v] for a, v in t.items()},
           "median_us": {a: round(v, 2) for a, v in med.items()},
           "bf16_minus_fp32_us": round(med["bf16"] - med["fp32"], 2),
           "step_read_bytes": {a: row_bytes(s, dt) for a, dt in DTYPES.items()}}
    del arms, params, batches
    torch.cuda.empty_cache()
    return res


def e2e(rounds, steps, nbuf=8, barrier=None):
    """Pinned-host end to end at cub_b64 (bench.py's e2e leg on one GPU), both token dtypes alternated."""
    s, mode, train = WORKLOADS["cub_b64"]
    sync = barrier.wait if barrier is not None else (lambda: None)
    batches = make_batches(s, nbuf, "cpu")
    runs = {}
    for name, dt in DTYPES.items():
        st, _ = make_step(s, mode, train, dt, 2)
        host = [{"tokens": tokens_of(b, dt).pin_memory(), "scores": b["scores"].pin_memory(),
                 "labels": b["labels"].pin_memory()} for b in batches]
        st.load(0, host[0]["tokens"], host[0]["scores"], host[0]["labels"])
        torch.cuda.synchronize()
        st.capture()
        st.capture_host_pipeline()
        pair = {(sl, j): st.capture_host_overlapped(sl, host[j]["tokens"], host[j]["scores"], host[j]["labels"])
                for sl in range(2) for j in range(nbuf) if j % 2 != sl}
        runs[name] = (st, host, pair)

    def loop(name, n):
        st, host, pair = runs[name]
        b0 = host[0]
        st.load_host(0, b0["tokens"], b0["scores"], b0["labels"])
        for i in range(n):
            pair[(i % 2, (i + 1) % nbuf)].replay()
        torch.cuda.synchronize()
        return st.loss_host[(n - 1) % 2].clone()

    last = {}
    t = {k: [] for k in runs}
    for _ in range(rounds):
        for name in runs:
            loop(name, 30)
            sync()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            last[name] = loop(name, steps)
            e1.record()
            torch.cuda.synchronize()
            t[name].append(s.B * steps / (e0.elapsed_time(e1) * 1e-3))
    assert torch.equal(last["bf16"], last["fp32"]), (last["bf16"], last["fp32"])
    med = {a: sorted(v)[len(v) // 2] for a, v in t.items()}
    return {"workload": "cub_b64", "leg": "e2e_pinned_host", "gpus": 1, "us_per_step": {
                a: [round(1e6 * s.B / x, 2) for x in v] for a, v in t.items()}, "steps": steps, "ring": nbuf,
            "images_per_s": {a: [round(x) for x in v] for a, v in t.items()},
            "median_images_per_s": {a: round(v) for a, v in med.items()},
            "h2d_bytes_per_step": {a: row_bytes(s, dt) for a, dt in DTYPES.items()},
            "launches": {k: v[0].kernel_launches_per_step for k, v in runs.items()}}


def _rank_e2e(rank, rounds, steps, barrier, q):
    torch.cuda.set_device(rank)
    try:
        q.put((rank, e2e(rounds, steps, barrier=barrier)))
    except Exception as exc:          # report, and release the others
        barrier.abort()
        q.put((rank, repr(exc)))


def e2e_multi(n, rounds, steps):
    """n pipelines, one process per GPU, every timed arm started behind one barrier: aggregate images/s = sum of ranks."""
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    barrier, q = ctx.Barrier(n), ctx.Queue()
    procs = [ctx.Process(target=_rank_e2e, args=(r, rounds, steps, barrier, q)) for r in range(n)]
    for p in procs:
        p.start()
    res = dict(q.get() for _ in procs)
    for p in procs:
        p.join()
    bad = {r: v for r, v in res.items() if not isinstance(v, dict)}
    assert not bad, bad
    agg = {a: [sum(res[r]["images_per_s"][a][i] for r in res) for i in range(rounds)] for a in DTYPES}
    med = {a: sorted(v)[len(v) // 2] for a, v in agg.items()}
    return {"workload": "cub_b64", "leg": "e2e_pinned_host", "gpus": n, "exchange": "none (independent pipelines)",
            "aggregate_images_per_s": agg, "median_aggregate_images_per_s": med,
            "per_rank_median_us_per_step": {a: [sorted(res[r]["us_per_step"][a])[rounds // 2] for r in sorted(res)]
                                            for a in DTYPES},
            "h2d_bytes_per_step_per_rank": res[0]["h2d_bytes_per_step"]}


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--workloads", default=",".join(WORKLOADS))
    ap.add_argument("--rounds", type=int, default=3, help="fp32 / bf16 alternations (>= 3)")
    ap.add_argument("--window", type=float, default=0.3, help="seconds of replays per timed device-resident arm (>= 0.2)")
    ap.add_argument("--e2e-steps", type=int, default=2000, help="steps per timed end-to-end arm (0: skip the leg)")
    ap.add_argument("--out", default=None, help="also write the report to this file")
    ap.add_argument("--dry-run", action="store_true", help="workloads and byte counts only (no device)")
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

    if args.dry_run:
        for w in names:
            s = WORKLOADS[w][0]
            emit(json.dumps({"workload": w, "slots": n_slots(s),
                             "step_read_bytes": {a: row_bytes(s, dt) for a, dt in DTYPES.items()}}))
        return
    assert torch.cuda.is_available(), "bf16_tokens_bench.py measures on a CUDA device (use --dry-run without one)"
    name, power = gpu_identity()
    emit(f"# GPU: {name} x {torch.cuda.device_count()}; power.limit, clocks.max.sm: {power}")
    for w in names:
        r = device_resident(w, args.rounds, args.window)
        emit(f"{w}: fp32 tokens {r['median_us']['fp32']:.2f} us/step, bf16 tokens {r['median_us']['bf16']:.2f} us/step "
             f"(difference {r['bf16_minus_fp32_us']:+.2f} us; rounds {r['us_per_step']})")
        emit(json.dumps(r))
    if args.e2e_steps > 0:
        r = e2e(args.rounds, args.e2e_steps)
        emit(f"e2e cub_b64, 1 GPU: fp32 tokens {r['median_images_per_s']['fp32']} img/s, bf16 tokens "
             f"{r['median_images_per_s']['bf16']} img/s; H2D bytes/step {r['h2d_bytes_per_step']}")
        emit(json.dumps(r))
    if args.e2e_steps > 0 and torch.cuda.device_count() >= 8:
        r = e2e_multi(8, args.rounds, args.e2e_steps)
        emit(f"e2e cub_b64, 8 GPUs, no exchange: fp32 tokens {r['median_aggregate_images_per_s']['fp32']} img/s, bf16 tokens "
             f"{r['median_aggregate_images_per_s']['bf16']} img/s (aggregate)")
        emit(json.dumps(r))
    elif args.e2e_steps > 0:
        emit(f"# e2e at 8 GPUs: not measured ({torch.cuda.device_count()} GPU(s) on this machine)")
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(report) + "\n")


if __name__ == "__main__":
    main()
