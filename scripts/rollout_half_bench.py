"""Attention rollout on half-precision maps: the bf16 / fp16 twins against the fp32 kernel and against widening first.

    python scripts/rollout_half_bench.py [--shapes "11,64,3,197;..."] [--dtypes bf16,fp16] [--rounds 5] [--reps 10]
                                         [--out FILE] [--dry-run]

Per shape (L, B, H, T) and half dtype, the arms are alternated --rounds times in ONE process:
  fp32  fp32 maps through pph_rollout_scores;
  cast  half maps widened to an fp32 copy ([m.float() for m in maps]) and then pph_rollout_scores, both timed;
  twin  half maps through pph_rollout_scores_{bf16,f16}attn, read as they are;
and, to separate the kernel's cost on half-precision VALUES from the cost of reading them, a fourth arm:
  wide  the fp32 widening of the half maps, made before timing, through pph_rollout_scores (the kernel time of "cast").
The arms are timed with CUDA events over --reps calls; every shape's maps exceed the 126 MB L2 of a B200 in every arm.
Reported per arm: median us per call over the rounds, the bytes the arm moves from and to the maps (fp32: 4 B per map
element read; cast: 2 B read + 4 B written + 4 B read; twin: 2 B read), that over the time, and the rise of peak
allocated memory during one call with a preallocated workspace.  The half arms are asserted bit-identical before timing.
The GPU name and power limit are read in the same call.  --dry-run prints the shapes and byte counts without a device.
"""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

SHAPES = [(11, 64, 3, 197), (11, 256, 3, 197), (11, 64, 6, 197), (24, 64, 4, 196), (11, 256, 6, 197)]
DTYPES = {"bf16": torch.bfloat16, "fp16": torch.float16}
ARM_BYTES_PER_ELEMENT = {"fp32": 4, "cast": 2 + 4 + 4, "twin": 2, "wide": 4}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--shapes", default=";".join(",".join(map(str, s)) for s in SHAPES))
    ap.add_argument("--dtypes", default="bf16,fp16")
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default=None)
    ap.add_argument("--dry-run", action="store_true")
    a = ap.parse_args()
    shapes = [tuple(int(x) for x in s.split(",")) for s in a.shapes.split(";")]
    dtypes = a.dtypes.split(",")
    out = open(a.out, "w") if a.out else None

    def emit(line):
        print(line, flush=True)
        if out:
            out.write(line + "\n")
            out.flush()

    if a.dry_run:
        for L, B, H, T in shapes:
            n = L * B * H * T * T
            emit(json.dumps({"L": L, "B": B, "H": H, "T": T,
                             "bytes": {k: n * v for k, v in ARM_BYTES_PER_ELEMENT.items()}}))
        return
    if not torch.cuda.is_available():
        raise SystemExit("rollout_half_bench.py measures on a CUDA device; none is available")
    from protopformer_b200 import ops
    dev = torch.device("cuda:0")
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True)
        power = q.stdout.strip() or "unknown"
    except OSError:
        power = "unknown"
    emit(f"# GPU: {torch.cuda.get_device_name(0)}; power.limit, clocks.max.sm: {power}")

    for L, B, H, T in shapes:
        g = torch.Generator(device=dev).manual_seed(0)
        maps32 = [torch.softmax(2.0 * torch.randn(B, H, T, T, device=dev, generator=g), dim=-1) for _ in range(L)]
        n = L * B * H * T * T
        k = int(T * T * 0.9)
        ws = ops.rollout_workspace(L, B, T, k, dev)
        for dname in dtypes:
            maps16 = [m.to(DTYPES[dname]) for m in maps32]
            wide = [m.float() for m in maps16]
            arms = {
                "fp32": lambda: ops.rollout_scores(maps32, workspace=ws),
                "cast": lambda: ops.rollout_scores([m.float() for m in maps16], workspace=ws),
                "twin": lambda: ops.rollout_scores(maps16, workspace=ws),
                "wide": lambda: ops.rollout_scores(wide, workspace=ws),
            }
            assert torch.equal(arms["cast"](), arms["twin"]())
            for f in arms.values():                     # warm-up: modules loaded, allocator blocks cached
                f()
            peak = {}
            for name, f in arms.items():
                torch.cuda.synchronize()
                torch.cuda.reset_peak_memory_stats()
                base = torch.cuda.memory_allocated()
                f()
                torch.cuda.synchronize()
                peak[name] = torch.cuda.max_memory_allocated() - base
            us = {name: [] for name in arms}
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            for _ in range(a.rounds):
                for name, f in arms.items():
                    torch.cuda.synchronize()
                    e0.record()
                    for _ in range(a.reps):
                        f()
                    e1.record()
                    torch.cuda.synchronize()
                    us[name].append(round(1e3 * e0.elapsed_time(e1) / a.reps, 1))
            med = {name: sorted(v)[len(v) // 2] for name, v in us.items()}
            nbytes = {name: n * ARM_BYTES_PER_ELEMENT[name] for name in arms}
            row = {"L": L, "B": B, "H": H, "T": T, "half": dname, "median_us": med, "us_rounds": us,
                   "bytes": nbytes, "gbs": {name: round(nbytes[name] / med[name] / 1e3, 1) for name in arms},
                   "peak_alloc_rise_bytes": peak,
                   "twin_vs_cast": round(med["cast"] / med["twin"], 2), "twin_vs_fp32": round(med["fp32"] / med["twin"], 2)}
            emit(f"({L},{B},{H},{T}) {dname}: fp32 {med['fp32']} us, cast {med['cast']} us, twin {med['twin']} us, "
                 f"wide {med['wide']} us")
            emit(json.dumps(row))
            del maps16, wide
        del maps32, ws
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
