"""Outputs of the attention rollout and of the class-row activation maps on seeded inputs, and a bitwise comparison of
two such sets: the check that a change around either kernel leaves its results as they were.

    python scripts/rollout_classmap_outputs.py --out A.pt [--root DIR]
    python scripts/rollout_classmap_outputs.py --compare A.pt B.pt

--root imports protopformer_b200 from another checkout (default: the one holding this script), so two builds run the
same inputs, one process each.  Rollout: the DeiT-Ti shape (L = 11, H = 3, T = 197, B = 64), fp32 / bf16 / fp16 maps,
discard ratios 0.9 (the reference's) and 0.2 (entry lists too long for the staged chain kernel), scores alone and with
the fused top-81.  Class maps: the CUB shape at B = 64.  --compare exits with 1 if any tensor differs in any bit.
"""
import argparse
import os
import sys

import torch


def outputs():
    from protopformer_b200 import ops, synth
    dev = torch.device("cuda:0")
    out = {}
    g = torch.Generator(device=dev).manual_seed(0)
    L, B, H, T = 11, 64, 3, 197
    maps = [torch.softmax(2.0 * torch.randn(B, H, T, T, device=dev, generator=g), dim=-1) for _ in range(L)]
    for name, dt in (("fp32", torch.float32), ("bf16", torch.bfloat16), ("fp16", torch.float16)):
        m = [a.to(dt) for a in maps]
        for ratio in (0.9, 0.2):
            out[f"rollout_{name}_{ratio}"] = ops.rollout_scores(m, ratio)
            out[f"rollout_{name}_{ratio}_top81_scores"], out[f"rollout_{name}_{ratio}_top81_idx"] = \
                ops.rollout_scores(m, ratio, topk=81)
    shape = synth.SHAPES["cub_b64"]
    case = {k: v.to(dev) for k, v in synth.make_case(shape, seed=1).items()}
    cfg = ops.HeadConfig(K=shape.K, mode="fp32_fma")
    idx = ops.select_topk(case["scores"], shape.K)
    tf = ops.addon(case["tokens"], idx, case["Wa"], case["ba"], False)
    out["class_maps"] = ops.class_activation_maps(cfg, tf, case["P"], case["labels"], shape.m, shape.N)
    torch.cuda.synchronize()
    return {k: v.cpu() for k, v in out.items()}


def compare(a_path, b_path) -> bool:
    a, b = torch.load(a_path), torch.load(b_path)
    same = set(a) == set(b)
    if not same:
        print("different keys:", sorted(set(a) ^ set(b)))
    for k in sorted(set(a) & set(b)):
        eq = a[k].dtype == b[k].dtype and a[k].shape == b[k].shape and torch.equal(a[k], b[k])
        diff = 0.0 if eq else (a[k].double() - b[k].double()).abs().max().item()
        print(f"{k:34s} {tuple(a[k].shape)} {'bit-identical' if eq else f'DIFFERS (max abs {diff:.3e})'}")
        same &= eq
    return same


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out")
    ap.add_argument("--root", default=os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    ap.add_argument("--compare", nargs=2, metavar=("A", "B"))
    a = ap.parse_args()
    if a.compare:
        sys.exit(0 if compare(*a.compare) else 1)
    if not a.out:
        ap.error("--out or --compare")
    sys.path.insert(0, os.path.abspath(a.root))
    with torch.no_grad():
        res = outputs()
    torch.save(res, a.out)
    print(f"{len(res)} tensors -> {a.out}")


if __name__ == "__main__":
    main()
