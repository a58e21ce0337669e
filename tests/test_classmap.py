"""Class-row activation maps on the original token grid (SURVEY.md §8(f) next #4, eval_interpretability.py:195-225).

The consumer is script code (argparse + dataset loading at import time), so it cannot be imported; its class-map lines
are plain tensor code, though, and `oracle/ref_script_lines.py` EXECUTES them as written (:196-202 gather, :213-225
scatter).  Pin: `tests/golden/classmap_*.npz` hold what those lines return on seeded inputs
(`tests/golden/make_classmap_golden.py`); the oracle's restatement must reproduce them bit-exactly (CPU suite, plus a
live run on fresh seeds where /root/reference exists); the CUDA kernel is fed the REFERENCE's own `proto_acts` from the
head fixtures through that restatement (GPU tests)."""
import numpy as np
import pytest
import torch

from oracle import protohead_oracle as O
from tests.util import load_golden, rel_close, max_rel


def _classmap_inputs(name):
    import importlib.util
    import os
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "make_classmap_golden.py")
    spec = importlib.util.spec_from_file_location("make_classmap_golden", path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod, mod.CASES[name]


@pytest.mark.parametrize("name", ["classmap_small", "classmap_cub_b4", "classmap_cars_b3"])
def test_oracle_reproduces_the_reference_scripts_own_lines(name):
    """Fixture = output of eval_interpretability.py:196-202 + :213-225 executed as written."""
    import os
    from protopformer_b200 import synth
    mod, (B, C, K, N, seed) = _classmap_inputs(name)
    proto_acts, scores, targets = mod.make_inputs(B, C, K, N, seed)
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", name + ".npz"))
    assert abs(synth.checksum(proto_acts) - float(g["chk_acts"])) <= 1e-9 * abs(float(g["chk_acts"]))      # same RNG stream
    assert np.array_equal(targets.numpy(), g["targets"])
    idx = O.select_tokens(scores, K)
    got = O.class_activation_maps(proto_acts.flatten(2), idx, targets, 10, N)
    assert np.array_equal(got.numpy().reshape(g["maps"].shape), g["maps"])


def test_oracle_matches_the_live_reference_lines_on_fresh_seeds():
    from oracle import ref_script_lines as S
    if not S.available():
        pytest.skip("/root/reference is absent (GPU box): the frozen fixtures above cover this row")
    mod, _ = _classmap_inputs("classmap_small")
    for seed, (B, C, K, N) in enumerate([(5, 9, 16, 36), (2, 30, 49, 196), (3, 4, 4, 9)], start=40):
        proto_acts, scores, targets = mod.make_inputs(B, C, K, N, seed)
        want = S.class_maps_by_reference_lines(proto_acts, scores, targets, K, 10)
        got = O.class_activation_maps(proto_acts.flatten(2), O.select_tokens(scores, K), targets, 10, N)
        assert np.array_equal(got.numpy().reshape(want.shape), want)


def test_oracle_gather_scatter_matches_index_loop():
    g = torch.Generator().manual_seed(0)
    B, P, K, m, N = 3, 12, 4, 3, 9
    act = torch.rand(B, P, K, generator=g)
    idx = torch.stack([torch.randperm(N, generator=g)[:K].sort()[0] for _ in range(B)])
    labels = torch.tensor([0, 3, 2])
    got = O.class_activation_maps(act, idx, labels, m, N)
    want = torch.zeros(B, m, N)
    for b in range(B):
        for q in range(m):
            for k in range(K):
                want[b, q, idx[b, k]] = act[b, int(labels[b]) * m + q, k]
    assert torch.equal(got, want)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["tiny_s1", "tiny_s2_linear", "small_s1", "small_s3_matched"])
def test_class_maps_match_reference_proto_acts(name):
    from protopformer_b200 import ops
    shape, case, g, fn = load_golden(name)
    dev = torch.device("cuda:0")
    d = {k: v.to(dev) for k, v in case.items()}
    cfg = ops.HeadConfig(K=shape.K, global_coe=shape.global_coe, act_fn=fn, mode="fp32_fma")
    idx = ops.select_topk(d["scores"], shape.K)
    tf = ops.addon(d["tokens"], idx, d["Wa"], d["ba"], False)
    maps = ops.class_activation_maps(cfg, tf, d["P"], d["labels"], shape.m, shape.N)
    side = int(round(shape.N ** 0.5))
    assert maps.shape == (shape.B, shape.m, side, side)
    # the reference's own push_forward activations (fixture), gathered / scattered as eval_interpretability.py does
    want = O.class_activation_maps(torch.from_numpy(g["act_map"]), torch.from_numpy(g["idx"]).long(), case["labels"],
                                   shape.m, shape.N)
    tol = 1e-3 if "matched" in name else 1e-4
    assert rel_close(maps.flatten(2).cpu(), want, tol), max_rel(maps.flatten(2).cpu(), want)
    assert int((maps.flatten(2) != 0).sum(-1).max()) <= shape.K          # pruned tokens stay exactly zero


@pytest.mark.gpu
def test_class_maps_full_size_against_materialised_map():
    from protopformer_b200 import synth
    from protopformer_b200 import ops
    shape = synth.SHAPES["cub_b64"].with_batch(16)
    case = synth.make_case(shape, seed=2)
    dev = torch.device("cuda:0")
    d = {k: v.to(dev) for k, v in case.items()}
    cfg = ops.HeadConfig(K=shape.K, mode="fp32_fma")
    idx = ops.select_topk(d["scores"], shape.K)
    tf = ops.addon(d["tokens"], idx, d["Wa"], d["ba"], False)
    maps = ops.class_activation_maps(cfg, tf, d["P"], d["labels"], shape.m, shape.N)
    _, act_map = ops.materialize_maps(cfg, tf, d["P"], d["Pg"])                    # (B,P,K) from the FP32-FMA kernel
    want = O.class_activation_maps(act_map.cpu(), idx.cpu().long(), case["labels"], shape.m, shape.N)
    assert rel_close(maps.flatten(2).cpu(), want, 1e-4), max_rel(maps.flatten(2).cpu(), want)
