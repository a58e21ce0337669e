"""The fused (autograd-free, CUDA-graph-captured) training step against the reference fixtures and the oracle:
same entry points as the modular path, so this mainly checks the sequencing, the accumulate-mode PPC backward, the
loss tail kernel and graph replay determinism."""
import numpy as np
import pytest
import torch

from oracle import protohead_oracle as O
from protopformer_b200 import synth
from tests.util import GOLDEN_CASES, load_golden, norm_rel, rel_close

pytestmark = pytest.mark.gpu


def _make(shape, case, mode, n_slots=1, train=True, fused=True):
    from protopformer_b200 import ops
    from protopformer_b200.graph import GraphedHeadStep
    dev = torch.device("cuda:0")
    params = {k: case[k].to(dev).clone() for k in ("Wa", "ba", "P", "Pg", "Wl", "Wg")}
    for k in ("Wa", "ba", "P", "Pg"):
        params[k].requires_grad_(train)
    cfg = ops.HeadConfig(K=shape.K, global_coe=shape.global_coe, mode=mode, ppc_cov_thresh=shape.ppc_cov_thresh,
                         ppc_mean_thresh=shape.ppc_mean_thresh)
    step = GraphedHeadStep(params, cfg, B=shape.B, N=shape.N, C=shape.C, m=shape.m, n_slots=n_slots, train=train,
                           fused=fused)
    for i in range(n_slots):
        step.load(i, case["tokens"], case["scores"], case["labels"])
    torch.cuda.synchronize()
    step.capture()
    return step, params


@pytest.mark.parametrize("name,mode", [("cub_b8_s1", "fp32"), ("cub_b8_s1", "bf16"), ("cars_b4_s1", "fp32"),
                                       ("dogs_b4_s1", "fp32"), ("small_s1", "fp32_fma"), ("tiny_s1", "fp32_fma"),
                                       ("cub_b8_s2_matched", "fp32")])
def test_fused_graphed_step_matches_reference(name, mode):
    shape, case, g, fn = load_golden(name)
    step, params = _make(shape, case, mode)
    step.run(0)
    step.run(0)                      # replay twice: counters / accumulate buffers must self-reset
    torch.cuda.synchronize()
    f = step.fused
    tol = 5e-3 if mode == "bf16" else (1e-3 if "matched" in name else 1e-4)
    assert np.array_equal(f.idx32.cpu().numpy(), g["idx"])
    assert rel_close(f.logits.cpu(), g["logits_train"], tol)
    losses = f.losses.cpu()
    assert rel_close(losses[0], g["loss"], tol) and rel_close(losses[1], g["ce"], tol)
    ptol = 1e-3 if "matched" in name else 1e-4
    assert rel_close(losses[2], g["ppc_cov"], ptol) and rel_close(losses[3], g["ppc_mean"], ptol)
    ref = O.head_train_step(case, shape, fn=fn, route=f.argmin.cpu().long())
    gt = 5e-2 if mode == "bf16" else 5 * tol
    got = dict(g_tokens=f.dtokens, g_P=params["P"].grad, g_Pg=params["Pg"].grad, g_Wa=params["Wa"].grad,
               g_ba=params["ba"].grad)
    for k, v in got.items():
        assert norm_rel(v.cpu().reshape(ref[k].shape), ref[k]) < gt, (k, norm_rel(v.cpu().reshape(ref[k].shape), ref[k]))


def test_fused_step_is_bit_reproducible_and_matches_modular_path():
    shape = synth.SHAPES["cub_b64"]
    case = synth.make_case(shape, seed=4)
    step, params = _make(shape, case, "fp32")
    step.run(0)
    torch.cuda.synchronize()
    a = {k: params[k].grad.clone() for k in ("P", "Pg")}
    la, dta = step.fused.losses.clone(), step.fused.dtokens.clone()
    step.run(0)
    torch.cuda.synchronize()
    # every reduction of the fused step is ordered except the split-K add-on weight gradient and the PPC rows of
    # images that share a label (both atomics)
    assert torch.equal(a["Pg"], params["Pg"].grad)
    assert norm_rel(a["P"], params["P"].grad) < 1e-6
    assert torch.equal(la, step.fused.losses) and torch.equal(dta, step.fused.dtokens)
    mod, mparams = _make(shape, case, "fp32", fused=False)
    mod.run(0)
    torch.cuda.synchronize()
    assert rel_close(mod.loss[0].cpu(), la[0].cpu(), 1e-6)
    # two different kernel sequences for the same gradients, each within 1e-4 of the float64 oracle on its own
    # (tests/test_gpu_parity.py, tests/test_step2_gpu.py): 2e-4 between them
    for k in ("P", "Pg", "Wa", "ba"):
        assert norm_rel(mparams[k].grad.cpu(), params[k].grad.cpu()) < 2e-4, k
    assert norm_rel(mod.dtokens[0].cpu(), dta.cpu()) < 2e-4


def test_fused_eval_step():
    shape, case, g, fn = load_golden("cub_b8_s1")
    step, _ = _make(shape, case, "fp32", train=False)
    step.run(0)
    torch.cuda.synchronize()
    assert rel_close(step.fused.logits.cpu(), g["logits"], 1e-4)
