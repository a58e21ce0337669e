"""Class-sum form of the last layers (pph_last_layer_pattern + the class-sum LL role of pph_head_mid).

The step checks on the device, every step, whether Wl and Wg still hold the class-connection pattern of
set_last_layer_incorrect_connection; only then does pph_head_mid take the O(B P) class-sum form.  Held here: the verdict
itself, both forms of the step against the CPU oracle (tolerances of tests/test_step2_gpu.py, fp32 mode), the switch
between them inside ONE captured graph when the weights change through .data, and bit-identical replays."""
import pytest
import torch

from oracle import protohead_oracle as O
from protopformer_b200 import synth
from tests.util import norm_rel, rel_close

pytestmark = pytest.mark.gpu

DEV = "cuda:0"


def _pattern(C, n, a, b):
    m = n // C
    own = (torch.arange(n)[None, :] // m) == torch.arange(C)[:, None]
    return torch.where(own, torch.tensor(a), torch.tensor(b)).float()


def _verdict(Wl, Wg, C):
    """Run the check; returns [(ok, a, b)] for Wl and Wg as the records in the workspace hold them."""
    from protopformer_b200 import _lib, ops
    ws = ops._ws("pph_head_mid_ws_bytes", 8, 9, 16, Wl.shape[1], Wg.shape[1] if Wg is not None else 0, C, 1, zero=True,
                 device=DEV)
    _lib.call("pph_last_layer_pattern", Wl.to(DEV).contiguous(), Wl.shape[1],
              None if Wg is None else Wg.to(DEV).contiguous(), 0 if Wg is None else Wg.shape[1], C, ws)
    torch.cuda.synchronize()
    ints, floats = ws[:32].view(torch.int32).cpu(), ws[:32].view(torch.float32).cpu()
    return [(int(ints[4 * i]), float(floats[4 * i + 1]), float(floats[4 * i + 2])) for i in range(2)]


def test_pattern_check_verdicts():
    C, P = 200, 2000
    ref = _pattern(C, P, 1.0, -0.5)                       # set_last_layer_incorrect_connection(-0.5)
    assert _verdict(ref, ref, C) == [(1, 1.0, -0.5)] * 2
    two = _pattern(C, P, 2.0, 0.0)
    assert _verdict(two, two, C) == [(1, 2.0, 0.0)] * 2
    bad = ref.clone()
    bad[C - 1, P - 1] = -0.25                            # last entry: the tail of the grid-stride loop
    assert [v[0] for v in _verdict(bad, ref, C)] == [0, 1]
    bad = ref.clone()
    bad[17, 3] = 1.0 + 2 ** -23                          # one ulp off: exact equality
    assert [v[0] for v in _verdict(ref, bad, C)] == [1, 0]
    perm = ref[:, torch.randperm(P, generator=torch.Generator().manual_seed(3))]     # prototypes moved to other classes
    assert [v[0] for v in _verdict(perm, perm, C)] == [0, 0]
    one = torch.full((1, 30), 3.0)                       # C = 1: b = a
    assert _verdict(one, one, 1) == [(1, 3.0, 3.0)] * 2
    odd = _pattern(3, 15, 1.0, -0.5)                     # n % 4 != 0: scalar loads
    assert _verdict(odd, None, 3) == [(1, 1.0, -0.5), (1, 0.0, 0.0)]
    assert _verdict(torch.ones(3, 16), None, 3)[0][0] == 0        # n % C != 0
    # the check resets its own counters: a bad verdict does not stick to the next call on the same workspace
    from protopformer_b200 import _lib, ops
    ws = ops._ws("pph_head_mid_ws_bytes", 8, 9, 16, P, P, C, 1, zero=True, device=DEV)
    for W, want in ((bad, 0), (ref, 1), (ref, 1)):
        _lib.call("pph_last_layer_pattern", W.to(DEV), P, W.to(DEV), P, C, ws)
        torch.cuda.synchronize()
        assert int(ws[:4].view(torch.int32).item()) == want


def _step(shape, case, variants=None, train=True):
    from protopformer_b200 import ops
    from protopformer_b200.graph import GraphedHeadStep
    cfg = ops.HeadConfig(K=shape.K, global_coe=shape.global_coe, mode="fp32", ppc_cov_thresh=shape.ppc_cov_thresh,
                         ppc_mean_thresh=shape.ppc_mean_thresh)
    params = {k: case[k].to(DEV).clone() for k in ("Wa", "ba", "P", "Pg", "Wl", "Wg")}
    for k in ("Wa", "ba", "P", "Pg"):
        params[k].requires_grad_(train)
    step = GraphedHeadStep(params, cfg, B=shape.B, N=shape.N, C=shape.C, m=shape.m, train=train, variants=variants)
    step.load(0, case["tokens"], case["scores"], case["labels"])
    torch.cuda.synchronize()
    step.capture()
    return step, params


def _class_sum_ran(step):
    """Only the class-sum role clears the verdicts it used: ok == 0 with the weights' a, b still in place."""
    rec = step.fused.ws_mid[:32].view(torch.int32).cpu()
    return int(rec[0]) == 0 and int(rec[4]) == 0 and float(step.fused.ws_mid[:32].view(torch.float32)[1]) != 0.0


def _check_against_oracle(step, params, case, shape, train=True):
    f = step.fused
    ref = O.head_train_step(case, shape, route=f.argmin.cpu().long())
    assert torch.equal(f.idx32.cpu().long(), ref["idx"])
    assert rel_close(f.logits.cpu(), ref["logits"], 1e-4)
    assert rel_close(f.logits_g.cpu(), ref["logits_global"], 1e-4) and rel_close(f.logits_l.cpu(), ref["logits_local"], 1e-4)
    if not train:
        return
    losses = f.losses.cpu()
    assert rel_close(losses[0], ref["loss"], 1e-4) and rel_close(losses[1], ref["ce"], 1e-4)
    assert rel_close(losses[2], ref["ppc_cov"], 1e-4) and rel_close(losses[3], ref["ppc_mean"], 1e-4)
    got = dict(g_tokens=f.dtokens, g_P=params["P"].grad, g_Pg=params["Pg"].grad, g_Wa=params["Wa"].grad,
               g_ba=params["ba"].grad)
    for k, v in got.items():
        e = norm_rel(v.cpu().reshape(ref[k].shape), ref[k])
        assert e < 1e-4, (k, e)


def _perturb(case):
    case = dict(case)
    case["Wl"] = case["Wl"].clone()
    case["Wl"][3, 17] = 0.75
    return case


@pytest.mark.parametrize("structured", [True, False])
@pytest.mark.parametrize("batch,variants,train", [(64, None, True), (64, None, False),
                                                  (65, dict(bwd="staged", ppc="split"), True)])
def test_both_last_layer_forms_match_the_oracle(structured, batch, variants, train):
    shape = synth.SHAPES["cub_b64"].with_batch(batch)
    case = synth.make_case(shape, seed=1)
    if not structured:
        case = _perturb(case)
    step, params = _step(shape, case, variants, train)
    step.run(0)
    torch.cuda.synchronize()
    assert _class_sum_ran(step) == structured
    _check_against_oracle(step, params, case, shape, train)


def test_form_switches_inside_one_graph_when_the_weights_change():
    shape = synth.SHAPES["cub_b64"]
    case = synth.make_case(shape, seed=2)
    step, params = _step(shape, case)
    pert = _perturb(case)
    for c, structured in ((case, True), (pert, False), (case, True)):
        params["Wl"].data.copy_(c["Wl"])              # no version bump, no recapture: the graph must notice by itself
        step.run(0)
        torch.cuda.synchronize()
        assert _class_sum_ran(step) == structured
        _check_against_oracle(step, params, c, shape)


@pytest.mark.parametrize("structured", [True, False])
def test_replays_are_bit_identical(structured):
    shape = synth.SHAPES["cub_b64"]
    case = synth.make_case(shape, seed=4)
    if not structured:
        case = _perturb(case)
    step, params = _step(shape, case)
    outs = []
    for _ in range(2):
        step.run(0)
        torch.cuda.synchronize()
        f = step.fused
        outs.append([t.clone() for t in (f.losses, f.logits, f.logits_g, f.logits_l, f.dlogits, f.g_l, f.g_g, f.dtokens,
                                         params["P"].grad, params["Pg"].grad, params["Wa"].grad, params["ba"].grad)])
    for a, b in zip(*outs):
        assert torch.equal(a, b)
