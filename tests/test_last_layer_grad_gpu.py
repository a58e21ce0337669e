"""Trainable last layers: pph_last_layer_wgrad and every layer above it.

The reference freezes Wl / Wg (protopformer.py:130-131); a user who sets their requires_grad gets, from the reference's
autograd, dWl = (1-gc) dlogits^T act_l and dWg = gc dlogits^T act_g (plus the upstream gradients of logits_local /
logits_global).  Held here: the kernel against float64, the autograd path of PPNet, the graphed step (both last-layer
forms, v1, the staged variant, bf16 mode) against the CPU restatement's float64 autograd -- with every output the frozen
step also produces bit-identical to it -- a training loop through the fused AdamW, and the data-parallel / optimizer
plumbing on the CPU."""
import ctypes
import os

import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F

from oracle import protohead_oracle as O
from protopformer_b200 import synth
from tests.util import norm_rel

DEV = "cuda:0"


class MyVisionTransformer(nn.Module):
    """Fake backbone handing the head preset tokens / CLS-attention (the class NAME matters, protopformer.py:78-81)."""

    def __init__(self, din, n):
        super().__init__()
        self.fc = nn.Linear(din, din)
        self.patch_embed = nn.Module()
        self.patch_embed.num_patches = n
        self.tokens = self.attn = None

    def forward_feature_patch_embed_all(self, x):
        return self.tokens[:, :1], self.tokens[:, 1:]

    def forward_feature_mask_train_direct(self, cls_embed, x_embed, token_attn, reserve_layer_nums):
        return self.tokens, (self.attn, None)


def _ppnet(shape, precision="fp32"):
    from protopformer_b200 import PPNet
    return PPNet(MyVisionTransformer(shape.Din, shape.N), 224, [shape.P, shape.D, 1, 1], [14, 16, 16, 8.0], shape.C,
                 reserve_layers=[11], reserve_token_nums=[shape.K], use_global=True, use_ppc_loss=True,
                 ppc_cov_thresh=shape.ppc_cov_thresh, ppc_mean_thresh=shape.ppc_mean_thresh, global_coe=shape.global_coe,
                 global_proto_per_class=shape.Pg // shape.C, add_on_layers_type='regular', precision=precision)


def _oracle(case, shape, route, extra=False):
    """float64 autograd of the CPU restatement with the last layers trainable: loss = CE + 0.1 L_cov + 0.5 L_mean
    (engine_proto.py:51-64), or extra=True: CE + terms on logits_local / logits_global.  Returns the gradients of every
    head input."""
    c = {k: (v.detach().clone().double() if v.is_floating_point() else v.clone()) for k, v in case.items()}
    for k in ("tokens", "P", "Pg", "Wa", "ba", "Wl", "Wg"):
        c[k].requires_grad_(True)
    out = O.head_forward(c, shape.K, shape.global_coe, route=route)
    loss = F.cross_entropy(out["logits"], c["labels"])
    if extra:
        loss = loss + _extra_terms(out["logits_local"], out["logits_global"], c["labels"])
    else:
        cov, mean = O.ppc_loss(out["act_map"], out["idx"], c["labels"], shape.m, shape.N, shape.ppc_cov_thresh,
                               shape.ppc_mean_thresh)
        loss = loss + 0.1 * cov + 0.5 * mean
    loss.backward()
    return {k: c[k].grad for k in ("tokens", "P", "Pg", "Wa", "ba", "Wl", "Wg")}


def _extra_terms(logits_local, logits_global, labels):
    return 0.3 * F.cross_entropy(logits_local, labels) + 0.2 * logits_global.square().mean()


# ----------------------------------------------------------------------------------------------------------------------
# CPU: data-parallel / optimizer plumbing and the C ABI's argument checks
# ----------------------------------------------------------------------------------------------------------------------
def test_head_parameters_list_the_last_layers_only_when_unfrozen():
    from protopformer_b200.dist import FlatGradReducer, head_parameters
    net = _ppnet(synth.SHAPES["tiny"])
    four = ["prototype_vectors", "prototype_vectors_global", "add_on_layers.0.weight", "add_on_layers.0.bias"]
    assert [n for n, _ in head_parameters(net)] == four
    net.last_layer_global.weight.requires_grad_(True)
    assert [n for n, _ in head_parameters(net)] == four + ["last_layer_global.weight"]
    net.last_layer.weight.requires_grad_(True)
    named = head_parameters(net)
    assert [n for n, _ in named] == four + ["last_layer.weight", "last_layer_global.weight"]
    # the graphed step's flat buffer: P | Pg | Wa | ba | Wl | Wg -- the last layers are one contiguous tail segment
    p = dict(named)
    red = FlatGradReducer([("P", p[four[0]]), ("Pg", p[four[1]]), ("Wa", p[four[2]]), ("ba", p[four[3]]),
                           ("Wl", net.last_layer.weight), ("Wg", net.last_layer_global.weight)])
    lo, hi = red.segment(("Wl", "Wg"))
    assert (lo, hi) == (red.segment(("Wa", "ba"))[1], red.flat.numel())
    assert hi - lo == net.last_layer.weight.numel() + net.last_layer_global.weight.numel()
    assert red.segment(("P", "Pg")) == (0, p[four[0]].numel() + p[four[1]].numel())
    assert net.last_layer.weight.grad.data_ptr() == red.flat[lo:].data_ptr()


def test_head_param_groups_add_the_last_layer_group_only_when_unfrozen():
    from protopformer_b200.optim import head_param_groups
    net = _ppnet(synth.SHAPES["tiny"])
    lrs = {"add_on_layers": 3e-3, "prototype_vectors": 2e-3}
    assert len(head_param_groups(net, lrs, 0.05)) == 3                  # frozen: the reference's groups, no new key needed
    net.last_layer.weight.requires_grad_(True)
    with pytest.raises(KeyError, match="last_layer"):
        head_param_groups(net, lrs, 0.05)
    groups = head_param_groups(net, dict(lrs, last_layer=1e-4), 0.05)
    assert len(groups) == 4 and groups[3]["lr"] == 1e-4 and groups[3]["weight_decay"] == 0.0
    assert groups[3]["params"] == [net.last_layer.weight]
    net.last_layer_global.weight.requires_grad_(True)
    g = head_param_groups(net, dict(lrs, last_layer=1e-4), 0.05)[3]["params"]
    assert len(g) == 2 and g[0] is net.last_layer.weight and g[1] is net.last_layer_global.weight


def test_last_layer_wgrad_rejects_bad_arguments_before_touching_a_device():
    from protopformer_b200 import _lib
    lib = _lib.load()
    fake = ctypes.c_void_p(0x1000)            # never dereferenced: every call below must fail (or finish) on the host
    ok = (fake, None, None, fake, fake, 64, 2000, 2000, 200, 0.5, fake, fake, None)
    for i, bad in ((5, 0), (6, 0), (8, 0), (7, -1), (5, -3)):               # B, P, C >= 1, Pg >= 0
        args = list(ok)
        args[i] = bad
        assert lib.pph_last_layer_wgrad(*args) == -1
        assert b"dims" in lib.pph_last_error_string()
    for i in (0, 3, 4):                                                      # dlogits, act_l, act_g for a requested output
        args = list(ok)
        args[i] = None
        assert lib.pph_last_layer_wgrad(*args) == -1
        assert b"null" in lib.pph_last_error_string()
    args = list(ok)
    args[3], args[10] = None, None                     # no dWl requested: act_l is not needed ...
    args[4], args[11] = None, None                     # ... nor act_g without dWg: nothing to do, no launch
    assert lib.pph_last_layer_wgrad(*args) == 0
    args = list(ok)
    args[4], args[7] = None, 0                         # Pg = 0: no global layer, dWg is ignored
    args[10] = None
    assert lib.pph_last_layer_wgrad(*args) == 0


def _gloo_worker(rank, world, port, q):
    import torch.distributed as dist
    from protopformer_b200.dist import FlatGradReducer, head_parameters
    dist.init_process_group("gloo", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world)
    torch.manual_seed(0)
    net = _ppnet(synth.SHAPES["tiny"])
    net.last_layer.weight.requires_grad_(True)
    net.last_layer_global.weight.requires_grad_(True)
    named = head_parameters(net)
    red = FlatGradReducer(named)
    red.zero()
    loss = sum((p * (rank + 1) * (i + 1)).sum() for i, (_, p) in enumerate(named))      # rank-dependent gradients
    loss.backward()
    lo, hi = red.segment(("last_layer.weight", "last_layer_global.weight"))
    before = red.flat.clone()
    red.allreduce(lo=lo, hi=hi)                         # the "last" exchange alone
    untouched = torch.equal(red.flat[:lo], before[:lo])
    q.put((rank, net.last_layer.weight.grad.tolist(), net.last_layer_global.weight.grad.tolist(), untouched,
           hi == red.flat.numel()))
    dist.destroy_process_group()


def test_last_layer_gradients_are_averaged_gloo_world2():
    import socket

    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    with socket.socket() as sk:
        sk.bind(("127.0.0.1", 0))
        port = sk.getsockname()[1]
    procs = [ctx.Process(target=_gloo_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted([q.get(timeout=300) for _ in procs], key=lambda t: t[0])
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    for _, gl, gg, untouched, tail in res:
        assert untouched and tail
        assert torch.allclose(torch.tensor(gl), torch.full_like(torch.tensor(gl), 1.5 * 5))     # mean of 5, 10
        assert torch.allclose(torch.tensor(gg), torch.full_like(torch.tensor(gg), 1.5 * 6))     # mean of 6, 12


# ----------------------------------------------------------------------------------------------------------------------
# GPU: the kernel
# ----------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("B,C,P,Pg", [(1, 200, 2000, 2000), (63, 7, 1960, 1000), (64, 200, 2000, 2000),
                                      (65, 256, 1000, 8000), (1024, 200, 2000, 2000), (64, 1, 8000, 1960),
                                      (65, 7, 1000, 1960), (1024, 256, 8000, 8000)])
def test_kernel_matches_float64(B, C, P, Pg):
    from protopformer_b200 import _lib
    g = torch.Generator(device=DEV).manual_seed(B * 7 + C)
    r = lambda *s: torch.randn(*s, device=DEV, generator=g)  # noqa: E731

    def upstream():      # what a cross-entropy produces, (softmax - onehot) / B, plus noise (C = 1 would be all zeros)
        onehot = F.one_hot(torch.randint(0, C, (B,), device=DEV, generator=g), C).float()
        return (torch.softmax(3 * r(B, C), dim=1) - onehot + 0.05 * r(B, C)) / B

    dl, dlg, dll = upstream(), upstream(), upstream()
    act_l = 5 * torch.rand(B, P, device=DEV, generator=g)
    act_g = 5 * torch.rand(B, Pg, device=DEV, generator=g)
    gc = 0.3
    want_l = ((1 - gc) * dl.double() + dll.double()).t() @ act_l.double()
    want_g = (gc * dl.double() + dlg.double()).t() @ act_g.double()
    plain_l, plain_g = ((1 - gc) * dl.double()).t() @ act_l.double(), (gc * dl.double()).t() @ act_g.double()
    # (extras, dWl wanted, dWg wanted): with / without the branch gradients, each output skipped once
    for extras, wl, wg in ((False, True, True), (True, True, True), (True, True, False), (False, False, True)):
        outs = []
        for _ in range(2):
            dWl = torch.full((C, P), float("nan"), device=DEV)
            dWg = torch.full((C, Pg), float("nan"), device=DEV)
            # the activations of a skipped output are not needed: pass NULL for them
            _lib.call("pph_last_layer_wgrad", dl, dlg if extras else None, dll if extras else None, act_l if wl else None,
                      act_g if wg else None, B, P, Pg, C, gc, dWl if wl else None, dWg if wg else None)
            torch.cuda.synchronize()
            outs.append((dWl, dWg))
        for (a, want, plain), wanted in zip(((outs[0][0], want_l, plain_l), (outs[0][1], want_g, plain_g)), (wl, wg)):
            if not wanted:
                assert torch.isnan(a).all()                    # skipped output untouched
                continue
            ref = want if extras else plain
            err = float((a.double() - ref).abs().max() / ref.abs().max())
            # 1e-6 up to B = 256; one sequential FP32 sum of 1024 terms per entry measured 1.8e-6 on B200
            assert err <= (1e-6 if B <= 256 else 4e-6), (B, C, P, Pg, extras, err)
        for a, b in zip(*outs):
            assert torch.equal(a, b) or (torch.isnan(a).all() and torch.isnan(b).all())     # bit-identical launches


# ----------------------------------------------------------------------------------------------------------------------
# GPU: autograd path (PPNet)
# ----------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("extra", [False, True])
def test_ppnet_unfrozen_last_layers_get_the_oracle_gradient(extra):
    shape = synth.SHAPES["cub_b8"]
    case = synth.make_case(shape, seed=5)
    net = _ppnet(shape).cuda()
    with torch.no_grad():
        net.prototype_vectors.copy_(case["P"].reshape(shape.P, shape.D, 1, 1))
        net.prototype_vectors_global.copy_(case["Pg"].reshape(shape.Pg, shape.D, 1, 1))
        net.add_on_layers[0].weight.copy_(case["Wa"].reshape(shape.D, shape.Din, 1, 1))
        net.add_on_layers[0].bias.copy_(case["ba"])
    net.last_layer.weight.requires_grad_(True)
    net.last_layer_global.weight.requires_grad_(True)
    feats = net.features
    feats.tokens, feats.attn = case["tokens"].cuda().requires_grad_(True), case["scores"].cuda()
    labels = case["labels"].cuda()
    net.train()
    if extra:
        # PPNet.head: the forward of PPNet.forward, with logits_local / logits_global (upstream gradients on both branches)
        out = net.head(feats.tokens, feats.attn)
        loss = F.cross_entropy(out.logits, labels) + _extra_terms(out.logits_local, out.logits_global, labels)
        route = out.argmin.long().cpu()
    else:
        logits, aux = net(None)
        cov, mean = net.get_PPC_loss(aux[2], aux[3], aux[4], labels)
        loss = F.cross_entropy(logits, labels) + 0.1 * cov + 0.5 * mean
        with torch.no_grad():
            route = net.head(feats.tokens, feats.attn).argmin.long().cpu()
    loss.backward()
    ref = _oracle(case, shape, route, extra)
    for k, p in (("Wl", net.last_layer.weight), ("Wg", net.last_layer_global.weight)):
        e = norm_rel(p.grad.cpu(), ref[k])
        assert e < 1e-4, (k, e)
    e = norm_rel(net.prototype_vectors.grad.reshape(shape.P, shape.D).cpu(), ref["P"])
    assert e < 1e-4, ("P", e)
    # frozen (the default): no gradient, as in the reference
    net2 = _ppnet(shape).cuda()
    net2.features.tokens, net2.features.attn = feats.tokens.detach(), feats.attn
    net2.train()
    logits2, aux2 = net2(None)
    F.cross_entropy(logits2, labels).backward()
    assert net2.last_layer.weight.grad is None and net2.last_layer_global.weight.grad is None


# ----------------------------------------------------------------------------------------------------------------------
# GPU: the graphed training step
# ----------------------------------------------------------------------------------------------------------------------
def _graphed(shape, case, train_ll, mode="fp32", variants=None, impl="auto"):
    from protopformer_b200 import ops
    from protopformer_b200.graph import GraphedHeadStep
    cfg = ops.HeadConfig(K=shape.K, global_coe=shape.global_coe, mode=mode, ppc_cov_thresh=shape.ppc_cov_thresh,
                         ppc_mean_thresh=shape.ppc_mean_thresh)
    params = {k: case[k].to(DEV).clone() for k in ("Wa", "ba", "P", "Pg", "Wl", "Wg")}
    for k in ("Wa", "ba", "P", "Pg") + (("Wl", "Wg") if train_ll else ()):
        params[k].requires_grad_(True)
    step = GraphedHeadStep(params, cfg, B=shape.B, N=shape.N, C=shape.C, m=shape.m, variants=variants, impl=impl)
    step.load(0, case["tokens"], case["scores"], case["labels"])
    torch.cuda.synchronize()
    step.capture()
    return step, params


def _shared_outputs(step, params):
    """Everything the frozen step produces (the trainable step must reproduce it bit for bit)."""
    f = step.fused
    return [t.clone() for t in (f.losses, f.logits, f.logits_g, f.logits_l, f.dlogits, f.dtokens, params["P"].grad,
                                params["Pg"].grad, params["Wa"].grad, params["ba"].grad)]


def _class_sum_ran(step):
    rec = step.fused.ws_mid[:32].view(torch.int32).cpu()
    return int(rec[0]) == 0 and int(rec[4]) == 0 and float(step.fused.ws_mid[:32].view(torch.float32)[1]) != 0.0


def _perturb(case):
    case = dict(case)
    case["Wl"] = case["Wl"].clone()
    case["Wl"][3, 17] = 0.75
    return case


def _check_step(shape, case, mode="fp32", variants=None, impl="auto", structured=True, tol=1e-4):
    frozen, fparams = _graphed(shape, case, False, mode, variants, impl)
    frozen.run(0)
    torch.cuda.synchronize()
    want = _shared_outputs(frozen, fparams)
    assert fparams["Wl"].grad is None and fparams["Wg"].grad is None
    step, params = _graphed(shape, case, True, mode, variants, impl)
    assert [n for n, _ in step.reducer.named] == ["P", "Pg", "Wa", "ba", "Wl", "Wg"]
    assert step.kernel_launches_per_step == frozen.kernel_launches_per_step + 1
    if shape.name == "cub_b64" and shape.B == 64 and impl != "v1" and variants is None:
        assert frozen.kernel_launches_per_step == 11
    runs = []
    for _ in range(2):
        step.run(0)
        torch.cuda.synchronize()
        runs.append(_shared_outputs(step, params) + [params["Wl"].grad.clone(), params["Wg"].grad.clone()])
    # the round-1 sequence adds the PPC prototype rows onto dP with float atomics: its outputs are reproducible to rounding
    # only (with or without trainable last layers); the v2 step is bit-reproducible, and dWl / dWg always are
    same = torch.equal if step.impl == "v2" else (lambda a, b: norm_rel(a.cpu(), b.cpu()) <= 1e-6)
    for a, b in zip(runs[0][-2:], runs[1][-2:]):
        assert torch.equal(a, b)                               # dWl, dWg: replays bit-identical
    for a, b in zip(*runs):
        assert same(a, b)                                      # replays
    for a, b in zip(want, runs[0]):
        assert same(a, b)                                      # the frozen step's outputs
    if step.impl == "v2":
        assert _class_sum_ran(step) == structured
    ref = _oracle(case, shape, step.fused.argmin.cpu().long())
    for k in ("Wl", "Wg"):
        e = norm_rel(params[k].grad.cpu(), ref[k])
        assert e < tol, (k, e)


@pytest.mark.gpu
@pytest.mark.parametrize("structured", [True, False])
@pytest.mark.parametrize("batch,variants,impl", [(64, None, "auto"), (65, dict(bwd="staged", ppc="split"), "auto"),
                                                 (64, None, "v1")])
def test_graphed_step_last_layer_gradients(structured, batch, variants, impl):
    shape = synth.SHAPES["cub_b64"].with_batch(batch)
    case = synth.make_case(shape, seed=1)
    if not structured:
        case = _perturb(case)
    _check_step(shape, case, variants=variants, impl=impl, structured=structured)


@pytest.mark.gpu
def test_graphed_step_last_layer_gradients_bf16_cars():
    shape = synth.SHAPES["cars_b64"]
    _check_step(shape, synth.make_case(shape, seed=1), mode="bf16", tol=2e-3)      # DESIGN.md section 3: bf16 gradients


@pytest.mark.gpu
def test_fused_adamw_training_loop_over_the_six_flat_views():
    from protopformer_b200 import _lib, ops
    from protopformer_b200.optim import FusedHeadAdamW
    shape = synth.SHAPES["cub_b64"]
    case = synth.make_case(shape, seed=3)
    step, params = _graphed(shape, case, True)
    p = params
    groups = [{"params": [p["P"]], "lr": 2e-3, "weight_decay": 0.05}, {"params": [p["Pg"]], "lr": 2e-3, "weight_decay": 0.05},
              {"params": [p["Wa"], p["ba"]], "lr": 3e-3, "weight_decay": 1e-3},
              {"params": [p["Wl"], p["Wg"]], "lr": 1e-2, "weight_decay": 0.0}]
    opt = FusedHeadAdamW(groups, grads=step.reducer.views)
    step.run(0)
    torch.cuda.synchronize()
    assert _class_sum_ran(step)                                # the reference init: class-sum form
    opt.step()
    step.run(0)                                                # the same graph, new weights
    torch.cuda.synchronize()
    # the update broke the class-connection pattern of both layers: the check in the replay found it (fresh check below
    # on the updated weights, same verdicts), so pph_head_mid took the general product -- and its gradients are right
    ws = ops._ws("pph_head_mid_ws_bytes", 8, 9, 16, shape.P, shape.Pg, shape.C, 1, zero=True, device=DEV)
    _lib.call("pph_last_layer_pattern", p["Wl"].detach(), shape.P, p["Wg"].detach(), shape.Pg, shape.C, ws)
    torch.cuda.synchronize()
    rec = ws[:32].view(torch.int32).cpu()
    assert int(rec[0]) == 0 and int(rec[4]) == 0
    upd = dict(case)
    for k in ("P", "Pg", "Wa", "ba", "Wl", "Wg"):
        upd[k] = p[k].detach().cpu()
    ref = _oracle(upd, shape, step.fused.argmin.cpu().long())
    for k in ("Wl", "Wg", "P", "Wa"):
        e = norm_rel(p[k].grad.cpu().reshape(ref[k].shape), ref[k])
        assert e < 1e-4, (k, e)
    # the checkpoint layout: loadable by torch.optim.AdamW over the same groups
    clones = {k: v.detach().clone().requires_grad_(True) for k, v in p.items()}
    tg = [{"params": [clones[k] for k in ks], "lr": g["lr"], "weight_decay": g["weight_decay"]}
          for ks, g in zip((("P",), ("Pg",), ("Wa", "ba"), ("Wl", "Wg")), groups)]
    ref_opt = torch.optim.AdamW(tg)
    ref_opt.load_state_dict(opt.state_dict())
    st = ref_opt.state[clones["Wl"]]
    assert float(st["step"]) == 1.0 and torch.equal(st["exp_avg"], opt.state[p["Wl"]]["exp_avg"])


# ----------------------------------------------------------------------------------------------------------------------
# multi-GPU: the third in-graph exchange
# ----------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.multigpu
@pytest.mark.parametrize("exchange", ["peer", "peer_nomc", "nccl"])
def test_in_graph_exchange_averages_the_last_layer_gradients(exchange):
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ)
    env.pop("PPH_TIMELINE", None)
    port = {"peer": 29541, "peer_nomc": 29542, "nccl": 29543}[exchange]
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
                        "127.0.0.1", "--master-port", str(port), os.path.join(root, "scripts", "ddp_check.py"),
                        "--train-last-layers", exchange],
                       env=env, cwd=root, capture_output=True, text=True, timeout=240)
    assert r.returncode == 0, (r.stdout[-2000:], r.stderr[-2000:])
    assert r.stdout.count("in-graph exchange vs averaged local gradients") == 2
    assert r.stdout.count("last layers") == 2
