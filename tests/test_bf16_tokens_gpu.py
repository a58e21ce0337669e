"""bf16 backbone tokens: the `_bf16tok` twins of every entry point that reads tokens, and every layer above them.

Every bf16 value is exact in fp32, so the contract is bit-identity: each twin, fed bf16 tokens, returns exactly what its
fp32 entry returns on the same tokens widened to fp32, and its token gradient equals that entry's gradient rounded once to
bf16 (round to nearest even).  Held here per entry point (CUB and Dogs widths, B = 1 and 65), for PPNet (training, eval,
push_forward, push_forward_class_maps) -- also against the float64 oracle -- and for the graphed step in v1 and v2, over the
variant sets of tests/test_step2_gpu.py, with trainable last layers and through the pinned-host pipeline.  On the CPU: the
twins' argument checks and the byte count of the bf16 host transfer."""
import ctypes

import pytest
import torch
import torch.nn.functional as F

from oracle import protohead_oracle as O
from protopformer_b200 import synth
from tests.util import norm_rel, rel_close

DEV = "cuda:0"
BF = torch.bfloat16


def _lib():
    from protopformer_b200 import _lib
    return _lib


def _ops():
    from protopformer_b200 import ops
    return ops


def _bf16_case(shape, seed):
    """A synthetic batch whose tokens are bf16 (`tokens_bf`); `tokens` holds the same values widened to fp32."""
    case = synth.make_case(shape, seed=seed)
    case["tokens_bf"] = case["tokens"].to(BF)
    case["tokens"] = case["tokens_bf"].float()
    return case


# ----------------------------------------------------------------------------------------------------------------------
# CPU: argument checks of the C ABI, the binding, the byte count of load_host
# ----------------------------------------------------------------------------------------------------------------------
TWINS = ("pph_addon_fwd", "pph_addon_bwd", "pph_addon_fwd2", "pph_select_addon_fwd", "pph_addon_bwd3", "pph_head_prep",
         "pph_addon_bwd2", "pph_gather_rows_host")


def test_every_token_entry_has_a_registered_bf16_twin_with_the_same_launch_count():
    L = _lib()
    assert set(L.BF16TOK_TWINS) == set(TWINS)
    lib = L.load()
    for n in TWINS:
        assert L.SIGNATURES[n + "_bf16tok"] == L.SIGNATURES[n]
        assert getattr(lib, n + "_bf16tok").argtypes is not None


def _twin_calls(Din):
    """(name, args) of every bf16 twin with fake, never dereferenced device pointers; B = 4, N = 196, D = 192, K = 81."""
    fake = ctypes.c_void_p(0x1000)
    B, N, D, K = 4, 196, 192, 81
    f = [fake] * 10
    calls = {
        "pph_addon_fwd_bf16tok": [fake, fake, fake, fake, B, N, Din, D, K, *f[:4], 0.5, *f[:8], None],
        "pph_addon_bwd_bf16tok": [fake] * 7 + [B, N, Din, D, K, fake, 3, fake, fake, fake, None],
        "pph_addon_fwd2_bf16tok": [fake, fake, fake, fake, B, N, Din, D, K, *f[:4], 0.5, *f[:8], fake, None],
        "pph_select_addon_fwd_bf16tok": [fake, 1, fake, fake, fake, B, N, Din, D, K, fake, *f[:4], 0.5, *f[:8], fake, None],
        "pph_addon_bwd3_bf16tok": [3] + [fake] * 6 + [B, N, Din, D, K, fake, fake, fake, fake, None],
        "pph_head_prep_bf16tok": [fake] * 4 + [B, 1, N, Din, D, K, 0.5] + [fake] * 14 + [fake, 8] + [fake] * 5 +
                                 [fake, 8] + [fake] * 5 + [None],
        "pph_addon_bwd2_bf16tok": [3] + [fake] * 5 + [B, N, Din, D, K, fake, fake, fake, fake, None],
        "pph_gather_rows_host_bf16tok": [fake, fake, B, N, Din, K, fake, 8, None],
    }
    return calls


# position of the tokens pointer in each twin's argument list
_TOKENS_AT = {"pph_addon_fwd_bf16tok": 0, "pph_addon_bwd_bf16tok": 0, "pph_addon_fwd2_bf16tok": 0,
              "pph_select_addon_fwd_bf16tok": 2, "pph_addon_bwd3_bf16tok": 1, "pph_head_prep_bf16tok": 1,
              "pph_addon_bwd2_bf16tok": 1, "pph_gather_rows_host_bf16tok": 0}


@pytest.mark.parametrize("name", sorted(_TOKENS_AT))
def test_bf16_twins_reject_bad_arguments_before_touching_a_device(name):
    lib = _lib().load()
    fn = getattr(lib, name)
    args = _twin_calls(196)[name]                        # Din = 196: a multiple of 4 but not of 8
    assert fn(*args) < 0
    msg = lib.pph_last_error_string()
    assert b"Din" in msg, msg
    args = _twin_calls(192)[name]
    args[_TOKENS_AT[name]] = None
    assert fn(*args) == -1
    assert b"null" in lib.pph_last_error_string()


def test_load_host_counts_half_the_token_bytes_for_bf16():
    """The byte count load_host returns: scores and labels whole, B (K+1) token rows of Din elements in the token dtype."""
    from protopformer_b200.graph import GraphedHeadStep
    shape = synth.SHAPES["cub_b64"]
    B, N, K, Din = shape.B, shape.N, shape.K, shape.Din
    scores, labels = torch.zeros(B, N), torch.zeros(B, dtype=torch.int64)
    n = {dt: GraphedHeadStep.host_transfer_bytes(torch.zeros(B, 1 + N, Din, dtype=dt), scores, labels, K)
         for dt in (torch.float32, BF)}
    assert n[torch.float32] == 4 * B * N + 8 * B + 4 * B * (K + 1) * Din == 4_081_152
    assert n[BF] == 4 * B * N + 8 * B + 2 * B * (K + 1) * Din == 2_065_920
    # the token rows are 98 % of what crosses the bus at this shape: bf16 nearly halves the transfer
    assert 0.50 < n[BF] / n[torch.float32] < 0.51


def test_token_dtype_policy_on_the_host():
    ops = _ops()
    assert ops.token_entry("pph_addon_fwd", torch.float32) == "pph_addon_fwd"
    assert ops.token_entry("pph_addon_fwd", BF) == "pph_addon_fwd_bf16tok"
    for dt in (torch.float16, torch.float64, torch.int8):
        with pytest.raises(TypeError, match=str(dt)):
            ops.token_entry("pph_addon_fwd", dt)
    t = torch.zeros(2, 5, 8, dtype=BF)
    ops.check_head_dtypes(t, torch.zeros(3, dtype=torch.float32))
    with pytest.raises(TypeError, match="bfloat16"):
        ops.check_head_dtypes(t, torch.zeros(3, dtype=BF))
    with pytest.raises(TypeError, match="float16"):
        ops.check_head_dtypes(t.half())


# ----------------------------------------------------------------------------------------------------------------------
# GPU: entry points against their fp32 twins
# ----------------------------------------------------------------------------------------------------------------------
def _e(*s, dt=torch.float32):
    return torch.empty(s, dtype=dt, device=DEV)


def _fwd_outputs(shape):
    B, K, D = shape.B, shape.K, shape.D
    return dict(Zs=_e(B, K, D), Zc=_e(B, D), z2s=_e(B, K), z2c=_e(B), z2s_ctr=_e(B, K), z2c_ctr=_e(B), z2s_hi=_e(B, K),
                z2c_hi=_e(B), Zs_hi=_e(B * K, D, dt=BF), Zs_lo=_e(B * K, D, dt=BF), Zc_hi=_e(B, D, dt=BF),
                Zc_lo=_e(B, D, dt=BF))


_FWD = ("Zs", "Zc", "z2s", "z2c", "z2s_ctr", "z2c_ctr", "z2s_hi", "z2c_hi", "Zs_hi", "Zs_lo", "Zc_hi", "Zc_lo")


def _assert_same(a: dict, b: dict, what):
    assert a.keys() == b.keys()
    for k in a:
        assert torch.equal(a[k], b[k]), (what, k)


def _assert_dtokens(d16, d32, idx, what):
    """bf16 dtokens == fp32 dtokens rounded once; rows of unselected tokens are zero."""
    assert d16.dtype == BF and d32.dtype == torch.float32
    assert torch.equal(d16, d32.to(BF)), (what, float((d16.float() - d32).abs().max()))
    B, n1, _ = d16.shape
    sel = torch.zeros(B, n1, dtype=torch.bool, device=DEV)
    sel[:, 0] = True
    sel.scatter_(1, idx.long() + 1, True)
    assert int((d16[~sel] != 0).sum()) == 0, what
    assert bool((d16[sel].abs().sum(-1) > 0).all()), what


ENTRY_SHAPES = [("cub_b64", 1), ("cub_b64", 65), ("dogs_b256", 1), ("dogs_b256", 65)]


@pytest.mark.gpu
@pytest.mark.parametrize("key,B", ENTRY_SHAPES)
def test_every_bf16_entry_is_bit_identical_to_its_fp32_twin(key, B):
    L, ops = _lib(), _ops()
    shape = synth.SHAPES[key].with_batch(B)
    case = _bf16_case(shape, seed=B)
    d = {k: v.to(DEV) for k, v in case.items()}
    N, Din, D, K, P, Pg = shape.N, shape.Din, shape.D, shape.K, shape.P, shape.Pg
    tok = {torch.float32: d["tokens"], BF: d["tokens_bf"]}
    idx = ops.select_topk(d["scores"], K)
    bits = L.load().pph_addon_tc2_supported(B, N, Din, D, K)
    ws_tc = ops._ws("pph_addon_tc2_ws_bytes", B, N, Din, D, K, zero=True, device=DEV)
    name = ops.token_entry
    ran = []

    def fwd(entry):
        out = {}
        for dt, t in tok.items():
            o = _fwd_outputs(shape)
            entry(name, dt, t, o)
            out[dt] = o
        torch.cuda.synchronize()
        return out

    # round 1: pph_addon_fwd
    r = fwd(lambda n, dt, t, o: L.call(n("pph_addon_fwd", dt), t, idx, d["Wa"], d["ba"], B, N, Din, D, K,
                                       *[o[k] for k in _FWD[:4]], 0.5, *[o[k] for k in _FWD[4:]]))
    _assert_same(r[BF], r[torch.float32], "pph_addon_fwd")
    Zs, Zc = r[torch.float32]["Zs"], r[torch.float32]["Zc"]
    ran.append("pph_addon_fwd")
    if bits & 1:
        r = fwd(lambda n, dt, t, o: L.call(n("pph_addon_fwd2", dt), t, idx, d["Wa"], d["ba"], B, N, Din, D, K,
                                           *[o[k] for k in _FWD[:4]], 0.5, *[o[k] for k in _FWD[4:]], ws_tc))
        _assert_same(r[BF], r[torch.float32], "pph_addon_fwd2")
        ran.append("pph_addon_fwd2")
    if bits & 8:
        sel = {}

        def sel_fwd(n, dt, t, o):
            o["idx32"] = _e(B, K, dt=torch.int32)
            L.call(n("pph_select_addon_fwd", dt), d["scores"], 1, t, d["Wa"], d["ba"], B, N, Din, D, K, o["idx32"],
                   *[o[k] for k in _FWD[:4]], 0.5, *[o[k] for k in _FWD[4:]], ws_tc)
        r = fwd(sel_fwd)
        _assert_same(r[BF], r[torch.float32], "pph_select_addon_fwd")
        assert torch.equal(r[BF]["idx32"], idx)
        ran.append("pph_select_addon_fwd")
    if L.load().pph_head_prep_supported(B, N, Din, D, K):
        def prep(n, dt, t, o):
            o.update(idx32=_e(B, K, dt=torch.int32), idx64=_e(B, K, dt=torch.int64), P_hi=_e(P, D, dt=BF),
                     P_lo=_e(P, D, dt=BF), p2=_e(P), p2_ctr=_e(P), p2_hi=_e(P), Pg_hi=_e(Pg, D, dt=BF),
                     Pg_lo=_e(Pg, D, dt=BF), pg2=_e(Pg), pg2_ctr=_e(Pg), pg2_hi=_e(Pg))
            L.call(n("pph_head_prep", dt), d["scores"], t, d["Wa"], d["ba"], B, 1, N, Din, D, K, 0.5, o["idx32"], o["idx64"],
                   *[o[k] for k in _FWD], d["P"], P, o["P_hi"], o["P_lo"], o["p2"], o["p2_ctr"], o["p2_hi"],
                   d["Pg"], Pg, o["Pg_hi"], o["Pg_lo"], o["pg2"], o["pg2_ctr"], o["pg2_hi"])
        r = fwd(prep)
        _assert_same(r[BF], r[torch.float32], "pph_head_prep")
        assert torch.equal(r[BF]["idx32"], idx)
        ran.append("pph_head_prep")

    # backward: random upstream gradients of Z (round 1) and of the pre-activation (bwd2 / bwd3)
    g = torch.Generator(device="cpu").manual_seed(B)
    dZs = torch.randn(B, K, D, generator=g).to(DEV)
    dZc = torch.randn(B, D, generator=g).to(DEV)
    dpre_s, dpre_c = (dZs * Zs * (1 - Zs)).contiguous(), (dZc * Zc * (1 - Zc)).contiguous()

    def bwd(entry, zero_dtokens):
        out = {}
        for dt, t in tok.items():
            o = dict(dWa=_e(D, Din), dba=_e(D), dtok=(torch.zeros if zero_dtokens else torch.empty)(
                B, 1 + N, Din, dtype=dt, device=DEV))
            if not zero_dtokens:
                o["dtok"].fill_(float("nan"))                 # every row must be written
            entry(name, dt, t, o)
            out[dt] = o
        torch.cuda.synchronize()
        a, b = out[BF], out[torch.float32]
        return a, b

    ws1 = ops.addon_bwd_workspace(B, N, Din, D, K, DEV)
    a, b = bwd(lambda n, dt, t, o: L.call(n("pph_addon_bwd", dt), t, idx, d["Wa"], Zs, Zc, dZs, dZc, B, N, Din, D, K, ws1,
                                          3, o["dWa"], o["dba"], o["dtok"]), False)
    assert torch.equal(a["dWa"], b["dWa"]) and torch.equal(a["dba"], b["dba"])
    _assert_dtokens(a["dtok"], b["dtok"], idx, "pph_addon_bwd")
    ran.append("pph_addon_bwd")
    if (bits & 6) == 6:
        a, b = bwd(lambda n, dt, t, o: L.call(n("pph_addon_bwd3", dt), 3, t, idx, d["Wa"], dpre_s, dpre_c, None, B, N, Din,
                                              D, K, ws_tc, o["dWa"], o["dba"], o["dtok"]), True)
        assert torch.equal(a["dWa"], b["dWa"]) and torch.equal(a["dba"], b["dba"])
        _assert_dtokens(a["dtok"], b["dtok"], idx, "pph_addon_bwd3")
        ran.append("pph_addon_bwd3")
    if L.load().pph_addon_bwd2_supported(B, N, Din, D, K):
        ws2 = ops._ws("pph_addon_bwd2_ws_bytes", B, N, Din, D, K, zero=True, device=DEV)
        a, b = bwd(lambda n, dt, t, o: L.call(n("pph_addon_bwd2", dt), 3, t, idx, d["Wa"], dpre_s, dpre_c, B, N, Din, D, K,
                                              ws2, o["dWa"], o["dba"], o["dtok"]), False)
        assert torch.equal(a["dWa"], b["dWa"]) and torch.equal(a["dba"], b["dba"])
        _assert_dtokens(a["dtok"], b["dtok"], idx, "pph_addon_bwd2")
        ran.append("pph_addon_bwd2")

    # pph_gather_rows_host: the selected rows of pinned bf16 tokens, bit for bit, nothing else
    host = case["tokens_bf"].pin_memory()
    dst = torch.full((B, 1 + N, Din), float("nan"), dtype=BF, device=DEV)
    L.call("pph_gather_rows_host_bf16tok", host.data_ptr(), idx, B, N, Din, K, dst, 48)
    torch.cuda.synchronize()
    sel = torch.zeros(B, 1 + N, dtype=torch.bool, device=DEV)
    sel[:, 0] = True
    sel.scatter_(1, idx.long() + 1, True)
    assert torch.equal(dst[sel], d["tokens_bf"][sel])
    assert bool(torch.isnan(dst[~sel].float()).all())
    ran.append("pph_gather_rows_host")
    # every twin ran at least at the CUB width (the single-shot forward needs Din <= 192)
    if key == "cub_b64":
        assert set(ran) == set(TWINS), ran


# ----------------------------------------------------------------------------------------------------------------------
# GPU: PPNet with a bf16 backbone
# ----------------------------------------------------------------------------------------------------------------------
class MyVisionTransformer(torch.nn.Module):
    """Fake backbone handing the head preset tokens / CLS-attention (the class NAME matters, protopformer.py:78-81)."""

    def __init__(self, din, n):
        super().__init__()
        self.fc = torch.nn.Linear(din, din)
        self.patch_embed = torch.nn.Module()
        self.patch_embed.num_patches = n
        self.tokens = self.attn = None

    def forward_feature_patch_embed_all(self, x):
        return self.tokens[:, :1], self.tokens[:, 1:]

    def forward_feature_mask_train_direct(self, cls_embed, x_embed, token_attn, reserve_layer_nums):
        return self.tokens, (self.attn, None)


def _ppnet(shape, case):
    from protopformer_b200 import PPNet
    net = PPNet(MyVisionTransformer(shape.Din, shape.N), 224, [shape.P, shape.D, 1, 1], [14, 16, 16, 8.0], shape.C,
                reserve_layers=[11], reserve_token_nums=[shape.K], use_global=True, use_ppc_loss=True,
                ppc_cov_thresh=shape.ppc_cov_thresh, ppc_mean_thresh=shape.ppc_mean_thresh, global_coe=shape.global_coe,
                global_proto_per_class=shape.Pg // shape.C, add_on_layers_type='regular').to(DEV)
    with torch.no_grad():
        net.add_on_layers[0].weight.copy_(case["Wa"].reshape(shape.D, shape.Din, 1, 1))
        net.add_on_layers[0].bias.copy_(case["ba"])
        net.prototype_vectors.copy_(case["P"].reshape(shape.P, shape.D, 1, 1))
        net.prototype_vectors_global.copy_(case["Pg"].reshape(shape.Pg, shape.D, 1, 1))
        net.last_layer.weight.copy_(case["Wl"])
        net.last_layer_global.weight.copy_(case["Wg"])
    net.features.attn = case["scores"].to(DEV)
    return net


def _train_pass(net, tokens, labels, N):
    net.train()
    net.zero_grad(set_to_none=True)
    leaf = tokens.clone().requires_grad_(True)
    net.features.tokens = leaf
    logits, aux = net(torch.zeros(1, device=DEV))
    cov, mean = net.get_PPC_loss(aux[2], aux[3], aux[4], labels)
    loss = F.cross_entropy(logits, labels) + 0.1 * cov + 0.5 * mean
    loss.backward()
    grads = {k: p.grad.clone() for k, p in (("Wa", net.add_on_layers[0].weight), ("ba", net.add_on_layers[0].bias),
                                             ("P", net.prototype_vectors), ("Pg", net.prototype_vectors_global))}
    return dict(logits=logits.detach(), loss=loss.detach(), cov=cov.detach(), mean=mean.detach(), dtokens=leaf.grad,
                **grads)


@pytest.mark.gpu
@pytest.mark.parametrize("key", ["cub_b8", "dogs_b256"])
def test_ppnet_with_a_bf16_backbone_equals_the_fp32_path_and_the_oracle(key):
    shape = synth.SHAPES[key] if key == "cub_b8" else synth.SHAPES[key].with_batch(6)
    case = _bf16_case(shape, seed=3)
    net = _ppnet(shape, case)
    labels = case["labels"].to(DEV)
    t32, t16 = case["tokens"].to(DEV), case["tokens_bf"].to(DEV)
    a, b = _train_pass(net, t16, labels, shape.N), _train_pass(net, t32, labels, shape.N)
    for k in a:
        if k == "dtokens":
            assert a[k].dtype == BF and torch.equal(a[k], b[k].to(BF))      # a bf16 leaf gets a bf16 gradient
        elif k == "P":
            # the autograd PPC backward adds the rows of images that share a label with float atomics (pph_ppc_bwd): dP is
            # reproducible to rounding only, in either token dtype
            assert norm_rel(a[k].cpu(), b[k].cpu()) <= 1e-6, k
        else:
            assert torch.equal(a[k], b[k]), k
    # eval forward, push_forward, push_forward_class_maps
    net.eval()
    outs = {}
    for dt, t in ((BF, t16), (torch.float32, t32)):
        net.features.tokens = t
        with torch.no_grad():
            logits, aux = net(torch.zeros(1, device=DEV))
            outs[dt] = [logits, aux[1].materialize(), aux[2], aux[3], net.push_forward(None)[1],
                        net.push_forward_class_maps(None, labels)[1]]
    torch.cuda.synchronize()
    for x, y in zip(outs[BF], outs[torch.float32]):
        assert torch.equal(x, y)
    # the float64 oracle on the widened tokens, at the tolerances of the fp32 path (tests/test_gpu_parity.py)
    with torch.no_grad():
        route = net.head(t16, net.features.attn).argmin.long().cpu()
    ref = O.head_train_step({k: v for k, v in case.items() if k != "tokens_bf"}, shape, dtype=torch.float64, route=route)
    assert rel_close(a["logits"].cpu(), ref["logits"].float(), 1e-4)
    assert rel_close(a["loss"].cpu(), ref["loss"].float(), 1e-4)
    for k, rk in (("P", "g_P"), ("Wa", "g_Wa"), ("ba", "g_ba")):
        assert norm_rel(a[k].cpu().reshape(ref[rk].shape), ref[rk].float()) < 2e-4, k
    # dtokens: the oracle's gradient within 2e-4 of its largest entry plus the one bf16 rounding (2^-9 relative)
    g_ref = ref["g_tokens"].float().reshape(a["dtokens"].shape)
    err = (a["dtokens"].float().cpu() - g_ref).abs()
    assert bool((err <= 2e-4 * g_ref.abs().max() + 2.0 ** -8 * g_ref.abs()).all())


@pytest.mark.gpu
def test_fp16_tokens_and_bf16_parameters_are_refused_before_any_launch():
    L, ops = _lib(), _ops()
    shape = synth.SHAPES["cub_b8"]
    case = _bf16_case(shape, seed=5)
    d = {k: v.to(DEV) for k, v in case.items()}
    cfg = ops.HeadConfig(K=shape.K)
    args = (d["scores"], d["Wa"], d["ba"], d["P"], d["Pg"], d["Wl"], d["Wg"])
    n0 = L.launch_count()
    with pytest.raises(TypeError, match="float16"):
        ops.head_forward(cfg, d["tokens"].half(), *args)
    with pytest.raises(TypeError, match="float16"):
        ops.addon(d["tokens"].half(), torch.zeros(shape.B, shape.K, dtype=torch.int32, device=DEV), d["Wa"], d["ba"], True)
    for i in range(1, 7):
        bad = list(args)
        bad[i] = bad[i].to(BF)
        with pytest.raises(TypeError, match="bfloat16"):
            ops.head_forward(cfg, d["tokens_bf"], *bad)
    assert L.launch_count() == n0
    from protopformer_b200.graph import GraphedHeadStep
    params = {k: d[k].clone() for k in ("Wa", "ba", "P", "Pg", "Wl", "Wg")}
    with pytest.raises(TypeError, match="float16"):
        GraphedHeadStep(params, cfg, B=shape.B, N=shape.N, C=shape.C, m=shape.m, token_dtype=torch.float16)
    # autocast keeps its float32 cast policy: fp16 tokens are cast there, as before
    with torch.autocast("cuda", dtype=torch.float16):
        out = ops.head_forward(cfg, d["tokens"].half(), *args)
    assert out.logits.dtype == torch.float32


# ----------------------------------------------------------------------------------------------------------------------
# GPU: the graphed step
# ----------------------------------------------------------------------------------------------------------------------
def _graphed(shape, case, token_dtype, variants=None, impl="auto", train_ll=False, mode="fp32"):
    from protopformer_b200.graph import GraphedHeadStep
    cfg = _ops().HeadConfig(K=shape.K, global_coe=shape.global_coe, mode=mode, ppc_cov_thresh=shape.ppc_cov_thresh,
                            ppc_mean_thresh=shape.ppc_mean_thresh)
    params = {k: case[k].to(DEV).clone() for k in ("Wa", "ba", "P", "Pg", "Wl", "Wg")}
    for k in ("Wa", "ba", "P", "Pg") + (("Wl", "Wg") if train_ll else ()):
        params[k].requires_grad_(True)
    step = GraphedHeadStep(params, cfg, B=shape.B, N=shape.N, C=shape.C, m=shape.m, n_slots=2, variants=variants,
                           impl=impl, token_dtype=token_dtype)
    step.load(0, case["tokens_bf"] if token_dtype == BF else case["tokens"], case["scores"], case["labels"])
    torch.cuda.synchronize()
    step.capture()
    return step, params


def _results(step, params):
    f = step.fused
    out = dict(losses=f.losses, logits=f.logits, logits_g=f.logits_g, logits_l=f.logits_l, act_l=f.act_l, dmin_l=f.dmin_l,
               argmin=f.argmin, idx32=f.idx32, Zs=f.Zs, Zc=f.Zc, dtokens=f.dtokens)
    out.update({k: p.grad for k, p in params.items() if p.grad is not None})
    return {k: v.clone() for k, v in out.items()}


def _compare_steps(s16, p16, s32, p32):
    a, b = _results(s16, p16), _results(s32, p32)
    assert a.keys() == b.keys()
    assert s16.impl == s32.impl and s16.kernel_launches_per_step == s32.kernel_launches_per_step
    for k in a:
        if k == "dtokens":
            assert a[k].dtype == BF and torch.equal(a[k], b[k].to(BF)), k
        elif k == "P" and s16.impl == "v1":
            # the round-1 sequence adds the PPC prototype rows with float atomics: reproducible to rounding only
            assert norm_rel(a[k].cpu(), b[k].cpu()) <= 1e-6, k
        else:
            assert torch.equal(a[k], b[k]), k


_S = dict(prep="simt", addon_bwd="simt", bwd="staged", ppc="inline", select="kernel")
_T = dict(prep="tc", addon_bwd="tc", bwd="gather", ppc="late", select="fused")
VARIANTS = [_S, _T, dict(_T, ppc="inline"), dict(_T, ppc="split"), dict(_T, bwd="staged", ppc="split"), dict(_S, bwd="gather"),
            dict(_S, ppc="split"), dict(_T, prep="simt"), dict(_T, addon_bwd="simt"), dict(_T, select="kernel"),
            dict(_T, prep="tc1")]


@pytest.mark.gpu
@pytest.mark.parametrize("variants", VARIANTS)
def test_graphed_bf16_step_equals_the_fp32_step_in_every_variant(variants):
    shape = synth.SHAPES["cub_b8"]
    case = _bf16_case(shape, seed=8)
    s16, p16 = _graphed(shape, case, BF, variants)
    s32, p32 = _graphed(shape, case, torch.float32, variants)
    assert s16.fused.variants == s32.fused.variants == variants
    for s in (s16, s32):
        s.run(0)
    torch.cuda.synchronize()
    _compare_steps(s16, p16, s32, p32)


@pytest.mark.gpu
@pytest.mark.parametrize("key,impl,train_ll,mode", [("cub_b64", "auto", False, "fp32"), ("cub_b64", "v1", False, "fp32"),
                                                    ("cub_b64", "auto", True, "fp32"), ("cub_b64", "v1", True, "fp32"),
                                                    ("cars_b64", "auto", False, "bf16"), ("dogs_b256", "auto", False, "fp32")])
def test_graphed_bf16_step_at_benchmark_shapes_v1_v2_and_trainable_last_layers(key, impl, train_ll, mode):
    shape = synth.SHAPES[key]
    case = _bf16_case(shape, seed=1)
    s16, p16 = _graphed(shape, case, BF, impl=impl, train_ll=train_ll, mode=mode)
    s32, p32 = _graphed(shape, case, torch.float32, impl=impl, train_ll=train_ll, mode=mode)
    if key == "cub_b64" and impl == "auto" and not train_ll:
        assert s16.kernel_launches_per_step == 11
    for _ in range(2):
        for s in (s16, s32):
            s.run(0)
    torch.cuda.synchronize()
    _compare_steps(s16, p16, s32, p32)
    if train_ll:
        assert p16["Wl"].grad is not None and p16["Wg"].grad is not None


@pytest.mark.gpu
def test_graphed_bf16_eval_step():
    shape = synth.SHAPES["dogs_b256"]
    case = _bf16_case(shape, seed=2)
    from protopformer_b200.graph import GraphedHeadStep
    steps = {}
    for dt in (BF, torch.float32):
        cfg = _ops().HeadConfig(K=shape.K, global_coe=shape.global_coe)
        params = {k: case[k].to(DEV).clone() for k in ("Wa", "ba", "P", "Pg", "Wl", "Wg")}
        s = GraphedHeadStep(params, cfg, B=shape.B, N=shape.N, C=shape.C, m=shape.m, train=False, token_dtype=dt)
        s.load(0, case["tokens_bf"] if dt == BF else case["tokens"], case["scores"], case["labels"])
        s.capture()
        s.run(0)
        steps[dt] = s
    torch.cuda.synchronize()
    assert steps[BF].tokens[0].dtype == BF
    assert torch.equal(steps[BF].fused.logits, steps[torch.float32].fused.logits)
    assert torch.equal(steps[BF].fused.losses, steps[torch.float32].fused.losses)


@pytest.mark.gpu
def test_bf16_host_pipeline_moves_half_the_bytes_and_feeds_the_same_step():
    """load_host / capture_load_host / capture_host_overlapped with pinned bf16 tokens: the step's results are bitwise those
    of the fp32 step fed the widened tokens through its own host pipeline."""
    shape = synth.SHAPES["cub_b64"]
    case = _bf16_case(shape, seed=12)
    nxt = _bf16_case(shape, seed=13)
    out = {}
    for dt in (BF, torch.float32):
        step, params = _graphed(shape, case, dt)
        key = "tokens_bf" if dt == BF else "tokens"
        host = [{k: c[k].pin_memory() for k in (key, "scores", "labels")} for c in (case, nxt)]
        step.tokens[0].detach().fill_(float("nan"))
        moved = step.load_host(0, host[0][key], host[0]["scores"], host[0]["labels"])
        B, N, K, Din = shape.B, shape.N, shape.K, shape.Din
        assert moved == 4 * B * N + 8 * B + (2 if dt == BF else 4) * B * (K + 1) * Din
        step.capture_host_pipeline()
        g_load = step.capture_load_host(1, host[1][key], host[1]["scores"], host[1]["labels"])
        g_over = step.capture_host_overlapped(0, host[1][key], host[1]["scores"], host[1]["labels"])
        step.load_host(0, host[0][key], host[0]["scores"], host[0]["labels"])
        lh0 = step.run_host(0).clone()
        torch.cuda.synchronize()
        r0 = _results(step, params)
        g_load.replay()
        lh1 = step.run_host(1).clone()
        torch.cuda.synchronize()
        r1 = _results(step, params)
        step.load_host(0, host[0][key], host[0]["scores"], host[0]["labels"])
        g_over.replay()                           # step of slot 0 || transfer of the next batch into slot 1
        torch.cuda.synchronize()
        r2 = _results(step, params)
        assert torch.equal(r2["losses"], r0["losses"])
        out[dt] = (lh0, lh1, r0, r1, step.kernel_launches_per_step)
        if dt == BF:
            with pytest.raises(TypeError):
                step.load_host(0, case["tokens"].pin_memory(), host[0]["scores"], host[0]["labels"])
    a, b = out[BF], out[torch.float32]
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1]) and a[4] == b[4] == 11
    for ra, rb in ((a[2], b[2]), (a[3], b[3])):
        for k in ra:
            if k == "dtokens":
                sel = torch.zeros(shape.B, shape.N + 1, dtype=torch.bool, device=DEV)
                sel[:, 0] = True
                sel.scatter_(1, ra["idx32"].long() + 1, True)
                assert torch.equal(ra[k][sel], rb[k][sel].to(BF))
            elif k != "idx32":                   # the host pipeline's selection lives in the transfer's own buffer
                assert torch.equal(ra[k], rb[k]), k
