"""Attention rollout on bf16 and fp16 attention maps (pph_rollout_scores_{bf16,f16}attn, pph_rollout_cls_rows_*attn).

Every half-precision value is exact in fp32, so the twins must give, bit for bit, what the fp32 entry points give on the
widened maps -- the result the rollout had on half maps when it made an fp32 copy of every layer first -- and must hold
the oracle's bar on those widened maps."""
import ctypes

import pytest
import torch

from oracle import rollout_oracle as R
from tests.test_rollout_oracle import CAIT_CASES, ROLLOUT_CASES, load_cait, load_rollout
from tests.util import FakeCait, FakeDeit, max_rel, rel_close

DEV = "cuda:0"
HALF = {"bf16": torch.bfloat16, "fp16": torch.float16}
TWINS = ("pph_rollout_scores_bf16attn", "pph_rollout_scores_f16attn",
         "pph_rollout_cls_rows_bf16attn", "pph_rollout_cls_rows_f16attn")
# the shapes of tests/test_rollout_gpu.py::test_rollout_against_oracle_shapes (T = 2, odd T*T, T = 224, H = 1 and the
# runtime-H kernel at H = 5, L = 24) and the DeiT-Ti / DeiT-S shapes at B = 64
ORACLE_SHAPES = [(1, 1, 1, 2, "mean"), (2, 3, 1, 33, "min"), (5, 4, 3, 64, "mean"), (3, 2, 5, 100, "mean"),
                 (12, 5, 6, 197, "mean"), (2, 1, 4, 224, "max"), (24, 3, 4, 196, "mean")]
DEIT_SHAPES = [(11, 64, 3, 197), (11, 64, 6, 197)]


def _ops():
    from protopformer_b200 import ops
    return ops


def _half_maps(maps, dt):
    return [m.to(DEV).to(dt) for m in maps]


def _widened(maps):
    return [m.float() for m in maps]


def _assert_same_as_widened(maps, **kw):
    """Half maps through the twin == their fp32 widening through the fp32 entry, bit for bit (scores and index lists)."""
    ops = _ops()
    got = ops.rollout_scores(maps, **kw)
    want = ops.rollout_scores(_widened(maps), **kw)
    if isinstance(got, tuple):
        for g, w in zip(got, want):
            assert torch.equal(g, w)
    else:
        assert torch.equal(got, want)
    return got


# ---------------------------------------------------------------------------------------------------------------------
# CPU: the C ABI refuses bad arguments before touching a device
# ---------------------------------------------------------------------------------------------------------------------
def test_twins_are_declared_and_validate_arguments_without_a_device():
    from protopformer_b200 import _lib
    from tests.test_host_cpu import _header_functions
    decl = _header_functions()
    for name in TWINS:
        assert name in decl and name in _lib.SIGNATURES
        base = name.rsplit("_", 1)[0]
        assert decl[name] == decl[base] and _lib.SIGNATURES[name] == _lib.SIGNATURES[base]
    lib = _lib.load()
    tbl = (ctypes.c_void_p * 33)(*([16] * 33))        # non-null fake device pointers: never dereferenced on refusal
    ws = ctypes.c_void_p(16)
    for name in TWINS[:2]:
        f = getattr(lib, name)
        assert f(None, 1, 1, 1, 8, 0, 0, 0.2, None, 1, ws, ws, 0, None, None, None) == -1
        assert name.encode() in lib.pph_last_error_string() and b"null" in lib.pph_last_error_string()
        assert f(tbl, 33, 1, 1, 8, 0, 0, 0.2, None, 1, ws, ws, 0, None, None, None) == -2          # L > 32
        assert f(tbl, 1, 1, 1, 225, 0, 0, 0.2, None, 1, ws, ws, 0, None, None, None) == -2         # T > 224
        assert f(tbl, 1, 1, 1, 8, 0, 3, 0.2, None, 1, ws, ws, 0, None, None, None) == -1           # bad fusion
        assert f(tbl, 1, 1, 1, 8, 0, -1, 0.2, None, 1, ws, ws, 0, None, None, None) == -1
    for name in TWINS[2:]:
        f = getattr(lib, name)
        assert f(None, 1, 1, 1, 8, 0, 0, 0.2, ws, None) == -1
        assert f(tbl, 33, 1, 1, 8, 0, 0, 0.2, ws, None) == -2
        assert f(tbl, 1, 1, 1, 257, 0, 0, 0.2, ws, None) == -2
        assert f(tbl, 1, 1, 1, 8, 0, 3, 0.2, ws, None) == -1


# ---------------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("dt", list(HALF))
@pytest.mark.parametrize("L,B,H,T,fusion", ORACLE_SHAPES)
def test_half_maps_equal_widened_maps_and_the_oracle(dt, L, B, H, T, fusion):
    attn = R.synth_attention(L, B, H, T, seed=L + T)
    maps = _half_maps(attn, HALF[dt])
    got = _assert_same_as_widened(maps, head_fusion=fusion)
    want = R.rollout_cls_row([m.float().cpu() for m in maps], 0.9, fusion)
    assert rel_close(got.cpu(), want, 1e-5, 1e-9), max_rel(got.cpu(), want, 1e-9)
    full = _assert_same_as_widened(maps, head_fusion=fusion, drop_first=False)
    assert rel_close(full.sum(-1).cpu(), torch.ones(B), 1e-5)


@pytest.mark.gpu
@pytest.mark.parametrize("dt", list(HALF))
@pytest.mark.parametrize("L,B,H,T", DEIT_SHAPES)
def test_half_maps_at_deit_shapes_all_fusions_and_fused_topk(dt, L, B, H, T):
    g = torch.Generator(device=DEV).manual_seed(L * H)
    maps = [torch.softmax(2.0 * torch.randn(B, H, T, T, device=DEV, generator=g), dim=-1).to(HALF[dt])
            for _ in range(L)]
    for fusion in ("mean", "max", "min"):
        _assert_same_as_widened(maps, head_fusion=fusion)
    s, i32, i64 = _assert_same_as_widened(maps, topk=81, want_int64=True)
    assert torch.equal(i32, _ops().select_topk(s, 81)) and torch.equal(i64, i32.long())


@pytest.mark.gpu
@pytest.mark.parametrize("dt", list(HALF))
def test_half_maps_discard_ratios_start_row_and_odd_base_address(dt):
    attn = R.synth_attention(4, 3, 2, 197, seed=11)
    maps = _half_maps(attn, HALF[dt])
    wide = [m.float().cpu() for m in maps]
    v0 = torch.rand(3, 197, generator=torch.Generator().manual_seed(1))
    got = _assert_same_as_widened(maps, v0=v0.to(DEV), drop_first=False)
    assert rel_close(got.cpu(), R.rollout_cls_row(wide, v0=v0, drop_first=False), 1e-5, 1e-9)
    for ratio in (0.0, 0.2, 0.5, 1.0):           # 0.0 and 0.2: entry lists too long for the staged chain kernel
        got = _assert_same_as_widened(maps, discard_ratio=ratio, drop_first=False)
        assert rel_close(got.cpu(), R.rollout_cls_row(wide, ratio, "mean", drop_first=False), 1e-5, 1e-9), ratio
    # maps whose storage starts 2 bytes past a 4-byte boundary (a view at an odd element offset)
    odd = []
    for m in maps:
        buf = torch.empty(m.numel() + 1, dtype=m.dtype, device=DEV)
        v = buf[1:].view(m.shape)
        v.copy_(m)
        assert v.data_ptr() % 4 == 2
        odd.append(v)
    assert torch.equal(_ops().rollout_scores(odd), _ops().rollout_scores(maps))


@pytest.mark.gpu
@pytest.mark.parametrize("dt", list(HALF))
def test_half_maps_ties_at_the_threshold(dt):
    """Half maps tie at the discard threshold far more often than fp32 maps; with H = 1 the fused values are half values
    themselves.  The rule is the oracle's: among equal entries the lowest flat index is discarded first."""
    g = torch.Generator().manual_seed(5)
    soft = [torch.softmax(2.0 * torch.randn(2, 1, 197, 197, generator=g), dim=-1) for _ in range(3)]
    quant = [torch.randint(1, 6, (2, 2, 40, 40), generator=g).float() / 8.0 for _ in range(3)]
    for attn in (soft, quant):
        maps = _half_maps(attn, HALF[dt])
        wide = [m.float().cpu() for m in maps]
        got = _assert_same_as_widened(maps)
        want = R.rollout_cls_row(wide, 0.9, "mean")
        assert rel_close(got.cpu(), want, 1e-5, 1e-9), max_rel(got.cpu(), want, 1e-9)
    s2, i32 = _assert_same_as_widened(_half_maps(quant, HALF[dt]), discard_ratio=1.0, topk=7)
    assert torch.equal(i32.cpu(), torch.arange(7, dtype=torch.int32).repeat(2, 1))


@pytest.mark.gpu
@pytest.mark.parametrize("dt", list(HALF))
@pytest.mark.parametrize("name", list(ROLLOUT_CASES))
def test_half_maps_of_the_reference_fixtures(dt, name):
    attn, _, fusion, K = load_rollout(name)
    _assert_same_as_widened(_half_maps(attn, HALF[dt]), head_fusion=fusion, topk=K, want_int64=True)


@pytest.mark.gpu
@pytest.mark.parametrize("dt", list(HALF))
@pytest.mark.parametrize("name", list(CAIT_CASES))
def test_cait_half_patch_and_class_maps(dt, name):
    attn, _, n_patch, _ = load_cait(name)
    ops = _ops()
    full = [a.to(DEV) for a in attn]
    half = [a.to(HALF[dt]) for a in full]
    want = ops.rollout_scores_cait([a.float() for a in half], n_patch)
    for maps in (half, half[:n_patch] + [a.float() for a in half[n_patch:]],
                 [a.float() for a in half[:n_patch]] + half[n_patch:]):
        assert torch.equal(ops.rollout_scores_cait(maps, n_patch), want)
    for fusion in ("max", "min"):
        assert torch.equal(ops.rollout_scores_cait(half, n_patch, head_fusion=fusion),
                           ops.rollout_scores_cait([a.float() for a in half], n_patch, head_fusion=fusion))


@pytest.mark.gpu
@pytest.mark.parametrize("dt", list(HALF))
def test_half_maps_make_no_fp32_copy(dt):
    L, B, H, T = DEIT_SHAPES[0]
    ops = _ops()
    g = torch.Generator(device=DEV).manual_seed(2)
    maps = [torch.softmax(2.0 * torch.randn(B, H, T, T, device=DEV, generator=g), dim=-1).to(HALF[dt])
            for _ in range(L)]
    ws = ops.rollout_workspace(L, B, T, int(T * T * 0.9), DEV)
    ops.rollout_scores(maps, workspace=ws, topk=81)                        # library loaded, kernels warm
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    s, i32 = ops.rollout_scores(maps, workspace=ws, topk=81)
    torch.cuda.synchronize()
    outputs = s.numel() * 4 + i32.numel() * 4
    rise = torch.cuda.max_memory_allocated() - base
    assert rise <= outputs + 2 * 512, (rise, outputs)                      # allocator rounds each block to 512 B


@pytest.mark.gpu
@pytest.mark.parametrize("dt", list(HALF))
def test_half_maps_reproducible_batch_independent_and_graph_capturable(dt):
    ops = _ops()
    maps = _half_maps(R.synth_attention(6, 4, 3, 197, seed=5), HALF[dt])
    a = ops.rollout_scores(maps).clone()
    assert torch.equal(a, ops.rollout_scores(maps))
    perm = torch.tensor([2, 0, 3, 1], device=DEV)
    assert torch.equal(ops.rollout_scores([m[perm].contiguous() for m in maps]), a[perm])
    ws = ops.rollout_workspace(6, 4, 197, int(197 * 197 * 0.9), DEV)
    want = ops.rollout_scores(maps, workspace=ws, topk=20)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        ops.rollout_scores(maps, workspace=ws, topk=20)
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        out = ops.rollout_scores(maps, workspace=ws, topk=20)
    for o in out:
        o.zero_()
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(out[0], want[0]) and torch.equal(out[1], want[1])


class _CastMaps(torch.nn.Module):
    """A block whose attention maps come out in `dtype`, as a half-precision backbone's do."""

    def __init__(self, blk, dtype):
        super().__init__()
        self.blk, self.dtype = blk, dtype

    def forward(self, *args):
        out, attn = self.blk(*args)
        return out, attn.to(self.dtype)


@pytest.mark.gpu
@pytest.mark.parametrize("dt", list(HALF))
def test_backbone_loops_with_half_maps(dt):
    from protopformer_b200.backbone import forward_feature_mask_train_direct, forward_feature_mask_train_direct_cait
    ops = _ops()
    dtype = HALF[dt]
    gen = torch.Generator().manual_seed(104)
    net = FakeDeit(24, 3, 7).to(DEV)
    net.blocks = torch.nn.ModuleList([_CastMaps(b, dtype) for b in net.blocks])
    cls_embed, x_embed = torch.randn(2, 1, 24, generator=gen).to(DEV), torch.randn(2, 49, 24, generator=gen).to(DEV)
    reserve = [(3, 25), (5, 9)]

    def widened(all_attn, **kw):
        assert all(a.dtype == dtype for a in all_attn)
        return ops.rollout_scores(_widened(all_attn), **kw)

    with torch.no_grad():
        x, (score, _) = forward_feature_mask_train_direct(net, cls_embed, x_embed, None, reserve)
        x2, (score2, _) = forward_feature_mask_train_direct(net, cls_embed, x_embed, None, reserve, rollout=widened)
    assert torch.equal(score, score2) and torch.equal(x, x2)

    cait = FakeCait(32, 2, 5, 2).to(DEV)
    cait.blocks = torch.nn.ModuleList([_CastMaps(b, dtype) for b in cait.blocks])
    cait.blocks_token_only = torch.nn.ModuleList([_CastMaps(b, dtype) for b in cait.blocks_token_only])
    cls_embed, x_embed = torch.randn(3, 1, 32, generator=gen).to(DEV), torch.randn(3, 36, 32, generator=gen).to(DEV)
    with torch.no_grad():
        x, (score, _) = forward_feature_mask_train_direct_cait(cait, cls_embed, x_embed, None, [(1, 16)])
        x2, (score2, _) = forward_feature_mask_train_direct_cait(
            cait, cls_embed, x_embed, None, [(1, 16)],
            rollout_cait=lambda a, pre: ops.rollout_scores_cait(_widened(a), pre))
    assert torch.equal(score, score2) and torch.equal(x, x2)
