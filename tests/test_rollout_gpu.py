"""GPU suite: pph_rollout_scores (csrc/pph_rollout.cu) against the reference fixtures and the oracle."""
import numpy as np
import pytest
import torch

from oracle import rollout_oracle as R
from tests.test_rollout_oracle import CAIT_CASES, ROLLOUT_CASES, load_cait, load_rollout
from tests.util import max_rel, rel_close

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _ops():
    from protopformer_b200 import ops
    return ops


@pytest.mark.parametrize("name", list(ROLLOUT_CASES))
def test_rollout_matches_reference_fixture(name):
    attn, g, fusion, K = load_rollout(name)
    ops = _ops()
    d_attn = [a.to(DEV) for a in attn]
    scores = ops.rollout_scores(d_attn, 0.9, fusion)
    assert scores.shape == g["scores"].shape
    # fp32 tolerance: same arithmetic as the reference in a different association order (vector-matrix chain
    # instead of matrix-matrix products): 1e-5 relative
    assert rel_close(scores.cpu(), g["scores"], 1e-5, 1e-9), max_rel(scores.cpu(), g["scores"], 1e-9)
    idx = ops.select_topk(scores, K)
    assert np.array_equal(idx.cpu().numpy(), g["idx"])                # bit-exact selection downstream
    # the fused form (score reduction + top-K in one launch sequence) returns the same scores and index lists
    s2, i32, i64 = ops.rollout_scores(d_attn, 0.9, fusion, topk=K, want_int64=True)
    assert torch.equal(s2, scores) and torch.equal(i32, idx) and torch.equal(i64, idx.long())


@pytest.mark.parametrize("L,B,H,T,fusion", [(1, 1, 1, 2, "mean"), (2, 3, 1, 33, "min"), (5, 4, 3, 64, "mean"),
                                            (3, 2, 5, 100, "mean"), (12, 5, 6, 197, "mean"), (2, 1, 4, 224, "max"),
                                            (24, 3, 4, 196, "mean")])
def test_rollout_against_oracle_shapes(L, B, H, T, fusion):
    attn = R.synth_attention(L, B, H, T, seed=L + T)
    want = R.rollout_cls_row(attn, 0.9, fusion)
    got = _ops().rollout_scores([a.to(DEV) for a in attn], 0.9, fusion)
    assert rel_close(got.cpu(), want, 1e-5, 1e-9), max_rel(got.cpu(), want, 1e-9)
    # every a_l is row-stochastic, so the CLS row of the product sums to 1 with the dropped CLS column
    full = _ops().rollout_scores([a.to(DEV) for a in attn], 0.9, fusion, drop_first=False)
    assert rel_close(full.sum(-1).cpu(), torch.ones(B), 1e-5)


def test_rollout_threshold_ties_discard_lowest_index_first():
    """A map quantised to few distinct values has massive ties at the threshold: the documented rule applies."""
    g = torch.Generator().manual_seed(3)
    attn = [torch.randint(1, 6, (2, 2, 40, 40), generator=g).float() / 8.0 for _ in range(3)]
    want = R.rollout_cls_row(attn, 0.9, "mean")
    got = _ops().rollout_scores([a.to(DEV) for a in attn], 0.9, "mean")
    assert rel_close(got.cpu(), want, 1e-5, 1e-9), max_rel(got.cpu(), want, 1e-9)
    # tied SCORES (rows the rollout leaves at exactly zero): the fused selection breaks ties like pph_select_topk
    s2, i32 = _ops().rollout_scores([a.to(DEV) for a in attn], 1.0, "mean", topk=7)
    assert torch.equal(i32, _ops().select_topk(s2, 7))
    assert torch.equal(i32.cpu(), torch.arange(7, dtype=torch.int32).repeat(2, 1))      # all-zero scores: first 7 tokens


def test_rollout_start_row_and_discard_ratio_edges():
    attn = R.synth_attention(4, 3, 2, 50, seed=11)
    v0 = torch.rand(3, 50, generator=torch.Generator().manual_seed(1))
    ops = _ops()
    d = [a.to(DEV) for a in attn]
    got = ops.rollout_scores(d, 0.9, "mean", v0=v0.to(DEV), drop_first=False)
    assert rel_close(got.cpu(), R.rollout_cls_row(attn, v0=v0, drop_first=False), 1e-5, 1e-9)
    for ratio in (0.0, 0.5, 1.0):                      # nothing / half / everything discarded (a_l = I at 1.0)
        got = ops.rollout_scores(d, ratio, "mean", drop_first=False)
        assert rel_close(got.cpu(), R.rollout_cls_row(attn, ratio, "mean", drop_first=False), 1e-5, 1e-9), ratio
    one = ops.rollout_scores(d, 1.0, "mean", drop_first=False).cpu()
    assert torch.equal(one, torch.eye(50)[:1].repeat(3, 1))
    # T = 197 below a ratio of about 0.3: a layer's entry list does not fit in shared memory, the chain reads it from
    # global memory instead
    big = R.synth_attention(3, 2, 3, 197, seed=12)
    d = [a.to(DEV) for a in big]
    for ratio in (0.0, 0.2):
        got, want = ops.rollout_scores(d, ratio, "mean").cpu(), R.rollout_cls_row(big, ratio, "mean")
        assert rel_close(got, want, 1e-5, 1e-9), (ratio, max_rel(got, want, 1e-9))


def test_rollout_is_bit_reproducible_and_batch_independent():
    attn = R.synth_attention(6, 4, 3, 197, seed=5)
    ops = _ops()
    d = [a.to(DEV) for a in attn]
    a = ops.rollout_scores(d).clone()
    b = ops.rollout_scores(d)
    assert torch.equal(a, b)
    perm = torch.tensor([2, 0, 3, 1])
    c = ops.rollout_scores([x[perm].contiguous() for x in d])
    assert torch.equal(c, a[perm.to(DEV)])


@pytest.mark.parametrize("name", list(CAIT_CASES))
def test_cait_rollout_matches_reference_fixture(name):
    """pph_rollout_cls_rows + pph_rollout_scores(v0) against the reference's attn_rollout_cait (fixture)."""
    attn, g, n_patch, K = load_cait(name)
    ops = _ops()
    scores = ops.rollout_scores_cait([a.to(DEV) for a in attn], n_patch, 0.9, "mean")
    assert scores.shape == g["scores"].shape
    assert rel_close(scores.cpu(), g["scores"], 1e-5, 1e-9), max_rel(scores.cpu(), g["scores"], 1e-9)
    assert np.array_equal(ops.select_topk(scores, K).cpu().numpy(), g["idx"])


def test_cait_start_row_ties_and_fusions_against_oracle():
    g = torch.Generator().manual_seed(8)
    for fusion in ("mean", "max", "min"):
        attn = R.synth_cait_attention(2, 3, 3, 3, 25, seed=4)
        attn[-1] = torch.randint(1, 4, attn[-1].shape, generator=g).float() / 4.0       # quantised row: ties everywhere
        got = _ops().rollout_scores_cait([a.to(DEV) for a in attn], 2, 0.9, fusion)
        want = R.rollout_cait(attn, 2, 0.9, fusion)
        assert rel_close(got.cpu(), want, 1e-5, 1e-9), (fusion, max_rel(got.cpu(), want, 1e-9))
