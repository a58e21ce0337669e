"""Last layers with dense weights, held to float64 at every class-count and batch-tiling switch of their kernels.

Every other test feeds the last layers the class-connection pattern of synth.make_case (+1 on the own class, -0.5
elsewhere).  With those weights most indexing mistakes in the general product cancel: every off-class entry is the same
-0.5, so reading W[c', p] for W[c, p] gives the same number whenever neither class owns p.  A last-layer fine-tune runs
the general product on every step after the first one, so here the weights are dense, N(0, 1) / sqrt(P), and the two
layers differ.

  1. kernel level, synthetic inputs against float64 computed here:
     pph_head_mid's three-phase LL role (CJ = 4 / 7 / 8; one slice per CTA, proportional split, several slices per CTA
     at one image tile, budget = 2 at B = 4736), its class-sum form on pattern weights (C = 1 ... 256, three (a, b)
     pairs), pph_logits_fwd / pph_logits_bwd (8-class tile tails, 256-prototype tails, the FP32-FMA kernel up to
     C = 1536 and the tcgen05 product at C = 1537);
  2. the graphed step (v2 default and staged / split variants, frozen and trainable last layers, eval; v1 above
     C = 256) and the autograd path (PPNet) against the float64 oracle;
  3. a last-layer fine-tune (GraphedHeadStep + FusedHeadAdamW) from the pattern: gradients against the oracle at the
     current weights after every step;
  4. on the CPU: where fused_step_supported switches, and pph_head_mid's host-side refusal of C > 256.

Bounds: max |a - b| / max |b| per tensor (CE and the losses: relative).  Each bound is at most twice the largest error
measured over its cases on one NVIDIA B200 (1000 W power limit), given in brackets:
  pph_head_mid, three-phase and class-sum forms, and the step's last layers on the step's own activations:
      logits 4e-6 [2.2e-6], CE 2e-6 [1.0e-6], dlogits 6e-6 [3.3e-6], g 6e-6 [3.2e-6]
  pph_logits_fwd 3e-7 [1.7e-7]; pph_logits_bwd FP32-FMA 2e-6 [1.1e-6]
  pph_logits_bwd tcgen05 (C = 1537: the upstream gradient is rounded to bf16 hi + lo, 2^-17 per element) 1.2e-5
      [6.8e-6]: not an FP32 bound, stated for what it is
  step level against the float64 oracle (graphed step v1 / v2, eval, PPNet, fine-tune):
      logits 3.5e-6 [1.9e-6], total loss 2e-7 [9.3e-8], CE 2e-7 [8.6e-8], PPC cov 5e-7 [2.6e-7], PPC mean 8e-7
      [4.3e-7], dtokens 1e-4 [6.5e-5], dP 2e-4 [1.2e-4], dPg 1.2e-5 [6.1e-6], dWa 6e-5 [3.2e-5], dba 4.5e-5
      [2.4e-5], dWl 8e-6 [4.1e-6], dWg 8e-6 [4.1e-6]
  dP is held to 2e-4, the bound tests/test_step2_gpu.py gives the fp32-mode step on its reference fixtures, not to
  1e-4: at B = 130 it measured 1.17e-4.  That error is not the last layers': the step's g is held to 6e-6 on its own
  inputs, and dP carries the similarity kernel's bf16x3 distances (the autograd path, other kernels, measured 9.3e-5).
"""
import ctypes
import math

import pytest
import torch
import torch.nn.functional as F

from oracle import protohead_oracle as O
from protopformer_b200 import synth
from tests.test_last_layer_grad_gpu import _ppnet
from tests.util import norm_rel

DEV = "cuda:0"
EPS = 1e-4
K_SYN = 81                    # token slots of the synthetic argmin (kernel level)

# kernel-level bounds (measured maxima in the module docstring)
TOL_LOGITS, TOL_CE, TOL_DLOGITS, TOL_G = 4e-6, 2e-6, 6e-6, 6e-6
TOL_FWD, TOL_BWD_FMA, TOL_BWD_TC = 3e-7, 2e-6, 1.2e-5
# step level, against the float64 oracle (the graphed step, the eval step, PPNet and the fine-tune loop)
STEP_TOL = dict(logits=3.5e-6, loss=2e-7, ce=2e-7, ppc_cov=5e-7, ppc_mean=8e-7, tokens=1e-4, P=2e-4, Pg=1.2e-5, Wa=6e-5,
                ba=4.5e-5, Wl=8e-6, Wg=8e-6)


def _report(what, err):
    print(f"dense-ll {what}: {err:.3e}")
    return err


def _lib():
    from protopformer_b200 import _lib
    return _lib


def _dense(C, n, g):
    return torch.randn(C, n, generator=g) / math.sqrt(max(n, 1))


def _pattern(C, n, a, b):
    m = n // C
    own = (torch.arange(n)[None, :] // m) == torch.arange(C)[:, None]
    return torch.where(own, torch.tensor(a), torch.tensor(b)).float()


def _dact(dmin):
    d = dmin.double()
    return torch.where(d > 0, 1 / (d + 1) - 1 / (d + EPS), torch.zeros_like(d))


def _synthetic(B, C, P, Pg, seed, W=None, act_hi=4.0):
    """Inputs of the last layers without a similarity kernel: positive activations in (0, act_hi], distances with
    exact zeros (the act'(0) branch), argmin in [0, K), labels that repeat; dense last layers unless W = (Wl, Wg)."""
    g = torch.Generator().manual_seed(seed)
    x = dict(act_l=act_hi * (1 - torch.rand(B, P, generator=g)), act_g=act_hi * (1 - torch.rand(B, Pg, generator=g)))
    for k, n in (("dmin_l", P), ("dmin_g", Pg)):
        # away from 0 (act'(d) ~ -1 / d there): g then spans a factor of 16, and a bound relative to its largest entry
        # holds every entry, not only those of the smallest distances
        d = 0.5 + 2.5 * torch.rand(B, n, generator=g)
        d[torch.rand(B, n, generator=g) < 0.05] = 0.0
        x[k] = d
    x["argmin"] = torch.randint(0, K_SYN, (B, P), generator=g, dtype=torch.int32)
    lab = torch.randint(0, C, (B,), generator=g)
    lab[1::3] = lab[0]
    x["labels"] = lab
    x["Wl"], x["Wg"] = W if W is not None else (_dense(C, P, g), _dense(C, Pg, g))
    return x


def _ref_last_layers(x, gc, upstream):
    """float64: logits, logits_l, logits_g, CE, dlogits = (softmax - onehot) upstream / B, g_l, g_g."""
    al, ag, Wl, Wg = x["act_l"].double(), x["act_g"].double(), x["Wl"].double(), x["Wg"].double()
    ll, lg = al @ Wl.T, ag @ Wg.T
    lt = gc * lg + (1 - gc) * ll
    B, C = lt.shape
    ce = F.cross_entropy(lt, x["labels"])
    dl = (torch.softmax(lt, 1) - F.one_hot(x["labels"], C).double()) * upstream / B
    g_l = (1 - gc) * (dl @ Wl) * _dact(x["dmin_l"])
    g_g = gc * (dl @ Wg) * _dact(x["dmin_g"])
    return dict(logits=lt, logits_l=ll, logits_g=lg, ce=ce, dlogits=dl, g_l=g_l, g_g=g_g)


# ----------------------------------------------------------------------------------------------------------------------
# pph_head_mid's plan, restated (pph_mid.cu mid_plan): which branch a case takes on this device
# ----------------------------------------------------------------------------------------------------------------------
def _plan(B, P, Pg, sms):
    tiles_b = -(-B // 64)
    nsl_l, nsl_g = -(-P // 32), -(-Pg // 32)
    budget = max(sms // tiles_b, 2 if Pg > 0 else 1)
    if nsl_l + nsl_g <= budget:
        S_l, S_g = nsl_l, nsl_g
    elif Pg > 0:
        S_l = min(max(budget * nsl_l // (nsl_l + nsl_g), 1), budget - 1)
        S_g = budget - S_l
        S_l, S_g = min(S_l, nsl_l), min(S_g, nsl_g)
    else:
        S_l, S_g = min(budget, nsl_l), 0
    if nsl_l + nsl_g <= budget:
        branch = "one-slice"                     # keepW: phase 3 reuses the W slice of phase 1
    elif budget == 2:
        branch = "budget2"
    else:
        branch = "split"
    multi = nsl_l > S_l or nsl_g > S_g           # some CTA walks several slices (phase 3 restages W)
    return dict(tiles_b=tiles_b, budget=budget, branch=branch, multi=multi, n_ll=tiles_b * (S_l + S_g))


def _mid_tail(ws, B, P, Pg, C):
    """The part of pph_head_mid's workspace only the three-phase role writes (dlT, then the partial logits): behind the
    pattern records, the counters, the PPC losses and the per-image CE and PPC terms (pph_mid.cu mid_carve).  The whole
    layout is restated and held to the size pph_head_mid_ws_bytes reports, so a change of mid_carve fails here instead
    of pointing the check at another region."""
    r = lambda n: (n + 255) // 256 * 256  # noqa: E731
    Cp, Bp = (C + 3) // 4 * 4, (B + 63) // 64 * 64
    S = -(-P // 32) + -(-Pg // 32)                    # the size query plans for unlimited CTAs: one slice each
    head = r(40) + r(4 * 8) + r(4 * 2) + r(4 * B) + r(8 * B)
    assert ws.numel() == max(head + r(4 * Cp * Bp) + r(4 * S * B * Cp) + 256, 256), "pph_mid.cu mid_carve changed"
    return ws[head:]


def _run_mid(x, B, C, P, Pg, gc, upstream, train, ws=None, pattern=False):
    """pph_head_mid with use_ppc = 0; a zeroed workspace carries no verdict (three-phase role) unless `pattern` runs
    pph_last_layer_pattern on it first.  Returns the outputs and the workspace."""
    L, ops = _lib(), _ops()
    d = {k: v.to(DEV).contiguous() for k, v in x.items()}
    Bp = (B + 63) // 64 * 64
    e = lambda *s: torch.full(s, float("nan"), device=DEV)  # noqa: E731
    o = dict(logits=e(B, C), logits_g=e(B, C), logits_l=e(B, C), losses=torch.zeros(4, device=DEV), dlogits=e(B, C),
             g_l=e(B, P), g_g=e(B, Pg), pairT=e(P + Pg, Bp, 2))
    if ws is None:
        ws = ops._ws("pph_head_mid_ws_bytes", B, K_SYN, 16, P, Pg, C, 1, zero=True, device=DEV)
    bins = ops._ws("pph_similarity_bwd2_ws_bytes", B, K_SYN, 16, P, zero=True, device=DEV)
    if pattern:
        L.call("pph_last_layer_pattern", d["Wl"], P, d["Wg"], Pg, C, ws)
    L.call("pph_head_mid", d["act_l"], d["act_g"], d["dmin_l"], d["dmin_g"], d["argmin"], d["Wl"], d["Wg"], d["labels"],
           B, K_SYN, 16, P, Pg, C, 1, 196, float(gc), 0, EPS, float(upstream), 1 if train else 0, 0,
           None, None, None, None, None, 0.0, 0.0, 0.0, 0.0, ws, bins if train else None,
           o["logits"], o["logits_g"], o["logits_l"], o["losses"], o["dlogits"] if train else None,
           o["g_l"] if train else None, o["g_g"] if train else None, o["pairT"] if train else None, None, None, None)
    torch.cuda.synchronize()
    return o, ws


def _ops():
    from protopformer_b200 import ops
    return ops


def _check_mid(o, x, ref, B, P, Pg, train, tag):
    for k, tol in (("logits", TOL_LOGITS), ("logits_l", TOL_LOGITS), ("logits_g", TOL_LOGITS)):
        if k == "logits_g" and Pg == 0:
            continue
        assert _report(f"{tag} {k}", norm_rel(o[k].cpu(), ref[k])) <= tol, k
    ce, want = float(o["losses"][1]), float(ref["ce"])
    if want == 0.0:                                       # C = 1: log-sum-exp of one logit minus itself, exactly
        assert ce == 0.0
    else:
        assert _report(f"{tag} ce", abs(ce - want) / abs(want)) <= TOL_CE
    assert float(o["losses"][0]) == ce                    # no PPC role: total = CE
    if not train:
        return
    assert _report(f"{tag} dlogits", norm_rel(o["dlogits"].cpu(), ref["dlogits"])) <= TOL_DLOGITS
    for k, n in (("g_l", P), ("g_g", Pg)):
        if n == 0:
            continue
        got = o[k].cpu()
        if float(ref[k].abs().max()) == 0.0:              # C = 1: softmax = onehot, nothing flows back
            assert float(got.abs().max()) == 0.0
        else:
            assert _report(f"{tag} {k}", norm_rel(got, ref[k])) <= TOL_G, k
        dz = (x["dmin_l"] if k == "g_l" else x["dmin_g"]) == 0
        assert bool((got[dz] == 0).all())                 # act'(0) = 0
    pt = o["pairT"].cpu()
    assert torch.equal(pt[:P, :B, 0], o["g_l"].cpu().T) and torch.equal(pt[P:, :B, 0], o["g_g"].cpu().T)
    assert torch.equal(pt[:P, :B, 1].contiguous().view(torch.int32), x["argmin"].T.contiguous())
    assert bool((pt[P:, :B, 1].contiguous().view(torch.int32) == K_SYN).all())
    assert bool((pt[:, B:] == 0).all())                   # the padded image columns are zeros


_OUTS = ("logits", "logits_g", "logits_l", "losses", "dlogits", "g_l", "g_g", "pairT")


def _same(a, b, train):
    for k in _OUTS if train else ("logits", "logits_g", "logits_l", "losses"):
        assert torch.equal(a[k].view(torch.int32), b[k].view(torch.int32)), k      # bitwise (NaN payloads included)


# (B, C, P, Pg, gc, upstream, train, branch, tiles_b): C covers CJ = 4 (C <= 128), 7 (<= 224) and 8 (<= 256) with
# the tails of the 32-class register blocks; P, Pg are never multiples of 32; branch is what mid_plan takes on a
# 148-SM B200 ("one-slice": every CTA keeps its W slice for phase 3, "split": prototype groups shared out between the
# layers, "budget2": B = 4736, the largest batch fused_step_supported admits, one CTA per SM).
MID_CASES = [
    (1, 2, 37, 23, 0.3, 1.0, True, "one-slice", 1),
    (63, 7, 3001, 1999, 0.0, 65536.0, True, "split", 1),          # P + Pg > 4736 at one image tile
    (64, 31, 6017, 1015, 1.0, 1.0, True, "split", 1),
    (65, 32, 1001, 501, 0.3, 1.0, True, "one-slice", 2),
    (129, 33, 2011, 1013, 0.3, 65536.0, True, "split", 3),
    (129, 33, 2011, 1013, 0.3, 1.0, False, "split", 3),
    (256, 128, 1990, 997, 0.3, 1.0, True, "split", 4),
    (1024, 129, 2003, 1001, 0.3, 65536.0, True, "split", 16),
    (64, 224, 161, 95, 0.3, 1.0, True, "one-slice", 1),
    (65, 225, 4001, 801, 0.0, 65536.0, True, "split", 2),
    (1, 256, 5000, 300, 0.3, 1.0, True, "split", 1),
    (63, 129, 4999, 0, 0.0, 1.0, True, "split", 1),                # no global layer
    (4736, 256, 2570, 1290, 0.3, 1.0, True, "budget2", 74),
    (4736, 200, 2010, 1990, 1.0, 65536.0, False, "budget2", 74),
]


@pytest.mark.gpu
@pytest.mark.parametrize("B,C,P,Pg,gc,upstream,train,branch,tiles_b", MID_CASES)
def test_head_mid_three_phase_role_matches_float64(B, C, P, Pg, gc, upstream, train, branch, tiles_b):
    sms = _lib().load().pph_sm_count()
    plan = _plan(B, P, Pg, sms)
    assert (plan["branch"], plan["tiles_b"]) == (branch, tiles_b), (sms, plan)
    assert plan["multi"] == (branch != "one-slice")          # a split leaves some CTA with several slices
    assert plan["n_ll"] <= sms                             # every LL CTA co-resident
    x = _synthetic(B, C, P, Pg, seed=B * 1000 + C)
    ref = _ref_last_layers(x, gc, upstream)
    o1, ws = _run_mid(x, B, C, P, Pg, gc, upstream, train)
    assert bool((_mid_tail(ws, B, P, Pg, C) != 0).any())   # the three-phase role ran (class-sum never writes there)
    tag = f"mid B{B} C{C}"
    _check_mid(o1, x, ref, B, P, Pg, train, tag)
    o2, _ = _run_mid(x, B, C, P, Pg, gc, upstream, train, ws=ws)       # replay on the same workspace
    _same(o1, o2, train)


# (B, C, m, mg, a, b, gc, upstream, act_hi).  act_hi = 0.06: activations of the initialised head (distances of ~30
# give log(31 / 30) ~ 0.03), where the pattern's b T offset of the logits is small and the general product is held to
# the same bound.  act_hi = 4 (every prototype near a token): the logits carry b T ~ 1e3, which costs the general
# product digits in FP32 (rounding of ~1e3 moves the softmax by ~1e-4); the class-sum form leaves that term out of the
# softmax, so only it is held to the bound there and the general product's error is reported.
CLASS_SUM_CASES = [
    (7, 1, 40, 9, 1.0, -0.5, 0.3, 1.0, 0.06),
    (9, 2, 13, 7, 2.0, -1.0, 0.3, 65536.0, 0.06),
    (64, 200, 10, 10, 1.0, -0.5, 0.5, 1.0, 0.06),
    (130, 200, 10, 5, 1.0, 0.0, 0.3, 1.0, 0.06),
    (65, 256, 10, 5, 2.0, -1.0, 0.3, 1.0, 0.06),
    (1, 256, 3, 1, 1.0, 0.0, 1.0, 65536.0, 0.06),
    (64, 200, 10, 10, 1.0, -0.5, 0.5, 1.0, 4.0),
    (65, 256, 10, 5, 2.0, -1.0, 0.3, 65536.0, 4.0),
]


@pytest.mark.gpu
@pytest.mark.parametrize("B,C,m,mg,a,b,gc,upstream,act_hi", CLASS_SUM_CASES)
def test_head_mid_class_sum_form_matches_float64_and_the_general_form(B, C, m, mg, a, b, gc, upstream, act_hi):
    P, Pg = C * m, C * mg
    W = (_pattern(C, P, a, b), _pattern(C, Pg, a, b))
    x = _synthetic(B, C, P, Pg, seed=7 * B + C, W=W, act_hi=act_hi)
    ref = _ref_last_layers(x, gc, upstream)
    runs = []
    for _ in range(2):
        o, ws = _run_mid(x, B, C, P, Pg, gc, upstream, True, pattern=True)
        rec_i, rec_f = ws[:32].view(torch.int32).cpu(), ws[:32].view(torch.float32).cpu()
        # the class-sum role cleared the verdicts it used and left (a, b); it never touches the three-phase scratch
        assert int(rec_i[0]) == 0 and int(rec_i[4]) == 0
        assert (float(rec_f[1]), float(rec_f[2])) == (a, b if C > 1 else a)
        assert not bool((_mid_tail(ws, B, P, Pg, C) != 0).any())
        runs.append(o)
    _same(runs[0], runs[1], True)
    tag = f"B{B} C{C} ({a},{b}) act<={act_hi}"
    _check_mid(runs[0], x, ref, B, P, Pg, True, f"class-sum {tag}")
    # the general product on the same pattern weights (no verdict)
    gen, ws = _run_mid(x, B, C, P, Pg, gc, upstream, True)
    assert bool((_mid_tail(ws, B, P, Pg, C) != 0).any())
    if act_hi < 1:
        _check_mid(gen, x, ref, B, P, Pg, True, f"general-on-pattern {tag}")
    else:
        for k in ("logits", "dlogits", "g_l", "g_g"):
            _report(f"general-on-pattern {tag} {k} (FP32 conditioning, not bounded)", norm_rel(gen[k].cpu(), ref[k]))


# (B, C, P, Pg): C with tails of the 8-class forward tile up to the largest FP32-FMA backward (8 C floats in 48 KB),
# P, Pg with tails of the 256-prototype blocks
LOGITS_CASES = [(1, 1, 257, 255), (7, 7, 511, 300), (8, 9, 1000, 513), (9, 9, 769, 0), (9, 200, 2049, 1999),
                (65, 257, 2570, 1285), (9, 800, 8000, 801), (8, 1000, 1001, 3000), (65, 1536, 769, 257)]


@pytest.mark.gpu
@pytest.mark.parametrize("extras", [False, True])
@pytest.mark.parametrize("B,C,P,Pg", LOGITS_CASES + [(9, 1537, 1537, 520)])
def test_logits_fwd_bwd_dense_match_float64(B, C, P, Pg, extras):
    L = _lib()
    gc = 0.3
    x = _synthetic(B, C, P, Pg, seed=B + 31 * C)
    d = {k: v.to(DEV).contiguous() for k, v in x.items()}
    g = torch.Generator().manual_seed(C)
    dl, dlg, dll = (torch.randn(B, C, generator=g) / B for _ in range(3))
    ref = _ref_last_layers(x, gc, 1.0)
    lt, lg, ll = (torch.full((B, C), float("nan"), device=DEV) for _ in range(3))
    L.call("pph_logits_fwd", d["act_l"], d["act_g"] if Pg else None, d["Wl"], d["Wg"] if Pg else None, B, P, Pg, C, gc,
           lt, lg, ll)
    up_l = (1 - gc) * dl.double() + (dll.double() if extras else 0)
    up_g = gc * dl.double() + (dlg.double() if extras else 0)
    ref_gl = (up_l @ x["Wl"].double()) * _dact(x["dmin_l"])
    ref_gg = (up_g @ x["Wg"].double()) * _dact(x["dmin_g"])
    outs = []
    for _ in range(2):
        g_l, g_g = torch.full((B, P), float("nan"), device=DEV), torch.full((B, Pg), float("nan"), device=DEV)
        L.call("pph_logits_bwd", dl.to(DEV), dlg.to(DEV) if extras else None, dll.to(DEV) if extras else None,
               d["Wl"], d["Wg"] if Pg else None, d["dmin_l"], d["dmin_g"] if Pg else None, B, P, Pg, C, gc, 0, EPS,
               g_l, g_g if Pg else None)
        torch.cuda.synchronize()
        outs.append((g_l.cpu(), g_g.cpu()))
    tag = f"logits B{B} C{C} P{P} Pg{Pg}"
    for k, got in (("logits", lt), ("logits_l", ll)) + ((("logits_g", lg),) if Pg else ()):
        assert _report(f"{tag} fwd {k}", norm_rel(got.cpu(), ref[k])) <= TOL_FWD, k
    tol = TOL_BWD_FMA if 8 * C * 4 <= 48 * 1024 else TOL_BWD_TC     # C = 1537: tcgen05, bf16 hi + lo upstream
    kind = "fma" if 8 * C * 4 <= 48 * 1024 else "tcgen05"
    for (got, want), n in ((outs[0][0], ref_gl), P), ((outs[0][1], ref_gg), Pg):
        if n:
            assert _report(f"{tag} bwd[{kind}] extras={extras}", norm_rel(got, want)) <= tol
    for a, b in zip(*outs):
        assert torch.equal(a, b)


# ----------------------------------------------------------------------------------------------------------------------
# 2. the training step against the float64 oracle
# ----------------------------------------------------------------------------------------------------------------------
def _shape(B, C, m=10, mg=5, P=None, Pg=None):
    P = C * m if P is None else P
    Pg = C * mg if Pg is None else Pg
    return synth.HeadShape(f"dense_b{B}_c{C}", B, 196, 192, 192, 81, P, Pg, C, 0.5, 1.0, 2.0)


def _dense_case(shape, seed):
    case = synth.make_case(shape, seed=seed)
    g = torch.Generator().manual_seed(500 + seed)
    case["Wl"], case["Wg"] = _dense(shape.C, shape.P, g), _dense(shape.C, shape.Pg, g)
    return case


def _oracle(case, shape, route):
    """float64 autograd of the CPU restatement with every head input trainable: loss = CE + 0.1 L_cov + 0.5 L_mean
    (tests/test_last_layer_grad_gpu.py::_oracle, with the forward values kept)."""
    c = {k: (v.detach().clone().double() if v.is_floating_point() else v.clone()) for k, v in case.items()}
    for k in ("tokens", "P", "Pg", "Wa", "ba", "Wl", "Wg"):
        c[k].requires_grad_(True)
    out = O.head_forward(c, shape.K, shape.global_coe, route=route)
    ce = F.cross_entropy(out["logits"], c["labels"])
    cov, mean = O.ppc_loss(out["act_map"], out["idx"], c["labels"], shape.m, shape.N, shape.ppc_cov_thresh,
                           shape.ppc_mean_thresh)
    loss = ce + 0.1 * cov + 0.5 * mean
    loss.backward()
    res = {k: c[k].grad for k in ("tokens", "P", "Pg", "Wa", "ba", "Wl", "Wg")}
    res.update(logits=out["logits"].detach(), losses=torch.stack([loss, ce, cov, mean]).detach(), idx=out["idx"])
    return res


def _make_step(shape, case, train=True, train_ll=False, variants=None, impl="auto"):
    from protopformer_b200 import ops
    from protopformer_b200.graph import GraphedHeadStep
    cfg = ops.HeadConfig(K=shape.K, global_coe=shape.global_coe, mode="fp32", ppc_cov_thresh=shape.ppc_cov_thresh,
                         ppc_mean_thresh=shape.ppc_mean_thresh)
    params = {k: case[k].to(DEV).clone() for k in ("Wa", "ba", "P", "Pg", "Wl", "Wg")}
    for k in ("Wa", "ba", "P", "Pg") + (("Wl", "Wg") if train_ll else ()):
        params[k].requires_grad_(train)
    step = GraphedHeadStep(params, cfg, B=shape.B, N=shape.N, C=shape.C, m=shape.m, train=train, variants=variants,
                           impl=impl)
    step.load(0, case["tokens"], case["scores"], case["labels"])
    torch.cuda.synchronize()
    step.capture()
    return step, params


def _run_step(step):
    """One replay; returns whether pph_head_mid took the three-phase LL role (v2 only)."""
    if step.impl != "v2":
        step.run(0)
        torch.cuda.synchronize()
        return True
    B, _, _, _, P, Pg, C, _, _ = step.fused.dims
    tail = _mid_tail(step.fused.ws_mid, B, P, Pg, C)
    tail.zero_()
    step.run(0)
    torch.cuda.synchronize()
    return bool((tail != 0).any())


def _check_ll_on_own_inputs(f, params, labels, gc, tag):
    """The step's last layers alone: its logits, dlogits and g against float64 over its own activations and distances
    (held to the kernel-level bounds; the oracle comparison below also carries the similarity kernel's rounding)."""
    x = dict(act_l=f.act_l.cpu(), act_g=f.act_g.cpu(), dmin_l=f.dmin_l.cpu(), dmin_g=f.dmin_g.cpu(), labels=labels,
             Wl=params["Wl"].detach().cpu(), Wg=params["Wg"].detach().cpu())
    ref = _ref_last_layers(x, gc, 1.0)
    for k, tol in (("logits", TOL_LOGITS), ("logits_l", TOL_LOGITS), ("logits_g", TOL_LOGITS), ("dlogits", TOL_DLOGITS),
                   ("g_l", TOL_G), ("g_g", TOL_G)):
        assert _report(f"{tag} own-input {k}", norm_rel(getattr(f, k).cpu(), ref[k])) <= tol, k


def _check_grads(params, f, ref, tag, train_ll):
    got = dict(tokens=f.dtokens, P=params["P"].grad, Pg=params["Pg"].grad, Wa=params["Wa"].grad, ba=params["ba"].grad)
    if train_ll:
        got.update(Wl=params["Wl"].grad, Wg=params["Wg"].grad)
    for k, v in got.items():
        e = _report(f"{tag} d{k}", norm_rel(v.cpu().reshape(ref[k].shape), ref[k]))
        assert e <= STEP_TOL[k], (tag, k, e)


# (B, C, extra shape arguments, impl that impl="auto" must choose)
STEP_CASES = [
    (65, 33, dict(m=5, mg=3), "v2"),
    (64, 129, {}, "v2"),
    (65, 225, {}, "v2"),
    (64, 256, {}, "v2"),
    (130, 200, {}, "v2"),                                # three image tiles
    (9, 200, dict(P=8000, Pg=2000), "v2"),               # P + Pg > 148 * 32: several slices per LL CTA
    (8, 257, {}, "v1"),
    (8, 800, dict(P=8000, Pg=800), "v1"),
]


@pytest.mark.gpu
@pytest.mark.parametrize("B,C,kw,impl", STEP_CASES)
def test_graphed_step_dense_last_layers_match_the_oracle(B, C, kw, impl):
    from protopformer_b200 import ops
    shape = _shape(B, C, **kw)
    assert ops.fused_step_supported(B, shape.N, shape.Din, shape.D, shape.K, shape.P, shape.Pg, C, shape.m) == (impl == "v2")
    case = _dense_case(shape, seed=C)
    oracles = {}

    def oracle(route):
        key = route.numpy().tobytes()
        if key not in oracles:
            oracles[key] = _oracle(case, shape, route)
        return oracles[key]

    runs = [(False, None), (True, None)] + ([(True, dict(bwd="staged", ppc="split"))] if impl == "v2" else [])
    for train_ll, variants in runs:
        step, params = _make_step(shape, case, train_ll=train_ll, variants=variants)
        assert step.impl == impl
        assert _run_step(step)                           # dense weights: the general product, never the class-sum form
        f = step.fused
        ref = oracle(f.argmin.cpu().long())
        tag = f"step B{B} C{C} {impl} ll={'train' if train_ll else 'frozen'} {variants or 'default'}"
        assert torch.equal(f.idx32.cpu().long(), ref["idx"])
        _check_ll_on_own_inputs(f, params, case["labels"], shape.global_coe, tag)
        assert _report(f"{tag} logits", norm_rel(f.logits.cpu(), ref["logits"])) <= STEP_TOL["logits"]
        for i, name in enumerate(("loss", "ce", "ppc_cov", "ppc_mean")):
            e = abs(float(f.losses[i]) - float(ref["losses"][i])) / abs(float(ref["losses"][i]))
            assert _report(f"{tag} {name}", e) <= STEP_TOL[name], name
        _check_grads(params, f, ref, tag, train_ll)
        if not train_ll:
            assert params["Wl"].grad is None and params["Wg"].grad is None
        del step, params
    ev, _ = _make_step(shape, case, train=False)
    assert ev.impl == impl and _run_step(ev)
    ref = next(iter(oracles.values()))
    assert _report(f"eval B{B} C{C} logits", norm_rel(ev.fused.logits.cpu(), ref["logits"])) <= STEP_TOL["logits"]
    e = abs(float(ev.fused.losses[1]) - float(ref["losses"][1])) / float(ref["losses"][1])
    assert _report(f"eval B{B} C{C} ce", e) <= STEP_TOL["ce"]


@pytest.mark.gpu
@pytest.mark.parametrize("B,C,kw", [(8, 200, {}), (8, 800, dict(P=8000, Pg=800))])
def test_ppnet_dense_unfrozen_last_layers_match_the_oracle(B, C, kw):
    shape = _shape(B, C, **kw)
    case = _dense_case(shape, seed=3)
    net = _ppnet(shape).cuda()
    with torch.no_grad():
        net.prototype_vectors.copy_(case["P"].reshape(shape.P, shape.D, 1, 1))
        net.prototype_vectors_global.copy_(case["Pg"].reshape(shape.Pg, shape.D, 1, 1))
        net.add_on_layers[0].weight.copy_(case["Wa"].reshape(shape.D, shape.Din, 1, 1))
        net.add_on_layers[0].bias.copy_(case["ba"])
        net.last_layer.weight.copy_(case["Wl"])
        net.last_layer_global.weight.copy_(case["Wg"])
    net.last_layer.weight.requires_grad_(True)
    net.last_layer_global.weight.requires_grad_(True)
    feats = net.features
    feats.tokens, feats.attn = case["tokens"].cuda().requires_grad_(True), case["scores"].cuda()
    labels = case["labels"].cuda()
    net.train()
    logits, aux = net(None)
    cov, mean = net.get_PPC_loss(aux[2], aux[3], aux[4], labels)
    loss = F.cross_entropy(logits, labels) + 0.1 * cov + 0.5 * mean
    loss.backward()
    with torch.no_grad():
        route = net.head(feats.tokens, feats.attn).argmin.long().cpu()
    ref = _oracle(case, shape, route)
    tag = f"ppnet B{B} C{C}"
    assert _report(f"{tag} logits", norm_rel(logits.detach().cpu(), ref["logits"])) <= STEP_TOL["logits"]
    e = abs(float(loss.detach()) - float(ref["losses"][0])) / float(ref["losses"][0])
    assert _report(f"{tag} loss", e) <= STEP_TOL["loss"]
    got = dict(tokens=feats.tokens.grad, P=net.prototype_vectors.grad, Pg=net.prototype_vectors_global.grad,
               Wa=net.add_on_layers[0].weight.grad, Wl=net.last_layer.weight.grad, Wg=net.last_layer_global.weight.grad)
    for k, v in got.items():
        e = _report(f"{tag} d{k}", norm_rel(v.cpu().reshape(ref[k].shape), ref[k]))
        assert e <= STEP_TOL[k], (k, e)


# ----------------------------------------------------------------------------------------------------------------------
# 3. a last-layer fine-tune from the pattern
# ----------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_last_layer_fine_tune_gradients_follow_the_oracle():
    from protopformer_b200.optim import FusedHeadAdamW
    shape = _shape(65, 256)
    case = synth.make_case(shape, seed=6)                 # the pattern init (+1 / -0.5)
    step, p = _make_step(shape, case, train_ll=True)
    assert step.impl == "v2"
    groups = [{"params": [p["P"]], "lr": 2e-3, "weight_decay": 0.05}, {"params": [p["Pg"]], "lr": 2e-3, "weight_decay": 0.05},
              {"params": [p["Wa"], p["ba"]], "lr": 3e-3, "weight_decay": 1e-3},
              {"params": [p["Wl"], p["Wg"]], "lr": 1e-2, "weight_decay": 0.0}]
    opt = FusedHeadAdamW(groups, grads=step.reducer.views)
    for it in range(4):
        general = _run_step(step)
        assert general == (it > 0), it                    # class-sum form on the pattern only: step 1
        cur = dict(case)
        for k in ("P", "Pg", "Wa", "ba", "Wl", "Wg"):
            cur[k] = p[k].detach().cpu()
        ref = _oracle(cur, shape, step.fused.argmin.cpu().long())
        _check_grads(p, step.fused, ref, f"fine-tune step {it + 1}", True)
        opt.step()


# ----------------------------------------------------------------------------------------------------------------------
# 4. CPU: where the step switches, and the host-side refusal
# ----------------------------------------------------------------------------------------------------------------------
def test_fused_step_supported_switches_at_the_class_and_batch_limits():
    from protopformer_b200 import ops
    dims = (196, 192, 192, 81)
    assert ops.fused_step_supported(64, *dims, 2560, 1280, 256, 10)
    assert not ops.fused_step_supported(64, *dims, 2570, 1285, 257, 10)
    assert not ops.fused_step_supported(4737, *dims, 2000, 2000, 200, 10)
    # B = 4736 (74 image tiles: two prototype groups per tile on 148 SMs) is a batch the v2 step takes, so the
    # budget = 2 cases of test_head_mid_three_phase_role_matches_float64 are shapes the step really runs
    assert ops.fused_step_supported(4736, *dims, 2000, 2000, 200, 10)
    assert ops.fused_step_supported(4736, *dims, 2570, 1290, 256, 10)


def test_head_mid_refuses_more_than_256_classes_before_touching_a_device():
    from protopformer_b200 import _lib
    lib = _lib.load()
    f = ctypes.c_void_p(0x1000)           # never dereferenced: the call must fail on the host
    args = [f] * 8 + [64, 81, 192, 2570, 1285, 257, 10, 196, 0.5, 0, EPS, 1.0, 1, 0] + [None] * 5 + [0.0] * 4 + \
        [f, f, f, f, f, f, f, f, f, None, None, None, None, None]
    assert lib.pph_head_mid(*args) == _lib_eunsup()
    assert b"C=257" in lib.pph_last_error_string()
    args[13] = 256                        # the same call at C = 256 passes the class check and stops at the next one,
    args[37] = None                       # a training call without dlogits
    assert lib.pph_head_mid(*args) != _lib_eunsup()
    assert b"null training pointer" in lib.pph_last_error_string()


def _lib_eunsup():
    return -2                             # PPH_EUNSUP (include/protohead.h)
