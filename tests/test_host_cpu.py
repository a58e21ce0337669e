"""CPU-side checks (no GPU): the C-ABI library loads and exports every symbol include/protohead.h declares, the
ctypes signatures agree with the header, the product never touches oracle/, host logic of the module and of the
multi-process plumbing (gloo, world_size 2)."""
import os
import re
import subprocess
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _header_functions():
    src = open(os.path.join(ROOT, "include", "protohead.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    out = {}
    for m in re.finditer(r"\b(?:int|const char\*)\s+(pph_\w+)\s*\(([^;]*?)\)\s*;", src, flags=re.S):
        args = m.group(2).strip()
        out[m.group(1)] = 0 if args == "void" else len([a for a in args.split(",") if a.strip()])
    return out


def test_library_builds_loads_and_exports_every_declared_symbol():
    from protopformer_b200 import _lib, build
    build.build()
    lib = _lib.load()
    decl = _header_functions()
    assert len(decl) >= 13
    for name, nargs in decl.items():
        assert hasattr(lib, name), f"{name} declared in protohead.h but not exported"
        assert name in _lib.SIGNATURES, f"{name} has no ctypes signature"
        assert len(_lib.SIGNATURES[name]) == nargs, f"{name}: header has {nargs} args, binding {len(_lib.SIGNATURES[name])}"
    assert set(_lib.SIGNATURES) == set(decl)
    assert lib.pph_version() == 203


def test_sass_contains_blackwell_tensor_and_tma_instructions():
    from protopformer_b200 import _lib, build
    cuobjdump = os.path.join(os.path.dirname(build._nvcc()), "cuobjdump")      # the toolkit that built the library
    sass = ""
    if os.path.exists(cuobjdump):
        sass = subprocess.run([cuobjdump, "-sass", _lib.LIB_PATH], capture_output=True, text=True).stdout
    if not sass:
        pytest.skip("cuobjdump unavailable")
    for mnemonic in ("UTCHMMA", "UTMALDG", "LDTM"):
        assert mnemonic in sass, f"{mnemonic} missing from the SASS of the similarity kernel"


def test_no_cpu_fallback_argument_errors_and_loud_failure_without_gpu():
    from protopformer_b200 import _lib, ops
    lib = _lib.load()
    # argument validation happens before any launch
    assert lib.pph_select_topk(None, 1, 1, 8, 4, None, None, None) == -1
    assert b"null" in lib.pph_last_error_string()
    if not torch.cuda.is_available():
        with pytest.raises((AssertionError, RuntimeError)):
            ops.select_topk(torch.rand(2, 16), 4)          # CPU tensors are refused, nothing falls back


def test_product_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "protopformer_b200")
    for dp, _, fs in os.walk(pkg):
        for f in fs:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                txt = open(os.path.join(dp, f)).read()
                assert "oracle" not in txt.replace("oracle/ is the checker", ""), f"{f} mentions the oracle"
                assert "/root/reference" not in txt or f.endswith(".py") and "Reference lines" in txt


def test_module_constructs_on_cpu_with_reference_attribute_names():
    import torch.nn as nn
    from protopformer_b200 import PPNet

    class MyVisionTransformer(nn.Module):
        def __init__(self):
            super().__init__()
            self.fc = nn.Linear(24, 24)
            self.patch_embed = nn.Module()
            self.patch_embed.num_patches = 16

    net = PPNet(MyVisionTransformer(), 224, [20, 16, 1, 1], [14, 16, 16, 8.0], 4, reserve_layers=[11],
                reserve_token_nums=[9], use_global=True, use_ppc_loss=True, global_proto_per_class=2,
                add_on_layers_type='regular')
    assert net.num_prototypes_per_class == 5 and net.num_prototypes_global == 8 and net.epsilon == 1e-4
    assert tuple(net.prototype_vectors.shape) == (20, 16, 1, 1) and tuple(net.prototype_vectors_global.shape) == (8, 16, 1, 1)
    assert not net.last_layer.weight.requires_grad and not net.ones.requires_grad
    w = net.last_layer.weight
    assert w[0, :5].eq(1).all() and w[0, 5:].eq(-0.5).all()                  # protopformer.py:367-386
    for attr in ("features", "add_on_layers", "prototype_vectors", "prototype_vectors_global"):
        assert hasattr(net, attr)                                            # tools/create_optimizer.py:31-39
    with pytest.raises(NotImplementedError):
        PPNet(MyVisionTransformer(), 224, [20, 16, 1, 1], [14, 16, 16, 8.0], 4, use_global=False)


def test_widened_rows_validate_arguments_and_refuse_cpu_tensors():
    """rollout / AdamW / class maps: argument errors come back through the C ABI before any launch, CPU tensors never
    reach a kernel, and the optimizer's parameter groups mirror tools/create_optimizer.py:31-39."""
    import ctypes
    import torch.nn as nn
    from protopformer_b200 import PPNet, _lib, ops
    from protopformer_b200.optim import FusedHeadAdamW, head_param_groups
    lib = _lib.load()
    n = ctypes.c_longlong(0)
    assert lib.pph_rollout_ws_bytes(11, 64, 197, 34928, ctypes.byref(n)) == 0
    cap = ((197 * 197 - 34928 + 197) + 7) // 8 * 8
    assert n.value >= 11 * 64 * (198 * 4 + cap * 6)                  # column pointers + (value, row) entries
    assert lib.pph_rollout_scores(None, 1, 1, 1, 8, 0, 0, 0.2, None, 1, None, None, 0, None, None, None) == -1
    assert lib.pph_adamw_step(0, None, None, None, None, None, None, None, 0.9, 0.999, 1e-8, 1.0, None, None) == -1
    assert lib.pph_class_maps(None, None, None, None, None, None, 1, 1, 1, 1, 1, 1, 0, 1e-4, None, None) == -1
    with pytest.raises((AssertionError, RuntimeError)):
        ops.rollout_scores([torch.rand(1, 2, 5, 5)])
    with pytest.raises(ValueError):
        FusedHeadAdamW([torch.zeros(4, 4)])

    class MyVisionTransformer(nn.Module):
        def __init__(self):
            super().__init__()
            self.fc = nn.Linear(24, 24)
            self.patch_embed = nn.Module()
            self.patch_embed.num_patches = 16

    net = PPNet(MyVisionTransformer(), 224, [20, 16, 1, 1], [14, 16, 16, 8.0], 4, reserve_layers=[11],
                reserve_token_nums=[9], use_global=True, use_ppc_loss=True, global_proto_per_class=2,
                add_on_layers_type='regular')
    groups = head_param_groups(net, {"add_on_layers": 3e-3, "prototype_vectors": 2e-3}, 0.05)
    assert [g["lr"] for g in groups] == [3e-3, 2e-3, 2e-3] and [g["weight_decay"] for g in groups] == [1e-3, 0.05, 0.05]
    assert groups[0]["params"][0] is net.add_on_layers[0].weight and groups[1]["params"][0] is net.prototype_vectors
    assert groups[2]["params"][0] is net.prototype_vectors_global


def _gloo_worker(rank, world, port, q):
    import torch.distributed as dist
    from protopformer_b200.dist import FlatGradReducer, shard_batch
    dist.init_process_group("gloo", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world)
    torch.manual_seed(0)
    P = torch.nn.Parameter(torch.rand(6, 4))
    W = torch.nn.Parameter(torch.rand(3))
    red = FlatGradReducer([("P", P), ("W", W)])
    red.zero()
    lo, hi = shard_batch(10, rank, world)
    x = torch.arange(10, dtype=torch.float32)[lo:hi]
    loss = (P.sum() * x.sum()) + (W * (rank + 1)).sum()
    loss.backward()
    assert P.grad.data_ptr() == red.views[0].data_ptr()       # autograd accumulated in place into the flat buffer
    # segment-wise exchange (what the in-graph hooks issue: prototypes first, add-on parameters later)
    seg_ok = red.segment(("P",)) == (0, 24) and red.segment(("W",)) == (24, 27) and red.segment(("P", "W")) == (0, 27)
    before = red.flat.clone()
    red.allreduce(lo=0, hi=24)
    seg_ok = seg_ok and torch.equal(red.flat[24:], before[24:])     # the other segment is untouched until its own call
    red.allreduce(lo=24, hi=27)
    gP, gW = P.grad.tolist(), W.grad.tolist()
    P.grad = None                                                   # a detached gradient is reported, not averaged silently
    try:
        red.allreduce()
        detached_reported = False
    except RuntimeError:
        detached_reported = True
    red.zero()                                                      # re-attaches the views
    red.check_attached()
    q.put((rank, lo, hi, gP, gW, seg_ok and detached_reported))     # plain lists: no fd passing that can outlive the worker
    dist.destroy_process_group()


def test_flat_gradient_allreduce_gloo_world2():
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    import socket
    with socket.socket() as sk:            # a port the kernel just handed out: no clash with a lingering listener
        sk.bind(("127.0.0.1", 0))
        port = sk.getsockname()[1]
    procs = [ctx.Process(target=_gloo_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted([q.get(timeout=300) for _ in procs], key=lambda t: t[0])
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    (_, lo0, hi0, gP0, gW0, ok0), (_, lo1, hi1, gP1, gW1, ok1) = res
    assert ok0 and ok1
    gP0, gW0, gP1, gW1 = (torch.tensor(t) for t in (gP0, gW0, gP1, gW1))
    assert (lo0, hi0, lo1, hi1) == (0, 5, 5, 10)
    assert torch.allclose(gP0, gP1) and torch.allclose(gW0, gW1)
    assert torch.allclose(gP0, torch.full((6, 4), 45.0 / 2))      # mean over ranks of sum(x_shard)
    assert torch.allclose(gW0, torch.full((3,), 1.5))


@pytest.mark.parametrize("mode", [1, 2])
def test_similarity_launch_plan_visits_every_tile_exactly_once(mode):
    """Host logic of the tcgen05 similarity kernel (CTA/job walk, global-branch chunking, stage budget) for the BASELINE
    shapes, the sweep corners and awkward sizes -- checked without a GPU through pph_similarity_plan."""
    import ctypes
    from protopformer_b200 import _lib
    lib = _lib.load()
    shapes = [(64, 81, 192, 2000, 2000), (8, 81, 192, 2000, 2000), (1, 81, 192, 2000, 2000), (256, 81, 384, 1200, 600),
              (64, 121, 192, 1960, 980), (1024, 81, 192, 2000, 2000), (300, 81, 192, 2000, 1000), (150, 81, 128, 300, 150),
              (1024, 196, 192, 8000, 8000), (512, 144, 384, 4000, 4000), (32, 49, 192, 1000, 1000), (10, 36, 64, 1000, 500),
              (3, 196, 192, 8000, 4000), (5, 256, 64, 129, 0), (1000, 1, 64, 20000, 128), (257, 100, 512, 2000, 2000)]
    for sms in (148, 132, 16):
        for B, K, D, P, Pg in shapes:
            out = (ctypes.c_int * 16)()
            assert lib.pph_similarity_plan(mode, B, K, D, P, Pg, sms, out, None) == 0
            v2, grid, lanes, n_local_ctas, stages, b_tile, smem, gN, MT_l, NG_l, MT_g, NB_g, G, un_l, un_g, n_tiles = out
            assert n_tiles == MT_l * NG_l + MT_g * NB_g and G == 256 // K and NG_l == -(-B // G)
            assert un_l % 16 == 0 and G * K <= un_l <= 256 and un_g % 16 == 0 and min(B, gN) <= un_g <= 256
            assert NB_g == (-(-B // gN) if Pg else 0) and gN in (128, 256)
            assert smem <= 232448 and grid >= 1
            if v2:
                assert stages >= 2 and 1 <= lanes <= NG_l and n_local_ctas == MT_l * lanes and grid >= n_local_ctas
                assert b_tile % 1024 == 0 and b_tile >= max(G * K, un_g if Pg else 0) * 128
            cov = (ctypes.c_int * n_tiles)()
            assert lib.pph_similarity_plan(mode, B, K, D, P, Pg, sms, out, cov) == 0
            assert list(cov) == [1] * n_tiles, (mode, sms, B, K, D, P, Pg)
    # the round-1 finding encoded in the default plan: 8 walkers per prototype tile + 16 global CTAs at the CUB shape
    out = (ctypes.c_int * 16)()
    lib.pph_similarity_plan(1, 64, 81, 192, 2000, 2000, 148, out, None)
    assert (out[0], out[1], out[2]) == (1, 144, 8)
    lib.pph_similarity_plan(1, 1024, 81, 192, 2000, 2000, 148, out, None)
    assert out[0] == 1 and out[7] == 128            # BF16X3 keeps the resident-prototype kernel by chunking the global branch
    assert lib.pph_similarity_plan(0, 64, 81, 192, 2000, 2000, 148, out, None) == -1


def test_bench_reference_arm_prints_the_contract_line():
    """`bench.py --impl reference` (the CPU port of the reference head, the one bench leg that may execute oracle/) runs
    without a GPU and prints ONE JSON line with the keys the driver reads."""
    import json
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "3"],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "prototype_head_train_images_per_sec" and d["unit"] == "images/s"
    for k in ("value", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype",
              "data", "config", "cpu_baseline", "e2e", "gpu_launches"):
        assert k in d, k
    assert d["config"]["workload"] == "cub_b64" and d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0 and d["value"] > 0


def test_bench_arms_build_identical_config_objects():
    """The driver compares the `config` of the two bench arms: both must come out of one function with the same arguments."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    for wl in ("cub_b64", "dogs_b256_eval", "cars_b64_bf16", "sweep:K=49,D=384,P=4000,B=32"):
        name, shape, mode, train = bench.parse_workload(wl, None)
        for world in (1, 2, 8):
            a = bench.make_config(name, shape, mode, train, world, 16, True, "peer")
            b = bench.make_config(name, shape, mode, train, world, 16, True, "peer")
            assert a == b and a["workload"] == wl and a["parallelism"] == f"dp{world}"
            assert ("all-reduce" in a["step"]) == (world > 1 and train)
    name, shape, mode, train = bench.parse_workload("dogs_b256_eval", None)
    assert not train and shape.D == 384 and mode == "fp32"
    assert bench.parse_workload("cars_b64_bf16", None)[2] == "bf16"
    assert bench.step_flops(shape, False) < bench.step_flops(shape, True)


def test_bench_dump_outputs_stays_in_budget_with_a_fixed_row_sample(tmp_path):
    """--dump-outputs: small arrays are written whole, a large one is cut to the same seeded rows on every call, and the
    data written stays within the budget."""
    import importlib.util
    import numpy as np
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    g = torch.Generator().manual_seed(3)
    arrays = {"loss": torch.tensor(1.5), "logits": torch.randn(8, 5, generator=g), "dtokens": torch.randn(300, 7, 4, generator=g)}
    budget = 4 * (1 + 40 + 100 * 28)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), arrays, budget)
    got = {k: np.load(tmp_path / "a" / f"{k}.npy") for k in arrays}
    assert got["loss"].dtype == np.float32 and float(got["loss"]) == 1.5
    assert np.array_equal(got["logits"], arrays["logits"].numpy())
    assert sum(a.nbytes for a in got.values()) <= budget and 1 <= got["dtokens"].shape[0] < 300
    assert np.array_equal(got["dtokens"], np.load(tmp_path / "b" / "dtokens.npy"))
    rows = [int(np.argmax((arrays["dtokens"].numpy() == r).all(axis=(1, 2)))) for r in got["dtokens"]]
    assert rows == sorted(set(rows))                       # distinct rows of the input, in their original order
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "0"], capture_output=True, text=True,
                       timeout=600, cwd=ROOT)
    assert r.returncode == 2 and "--steps" in r.stderr


def test_round2_entry_points_validate_arguments_before_touching_the_device():
    """Every entry point added in round 2 checks its arguments first (negative PPH_E* codes), so the error behaviour of the
    boundary can be held without a GPU; support queries and workspace sizes are pure host functions."""
    import ctypes
    from protopformer_b200 import _lib
    lib = _lib.load()
    n = ctypes.c_longlong(0)
    # support queries / sizes (CUB shape and shapes outside the kernels' range)
    assert lib.pph_addon_tc2_supported(64, 196, 192, 192, 81) == 15            # fwd | dgrad | wgrad | fused selection
    assert lib.pph_addon_tc2_supported(256, 196, 384, 384, 81) & 1 == 0        # Din = 384: k range not resident
    assert lib.pph_addon_tc2_supported(64, 400, 192, 192, 81) & 8 == 0         # N > 256: selection stays a separate launch
    assert lib.pph_addon_tc2_supported(0, 196, 192, 192, 81) == 0
    assert lib.pph_head_prep_supported(64, 196, 192, 192, 81) == 1
    assert lib.pph_similarity_bwd2_supported(64, 81, 192, 2000, 2000) == 1 and lib.pph_similarity_bwd2_supported(64, 196, 192, 1000, 1000) == 1
    for fn, dims in (("pph_head_mid_ws_bytes", (64, 81, 192, 2000, 2000, 200, 10)), ("pph_addon_tc2_ws_bytes", (64, 196, 192, 192, 81)),
                     ("pph_similarity_bwd2_ws_bytes", (64, 81, 192, 2000)), ("pph_addon_bwd2_ws_bytes", (64, 196, 192, 192, 81))):
        assert getattr(lib, fn)(*dims, ctypes.byref(n)) == 0 and n.value > 0, fn
        assert getattr(lib, fn)(*dims, None) == -1, fn
    assert lib.pph_peer_flag_bytes(ctypes.byref(n)) == 0 and n.value % 16 == 0 and n.value > 0
    assert lib.pph_peer_flag_bytes(None) == -1
    # argument errors
    tbl = (ctypes.c_ulonglong * 2)(0x1000, 0x2000)
    assert lib.pph_peer_allreduce(None, 0, 1024, 0, 2, 0, 64, 8, 0, None) == -1                 # no buffer table
    assert lib.pph_peer_allreduce(ctypes.cast(tbl, ctypes.c_void_p), 0, 1024, 2, 2, 0, 64, 8, 0, None) == -1    # rank out of range
    assert lib.pph_peer_allreduce(ctypes.cast(tbl, ctypes.c_void_p), 0, 1024, 0, 2, 2, 64, 8, 0, None) == -1    # lo not a multiple of 4
    assert lib.pph_peer_allreduce(ctypes.cast(tbl, ctypes.c_void_p), 0, 100, 0, 2, 0, 64, 8, 0, None) == -1     # flag block inside the data
    assert lib.pph_peer_allreduce(ctypes.cast(tbl, ctypes.c_void_p), 0, 1024, 0, 2, 0, 64, 65, 0, None) == -1   # too many CTAs
    assert lib.pph_peer_allreduce(ctypes.cast(tbl, ctypes.c_void_p), 0, 1024, 0, 1, 0, 64, 8, 0, None) == 0     # world 1: nothing to do
    assert lib.pph_gather_rows_host(None, None, 1, 196, 192, 81, None, 8, None) == -1
    assert lib.pph_ppc_dense_fwd(None, None, None, 1, 20, 9, 5, 16, 1.0, 2.0, None, None, None, None, None) == -1
    assert lib.pph_ppc_dense_bwd(None, None, None, None, None, None, 1, 20, 9, 5, 16, 2.0, None, None) == -1
    assert lib.pph_select_addon_fwd(None, 1, None, None, None, 1, 196, 192, 192, 81, None, None, None, None, None, 0.5,
                                    None, None, None, None, None, None, None, None, None, None) == -1
    assert lib.pph_head_mid(*([None] * 8), 1, 81, 192, 2000, 2000, 200, 10, 196, 0.5, 0, 1e-4, 1.0, 1, 1, *([None] * 5),
                            1.0, 2.0, 0.1, 0.5, *([None] * 14)) == -1
    assert lib.pph_rollout_ws_bytes(1, 1, 2, 0, None) == -1
    assert b"pph_rollout_ws_bytes" in lib.pph_last_error_string()
    # kernel choice is left to the shapes alone: no run-time switch is exported
    assert not hasattr(lib, "pph_set_option")
