"""N ranks, one per GPU: the step with the gradient all-reduce recorded inside the CUDA graph (overlapped with the
add-on backward) must leave, on every rank, the average of the per-rank gradients of the same step run without the
exchange.  Launch:  python -m torch.distributed.run --nproc-per-node 2 --master-addr 127.0.0.1 scripts/ddp_check.py
[--train-last-layers] [peer|peer_nomc|nccl ...]
--train-last-layers unfreezes Wl and Wg: their gradients join the flat buffer and the step's third exchange ("last")."""
import os
import sys

import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from protopformer_b200 import ops, synth  # noqa: E402
from protopformer_b200.graph import GraphedHeadStep  # noqa: E402


def main():
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    args = [a for a in sys.argv[1:] if a != "--train-last-layers"]
    train_ll = len(args) != len(sys.argv) - 1
    shape = synth.SHAPES["cub_b64"]
    case = synth.make_case(shape, seed=1)
    batch = synth.make_case(shape, seed=50 + rank)
    cfg = ops.HeadConfig(K=shape.K, global_coe=shape.global_coe, mode="fp32", ppc_cov_thresh=shape.ppc_cov_thresh,
                         ppc_mean_thresh=shape.ppc_mean_thresh)

    def make(in_graph, exchange="nccl"):
        params = {k: case[k].to(dev) for k in ("Wa", "ba", "P", "Pg", "Wl", "Wg")}
        for k in ("Wa", "ba", "P", "Pg") + (("Wl", "Wg") if train_ll else ()):
            params[k].requires_grad_(True)
        st = GraphedHeadStep(params, cfg, B=shape.B, N=shape.N, C=shape.C, m=shape.m, n_slots=2,
                             allreduce_in_graph=in_graph, exchange=exchange)
        for s in range(2):
            st.load(s, batch["tokens"], batch["scores"], batch["labels"])
        torch.cuda.synchronize()
        st.capture()
        return st

    local_step = make(False)
    local_step.run(0)
    torch.cuda.synchronize()
    want = local_step.reducer.flat.clone()
    dist.all_reduce(want, op=dist.ReduceOp.AVG)
    for exchange in (args or ["peer", "peer_nomc", "nccl"]):
        graphed = make(True, exchange)
        for i in range(50):                       # repeated replays: no hang, no drift
            graphed.run(i % 2)
        torch.cuda.synchronize()
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        dist.barrier()
        torch.cuda.synchronize()
        ev[0].record()
        for i in range(500):
            graphed.run(i % 2)
        ev[1].record()
        torch.cuda.synchronize()
        got = graphed.reducer.flat
        err = float((got - want).abs().max() / want.abs().max())
        own = float((got - local_step.reducer.flat).abs().max() / want.abs().max())
        print(f"rank {rank}/{world} [{graphed.exchange}]: in-graph exchange vs averaged local gradients: {err:.3e} "
              f"(vs own gradients {own:.3e}); {1e3 * ev[0].elapsed_time(ev[1]) / 500:.1f} us/step", flush=True)
        assert err < 1e-6, err
        if train_ll:
            lo, hi = graphed.reducer.segment(("Wl", "Wg"))
            assert hi - lo == case["Wl"].numel() + case["Wg"].numel()
            err_ll = float((got[lo:hi] - want[lo:hi]).abs().max() / want[lo:hi].abs().max())
            own_ll = float((got[lo:hi] - local_step.reducer.flat[lo:hi]).abs().max() / want[lo:hi].abs().max())
            print(f"rank {rank}/{world} [{graphed.exchange}]: last layers {err_ll:.3e} (vs own {own_ll:.3e})", flush=True)
            assert err_ll < 1e-6 and own_ll > 1e-3, (err_ll, own_ll)
        assert own > 1e-3, "ranks hold different batches: the averaged gradient must differ from the local one"
        if os.environ.get("PPH_TIMELINE") and rank != 0:
            for i in range(6):                # every rank replays: the exchange is a cross-rank barrier
                graphed.run(i % 2)
            torch.cuda.synchronize()
        if os.environ.get("PPH_TIMELINE") and rank == 0:
            from torch.profiler import ProfilerActivity, profile
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                for i in range(6):
                    graphed.run(i % 2)
                torch.cuda.synchronize()
            evs = sorted((e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA),
                         key=lambda e: e.time_range.start)
            per = len(evs) // 6
            one = evs[4 * per:5 * per]
            t0 = one[0].time_range.start
            print(f"# [{graphed.exchange}] {per} device activities per replay")
            for e in one:
                print(f"{e.time_range.start - t0:9.2f} us  +{e.time_range.end - e.time_range.start:8.2f} us  {e.name[:70]}")
            print(f"# next replay starts at {evs[5 * per].time_range.start - t0:.2f} us", flush=True)
        dist.barrier()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    ev[0].record()
    for i in range(500):
        local_step.run(i % 2)
    ev[1].record()
    torch.cuda.synchronize()
    print(f"rank {rank}/{world} [no exchange]: {1e3 * ev[0].elapsed_time(ev[1]) / 500:.1f} us/step", flush=True)
    sys.stdout.flush()
    os._exit(0)            # graphs that recorded NCCL kernels make destroy_process_group() wait forever


if __name__ == "__main__":
    main()
