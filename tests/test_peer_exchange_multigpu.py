"""The gradient exchange over peer memory on two ranks of one box (one process per GPU, torch.distributed.run on 127.0.0.1):
scripts/ddp_check.py holds the graphed step with the exchange recorded in its CUDA graph -- multicast, plain peer pointers
and NCCL -- to the averaged per-rank gradients of the same step without the exchange.  Skipped where fewer than 2 GPUs exist."""
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.gpu
@pytest.mark.multigpu
@pytest.mark.parametrize("exchange", ["peer", "peer_nomc", "nccl"])
def test_in_graph_exchange_matches_averaged_local_gradients(exchange):
    env = dict(os.environ)
    env.pop("PPH_TIMELINE", None)
    port = {"peer": 29531, "peer_nomc": 29532, "nccl": 29533}[exchange]
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
                        "127.0.0.1", "--master-port", str(port), os.path.join(ROOT, "scripts", "ddp_check.py"), exchange],
                       env=env, cwd=ROOT, capture_output=True, text=True, timeout=240)
    assert r.returncode == 0, (r.stdout[-2000:], r.stderr[-2000:])
    assert r.stdout.count("in-graph exchange vs averaged local gradients") == 2
