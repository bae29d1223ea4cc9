"""GPU, two or more devices (self-skips otherwise; run by the builder with `gpurun --gpus 2`): the REAL multi-rank
paths -- NCCL, torch symmetric memory, system-scope loads and posted NVLink stores between processes -- that the
simulated-rank tests of test_gpu_parallel.py cannot reach.  One torchrun-style launch per case: the distributed
trainer (dist_train.py) trains 3 epochs on N ranks and then re-assigns the environments once; rank 0 does the same with
the single-GPU trainer and compares losses, every gathered table and the environment assignments."""
import json
import os
import socket
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


@pytest.mark.parametrize("exchange", ["push", "nccl"])
@pytest.mark.parametrize("case", ["explicit", "implicit"])
def test_distributed_trainer_matches_single_gpu_on_real_ranks(case, exchange):
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs >= 2 GPUs (gpurun --gpus 2)")
    world = 2 if n < 4 else 4
    port = _free_port()
    procs = []
    for r in range(world):
        env = dict(os.environ, RANK=str(r), LOCAL_RANK=str(r), WORLD_SIZE=str(world), MASTER_ADDR="127.0.0.1",
                   MASTER_PORT=str(port))
        procs.append(subprocess.Popen([sys.executable, os.path.join(HERE, "_nccl_worker.py"), case, exchange], env=env,
                                      stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True))
    outs = []
    for p in procs:
        out, err = p.communicate(timeout=600)
        assert p.returncode == 0, err[-3000:]
        outs.append(json.loads(out.strip().splitlines()[-1]))
    r0 = [o for o in outs if o["rank"] == 0][0]
    assert r0["ok"], r0
    assert r0["exchange"] == exchange
    if exchange == "push":      # epochs 2 and 3 ran as CUDA-graph replays with the peer-memory all-reduce / barriers
        assert r0["peer_sync"] and r0["graph_epochs"], r0
    # environments after one re-assignment on the trained tables: only fp32 near-ties may differ (the tables of the
    # two runs differ by ~1e-5: a different, fixed summation order of the item partials)
    assert r0["env_mismatch"] <= 0.01 * r0["N"], r0
    assert abs(r0["diff"] - r0["ref_diff"]) <= r0["env_mismatch"]
