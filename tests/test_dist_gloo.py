"""CPU, world_size 2 and 3 over gloo: the collective driver (DistDriver) and the static item routing of the
row-sharded path (parallel.build_route_gen): every rank fetches exactly the rows its interactions need from
their owners, and partial gradients return to the owning rank -- through the all-to-all path and through the
tables of the push exchange (slot_owner / want_rows for the fetch, push_index / spos for the partial gradients
staged at the owner, pos[rank][row] for the owner's row push), with the peers' memory emulated by all_gather."""
import json
import os
import socket
import subprocess
import sys

import pytest

HERE = os.path.dirname(os.path.abspath(__file__))


def free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


@pytest.mark.parametrize("world", [2, 3])
def test_item_routing_over_gloo(world):
    port = free_port()
    procs = []
    for r in range(world):
        env = dict(os.environ, RANK=str(r), WORLD_SIZE=str(world), MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port),
                   OMP_NUM_THREADS="1")
        procs.append(subprocess.Popen([sys.executable, os.path.join(HERE, "_gloo_worker.py")], env=env,
                                      stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True))
    outs = []
    for p in procs:
        out, err = p.communicate(timeout=240)
        assert p.returncode == 0, err[-2000:]
        outs.append(json.loads(out.strip().splitlines()[-1]))
    assert sorted(o["rank"] for o in outs) == list(range(world))
    for o in outs:
        assert o["fetch"] and o["back"], o
        assert o["fetch_p2p"], o                        # routing tables of the peer-memory fetch
        assert o["push"], o                             # ... and of the push exchange (staging rows, spos, pos)
        assert sum(o["recv"]) == o["n_cache"]
    # what rank a receives from b is what b sends to a
    by = {o["rank"]: o for o in outs}
    for a in range(world):
        for b in range(world):
            assert by[a]["recv"][b] == by[b]["send"][a]


def test_replicated_chunks_partition_every_batch():
    """Host logic of the replicated-tables trainer (SURVEY.md 8e): the ranks' contiguous chunks of a global batch slice
    [lo, hi) are disjoint, ordered and cover it, for any world size (empty chunks allowed)."""
    from types import SimpleNamespace
    from invpref_kdd_2022_b200.parallel import ReplicatedTrainer
    for world in (1, 2, 3, 4, 8):
        for lo, hi in ((0, 0), (0, 1), (5, 12), (0, 262144), (262144, 311704), (7, 7 + world - 1)):
            cuts = [ReplicatedTrainer.chunk(SimpleNamespace(rank=r, world=world), lo, hi) for r in range(world)]
            assert cuts[0][0] == lo and cuts[-1][1] == hi
            for (a0, a1), (b0, b1) in zip(cuts[:-1], cuts[1:]):
                assert a0 <= a1 == b0 <= b1
            assert sum(b - a for a, b in cuts) == hi - lo
