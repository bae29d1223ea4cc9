"""Worker of tests/test_dist_gloo.py: one of WORLD_SIZE CPU processes talking over gloo."""
import json
import os
import sys

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from invpref_kdd_2022_b200.parallel import DistDriver, ItemRoute, build_route_gen, build_slot_table  # noqa: E402


def main():
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    dist.init_process_group("gloo", rank=rank, world_size=world)
    drv = DistDriver()
    n_items, dim = 97, 4
    g = torch.Generator().manual_seed(100 + rank)
    items = torch.randint(0, n_items, (300 + 50 * rank,), generator=g)
    route = ItemRoute()
    drv.run(build_route_gen(items, world, route))
    # row-sharded "table": row r of rank p holds global id r*world + p; value = id in every column
    shard = (torch.arange(n_items)[rank::world].float()[:, None] * torch.ones(dim)).contiguous()
    cache = torch.zeros((route.n_cache, dim))

    def fetch():
        yield ("all_to_all", cache, shard[route.send_rows].contiguous(), route.recv_splits, route.send_splits)

    drv.run(fetch())
    ok_fetch = bool(torch.equal(cache[route.slots][:, 0], items.float()))
    # gradients back: every requester sends ones for each cached row; the owner counts requesters per row
    recv = torch.zeros((int(route.send_rows.numel()), dim))

    def back():
        yield ("all_to_all", recv, torch.ones((route.n_cache, dim)), route.send_splits, route.recv_splits)

    drv.run(back())
    gshard = torch.zeros_like(shard)
    o = 0
    for p in range(world):
        n = route.send_splits[p]
        gshard[route.send_rows[o:o + n]] += recv[o:o + n]
        o += n
    # expected: number of ranks whose local batch contains the item
    present = torch.zeros(n_items)
    present[torch.unique(items)] = 1

    def red():
        yield ("all_reduce", present)

    drv.run(red())
    ok_back = bool(torch.equal(gshard[:, 0], present[rank::world]))

    # ---- the peer-memory exchange's host-side tables, with "peer memory" emulated by all_gather ----
    def gather_padded(t, rows_max):
        pad = torch.zeros((rows_max,) + tuple(t.shape[1:]), dtype=t.dtype)
        pad[:t.shape[0]] = t
        bufs = [torch.zeros_like(pad) for _ in range(world)]
        dist.all_gather(bufs, pad)
        return bufs

    rows_max = (n_items + world - 1) // world
    shards = gather_padded(shard, rows_max)                       # what invpref_fetch_rows_p2p reads
    cache2 = torch.stack([shards[int(o)][int(r)] for o, r in zip(route.slot_owner.tolist(), route.want_rows.tolist())]) \
        if route.n_cache else torch.zeros((0, dim))
    ok_fetch_p2p = bool(torch.equal(cache2, cache))

    # ---- the PUSH exchange's tables.  Every requester "stores" (rank + 1) * 1000 + slot for cache slot c into owner
    # slot_owner[c]'s staging row push_index[c] (emulated: gather every rank's (owner, index, value) triples); the
    # owner then reads its staging through spos[p, j] and must find, for each requester p, that requester's value
    # for row j -- and the staging rows written by different requesters never collide.
    vals = (rank + 1) * 1000.0 + torch.arange(route.n_cache, dtype=torch.float32)
    trip = torch.stack([route.slot_owner.float(), route.push_index.float(), vals], dim=1) if route.n_cache \
        else torch.zeros((0, 3))
    trips = gather_padded(torch.cat([trip, torch.full((1, 3), -1.0)]), n_items + 1)       # -1 row = terminator
    staging = torch.full((max(route.n_stage, 1),), float("nan"))
    writes = 0
    for p in range(world):
        tp = trips[p]
        tp = tp[: int((tp[:, 0] < 0).nonzero()[0])]
        mine = tp[tp[:, 0] == rank]
        idx = mine[:, 1].long()
        assert bool(torch.isnan(staging[idx]).all())                  # no two writers share a staging row
        staging[idx] = mine[:, 2]
        writes += int(idx.numel())
    ok_push = writes == route.n_stage and not bool(torch.isnan(staging[:route.n_stage]).any())
    pos = build_slot_table(route, world, shard.shape[0], route.peer_first)
    spos = build_slot_table(route, world, shard.shape[0], [sum(route.send_splits[:p]) for p in range(world)])
    # requester p's slot of my row j = pos[p, j]  =>  the staged value must be (p + 1) * 1000 + pos[p, j]
    for p in range(world):
        has = spos[p] >= 0
        ok_push = ok_push and bool(torch.equal(has, pos[p] >= 0))
        got = staging[spos[p][has].long()]
        ok_push = ok_push and bool(torch.equal(got, (p + 1) * 1000.0 + pos[p][has].float()))
    print(json.dumps({"rank": rank, "fetch": ok_fetch, "back": ok_back, "fetch_p2p": ok_fetch_p2p,
                      "push": ok_push, "n_cache": route.n_cache,
                      "recv": route.recv_splits, "send": route.send_splits}), flush=True)
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
