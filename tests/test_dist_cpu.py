"""World-size-2 gloo tests of the host-side multi-GPU logic (no GPU): the single weight-arena
broadcast and the member partition (SURVEY.md §8(e))."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from skyrim_b200.config import pangu_small
from skyrim_b200.ensemble import broadcast_arena, mean_and_spread, member_range
from skyrim_b200.weights import make_pangu_weights, pangu_param_shapes


def _free_port():
    """a port no other process on the host holds right now: the rendezvous must not depend on a fixed one being free"""
    with socket.socket(socket.AF_INET, socket.SOCK_STREAM) as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _worker(rank, world, port, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    cfg = pangu_small(24, 96)
    w = make_pangu_weights(cfg, 3) if rank == 0 else None
    arena, manifest = broadcast_arena(w, pangu_param_shapes(cfg), torch.device("cpu"), rank, world)
    ref = make_pangu_weights(cfg, 3)
    ok = True
    for d, (k, a) in zip(manifest, ref.items()):
        ok &= d.name.decode() == k and np.array_equal(arena[d.offset:d.offset + d.count].numpy(), a.reshape(-1))
    # ensemble statistics across ranks: 2 members per rank of a field with a large mean and a small spread
    g = torch.Generator().manual_seed(7)
    allm = 5.0e4 + 0.5 * torch.randn(4, 2, 8, 16, generator=g)
    mean, spread = mean_and_spread(allm[2 * rank:2 * rank + 2].clone(), world)
    ok &= bool(torch.allclose(mean, allm.mean(0), rtol=0, atol=1e-2))
    ok &= bool(torch.allclose(spread, allm.double().std(0, unbiased=False).float(), rtol=1e-3, atol=1e-4))
    q.put((rank, bool(ok), list(member_range(rank, 4)), float(arena.sum())))
    dist.destroy_process_group()


def test_weight_broadcast_and_member_partition():
    world, port = 2, _free_port()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    ps = [ctx.Process(target=_worker, args=(r, world, port, q)) for r in range(world)]
    [p.start() for p in ps]
    res = sorted(q.get(timeout=120) for _ in range(world))
    [p.join(30) for p in ps]
    assert all(r[1] for r in res), res
    assert res[0][2] == [0, 1, 2, 3] and res[1][2] == [4, 5, 6, 7]
    assert res[0][3] == res[1][3]


def test_member_ranges_cover_ensemble_exactly_once():
    for world, m in [(1, 1), (2, 4), (8, 4)]:
        ids = [i for r in range(world) for i in member_range(r, m)]
        assert ids == list(range(world * m))


def _worker_graphcast(rank, world, port, q):
    """GraphCast: the arena also carries the graph tables (built on every rank: their shapes size the manifest)"""
    from skyrim_b200.config import graphcast_small
    from skyrim_b200.icomesh import build_graph, graph_arena_entries
    from skyrim_b200.weights import graphcast_param_shapes, make_graphcast_weights
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    cfg = graphcast_small(21, 48, 1, 512, 1)
    gent = graph_arena_entries(build_graph(cfg.nlat, cfg.nlon, cfg.mesh_levels, cfg.radius_frac))
    shapes = graphcast_param_shapes(cfg)
    shapes.update({k: v.shape for k, v in gent.items()})
    w = None
    if rank == 0:
        w = make_graphcast_weights(cfg, 3); w.update(gent)
    arena, manifest = broadcast_arena(w, shapes, torch.device("cpu"), rank, world)
    ref = make_graphcast_weights(cfg, 3); ref.update(gent)
    ok = len(manifest) == len(ref)
    for d, (k, a) in zip(manifest, ref.items()):
        ok &= d.name.decode() == k and np.array_equal(arena[d.offset:d.offset + d.count].numpy(), np.asarray(a, np.float32).reshape(-1))
    q.put((rank, bool(ok), float(arena.double().sum())))
    dist.destroy_process_group()


def test_graphcast_arena_with_graph_tables_broadcasts():
    world, port = 2, _free_port()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    ps = [ctx.Process(target=_worker_graphcast, args=(r, world, port, q)) for r in range(world)]
    [p.start() for p in ps]
    res = sorted(q.get(timeout=180) for _ in range(world))
    [p.join(30) for p in ps]
    assert all(r[1] for r in res), res
    assert res[0][2] == res[1][2]
