"""Multi-GPU path on real devices (needs >= 2 GPUs): each rank culls its index-range shard on its own GPU,
lb200_culling_allgather exchanges the compacted visible lists over NCCL, and the merged result equals the oracle's unsharded cull.
The bitmask exchange fused into the cull kernel (lb200_culling_cull_exchange) is also run with a world of ONE rank, so that its
peer-store / epoch-flag path is covered on a single-GPU box."""
import os
import socket
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
pytestmark = pytest.mark.gpu


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, world, port, q):
    sys.path.insert(0, ROOT)
    import torch
    import torch.distributed as dist

    import lumixengine_b200 as lb
    from lumixengine_b200 import scenes, sharding
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)  # rendezvous only; the data path is our own NCCL communicator
    ctx = lb.Context(rank)
    uid = torch.zeros(128, dtype=torch.uint8)
    if rank == 0:
        uid.copy_(torch.from_numpy(ctx.comm_unique_id()))
    dist.broadcast(uid, 0)
    ctx.comm_init(world, rank, uid.numpy())
    scene = scenes.cull_scene(300_001, (3000.0, 300.0, 3000.0), seed=23, big_fraction=0.002, type_probs=(0.6, 0.3, 0.1))
    mine = sharding.shard_scene(scene, rank, world)
    cs = lb.CullingSystem(ctx)
    cs.add(mine["entities"], mine["types"], mine["pos"], mine["radius"])
    f = lb.frustum_perspective(**dict(scenes.c1_frustum_args(), far=2500.0))
    _, res = cs.cull_device(f, want_counts=True)
    n = torch.tensor([int(res.total)])
    dist.all_reduce(n, op=dist.ReduceOp.MAX)
    slab = int(n.item()) + 64
    dev_ptr, counts = cs.allgather(slab, world)
    slabs, counts2 = cs.read_gathered(dev_ptr, slab, world, stride=256 + slab)
    assert np.array_equal(counts, counts2)
    merged = sharding.merge_gathered(slabs, counts)
    # the asynchronous per-frame form gives the same buffer: first over NCCL, then over the NVLink peer path (several epochs)
    def check_async():
        dev2 = cs.cull_gather(f, slab)
        slabs_b, counts_b = cs.read_gathered(dev2, slab, world)
        assert np.array_equal(counts_b, counts)
        for r in range(world):
            for t in range(3):
                o = int(counts[r, :t].sum())
                assert np.array_equal(np.sort(slabs_b[r][o:o + counts[r, t]]), np.sort(slabs[r][o:o + counts[r, t]]))
    check_async()
    ctx.comm_enable_p2p(slab)
    for _ in range(5):
        check_async()
    for _ in range(50):  # back-to-back epochs without host synchronisation in between
        cs.cull_gather(f, slab)
    check_async()
    ok = True
    if rank == 0:
        from oracle import pyoracle as po
        oc = po.OracleCulling()
        oc.add(scene["entities"], scene["types"], scene["pos"], scene["radius"])
        oi, ot, _ = oc.cull(lb.culling.frustum_bytes(f))
        for t in range(3):
            ok &= np.array_equal(np.sort(merged.get(t, np.zeros(0, np.uint32))).astype(np.int64), np.sort(oi[ot == t]).astype(np.int64))
        ok &= len(oi) > 5000
    # every rank sees the same gathered data
    digest = torch.tensor([sum(int(np.sort(v).astype(np.uint64).sum()) % (1 << 40) for v in merged.values())])
    gathered = [torch.zeros_like(digest) for _ in range(world)]
    dist.all_gather(gathered, digest)
    ok &= all(int(g.item()) == int(digest.item()) for g in gathered)
    q.put((rank, bool(ok)))
    dist.barrier()
    cs.close()
    ctx.close()
    dist.destroy_process_group()


def _exchange_worker(rank, world, port, q):
    sys.path.insert(0, ROOT)
    import torch
    import torch.distributed as dist

    import lumixengine_b200 as lb
    from lumixengine_b200 import scenes, sharding
    from oracle import pyoracle as po
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    ctx = lb.Context(rank)
    uid = torch.zeros(128, dtype=torch.uint8)
    if rank == 0:
        uid.copy_(torch.from_numpy(ctx.comm_unique_id()))
    dist.broadcast(uid, 0)
    ctx.comm_init(world, rank, uid.numpy())
    scene = scenes.cull_scene(240_007, (3000.0, 300.0, 3000.0), seed=29, big_fraction=0.002, type_probs=(0.6, 0.3, 0.1))
    shards = [sharding.shard_scene(scene, r, world) for r in range(world)]
    systems = []
    for r in range(world):  # host bookkeeping of every shard (page -> entity ids); only this rank's shard is culled here
        c = lb.CullingSystem(ctx)
        c.add(shards[r]["entities"], shards[r]["types"], shards[r]["pos"], shards[r]["radius"])
        systems.append(c)
    cs = systems[rank]
    words = torch.tensor([cs.exchange_slab_words()])
    dist.all_reduce(words, op=dist.ReduceOp.MAX)
    ctx.comm_enable_p2p(int(words.item()) - 256)
    fails = []

    def chk(cond, msg):
        if not cond:
            fails.append(msg)
    tables = [(systems[r].pages(), systems[r].page_ids()) for r in range(world)]
    frusta = [lb.frustum_perspective(**dict(scenes.c1_frustum_args(), far=2500.0)),
              lb.frustum_perspective(position=(500.0, 20.0, -300.0), direction=(0.6, -0.1, 0.79), up=(0, 1, 0), fov=0.9, ratio=1.6, near=0.5, far=1800.0)]
    for step in range(14):  # many epochs: every exchange buffer and lane; single steps and batches on the internal streams
        f = frusta[step % 2]
        fb = lb.culling.frustum_bytes(f)
        if step % 3 == 2:
            cs.cull_exchange_n(frusta[(step + 1) % 2], 1 + step % 4)  # unread steps of the other view right before
            ids_ptr, slabs_ptr, stride = cs.cull_exchange_n(f, 2 + step)
        else:
            ids_ptr, slabs_ptr, stride = cs.cull_exchange(f)
        got = cs.read_exchanged(slabs_ptr, stride, world)
        for r in range(world):
            oc = po.OracleCulling()
            oc.add(shards[r]["entities"], shards[r]["types"], shards[r]["pos"], shards[r]["radius"])
            oi, ot, _ = oc.cull(fb)
            chk(len(oi) > 1000, f'step {step} rank {r}: scene too empty')
            # per-type counts of rank r as seen from here
            for t in range(3):
                chk(int(got[r]["counts"][t]) == int((ot == t).sum()), f'step {step} rank {r} type {t}: count {got[r]["counts"][t]} != {(ot == t).sum()}')
            # visibility rows of rank r -> entity ids through rank r's page table
            pages, pid = tables[r]
            chk(got[r]["n_pages"] == int(pid.max()) + 1, f'step {step} rank {r}: n_pages {got[r]["n_pages"]}')
            vis = []
            for i, pg in enumerate(pages):
                row = got[r]["mask"][pid[i]]
                bits = np.unpackbits(row.view(np.uint8), bitorder="little")[:pg["count"]]
                chk(int(np.unpackbits(row.view(np.uint8), bitorder="little")[pg["count"]:].sum()) == 0, f'step {step} rank {r} page {i}: bits beyond count')
                vis.append(pg["entities"][bits.astype(bool)])
            vis = np.sort(np.concatenate(vis)).astype(np.int64)
            chk(np.array_equal(vis, np.sort(oi).astype(np.int64)), f'step {step} rank {r}: mask rows decode to {len(vis)} ids, oracle {len(oi)}')
            if r == rank:  # the sharded id list of this rank agrees with its own rows
                total = int(got[r]["counts"].sum())
                base = np.concatenate([[0], np.cumsum(np.bincount(shards[r]["types"], minlength=256))])
                mine = [ctx.copy_to_host(ids_ptr + 4 * int(base[t]), int(got[r]["counts"][t]), np.uint32) for t in range(3)]
                chk(np.array_equal(np.sort(np.concatenate(mine)).astype(np.int64), vis) and total == len(vis), f'step {step}: own id list differs from own rows')
    for _ in range(10):  # back-to-back epochs without host synchronisation in between
        cs.cull_exchange(frusta[0])
    cs.cull_exchange_n(frusta[0], 40)
    _, slabs_ptr, stride = cs.cull_exchange_n(frusta[1], 5)
    got = cs.read_exchanged(slabs_ptr, stride, world)
    digest = torch.tensor([sum(int(g["mask"].astype(np.uint64).sum()) + int(g["counts"].sum()) for g in got)])
    gathered = [torch.zeros_like(digest) for _ in range(world)]
    dist.all_gather(gathered, digest)
    chk(all(int(g.item()) == int(digest.item()) for g in gathered), 'ranks disagree on the exchanged slabs')
    q.put((rank, not fails, fails[:5]))
    dist.barrier()
    for c in systems:
        c.close()
    ctx.close()
    dist.destroy_process_group()


def _run(target, world):
    import torch.multiprocessing as mp
    mpctx = mp.get_context("spawn")
    q = mpctx.Queue()
    port = _free_port()
    procs = [mpctx.Process(target=target, args=(r, world, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    results = [q.get(timeout=300) for _ in range(world)]
    for p in procs:
        p.join(timeout=120)
    assert all(r[1] for r in results), results
    assert all(p.exitcode == 0 for p in procs)


def test_bitmask_exchange_one_rank():
    _run(_exchange_worker, 1)


def test_bitmask_exchange_two_gpus():
    import lumixengine_b200 as lb
    if lb.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    _run(_exchange_worker, 2)


def test_two_gpu_cull_allgather():
    import lumixengine_b200 as lb
    if lb.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import torch.multiprocessing as mp
    mpctx = mp.get_context("spawn")
    q = mpctx.Queue()
    port = _free_port()
    procs = [mpctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    results = [q.get(timeout=300) for _ in range(2)]
    for p in procs:
        p.join(timeout=120)
    assert all(ok for _, ok in results), results
    assert all(p.exitcode == 0 for p in procs)
