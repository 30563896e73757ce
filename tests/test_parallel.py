"""Multi-process tests of the node-partitioned path.
CPU (gloo, world_size 2): partition arithmetic, owner-computes seed routing, locality relabelling.
GPU (nccl, 2 GPUs, skipped on a 1-GPU box): partitioned forward over peer-mapped shards == single-GPU forward."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from conftest import ROOT, rel_err  # noqa: F401


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _init(rank, world, port, backend):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world),
                      LOCAL_RANK=str(rank))
    if backend == "nccl":
        torch.cuda.set_device(rank)
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    else:
        dist.init_process_group("gloo", rank=rank, world_size=world)


def _cpu_worker(rank, world, port, q):
    try:
        from graphsage_b200 import parallel
        _init(rank, world, port, "gloo")
        n_nodes = 1001
        R = parallel.rows_per_shard(n_nodes, world)
        assert R == 501
        rs = np.random.RandomState(rank)
        seeds = torch.from_numpy(rs.randint(0, n_nodes, size=300 + 17 * rank).astype(np.int32))
        mine = parallel.route_seeds(seeds, n_nodes)
        assert mine.dtype == torch.int32
        own = parallel.owner_of(mine, n_nodes, world)
        assert bool((own == rank).all())
        # nothing lost, nothing duplicated: gather every rank's routed seeds and compare multisets
        got, sent = [None] * world, [None] * world
        dist.all_gather_object(got, mine.tolist())
        dist.all_gather_object(sent, seeds.tolist())
        assert sorted(sum(got, [])) == sorted(sum(sent, []))
        # dummy / out-of-range ids have no owner
        assert parallel.owner_of(np.array([n_nodes, -1, 0, n_nodes - 1]), n_nodes, world).tolist() == [-1, -1, 0, world - 1]
        # non-uniform (community-aligned) bounds: numpy and torch agree, routing follows them
        bounds = [0, 300, n_nodes]
        ids = np.array([0, 299, 300, 1000, n_nodes, -3])
        assert parallel.owner_of(ids, n_nodes, world, bounds).tolist() == [0, 0, 1, 1, -1, -1]
        assert parallel.owner_of(torch.from_numpy(ids), n_nodes, world, bounds).tolist() == [0, 0, 1, 1, -1, -1]
        mine_b = parallel.route_seeds(seeds, n_nodes, row_start=bounds)
        assert bool(((mine_b >= bounds[rank]) & (mine_b < bounds[rank + 1])).all())
        dist.all_gather_object(got, mine_b.tolist())
        assert sorted(sum(got, [])) == sorted(sum(sent, []))
        # data-parallel training plumbing: broadcast of the initial weights, ONE packed gradient all-reduce per step
        torch.manual_seed(rank)
        params = [torch.randn(3, 4, requires_grad=True), torch.randn(5, requires_grad=True), torch.randn(2, requires_grad=True)]
        parallel.broadcast_parameters(params, 0)
        ref = [None] * world
        dist.all_gather_object(ref, [p.detach().clone() for p in params])
        assert all(torch.equal(a, b) for a, b in zip(ref[0], ref[1]))
        params[0].grad = torch.full((3, 4), float(rank + 1))
        params[1].grad = torch.arange(5, dtype=torch.float32) * (rank + 1)
        if rank == 0:
            params[2].grad = torch.ones(2)                    # rank 1 has no gradient for this one: counts as zeros
        nbytes = parallel.allreduce_gradients(params)
        assert nbytes == (12 + 5 + 2) * 4
        assert torch.equal(params[0].grad, torch.full((3, 4), 1.5))
        assert torch.equal(params[1].grad, torch.arange(5, dtype=torch.float32) * 1.5)
        assert torch.equal(params[2].grad, torch.full((2,), 0.5))
        q.put((rank, "ok"))
    except Exception as e:  # pragma: no cover
        import traceback
        q.put((rank, traceback.format_exc()))
    finally:
        if dist.is_initialized():
            dist.destroy_process_group()


def _run(worker, world, *args):
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=worker, args=(r, world, port, q) + args) for r in range(world)]
    for p in procs:
        p.start()
    res = [q.get(timeout=300) for _ in procs]
    for p in procs:
        p.join(timeout=60)
    for rank, msg in res:
        assert msg == "ok", "rank %d failed:\n%s" % (rank, msg)


def test_route_seeds_gloo_world2():
    _run(_cpu_worker, 2)


def _cpu_worker_world4(rank, world, port, q):
    """The same host logic at four ranks (the driver's scaling run also uses N = 4): uneven bounds with an EMPTY shard,
    routing, and the packed gradient all-reduce."""
    try:
        from graphsage_b200 import parallel
        _init(rank, world, port, "gloo")
        n_nodes = 1003
        assert parallel.uniform_bounds(n_nodes, world) == [0, 251, 502, 753, 1003]
        bounds = [0, 400, 400, 900, n_nodes]                    # shard 1 owns nothing
        rs = np.random.RandomState(10 + rank)
        seeds = torch.from_numpy(rs.randint(0, n_nodes, size=200 + 31 * rank).astype(np.int32))
        for b in (None, bounds):
            mine = parallel.route_seeds(seeds, n_nodes, row_start=b)
            lo, hi = (parallel.uniform_bounds(n_nodes, world) if b is None else b)[rank:rank + 2]
            assert bool(((mine >= lo) & (mine < hi)).all())
            got, sent = [None] * world, [None] * world
            dist.all_gather_object(got, mine.tolist())
            dist.all_gather_object(sent, seeds.tolist())
            assert sorted(sum(got, [])) == sorted(sum(sent, []))
            if b is not None:
                assert len(got[1]) == 0
        p = [torch.zeros(7, requires_grad=True)]
        p[0].grad = torch.full((7,), float(rank))
        assert parallel.allreduce_gradients(p) == 28
        assert torch.equal(p[0].grad, torch.full((7,), 1.5))     # mean of 0, 1, 2, 3
        q.put((rank, "ok"))
    except Exception:  # pragma: no cover
        import traceback
        q.put((rank, traceback.format_exc()))
    finally:
        if dist.is_initialized():
            dist.destroy_process_group()


def test_route_seeds_gloo_world4():
    _run(_cpu_worker_world4, 4)


def test_locality_relabel_preserves_graph():
    from graphsage_b200 import parallel
    from graphsage_b200.synthetic import community_graph_csr
    indptr, indices, comm = community_graph_csr(2000, n_comm=7, mean_deg=12, seed=3)
    order, inv = parallel.locality_order(comm)
    assert (np.diff(comm[order]) >= 0).all()                      # communities are contiguous in the new labelling
    p2, i2 = parallel.relabel_graph(indptr, indices, order, inv)
    assert p2[-1] == indptr[-1]
    for new in range(0, 2000, 97):
        old = order[new]
        want = sorted(inv[indices[indptr[old]:indptr[old + 1]]].tolist())
        assert sorted(i2[p2[new]:p2[new + 1]].tolist()) == want
    # locality: with a contiguous 4-way split most neighbours share their node's part
    R = parallel.rows_per_shard(2000, 4)
    src = np.repeat(np.arange(2000), np.diff(p2))
    assert ((src // R) == (i2 // R)).mean() > 0.6


def test_community_bounds_and_hot_rows():
    from graphsage_b200 import parallel
    from graphsage_b200.synthetic import reddit_like
    g = reddit_like(n=6000, f=4, max_degree=16, seed=5, with_features=False)
    world = 4
    b = parallel.community_bounds(g["comm"], world)
    assert b[0] == 0 and b[-1] == 6000 and len(b) == world + 1 and all(x <= y for x, y in zip(b, b[1:]))
    for cut in b[1:-1]:
        assert g["comm"][cut] != g["comm"][cut - 1]                 # every cut sits on a community start
    assert parallel.uniform_bounds(10, 4) == [0, 3, 6, 9, 10] and parallel.uniform_bounds(2, 4) == [0, 1, 2, 2, 2]
    # aligned cuts cross fewer table entries than equal ranges
    def cross(bounds):
        own = parallel.owner_of(np.arange(6000), 6000, world, bounds)
        ent = g["adj"][:6000]
        o2 = parallel.owner_of(ent, 6000, world, bounds)
        return float(((o2 != own[:, None]) & (o2 >= 0)).mean())
    assert cross(b) <= cross(parallel.uniform_bounds(6000, world)) + 1e-9
    # hot rows: remote only, sorted unique, and they cover more reads than the same number of arbitrary remote rows
    rank = 1
    hot = parallel.hot_remote_rows(g["adj"], 6000, world, rank, 400, row_start=b)
    assert len(hot) == 400 and (np.diff(hot) > 0).all() and not ((hot >= b[rank]) & (hot < b[rank + 1])).any()
    import oracle
    rs = np.random.RandomState(0)
    seeds = rs.randint(b[rank], b[rank + 1], size=256).astype(np.int32)
    samples, _ = oracle.sample_khop(g["adj"], seeds, [5, 4], 1, 0)
    ids = np.concatenate(samples)
    remote = ids[(parallel.owner_of(ids, 6000, world, b) != rank) & (ids < 6000)]
    cov_hot = np.isin(remote, hot).mean()
    others = np.setdiff1d(np.arange(6000), np.arange(b[rank], b[rank + 1]))
    cov_rand = np.isin(remote, rs.choice(others, size=400, replace=False)).mean()
    assert cov_hot > cov_rand
    assert len(parallel.hot_remote_rows(g["adj"], 6000, 1, 0, 100)) == 0


def _gpu_worker(rank, world, port, q):
    try:
        _init(rank, world, port, "nccl")
        import graphsage_b200 as gs
        from graphsage_b200 import parallel
        rs = np.random.RandomState(0)                      # identical on every rank
        n, md, f, B = 3001, 32, 602, 64
        adj = rs.randint(0, n, size=(n + 1, md)).astype(np.int32)
        adj[n] = n
        adj[5] = n                                         # an isolated node -> dummy neighbours
        feats = rs.randn(n, f).astype(np.float32)
        seeds = rs.randint(0, n, size=B).astype(np.int32)
        seeds[0] = 5
        dev = torch.device("cuda", rank)
        bounds = [0, 1300, n]                               # deliberately unequal ranges
        lo, hi = bounds[rank], bounds[rank + 1]
        hot = parallel.hot_remote_rows(adj, n, world, rank, 200, row_start=bounds)
        assert len(hot) == 200
        shard = parallel.ShardedFeatures(feats[lo:hi], n, row_start=bounds, replica_ids=hot, replica_rows=feats[hot])
        adj_dev = torch.from_numpy(adj).to(dev)
        full = torch.from_numpy(np.vstack([feats, np.zeros((1, f), np.float32)])).to(dev)
        outs = {}
        for kind, concat, dim in (("mean", True, 128), ("gcn", False, 256), ("maxpool", True, 32)):
            res = []
            shard.stage_halo = kind != "gcn"               # both partitioned data paths: halo staging / direct peer copies
            for table in (shard, full):
                gs.inits.manual_seed(7, dev)
                sampler = gs.UniformNeighborSampler(adj_dev, seed=123)
                infos = [gs.SAGEInfo("node", sampler, 25, dim), gs.SAGEInfo("node", sampler, 10, dim)]
                m = gs.SampleAndAggregate({"batch_size": B, "dropout": 0.}, table, adj_dev, None, infos, concat=concat,
                                          aggregator_type=kind, device=dev)
                res.append(m.forward(torch.from_numpy(seeds), normalize=True).cpu().numpy())
            assert np.array_equal(res[0], res[1]), "partitioned != single-table for %s (max diff %g)" % (
                kind, np.abs(res[0] - res[1]).max())
            outs[kind] = res[0]
        ids = torch.from_numpy(rs.randint(0, n + 1, size=5000).astype(np.int32)).to(dev)
        rows = gs.ops.gather_rows(shard, ids)
        assert torch.equal(rows, full[ids.long()])
        frac0, frac = shard.remote_fraction(ids, use_replicas=False), shard.remote_fraction(ids)
        assert 0.3 < frac0 < 0.7 and frac < frac0
        # both data paths of the partitioned gather (bulk copies over the peer mapping / 128-bit loads) agree bit for bit
        s0 = torch.from_numpy(rs.randint(0, n, size=64).astype(np.int32)).to(dev)
        s1 = torch.from_numpy(rs.randint(0, n + 1, size=64 * 25).astype(np.int32)).to(dev)
        seg = [gs.ops.Seg(64, 25, self_ids=s0, neigh_ids=s1)]
        a = gs.ops.gather_mean(shard, seg)
        gs._lib.set_tuning("gather_variant", 0)
        b = gs.ops.gather_mean(shard, seg)
        gs._lib.set_tuning("gather_variant", 2)
        assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])
        ref_self = full[s0.long()]
        assert torch.equal(a[0][:, :f], ref_self)
        shard.close()
        q.put((rank, "ok"))
    except Exception:  # pragma: no cover
        import traceback
        q.put((rank, traceback.format_exc()))
    finally:
        if dist.is_initialized():
            dist.destroy_process_group()


@pytest.mark.gpu
def test_partitioned_forward_two_gpus():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    _run(_gpu_worker, 2)


@pytest.mark.gpu
def test_sharded_table_single_rank_matches_dense():
    """world_size 1: the sharded kernels with one shard must reproduce the dense-table kernels exactly."""
    import graphsage_b200 as gs
    from graphsage_b200 import parallel
    rs = np.random.RandomState(1)
    n, f = 2000, 602
    feats = rs.randn(n, f).astype(np.float32)
    shard = parallel.ShardedFeatures(feats, n)
    full = torch.from_numpy(np.vstack([feats, np.zeros((1, f), np.float32)])).cuda()
    ids = torch.from_numpy(rs.randint(-3, n + 5, size=4000).astype(np.int32)).cuda()
    clamp = ids.clone().long()
    clamp[(clamp < 0) | (clamp >= n)] = n
    assert torch.equal(gs.ops.gather_rows(shard, ids), full[clamp])
    s0 = torch.from_numpy(rs.randint(0, n, size=40).astype(np.int32)).cuda()
    s1 = torch.from_numpy(rs.randint(0, n + 1, size=400).astype(np.int32)).cuda()
    seg = [gs.ops.Seg(40, 10, self_ids=s0, neigh_ids=s1)]
    a = gs.ops.gather_mean(shard, seg, include_self=True)
    gs._lib.set_tuning("gather_variant", 0)
    b = gs.ops.gather_mean(full, seg, include_self=True)
    gs._lib.set_tuning("gather_variant", 2)
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])
    shard.close()


@pytest.mark.gpu
@pytest.mark.parametrize("kind,concat,dim", [("mean", True, 128), ("gcn", False, 256)])
def test_partitioned_forward_single_rank_vs_oracle(kind, concat, dim):
    """The node-partitioned path (ShardedFeatures + the sharded gather kernels) against the ORACLE, runnable on a
    1-GPU box: one shard, same kernels and address arithmetic as with N ranks (reference models.py:254-330)."""
    import graphsage_b200 as gs
    import oracle
    from conftest import rel_err
    from graphsage_b200 import parallel
    rs = np.random.RandomState(2)
    n, md, f, B = 3001, 32, 602, 64
    adj = rs.randint(0, n, size=(n + 1, md)).astype(np.int32)
    adj[n] = n
    adj[7] = n                                             # isolated node: dummy neighbours (zero row)
    feats = rs.randn(n, f).astype(np.float32)
    seeds = rs.randint(0, n, size=B).astype(np.int32)
    seeds[0] = 7
    shard = parallel.ShardedFeatures(feats, n)
    adj_dev = torch.from_numpy(adj).cuda()
    for math in ("fp32", "tf32x3"):
        gs.set_default_math(math)
        sampler = gs.UniformNeighborSampler(adj_dev, seed=123)
        infos = [gs.SAGEInfo("node", sampler, 25, dim), gs.SAGEInfo("node", sampler, 10, dim)]
        m = gs.SampleAndAggregate({"batch_size": B, "dropout": 0.}, shard, adj_dev, None, infos, concat=concat,
                                  aggregator_type=kind)
        out = m.forward(torch.from_numpy(seeds), normalize=True).cpu().numpy()
        aggs = [dict(type=kind, **{k: v.cpu().numpy() for k, v in a.vars.items()}) for a in m.aggregators]
        ref = oracle.forward_2hop(adj, np.vstack([feats, np.zeros((1, f), np.float32)]), seeds, [25, 10], aggs, concat,
                                  123, 0, normalize=True)
        assert rel_err(out, ref) < 1e-4, (kind, math)
    gs.set_default_math("fp32")
    shard.close()


def _gpu_train_worker(rank, world, port, q):
    """config 4 in miniature: unsupervised GraphSAGE, node-partitioned features, data-parallel over 2 GPUs - the weights
    must stay bit-identical on both ranks after every step (same initial weights, one gradient all-reduce per step), and
    a 1-rank run on the union batch with averaged loss must give the same first update."""
    try:
        _init(rank, world, port, "nccl")
        import graphsage_b200 as gs
        from graphsage_b200 import parallel
        rs = np.random.RandomState(0)
        n, md, f, B = 2000, 16, 32, 48
        adj = rs.randint(0, n, size=(n + 1, md)).astype(np.int32)
        adj[n] = n
        feats = rs.randn(n, f).astype(np.float32)
        deg = rs.randint(1, 30, size=n).astype(np.float64)
        dev = torch.device("cuda", rank)
        bounds = parallel.uniform_bounds(n, world)
        lo, hi = bounds[rank], bounds[rank + 1]
        shard = parallel.ShardedFeatures(feats[lo:hi], n, row_start=bounds)
        adj_dev = torch.from_numpy(adj).to(dev)
        gs.set_default_math("fp32")
        gs.inits.manual_seed(100 + rank, dev)                     # DIFFERENT initial weights per rank: the broadcast must fix that
        sampler = gs.UniformNeighborSampler(adj_dev, seed=123)
        infos = [gs.SAGEInfo("node", sampler, 5, 16), gs.SAGEInfo("node", sampler, 3, 16)]
        m = gs.UnsupervisedGraphsage({"batch_size": B, "dropout": 0.}, shard, adj_dev, deg, infos, concat=True,
                                     aggregator_type="mean", neg_sample_size=7, learning_rate=0.01, device=dev,
                                     distributed=True, seed=50 + rank)
        for step in range(3):
            b1 = torch.from_numpy(rs.randint(lo, hi, size=B).astype(np.int32))
            b2 = torch.from_numpy(adj[b1.numpy(), step % md].astype(np.int32))
            loss = m.train_step(b1, b2)
            assert np.isfinite(float(loss)) and m.last_allreduce_bytes == sum(p.numel() for p in m.parameters()) * 4
            mine = torch.cat([p.detach().reshape(-1) for p in m.parameters()]).cpu()
            both = [None] * world
            dist.all_gather_object(both, mine)
            assert torch.equal(both[0], both[1]), "weights diverged after step %d" % step
        shard.close()
        q.put((rank, "ok"))
    except Exception:  # pragma: no cover
        import traceback
        q.put((rank, traceback.format_exc()))
    finally:
        if dist.is_initialized():
            dist.destroy_process_group()


@pytest.mark.gpu
def test_unsupervised_data_parallel_two_gpus():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    _run(_gpu_train_worker, 2)
