"""Callers / data formats on the input side of the hot path (SURVEY section 8 row f3): dataset ingest
(reference graphsage/utils.py:19-92) and the minibatch iterators (reference graphsage/minibatch.py).  CPU only.

The iterator fixtures in tests/golden/iterators.npz were produced by the reference's OWN iterator classes
(tests/golden/make_golden.py: golden_iterators) running over graphsage_b200.graph.Graph with numpy's legacy global
generator seeded as noted there; these tests replay the same seeds through graphsage_b200.minibatch.
"""
import json
import os
import random

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))

from graphsage_b200 import minibatch, utils  # noqa: E402
from graphsage_b200.graph import Graph, node_link_graph, to_csr  # noqa: E402

GOLD = os.path.join(HERE, "golden", "iterators.npz")
TOY_GOLD = os.path.join(HERE, "golden", "toy_ppi.npz")


def fixture_graph():
    """Same construction as tests/golden/make_golden.py:iterator_fixture_graph (kept in step by test_fixture_graph_is_the_golden_one)."""
    r = np.random.RandomState(31)
    n = 90
    G = Graph()
    ids = [int(i) for i in r.permutation(n) + 100]
    for u in ids:
        G.add_node(u, val=bool(r.rand() < 0.12), test=bool(r.rand() < 0.15))
    for u in ids:
        if G.node[u]["val"] and G.node[u]["test"]:
            G.node[u]["test"] = False
    for u in ids[:-4]:
        for v in r.choice(ids[:-4], size=[1, 2, 5, 9, 14][r.randint(5)], replace=False):
            if int(v) != u:
                G.add_edge(u, int(v))
    for u, v in G.edges():
        a, b = G.node[u], G.node[v]
        G[u][v]["train_removed"] = bool(a["val"] or b["val"] or a["test"] or b["test"])
    return G, {u: i for i, u in enumerate(sorted(ids))}


@pytest.fixture(scope="module")
def gold():
    return np.load(GOLD)


def eq(a, b):
    a, b = np.asarray(a), np.asarray(b)
    assert a.shape == b.shape, (a.shape, b.shape)
    assert np.array_equal(a, b)


# ---------------------------------------------------------------------------------------------------- graph surface
def test_graph_surface_matches_networkx_1x_conventions():
    G = Graph()
    G.add_node("a", val=False)
    G.add_edge("a", "b", w=1)
    G.add_edge("b", "c")
    G.add_edge("c", "a")
    G.add_edge("c", "c")                                   # self loop
    G.add_node("z")
    assert G.nodes() == ["a", "b", "c", "z"]
    assert G.neighbors("a") == ["b", "c"] and G.neighbors("c") == ["b", "a", "c"]
    assert G.edges() == [("a", "b"), ("a", "c"), ("b", "c"), ("c", "c")]      # every undirected edge once
    assert G["a"]["b"] is G["b"]["a"] and G["a"]["b"]["w"] == 1               # one attribute dict per edge
    assert G.degree("z") == 0 and G.degree("c") == 4                          # self loop counts twice
    assert "a" in G and len(G) == 4
    H = G.subgraph(["a", "c", "z"])
    assert H.nodes() == ["a", "c", "z"] and H.edges() == [("a", "c"), ("c", "c")]
    G.remove_node("c")
    assert G.nodes() == ["a", "b", "z"] and G.edges() == [("a", "b")] and G.neighbors("b") == ["a"]


def test_node_link_graph_uses_positions_and_rejects_directed():
    data = {"directed": False, "multigraph": False, "graph": {},
            "nodes": [{"id": "x", "val": False, "test": False}, {"id": "y", "val": True, "test": False}, {"id": "w", "val": False, "test": True}],
            "links": [{"source": 0, "target": 2, "k": 3}, {"source": 2, "target": 1}]}
    G = node_link_graph(data)
    assert G.nodes() == ["x", "y", "w"] and G.edges() == [("x", "w"), ("y", "w")]
    assert G["x"]["w"]["k"] == 3 and G.node["y"]["val"] is True
    with pytest.raises(ValueError):
        node_link_graph(dict(data, directed=True))


def test_to_csr_orders_and_flags():
    G, id2idx = fixture_graph()
    c = to_csr(G, id2idx)
    n = len(id2idx)
    assert c["indptr"].shape == (n + 1,) and c["indptr"][-1] == 2 * len(G.edges())
    for u in G.nodes()[:20]:
        iu = id2idx[u]
        row = c["indices"][c["indptr"][iu]:c["indptr"][iu + 1]]
        assert list(row) == [id2idx[v] for v in G.neighbors(u)]
        flags = c["edge_removed"][c["indptr"][iu]:c["indptr"][iu + 1]]
        assert list(flags) == [G[u][v]["train_removed"] for v in G.neighbors(u)]
        assert c["val_or_test"][iu] == (G.node[u]["val"] or G.node[u]["test"])
    assert list(c["node_order"]) == [id2idx[u] for u in G.nodes()]


# ---------------------------------------------------------------------------------------------------- iterators
def test_fixture_graph_is_the_golden_one(gold):
    G, id2idx = fixture_graph()
    np.random.seed(123)
    it = minibatch.NodeMinibatchIterator(G, id2idx, None, {u: 0 for u in G.nodes()}, 4, batch_size=7, max_degree=6)
    eq(it.adj, gold["n_adj"])
    assert it.adj.dtype == np.int32 and it.adj.shape == (91, 6) and (it.adj[90] == 90).all()


def test_node_iterator_matches_reference(gold):
    G, id2idx = fixture_graph()
    lab = {u: int(u % 4) for u in G.nodes()}
    np.random.seed(123)
    it = minibatch.NodeMinibatchIterator(G, id2idx, None, lab, 4, batch_size=7, max_degree=6, context_pairs="swallowed")
    eq(it.adj, gold["n_adj"]); eq(it.deg, gold["n_deg"]); eq(it.test_adj, gold["n_test_adj"])
    eq(it.train_nodes, gold["n_train_nodes"]); eq(it.val_nodes, gold["n_val_nodes"]); eq(it.test_nodes, gold["n_test_nodes"])
    assert it.num_training_batches() == int(gold["n_num_batches"])
    f, l = it.next_minibatch_feed_dict()
    eq(f["batch"], gold["n_b0"]); eq(l, gold["n_l0"]); assert f["batch_size"] == int(gold["n_bs0"]) and f["labels"] is l
    f, l = it.next_minibatch_feed_dict()
    eq(f["batch"], gold["n_b1"]); eq(l, gold["n_l1"])
    f, l = it.node_val_feed_dict(size=5)
    eq(f["batch"], gold["n_val5"]); eq(l, gold["n_val5_labels"])
    f, l = it.node_val_feed_dict(test=True)
    eq(f["batch"], gold["n_test_all"])
    f, l, done, sub = it.incremental_node_val_feed_dict(4, 1)
    eq(f["batch"], gold["n_inc"]); assert done == bool(gold["n_inc_done"]); eq(sub, gold["n_inc_nodes"])
    (f, l), done, sub = it.incremental_embed_feed_dict(8, 2)
    eq(f["batch"], gold["n_emb"]); assert done == bool(gold["n_emb_done"])
    it.shuffle()
    assert it.batch_num == 0
    f, l = it.next_minibatch_feed_dict()
    eq(f["batch"], gold["n_shuf_b0"]); eq(it.train_nodes, gold["n_shuf_train"])
    n = 0
    while not it.end():
        it.next_minibatch_feed_dict()
        n += 1
    assert n == int(gold["n_batches_to_end"])


def test_node_iterator_list_labels_and_placeholder_keys(gold):
    G, id2idx = fixture_graph()
    lab2 = {u: [int(u % 2), int(u % 3 == 0), 1] for u in G.nodes()}
    ph = {"batch_size": ("ph", 0), "batch": ("ph", 1), "labels": ("ph", 2)}       # any hashable stands in for a placeholder
    np.random.seed(5)
    it = minibatch.NodeMinibatchIterator(G, id2idx, ph, lab2, 3, batch_size=5, max_degree=6)
    f, l = it.next_minibatch_feed_dict()
    assert set(f) == set(ph.values())
    eq(f[("ph", 1)], gold["n2_b0"]); eq(l, gold["n2_l0"])


def test_edge_iterator_matches_reference(gold):
    G, id2idx = fixture_graph()
    np.random.seed(123)
    it = minibatch.EdgeMinibatchIterator(G, id2idx, None, batch_size=9, max_degree=6)
    eq(it.nodes, gold["e_nodes"]); eq(it.adj, gold["e_adj"]); eq(it.deg, gold["e_deg"]); eq(it.test_adj, gold["e_test_adj"])
    eq(it.train_edges, gold["e_train_edges"]); eq(it.val_edges, gold["e_val_edges"])
    assert it.val_set_size == len(gold["e_val_edges"]) and it.num_training_batches() == int(gold["e_num_batches"])
    assert it.missing == 0
    f = it.next_minibatch_feed_dict()
    eq(f["batch1"], gold["e_b1"]); eq(f["batch2"], gold["e_b2"]); assert f["batch_size"] == int(gold["e_bs"])
    f = it.val_feed_dict(size=6)
    eq(f["batch1"], gold["e_val6_1"]); eq(f["batch2"], gold["e_val6_2"])
    f, done, sub = it.incremental_val_feed_dict(5, 1)
    eq(f["batch1"], gold["e_inc1"]); eq(f["batch2"], gold["e_inc2"]); assert done == bool(gold["e_inc_done"])
    f, done, sub = it.incremental_embed_feed_dict(10, 3)
    eq(f["batch1"], gold["e_emb1"]); eq(f["batch2"], gold["e_emb1"]); assert done == bool(gold["e_emb_done"])
    tr, va = it.label_val()
    eq(tr, gold["e_label_train"]); eq(va, gold["e_label_val"])
    it.shuffle()
    f = it.next_minibatch_feed_dict()
    eq(f["batch1"], gold["e_shuf_b1"]); eq(it.nodes, gold["e_shuf_nodes"])


def test_edge_iterator_context_pairs_and_n2v_modes(gold):
    G, id2idx = fixture_graph()
    pairs = [tuple(int(x) for x in p) for p in gold["c_pairs"]]
    np.random.seed(77)
    it = minibatch.EdgeMinibatchIterator(G, id2idx, None, context_pairs=pairs, batch_size=9, max_degree=6)
    eq(it.train_edges, gold["c_train_edges"])
    assert len(it.train_edges) < len(pairs)                      # _remove_isolated dropped some pairs
    np.random.seed(78)
    it = minibatch.EdgeMinibatchIterator(G, id2idx, None, context_pairs=pairs, batch_size=9, max_degree=6, n2v_retrain=True,
                                         fixed_n2v=True)
    eq(it.train_edges, gold["c_n2v_fixed"]); assert it.val_edges is it.train_edges
    np.random.seed(79)
    it = minibatch.EdgeMinibatchIterator(G, id2idx, None, context_pairs=pairs, batch_size=9, max_degree=6, n2v_retrain=True)
    eq(it.train_edges, gold["c_n2v"])


def test_iterator_rng_argument_is_isolated_from_global_state(gold):
    G, id2idx = fixture_graph()
    np.random.seed(999)
    before = np.random.get_state()[1].copy()
    it = minibatch.NodeMinibatchIterator(G, id2idx, None, {u: 0 for u in G.nodes()}, 4, batch_size=7, max_degree=6,
                                         rng=np.random.RandomState(123))
    eq(it.adj, gold["n_adj"])
    assert np.array_equal(before, np.random.get_state()[1])


# ---------------------------------------------------------------------------------------------------- ingest
def test_standard_scale_equals_sklearn():
    sk = pytest.importorskip("sklearn.preprocessing")
    r = np.random.RandomState(0)
    x = r.randn(200, 7) * np.array([1, 5, 0.1, 1, 1, 100, 1]) + np.array([0, 3, -2, 0, 0, 50, 0])
    x[:, 3] = 2.5                                         # a constant column is only centred
    train = r.choice(200, 120, replace=False)
    ref = sk.StandardScaler().fit(x[train]).transform(x)
    got = utils.standard_scale(x, train)
    assert np.allclose(got, ref, rtol=0, atol=1e-12)
    assert np.all(got[:, 3] == 0.0)


def test_write_then_load_roundtrip(tmp_path):
    G, id2idx = fixture_graph()
    feats = np.random.RandomState(4).randn(len(id2idx), 5)
    cls = {u: [int(u % 2), 1] for u in G.nodes()}
    walks = [(G.nodes()[0], G.nodes()[1]), (G.nodes()[2], G.nodes()[0])]
    # one node without val/test annotations must be dropped by the loader (reference utils.py:45-49)
    G.add_node(999)
    G.add_edge(999, G.nodes()[0])
    id2idx[999] = len(id2idx)
    cls[999] = [0, 0]
    feats = np.vstack([feats, np.zeros((1, 5))])
    prefix = str(tmp_path / "toy")
    utils.write_dataset(prefix, G, feats, id2idx, cls, walks)
    G2, f2, id2, w2, c2 = utils.load_data(prefix, normalize=False, load_walks=True)
    assert 999 not in G2 and len(G2) == len(G) - 1
    assert G2.nodes() == [n for n in G.nodes() if n != 999]
    assert sorted(map(sorted, G2.edges())) == sorted(sorted(e) for e in G.edges() if 999 not in e)
    for u, v in G2.edges():
        a, b = G2.node[u], G2.node[v]
        assert G2[u][v]["train_removed"] == bool(a["val"] or b["val"] or a["test"] or b["test"])
    assert np.array_equal(f2, feats) and id2 == id2idx and c2 == cls and w2 == walks
    assert isinstance(next(iter(id2)), int)                # int node ids stay ints (utils.py:22-25)
    _, f3, _, _, _ = utils.load_data(prefix, normalize=True)
    tr = np.array([id2[n] for n in G2.nodes() if not G2.node[n]["val"] and not G2.node[n]["test"]])
    assert np.allclose(f3[tr].mean(axis=0), 0, atol=1e-12) and np.allclose(f3[tr].std(axis=0), 1, atol=1e-12)
    os.remove(prefix + "-feats.npy")
    assert utils.load_data(prefix)[1] is None              # no features: identity features only (utils.py:27-31)


def test_random_walk_pairs():
    G, _ = fixture_graph()
    nodes = [n for n in G.nodes() if not G.node[n]["val"] and not G.node[n]["test"]]
    H = G.subgraph(nodes)                                  # as the reference's __main__ does (utils.py:99-100)
    random.seed(1)
    pairs = utils.run_random_walks(H, nodes, num_walks=3)
    random.seed(1)
    assert pairs == utils.run_random_walks(H, nodes, num_walks=3)
    assert pairs and all(a != b for a, b in pairs)
    assert all(a in H and b in H for a, b in pairs)
    per_start = {}
    for a, _ in pairs:
        per_start[a] = per_start.get(a, 0) + 1
    assert max(per_start.values()) <= 3 * (utils.WALK_LEN - 1)          # the start itself is never paired with itself
    assert all(H.degree(a) > 0 for a in per_start)


@pytest.fixture(scope="module")
def toy(tmp_path_factory):
    """tests/golden/toy_ppi.npz - a 2,300-node sample of the reference's example_data/toy-ppi (make_golden.py:
    golden_toy_ppi) - written back out in that dataset's file format; returns the path prefix."""
    t = np.load(TOY_GOLD)
    ids, feats, labels = [int(i) for i in t["ids"]], t["feats"].astype(np.float64), t["labels"].tolist()
    nodes = [{"test": bool(te), "id": i, "feature": f.tolist(), "val": bool(va), "label": lab}
             for i, va, te, f, lab in zip(ids, t["val"], t["test"], feats, labels)]
    links = [{"test_removed": bool(te), "train_removed": bool(tr), "target": int(d), "source": int(s)}
             for s, d, tr, te in zip(t["link_source"], t["link_target"], t["link_train_removed"], t["link_test_removed"])]
    prefix = str(tmp_path_factory.mktemp("toy") / "toy-ppi")
    with open(prefix + "-G.json", "w") as fp:
        json.dump({"directed": False, "graph": {"name": str(t["graph_name"])}, "nodes": nodes, "links": links,
                   "multigraph": False}, fp)
    with open(prefix + "-id_map.json", "w") as fp:
        json.dump({str(i): r for r, i in enumerate(ids)}, fp)
    with open(prefix + "-class_map.json", "w") as fp:
        json.dump({str(i): lab for i, lab in zip(ids, labels)}, fp)
    np.save(prefix + "-feats.npy", feats)
    return prefix


def test_toy_ppi_ingest_and_tables(toy):
    G, feats, id_map, walks, class_map = utils.load_data(toy, normalize=True, load_walks=False)
    assert len(G) == 2300 and len(G.edges()) == 41857 and feats.shape == (2300, 50) and len(id_map) == 2300
    assert len(next(iter(class_map.values()))) == 121 and isinstance(next(iter(id_map)), int)
    kinds = [(G.node[n]["val"], G.node[n]["test"]) for n in G.nodes()]
    assert kinds.count((False, False)) == 1500 and kinds.count((True, False)) == 300 and kinds.count((False, True)) == 500
    tr = np.array([id_map[n] for n in G.nodes() if not G.node[n]["val"] and not G.node[n]["test"]])
    assert np.allclose(feats[tr].mean(axis=0), 0, atol=1e-9)
    np.random.seed(123)
    it = minibatch.NodeMinibatchIterator(G, id_map, None, class_map, 121, batch_size=512, max_degree=128)
    n = len(id_map)
    assert it.adj.shape == (n + 1, 128) and it.adj.dtype == np.int32 and (it.adj[n] == n).all()
    vt = np.array([id_map[u] for u in G.nodes() if G.node[u]["val"] or G.node[u]["test"]])
    assert (it.adj[vt] == n).all() and (it.deg[vt] == 0).all()                       # val/test rows stay all-dummy
    has = it.deg > 0
    assert ((it.adj[:n][has] < n).all()) and ((it.adj[:n][~has] == n).all())
    # every train-table entry is a real train-graph neighbour
    c = to_csr(G, id_map)
    for u in tr[:200]:
        nb = c["indices"][c["indptr"][u]:c["indptr"][u + 1]][~c["edge_removed"][c["indptr"][u]:c["indptr"][u + 1]]]
        assert it.deg[u] == len(nb) and (len(nb) == 0 or set(it.adj[u]) <= set(nb))
    assert (it.test_adj[:n] < n).sum() >= (it.adj[:n] < n).sum()
    f, l = it.next_minibatch_feed_dict()
    assert f["batch_size"] == 512 and l.shape == (512, 121) and set(np.unique(l)) <= {0, 1}
    assert all(it.deg[id_map[u]] > 0 for u in it.train_nodes)


def test_config1_toy_ppi_cpu_oracle_path_loss_decreases(toy):
    """SURVEY 8d config 1: toy-ppi, graphsage_mean, B = 512, max_degree 128, dims [50, 128, 128], 121 sigmoid classes,
    fanouts [25, 10], lr 0.01 (reference supervised_train.py:32-49) on the CPU oracle path (oracle/torch_ref.py):
    ingest -> iterator -> sample -> gather -> aggregate -> l2-normalise -> Dense head -> sigmoid xent -> clipped Adam.
    The sample's train nodes last three batches, so the steps run over epochs, reshuffled as supervised_train.py does."""
    import torch
    from oracle import torch_ref
    G, feats, id_map, _, class_map = utils.load_data(toy, normalize=True)
    np.random.seed(123)
    it = minibatch.NodeMinibatchIterator(G, id_map, None, class_map, 121, batch_size=512, max_degree=128)
    n, F, D, C = len(id_map), feats.shape[1], 128, 121
    feats_t = torch.from_numpy(np.vstack([feats, np.zeros((1, F))]).astype(np.float32))     # zero dummy row (supervised_train.py:133-135)
    adj_t = torch.from_numpy(it.adj)
    g = torch.Generator().manual_seed(0)

    def glorot(shape):
        r = float(np.sqrt(6.0 / (shape[0] + shape[1])))
        return ((torch.rand(shape, generator=g) * 2 - 1) * r).requires_grad_(True)

    aggs = [{"neigh_weights": glorot((F, D)), "self_weights": glorot((F, D))},
            {"neigh_weights": glorot((2 * D, D)), "self_weights": glorot((2 * D, D))}]
    head = {"weights": glorot((2 * D, C)), "bias": torch.zeros(C, requires_grad=True)}
    params = [v for a in aggs for v in a.values()] + list(head.values())
    opt = torch.optim.Adam(params, lr=0.01)
    it.shuffle()
    losses = []
    for step in range(12):
        if it.end():
            it.shuffle()
        feed, labels = it.next_minibatch_feed_dict()
        seeds = torch.tensor(feed["batch"], dtype=torch.int32)
        out = torch_ref.forward(adj_t, feats_t, seeds, [25, 10], aggs, True, "mean", 123, 2 * step, normalize=True)
        logits = out @ head["weights"] + head["bias"]
        loss = torch.nn.functional.binary_cross_entropy_with_logits(logits, torch.from_numpy(labels.astype(np.float32)))
        opt.zero_grad()
        loss.backward()
        for p in params:
            p.grad.clamp_(-5.0, 5.0)                                  # supervised_models.py:101-103
        opt.step()
        losses.append(float(loss.detach()))
    assert np.isfinite(losses).all()
    assert np.mean(losses[-3:]) < 0.9 * np.mean(losses[:3]), losses


@pytest.mark.parametrize("seed", [0, 1, 2, 3])
def test_random_graphs_tables_are_consistent_with_the_graph(seed):
    """Randomised cross-check of graph.py -> to_csr -> construct_adj against a plain set-of-edges model."""
    r = np.random.RandomState(seed)
    n, md = int(r.randint(5, 60)), int(r.randint(1, 9))
    names = ["v%d" % i for i in r.permutation(n)]
    G = Graph()
    edges = set()
    for u in names:
        G.add_node(u, val=bool(r.rand() < 0.2), test=bool(r.rand() < 0.2))
    for _ in range(int(r.randint(0, 4 * n))):
        a, b = names[r.randint(n)], names[r.randint(n)]
        G.add_edge(a, b)
        edges.add(frozenset((a, b)))
    assert {frozenset(e) for e in G.edges()} == edges and len(G.edges()) == len(edges)
    for u, v in G.edges():
        G[u][v]["train_removed"] = bool(G.node[u]["val"] or G.node[u]["test"] or G.node[v]["val"] or G.node[v]["test"])
    id2idx = {u: i for i, u in enumerate(sorted(names))}
    it = minibatch.NodeMinibatchIterator(G, id2idx, None, {u: 0 for u in names}, 2, batch_size=3, max_degree=md,
                                         rng=np.random.RandomState(seed))
    idx2id = {i: u for u, i in id2idx.items()}
    for u in names:
        iu = id2idx[u]
        vt = G.node[u]["val"] or G.node[u]["test"]
        train_nb = {id2idx[v] for v in G.neighbors(u) if not G[u][v]["train_removed"]}
        all_nb = {id2idx[v] for v in G.neighbors(u)}
        if vt or not train_nb:
            assert (it.adj[iu] == n).all()
            assert it.deg[iu] == (0 if vt else len(train_nb))
        else:
            assert set(it.adj[iu]) <= train_nb and it.deg[iu] == len(train_nb)
            if len(train_nb) >= md:
                assert len(set(it.adj[iu])) == md                    # subsampled without replacement
            else:
                assert set(it.adj[iu]) <= train_nb and len(it.adj[iu]) == md
        if all_nb:
            assert set(it.test_adj[iu]) <= all_nb
            assert len(set(it.test_adj[iu])) == min(md, len(all_nb)) or len(all_nb) < md
        else:
            assert (it.test_adj[iu] == n).all()
    assert (it.adj[n] == n).all() and (it.test_adj[n] == n).all()
    assert set(it.train_nodes) == {u for u in names if not (G.node[u]["val"] or G.node[u]["test"]) and it.deg[id2idx[u]] > 0}
    assert idx2id[0] == sorted(names)[0]
