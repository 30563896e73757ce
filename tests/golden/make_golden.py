"""Generate tests/golden/*.npz by executing the reference's own hot-path python
(graphsage/{neigh_samplers,aggregators,layers,inits,models,minibatch}.py of a williamleif/GraphSAGE
checkout) under the numpy TF shim (tf_shim.py).  The tests only read the committed .npz files.

    GRAPHSAGE_REFERENCE=<checkout of williamleif/GraphSAGE> python tests/golden/make_golden.py [name]

Nothing from the reference is copied: the modules are imported from where they lie.
"""
import json
import os
import sys
import types

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
REFERENCE = os.environ.get("GRAPHSAGE_REFERENCE", "")
if not os.path.isdir(os.path.join(REFERENCE, "graphsage")):
    sys.exit("set GRAPHSAGE_REFERENCE to a checkout of williamleif/GraphSAGE")
sys.path.insert(0, ROOT)
sys.path.insert(0, HERE)
sys.path.insert(0, REFERENCE)

import tf_shim  # noqa: E402

tf = tf_shim.install()

from graphsage.neigh_samplers import UniformNeighborSampler  # noqa: E402
from graphsage.aggregators import MeanAggregator, GCNAggregator, MaxPoolingAggregator, MeanPoolingAggregator  # noqa: E402
from graphsage.models import SampleAndAggregate, SAGEInfo  # noqa: E402
from graphsage.minibatch import NodeMinibatchIterator  # noqa: E402
from graphsage.inits import glorot  # noqa: E402

rs = np.random.RandomState(7)


def save(name, **kw):
    path = os.path.join(HERE, name + ".npz")
    np.savez_compressed(path, **kw)
    print("wrote", path, {k: np.asarray(v).shape for k, v in kw.items()})


# ------------------------------------------------------------------ sampler
def make_adj(n, md):
    adj = rs.randint(0, n, size=(n + 1, md)).astype(np.int32)
    adj[n, :] = n                       # dummy row (minibatch.py:228)
    adj[3, :] = n                       # an isolated node
    return adj


def golden_sampler():
    cases = {}
    for ci, (n, md, nid, k, seed, counter) in enumerate(
            [(50, 16, 23, 5, 123, 0), (200, 128, 64, 25, 123, 1), (200, 128, 7, 10, 99, 1 << 33), (30, 8, 11, 8, 5, 2)]):
        adj = make_adj(n, md)
        ids = rs.randint(0, n + 1, size=nid).astype(np.int32)
        ids[0] = n                      # dummy id -> all outputs n
        tf_shim.SHUFFLE_SEED, tf_shim.SHUFFLE_COUNTER = seed, counter
        sampler = UniformNeighborSampler(adj)
        out = sampler((ids, k))
        cases.update({"adj%d" % ci: adj, "ids%d" % ci: ids, "k%d" % ci: k, "seed%d" % ci: seed,
                      "counter%d" % ci: np.uint64(counter), "out%d" % ci: out.astype(np.int32)})
    cases["n_cases"] = ci + 1
    save("sampler", **cases)


# ------------------------------------------------------------------ aggregators
def golden_aggregators():
    n, k, din, dout = 37, 10, 50, 16
    selfv = rs.randn(n, din).astype(np.float32)
    neigh = rs.randn(n, k, din).astype(np.float32)
    neigh[5] = 0.0                      # a node whose neighbours are all the dummy zero row
    out = {"self": selfv, "neigh": neigh}
    for concat in (False, True):
        agg = MeanAggregator(din, dout, concat=concat)
        tag = "mean_c%d" % concat
        out[tag + "_nw"], out[tag + "_sw"] = agg.vars["neigh_weights"], agg.vars["self_weights"]
        out[tag + "_out"] = agg((selfv, neigh))
        agg = MaxPoolingAggregator(din, dout, concat=concat)
        tag = "maxpool_c%d" % concat
        out[tag + "_nw"], out[tag + "_sw"] = agg.vars["neigh_weights"], agg.vars["self_weights"]
        out[tag + "_mw"], out[tag + "_mb"] = agg.mlp_layers[0].vars["weights"], agg.mlp_layers[0].vars["bias"] + \
            rs.randn(agg.hidden_dim).astype(np.float32) * 0.1
        agg.mlp_layers[0].vars["bias"] = out[tag + "_mb"]     # non-zero bias so the bias add is exercised
        out[tag + "_hidden"] = agg.hidden_dim
        out[tag + "_out"] = agg((selfv, neigh))
    agg = GCNAggregator(din, dout)
    out["gcn_w"] = agg.vars["weights"]
    out["gcn_out"] = agg((selfv, neigh))
    # identity activation (last layer, models.py:307-310) and distinct neigh_input_dim
    neigh2 = rs.randn(n, k, 24).astype(np.float32)
    agg = MeanAggregator(din, dout, neigh_input_dim=24, act=lambda x: x, concat=True)
    out["mean_id_nw"], out["mean_id_sw"], out["neigh2"] = agg.vars["neigh_weights"], agg.vars["self_weights"], neigh2
    out["mean_id_out"] = agg((selfv, neigh2))
    out["glorot_sample"] = glorot([50, 16])
    save("aggregators", **out)


# ------------------------------------------------------------------ K-hop recursion
class _Stub(object):
    """Just the attributes SampleAndAggregate.sample/.aggregate read (models.py:254-330)."""


def golden_khop():
    out = {}
    n, md, f = 300, 32, 20
    adj = make_adj(n, md)
    feats = np.vstack([rs.randn(n, f).astype(np.float32), np.zeros((1, f), np.float32)])   # supervised_train.py:133-135
    B = 9
    seeds = rs.randint(0, n, size=B).astype(np.int32)
    out.update(adj=adj, feats=feats, seeds=seeds)
    for model, cls, concat, dims, fan in [("mean", MeanAggregator, True, [f, 12, 8], [5, 3]),
                                          ("gcn", GCNAggregator, False, [f, 16, 16], [5, 3]),
                                          ("maxpool", MaxPoolingAggregator, True, [f, 12, 8], [4, 2]),
                                          ("mean3", MeanAggregator, True, [f, 8, 8, 6], [4, 3, 2])]:
        tf_shim.SHUFFLE_SEED, tf_shim.SHUFFLE_COUNTER = 123, 40
        sampler = UniformNeighborSampler(adj)
        infos = [SAGEInfo("node", sampler, fan[i], dims[i + 1]) for i in range(len(fan))]
        stub = _Stub()
        stub.batch_size = B
        stub.aggregator_cls = cls
        stub.placeholders = {"dropout": 0.0}
        samples, support = SampleAndAggregate.sample(stub, seeds, infos)
        hidden, aggs = SampleAndAggregate.aggregate(stub, samples, [feats][0], dims, fan, support, concat=concat)
        for h, s in enumerate(samples):
            out["%s_samples%d" % (model, h)] = np.asarray(s).astype(np.int32)
        out[model + "_support"] = np.array(support)
        out[model + "_fanout"] = np.array(fan)
        out[model + "_dims"] = np.array(dims)
        out[model + "_concat"] = concat
        out[model + "_out"] = hidden
        out[model + "_out_l2"] = tf.nn.l2_normalize(hidden, 1)          # models.py:368
        for li, a in enumerate(aggs):
            for key, v in a.vars.items():
                out["%s_L%d_%s" % (model, li, key)] = v
            if hasattr(a, "mlp_layers"):
                out["%s_L%d_mlp_weights" % (model, li)] = a.mlp_layers[0].vars["weights"]
                out["%s_L%d_mlp_bias" % (model, li)] = a.mlp_layers[0].vars["bias"]
    save("khop", **out)


# ------------------------------------------------------------------ padded adjacency
class _FakeG(object):
    """networkx-1.11-shaped view (G.nodes(), G.node[n], G.neighbors(n), G[u][v]) over plain dicts."""

    def __init__(self, nodes, nbrs, attrs, eattrs):
        self._nodes, self._nbrs, self.node, self._e = nodes, nbrs, attrs, eattrs

    def nodes(self):
        return list(self._nodes)

    def neighbors(self, n):
        return list(self._nbrs[n])

    def __getitem__(self, u):
        return {v: self._e[(u, v)] for v in self._nbrs[u]}


def golden_adjacency():
    n, md = 60, 8
    nodes = ["n%d" % i for i in rs.permutation(n)]
    id2idx = {"n%d" % i: i for i in range(n)}
    nbrs = {u: [] for u in nodes}
    for i in range(n):
        deg = [0, 1, 3, 8, 12, 20][rs.randint(6)]
        for j in rs.choice(n, size=deg, replace=False):
            u, v = "n%d" % i, "n%d" % j
            if u != v and v not in nbrs[u]:
                nbrs[u].append(v)
                nbrs[v].append(u)
    attrs = {u: {"val": bool(rs.rand() < 0.1), "test": bool(rs.rand() < 0.15)} for u in nodes}
    eattrs = {}
    for u in nodes:
        for v in nbrs[u]:
            eattrs[(u, v)] = {"train_removed": attrs[u]["val"] or attrs[u]["test"] or attrs[v]["val"] or attrs[v]["test"]}
    G = _FakeG(nodes, nbrs, attrs, eattrs)
    np.random.seed(123)
    it = NodeMinibatchIterator(G, id2idx, None, {u: 0 for u in nodes}, 2, batch_size=4, max_degree=md)
    flat_nb = np.array([id2idx[v] for u in nodes for v in nbrs[u]], dtype=np.int32)
    nb_ptr = np.cumsum([0] + [len(nbrs[u]) for u in nodes]).astype(np.int64)
    flat_removed = np.array([eattrs[(u, v)]["train_removed"] for u in nodes for v in nbrs[u]], dtype=bool)
    save("adjacency", node_order=np.array([id2idx[u] for u in nodes], dtype=np.int32), nb_ptr=nb_ptr, nb_idx=flat_nb,
         nb_removed=flat_removed, val_or_test=np.array([attrs[u]["val"] or attrs[u]["test"] for u in nodes]),
         max_degree=md, adj=it.adj.astype(np.int32), deg=it.deg, test_adj=it.test_adj.astype(np.int32))


def golden_meanpool():
    """MeanPoolingAggregator (reference aggregators.py:197-273), generated separately so the older fixtures keep their bytes."""
    rs2 = np.random.RandomState(21)
    n, k, din, dout = 29, 7, 40, 16
    selfv = rs2.randn(n, din).astype(np.float32)
    neigh = rs2.randn(n, k, din).astype(np.float32)
    out = {"self": selfv, "neigh": neigh}
    for concat in (False, True):
        agg = MeanPoolingAggregator(din, dout, concat=concat)
        tag = "c%d" % concat
        agg.mlp_layers[0].vars["bias"] = agg.mlp_layers[0].vars["bias"] + rs2.randn(agg.hidden_dim).astype(np.float32) * 0.1
        out[tag + "_nw"], out[tag + "_sw"] = agg.vars["neigh_weights"], agg.vars["self_weights"]
        out[tag + "_mw"], out[tag + "_mb"] = agg.mlp_layers[0].vars["weights"], agg.mlp_layers[0].vars["bias"]
        out[tag + "_out"] = agg((selfv, neigh))
    save("meanpool", **out)


def iterator_fixture_graph(seed=31, n=90):
    """Deterministic small graph with val/test annotations, isolated nodes, a node whose edges all lead to val/test nodes,
    and degrees on both sides of max_degree.  Node ids are ints (so that CPython's set order is reproducible)."""
    from graphsage_b200.graph import Graph
    r = np.random.RandomState(seed)
    G = Graph()
    ids = [int(i) for i in r.permutation(n) + 100]            # node ids 100..189, inserted in shuffled order
    for u in ids:
        G.add_node(u, val=bool(r.rand() < 0.12), test=bool(r.rand() < 0.15))
    for u in ids:
        if G.node[u]["val"] and G.node[u]["test"]:
            G.node[u]["test"] = False
    for u in ids[:-4]:                                           # the last four stay isolated
        for v in r.choice(ids[:-4], size=[1, 2, 5, 9, 14][r.randint(5)], replace=False):
            if int(v) != u:
                G.add_edge(u, int(v))
    for u, v in G.edges():
        a, b = G.node[u], G.node[v]
        G[u][v]["train_removed"] = bool(a["val"] or b["val"] or a["test"] or b["test"])
    id2idx = {u: i for i, u in enumerate(sorted(ids))}
    return G, id2idx


def golden_iterators():
    """NodeMinibatchIterator / EdgeMinibatchIterator (reference minibatch.py) driven over graphsage_b200.graph.Graph."""
    from graphsage.minibatch import EdgeMinibatchIterator
    G, id2idx = iterator_fixture_graph()
    ph = {k: k for k in ("batch_size", "batch", "labels", "batch1", "batch2")}
    out = {}
    # ---- node iterator, integer class labels
    lab = {u: int(u % 4) for u in G.nodes()}
    np.random.seed(123)
    it = NodeMinibatchIterator(G, id2idx, ph, lab, 4, batch_size=7, max_degree=6)
    out.update(n_adj=it.adj.astype(np.int32), n_deg=it.deg, n_test_adj=it.test_adj.astype(np.int32),
               n_train_nodes=np.array(it.train_nodes), n_val_nodes=np.array(it.val_nodes), n_test_nodes=np.array(it.test_nodes),
               n_num_batches=it.num_training_batches())
    f, l = it.next_minibatch_feed_dict()
    out.update(n_b0=np.array(f["batch"]), n_l0=l, n_bs0=f["batch_size"])
    f, l = it.next_minibatch_feed_dict()
    out.update(n_b1=np.array(f["batch"]), n_l1=l)
    f, l = it.node_val_feed_dict(size=5)
    out.update(n_val5=np.array(f["batch"]), n_val5_labels=l)
    f, l = it.node_val_feed_dict(test=True)
    out.update(n_test_all=np.array(f["batch"]))
    f, l, done, sub = it.incremental_node_val_feed_dict(4, 1)
    out.update(n_inc=np.array(f["batch"]), n_inc_done=done, n_inc_nodes=np.array(sub))
    (f, l), done, sub = it.incremental_embed_feed_dict(8, 2)
    out.update(n_emb=np.array(f["batch"]), n_emb_done=done)
    it.shuffle()
    f, l = it.next_minibatch_feed_dict()
    out.update(n_shuf_b0=np.array(f["batch"]), n_shuf_train=np.array(it.train_nodes))
    n = 0
    while not it.end():
        it.next_minibatch_feed_dict()
        n += 1
    out.update(n_batches_to_end=n)
    # ---- node iterator, multi-hot list labels
    lab2 = {u: [int(u % 2), int(u % 3 == 0), 1] for u in G.nodes()}
    np.random.seed(5)
    it = NodeMinibatchIterator(G, id2idx, ph, lab2, 3, batch_size=5, max_degree=6)
    f, l = it.next_minibatch_feed_dict()
    out.update(n2_b0=np.array(f["batch"]), n2_l0=l)
    # ---- edge iterator over graph edges
    np.random.seed(123)
    it = EdgeMinibatchIterator(G, id2idx, ph, batch_size=9, max_degree=6)
    out.update(e_nodes=np.array(it.nodes), e_adj=it.adj.astype(np.int32), e_deg=it.deg, e_test_adj=it.test_adj.astype(np.int32),
               e_train_edges=np.array(it.train_edges), e_val_edges=np.array(it.val_edges), e_num_batches=it.num_training_batches())
    f = it.next_minibatch_feed_dict()
    out.update(e_b1=np.array(f["batch1"]), e_b2=np.array(f["batch2"]), e_bs=f["batch_size"])
    f = it.val_feed_dict(size=6)
    out.update(e_val6_1=np.array(f["batch1"]), e_val6_2=np.array(f["batch2"]))
    f, done, sub = it.incremental_val_feed_dict(5, 1)
    out.update(e_inc1=np.array(f["batch1"]), e_inc2=np.array(f["batch2"]), e_inc_done=done)
    f, done, sub = it.incremental_embed_feed_dict(10, 3)
    out.update(e_emb1=np.array(f["batch1"]), e_emb_done=done)
    tr, va = it.label_val()
    out.update(e_label_train=np.array(tr), e_label_val=np.array(va))
    it.shuffle()
    f = it.next_minibatch_feed_dict()
    out.update(e_shuf_b1=np.array(f["batch1"]), e_shuf_nodes=np.array(it.nodes))
    # ---- edge iterator over context pairs (random-walk co-occurrences), n2v modes
    r = np.random.RandomState(3)
    nodes = G.nodes()
    pairs = [(nodes[i], nodes[j]) for i, j in r.randint(0, len(nodes), size=(60, 2))]
    np.random.seed(77)
    it = EdgeMinibatchIterator(G, id2idx, ph, context_pairs=pairs, batch_size=9, max_degree=6)
    out.update(c_pairs=np.array(pairs), c_train_edges=np.array(it.train_edges))
    np.random.seed(78)
    it = EdgeMinibatchIterator(G, id2idx, ph, context_pairs=pairs, batch_size=9, max_degree=6, n2v_retrain=True, fixed_n2v=True)
    out.update(c_n2v_fixed=np.array(it.train_edges))
    np.random.seed(79)
    it = EdgeMinibatchIterator(G, id2idx, ph, context_pairs=pairs, batch_size=9, max_degree=6, n2v_retrain=True)
    out.update(c_n2v=np.array(it.train_edges))
    save("iterators", **out)


def golden_heads():
    """Loss heads either side of the hot path's output: BipartiteEdgePredLayer (reference prediction.py:68-122),
    the MRR of SampleAndAggregate._accuracy (models.py:393-405) and SupervisedGraphsage._loss / predict
    (supervised_models.py:101-126), executed from the reference's own files."""
    from graphsage.prediction import BipartiteEdgePredLayer
    from graphsage.supervised_models import SupervisedGraphsage
    r = np.random.RandomState(11)
    B, NEG, D, C = 13, 20, 16, 6

    def unit(x):
        return (x / np.linalg.norm(x, axis=1, keepdims=True)).astype(np.float32)

    o1, o2, on = unit(r.randn(B, D)), unit(r.randn(B, D)), unit(r.randn(NEG, D))
    o2[3] = o1[3]                                   # a pair that ranks first
    on[5] = o1[7]                                   # a negative that beats a true pair
    out = {"o1": o1, "o2": o2, "on": on}
    ph = {"dropout": 0.0}
    for fn in ("xent", "skipgram", "hinge"):
        layer = BipartiteEdgePredLayer(D, D, ph, act=tf.nn.sigmoid, loss_fn=fn, bilinear_weights=False, name="edge_predict")
        out["loss_" + fn] = np.float64(layer.loss(o1, o2, on))
    out["aff"] = layer.affinity(o1, o2)
    out["neg_aff"] = layer.neg_cost(o1, on)
    layer = BipartiteEdgePredLayer(D, D, ph, loss_fn="xent", neg_sample_weights=0.25, bilinear_weights=True, name="bil")
    out["bil_w"] = layer.vars["weights"]
    out["bil_aff"], out["bil_neg_aff"] = layer.affinity(o1, o2), layer.neg_cost(o1, on)
    out["bil_loss"] = np.float64(layer.loss(o1, o2, on))
    # ---- MRR
    stub = _Stub()
    stub.link_pred_layer = BipartiteEdgePredLayer(D, D, ph, bilinear_weights=False, name="edge_predict2")
    stub.outputs1, stub.outputs2, stub.neg_outputs, stub.batch_size = o1, o2, on, B
    tf.app.flags.FLAGS.neg_sample_size = NEG
    SampleAndAggregate._accuracy(stub)
    out["mrr"], out["ranks"] = np.float64(stub.mrr), stub.ranks
    # ---- supervised loss / predictions
    logits = r.randn(B, C).astype(np.float32) * 2
    multi = (r.rand(B, C) < 0.3).astype(np.float32)
    onehot = np.eye(C, dtype=np.float32)[r.randint(0, C, size=B)]
    agg_vars = [{"neigh_weights": r.randn(5, 4).astype(np.float32), "self_weights": r.randn(5, 4).astype(np.float32)},
                {"weights": r.randn(4, 3).astype(np.float32)}]
    head_vars = {"weights": r.randn(8, C).astype(np.float32), "bias": r.randn(C).astype(np.float32)}
    out.update(logits=logits, multi=multi, onehot=onehot, head_w=head_vars["weights"], head_b=head_vars["bias"],
               a0_nw=agg_vars[0]["neigh_weights"], a0_sw=agg_vars[0]["self_weights"], a1_w=agg_vars[1]["weights"])
    for sig, labels, tag in ((True, multi, "sig"), (False, onehot, "soft")):
        for wd in (0.0, 0.05):
            st = _Stub()
            st.aggregators = [types.SimpleNamespace(vars=v) for v in agg_vars]
            st.node_pred = types.SimpleNamespace(vars=head_vars)
            st.node_preds, st.sigmoid_loss, st.placeholders, st.loss = logits, sig, {"labels": labels}, 0
            tf.app.flags.FLAGS.weight_decay = wd
            SupervisedGraphsage._loss(st)
            out["sup_%s_wd%d" % (tag, int(wd > 0))] = np.float64(st.loss)
        out["pred_" + tag] = SupervisedGraphsage.predict(st)
    tf.app.flags.FLAGS.weight_decay = 0.0
    save("heads", **out)


def golden_toy_ppi(quota=(1500, 300, 500)):
    """A sample of the reference's example_data/toy-ppi small enough to commit: for train, val and test nodes in turn, a
    breadth-first ball (neighbours in id order) from the first node of that kind, grown until it holds `quota` nodes,
    then the induced subgraph.  Node ids, flags, links (in file order, with their flags), features and labels keep the
    file's values; tests/test_data_cpu.py writes them back out in the file format."""
    prefix = os.path.join(REFERENCE, "example_data", "toy-ppi")
    with open(prefix + "-G.json") as fp:
        g = json.load(fp)
    nodes, links = g["nodes"], g["links"]
    kind = np.array([2 if nd["test"] else 1 if nd["val"] else 0 for nd in nodes])
    nbrs = [[] for _ in nodes]
    for ln in links:
        nbrs[ln["source"]].append(ln["target"])
        nbrs[ln["target"]].append(ln["source"])
    keep = set()
    for k, q in enumerate(quota):
        taken = []
        for start in np.nonzero(kind == k)[0]:
            if len(taken) == q:
                break
            if int(start) in keep:
                continue
            frontier = [int(start)]
            keep.add(int(start))
            taken.append(int(start))
            while frontier and len(taken) < q:
                nxt = []
                for u in frontier:
                    for v in sorted(set(nbrs[u])):
                        if v not in keep and len(taken) < q:
                            keep.add(v)
                            taken.append(v)
                            nxt.append(v)
                frontier = nxt
    pos = sorted(keep)
    row = {p: i for i, p in enumerate(pos)}
    sub = [ln for ln in links if ln["source"] in row and ln["target"] in row]
    feats = np.load(prefix + "-feats.npy")[pos]
    with open(prefix + "-id_map.json") as fp:
        id_map = json.load(fp)
    with open(prefix + "-class_map.json") as fp:
        class_map = json.load(fp)
    ids = [nodes[p]["id"] for p in pos]
    assert all(id_map[str(i)] == p for i, p in zip(ids, pos))
    assert set(np.unique(feats)) <= {0.0, 1.0}
    save("toy_ppi", ids=np.array(ids, np.int32), val=np.array([nodes[p]["val"] for p in pos]),
         test=np.array([nodes[p]["test"] for p in pos]),
         feats=feats.astype(np.uint8), labels=np.array([class_map[str(i)] for i in ids], np.uint8),
         link_source=np.array([row[ln["source"]] for ln in sub], np.int16),
         link_target=np.array([row[ln["target"]] for ln in sub], np.int16),
         link_train_removed=np.array([ln["train_removed"] for ln in sub]),
         link_test_removed=np.array([ln["test_removed"] for ln in sub]), graph_name=g["graph"]["name"])


def _standalone(fn):
    """meanpool / iterators / heads were added after the first four fixtures: each starts from a fresh initialiser
    stream, so regenerating everything reproduces every committed file."""
    tf_shim.INIT_RNG.seed(2024)
    fn()


if __name__ == "__main__":
    later = {"meanpool": golden_meanpool, "iterators": golden_iterators, "heads": golden_heads, "toy_ppi": golden_toy_ppi}
    if len(sys.argv) > 1:
        _standalone(later[sys.argv[1]])
        sys.exit(0)
    golden_sampler()
    golden_aggregators()
    golden_khop()
    golden_adjacency()
    for fn in later.values():
        _standalone(fn)
