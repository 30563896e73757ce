"""Generate tests/golden/seq.npz by executing the reference's own SeqAggregator (graphsage/aggregators.py:363-449) and
its SampleAndAggregate.sample / .aggregate recursion under the numpy TF shim (tf_shim.py + tf_shim_rnn.py).

    GRAPHSAGE_REFERENCE=<checkout of williamleif/GraphSAGE> python tests/golden/make_golden_seq.py

Nothing from the reference is copied: the modules are imported from where they lie (through make_golden.py).
"""
import numpy as np

import make_golden  # noqa: F401  (exits unless GRAPHSAGE_REFERENCE is set; installs tf_shim, puts the reference on the path)
import tf_shim_rnn
from make_golden import _Stub, save, tf, tf_shim

tf_shim_rnn.install(tf)

from graphsage.aggregators import SeqAggregator  # noqa: E402
from graphsage.models import SAGEInfo, SampleAndAggregate  # noqa: E402
from graphsage.neigh_samplers import UniformNeighborSampler  # noqa: E402


def golden_seq():
    """SeqAggregator (reference aggregators.py:363-449) through the shim's BasicLSTMCell / dynamic_rnn, and one K-hop
    recursion with it.  LSTM kernels are stored as their seeds (tf_shim_rnn.lstm_kernel).  Neighbour sets include zero
    rows in the middle (dynamic_rnn still consumes them: len counts the
    non-zero rows but the FIRST len rows are fed), an all-zero set, full sets and fanout 1."""
    r = np.random.RandomState(41)
    tf_shim_rnn.LSTM_BUILT = 0
    out = {}

    def neigh_set(n, k, d):
        x = r.randn(n, k, d).astype(np.float32)
        x[r.rand(n, k) < 0.2] = 0.0                  # scattered dummy rows
        if k > 4:
            x[0, 1] = x[0, 4] = 0.0                  # zero rows in the middle of a set
        x[1] = 0.0                                   # an all-zero set (len = max(1, 0) = 1)
        x[2] = r.randn(k, d)                         # a full set
        if k > 2:
            x[3, :k - 2] = 0.0                       # zeros first: len 2 feeds two ZERO rows, the data rows are dropped
        return x

    cases = [("c0", dict(concat=False), 24, 24, 10, 0.0),
             ("c1", dict(concat=True), 24, 24, 10, 0.0),
             ("id", dict(concat=True, act=lambda x: x, neigh_input_dim=12), 24, 12, 10, 0.0),
             ("big", dict(concat=False, model_size="big"), 24, 24, 7, 0.0),
             ("cb", dict(concat=True), 24, 24, 10, 0.5),
             ("k1", dict(concat=False), 24, 24, 1, 0.3)]
    n, dout = 21, 16
    for tag, kw, din, dneigh, k, bias_scale in cases:
        selfv = r.randn(n, din).astype(np.float32)
        neigh = neigh_set(n, k, dneigh)
        agg = SeqAggregator(din, dout, **kw)
        agg.cell.build(dneigh)
        if bias_scale:
            agg.cell.bias = (r.randn(4 * agg.hidden_dim) * bias_scale).astype(np.float32)
        y = agg((selfv, neigh))
        out.update({tag + "_self": selfv, tag + "_neigh": neigh, tag + "_nw": agg.vars["neigh_weights"],
                    tag + "_sw": agg.vars["self_weights"], tag + "_kseed": agg.cell.kernel_seed, tag + "_bias": agg.cell.bias,
                    tag + "_concat": bool(agg.concat), tag + "_identity": "act" in kw, tag + "_hidden": agg.hidden_dim,
                    tag + "_out": y})
    out["cases"] = np.array([c[0] for c in cases])
    # ---- K-hop recursion (models.py:254-330) with SeqAggregator, as golden_khop
    nn, md, f, B = 120, 16, 20, 7
    adj = r.randint(0, nn, size=(nn + 1, md)).astype(np.int32)
    adj[nn, :] = nn
    adj[3, :] = nn                                   # an isolated node: its fanout is all dummy (zero) rows
    adj[r.rand(nn + 1, md) < 0.15] = nn              # scattered dummy ids -> zero rows inside the neighbour sets
    feats = np.vstack([r.randn(nn, f).astype(np.float32), np.zeros((1, f), np.float32)])
    seeds = r.randint(0, nn, size=B).astype(np.int32)
    seeds[0] = 3
    dims, fan = [f, 12, 8], [5, 3]
    tf_shim.SHUFFLE_SEED, tf_shim.SHUFFLE_COUNTER = 123, 40
    sampler = UniformNeighborSampler(adj)
    infos = [SAGEInfo("node", sampler, fan[i], dims[i + 1]) for i in range(len(fan))]
    stub = _Stub()
    stub.batch_size = B
    stub.aggregator_cls = SeqAggregator
    stub.placeholders = {"dropout": 0.0}
    samples, support = SampleAndAggregate.sample(stub, seeds, infos)
    hidden, aggs = SampleAndAggregate.aggregate(stub, samples, [feats][0], dims, fan, support, concat=True)
    out.update(khop_adj=adj, khop_feats=feats, khop_seeds=seeds, khop_dims=np.array(dims), khop_fanout=np.array(fan),
               khop_support=np.array(support), khop_out=hidden)
    for h, s in enumerate(samples):
        out["khop_samples%d" % h] = np.asarray(s).astype(np.int32)
    for li, a in enumerate(aggs):
        for key, v in a.vars.items():
            out["khop_L%d_%s" % (li, key)] = v
        out["khop_L%d_kseed" % li], out["khop_L%d_bias" % li] = a.cell.kernel_seed, a.cell.bias
    save("seq", **out)


if __name__ == "__main__":
    tf_shim.INIT_RNG.seed(2024)          # a fresh initialiser stream, as make_golden.py gives its later fixtures
    golden_seq()
