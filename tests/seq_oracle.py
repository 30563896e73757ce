"""Oracle for the LSTM neighbour aggregator (reference graphsage/aggregators.py:363-449) and the K-hop recursion with it.
Plain numpy fp32, like oracle/aggregate.py, whose gather / sampling / l2_normalize it reuses; each function cites the
reference lines it restates.  Test infrastructure - not imported by the product."""
import numpy as np

from oracle.aggregate import _apply, gather_rows, identity, l2_normalize, relu, sample_khop


def lstm_kernel(seed, shape):
    """The fixture's LSTM kernels (tests/golden/tf_shim_rnn.py): glorot-uniform float32 from RandomState(seed)."""
    r = np.sqrt(6.0 / (shape[0] + shape[1]))
    return np.random.RandomState(int(seed)).uniform(-r, r, size=shape).astype(np.float32)


def _sigmoid(x):
    return (1.0 / (1.0 + np.exp(-x))).astype(x.dtype)


def lstm_cell(x, h, c, kernel, bias, forget_bias=1.0):
    """tf.contrib.rnn.BasicLSTMCell (aggregators.py:403): gates = [x, h] @ kernel + bias split i, j, f, o;
    c' = c * sigmoid(f + forget_bias) + sigmoid(i) * tanh(j);  h' = tanh(c') * sigmoid(o)."""
    gates = np.concatenate([x, h], axis=1) @ kernel + bias
    i, j, f, o = np.split(gates, 4, axis=1)
    c = c * _sigmoid(f + np.asarray(forget_bias, dtype=gates.dtype)) + _sigmoid(i) * np.tanh(j)
    return np.tanh(c) * _sigmoid(o), c


def seq_lengths(neigh_vecs):
    """aggregators.py:411-414: len = max(1, number of rows with a non-zero element)."""
    used = (np.abs(neigh_vecs).max(axis=2) > 0)
    return np.maximum(used.sum(axis=1), 1).astype(np.int64)


def lstm_last(neigh_vecs, kernel, bias):
    """dynamic_rnn(cell, neigh_vecs, sequence_length=len) and the gather of output len - 1 (aggregators.py:416-433):
    the FIRST len rows are consumed, zero rows included."""
    n, k, _ = neigh_vecs.shape
    H = kernel.shape[1] // 4
    lens = seq_lengths(neigh_vecs)
    h = np.zeros((n, H), neigh_vecs.dtype)
    c = np.zeros((n, H), neigh_vecs.dtype)
    out = np.zeros((n, H), neigh_vecs.dtype)
    for t in range(k):
        h, c = lstm_cell(neigh_vecs[:, t], h, c, kernel, bias)
        last = lens == t + 1
        out[last] = h[last]
    return out


def seq_aggregator(self_vecs, neigh_vecs, kernel, bias, neigh_weights, self_weights, concat=False, act=relu,
                   agg_bias=None):
    """aggregators.py:405-449 (dropout stored but not applied by the reference)."""
    neigh_h = lstm_last(neigh_vecs, kernel, bias)
    from_neighs = neigh_h @ neigh_weights                                   # :435
    from_self = self_vecs @ self_weights                                    # :436
    out = np.concatenate([from_self, from_neighs], axis=1) if concat else from_self + from_neighs   # :440-443
    if agg_bias is not None:
        out = out + agg_bias                                                # :446-447
    return act(out)


def apply(agg, self_vecs, neigh_vecs, concat, act):
    if agg["type"] == "seq":
        return seq_aggregator(self_vecs, neigh_vecs, agg["kernel"], agg["bias"], agg["neigh_weights"],
                              agg["self_weights"], concat, act, agg.get("agg_bias"))
    return _apply(agg, self_vecs, neigh_vecs, concat, act)


def aggregate_khop(samples, features, num_samples, support_sizes, batch_size, aggregators, concat):
    """reference graphsage/models.py:278-330 with the seq aggregator routed (oracle.aggregate.aggregate_khop's loop)."""
    hidden = [gather_rows(features, s) for s in samples]                    # :299
    L = len(num_samples)
    for layer in range(L):
        act = identity if layer == L - 1 else relu
        nxt = []
        for hop in range(L - layer):
            d = hidden[hop + 1].shape[1]
            neigh = hidden[hop + 1].reshape(batch_size * support_sizes[hop], num_samples[L - hop - 1], d)
            nxt.append(apply(aggregators[layer], hidden[hop], neigh, concat, act))
        hidden = nxt
    return hidden[0]


def forward_2hop(adj, features, seeds, num_samples, aggregators, concat, seed, counter0, normalize=False):
    samples, support = sample_khop(adj, seeds, num_samples, seed, counter0)
    out = aggregate_khop(samples, features, num_samples, support, len(seeds), aggregators, concat)
    return l2_normalize(out) if normalize else out


def golden_case(g, tag):
    """(self, neigh, agg dict, concat, act) of one aggregator case of tests/golden/seq.npz."""
    neigh = g[tag + "_neigh"]
    H = int(g[tag + "_hidden"])
    agg = {"type": "seq", "kernel": lstm_kernel(g[tag + "_kseed"], (neigh.shape[2] + H, 4 * H)), "bias": g[tag + "_bias"],
           "neigh_weights": g[tag + "_nw"], "self_weights": g[tag + "_sw"]}
    act = identity if bool(g[tag + "_identity"]) else relu
    return g[tag + "_self"], neigh, agg, bool(g[tag + "_concat"]), act


def golden_khop_aggs(g):
    dims, L = g["khop_dims"], len(g["khop_fanout"])
    aggs = []
    for li in range(L):
        din = (2 if li else 1) * int(dims[li])
        H = g["khop_L%d_neigh_weights" % li].shape[0]
        aggs.append({"type": "seq", "kernel": lstm_kernel(g["khop_L%d_kseed" % li], (din + H, 4 * H)),
                     "bias": g["khop_L%d_bias" % li], "neigh_weights": g["khop_L%d_neigh_weights" % li],
                     "self_weights": g["khop_L%d_self_weights" % li]})
    return aggs
