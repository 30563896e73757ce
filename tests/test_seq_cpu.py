"""The LSTM neighbour aggregator without a GPU: the oracle against the reference's own output (tests/golden/seq.npz), the
fixture against torch.nn.LSTMCell, the BPTT backward against torch autograd (kernels replaced by torch stand-ins with
the semantics documented in ops.py - TEST mocks only, the product has no such path), and the parameter lists."""
import numpy as np
import pytest
import torch

import graphsage_b200 as gs
import seq_oracle as so
from conftest import load_golden, rel_err
from graphsage_b200 import ops, supervised_models as sm

CASES = ["c0", "c1", "id", "big", "cb", "k1"]


@pytest.mark.parametrize("tag", CASES)
def test_oracle_matches_reference_seq_aggregator(tag):
    g = load_golden("seq")
    selfv, neigh, agg, concat, act = so.golden_case(g, tag)
    y = so.apply(agg, selfv, neigh, concat, act)
    assert y.shape == g[tag + "_out"].shape
    assert rel_err(y, g[tag + "_out"]) < 1e-5


def test_oracle_matches_reference_khop():
    g = load_golden("seq")
    samples = [g["khop_samples%d" % h] for h in range(3)]
    fan = [int(x) for x in g["khop_fanout"]]
    out = so.aggregate_khop(samples, g["khop_feats"], fan, [int(x) for x in g["khop_support"]], len(g["khop_seeds"]),
                            so.golden_khop_aggs(g), True)
    assert rel_err(out, g["khop_out"]) < 1e-5


def test_len_counts_nonzero_rows_but_feeds_the_first_len_rows():
    """The reference's quirk (aggregators.py:411-427): zero rows in the middle are fed to the LSTM, and data rows after
    the first len are dropped."""
    g = load_golden("seq")
    selfv, neigh, agg, concat, act = so.golden_case(g, "c0")
    k = neigh.shape[1]
    lens = so.seq_lengths(neigh)
    assert (np.abs(neigh[0]).max(axis=1) == 0)[[1, 4]].all() and lens[0] < k          # zero rows in the middle
    assert lens[1] == 1 and not neigh[1].any()                                           # all-zero set
    assert lens[2] == k                                                                  # full set
    assert not neigh[3, :lens[3]].any()                     # set 3: its first len rows are all zero, its data comes later
    ref = g["c0_out"]
    # skipping the zero rows instead (what the count suggests) gives a different answer for sets 0 and 3
    packed = np.zeros_like(neigh)
    for r in range(len(neigh)):
        rows = neigh[r][np.abs(neigh[r]).max(axis=1) > 0]
        packed[r, :len(rows)] = rows
    alt = so.apply(agg, selfv, packed, concat, act)
    assert rel_err(alt[[0, 3]], ref[[0, 3]]) > 1e-3
    # set 3's output saw only zero inputs: its data rows lie past len
    h_ref = so.lstm_last(neigh[3:4], agg["kernel"], agg["bias"])
    h_trunc = so.lstm_last(np.zeros_like(neigh[3:4, :lens[3]]), agg["kernel"], agg["bias"])
    assert np.allclose(h_ref, h_trunc, rtol=1e-6, atol=1e-7)


def _torch_lstm_last(neigh, kernel, bias):
    """The same recurrence on torch.nn.LSTMCell: gates permuted from TF's i, j, f, o to torch's i, f, g, o, and the
    forget bias 1.0 folded into b_ih."""
    n, k, d = neigh.shape
    H = kernel.shape[1] // 4
    K = torch.from_numpy(kernel).double()
    b = torch.from_numpy(bias).double()
    blk = lambda M, q: M[..., q * H:(q + 1) * H]                                 # noqa: E731
    order = [0, 2, 1, 3]                                                         # torch i, f, g, o <- TF i, j, f, o
    cell = torch.nn.LSTMCell(d, H).double()
    with torch.no_grad():
        cell.weight_ih.copy_(torch.cat([blk(K[:d], q).t() for q in order], dim=0))
        cell.weight_hh.copy_(torch.cat([blk(K[d:], q).t() for q in order], dim=0))
        cell.bias_ih.copy_(torch.cat([blk(b, q) + (1.0 if q == 2 else 0.0) for q in order]))
        cell.bias_hh.zero_()
        x = torch.from_numpy(neigh).double()
        lens = so.seq_lengths(neigh)
        h = torch.zeros(n, H, dtype=torch.float64)
        c = torch.zeros_like(h)
        out = torch.zeros_like(h)
        for t in range(k):
            h, c = cell(x[:, t], (h, c))
            last = torch.from_numpy(lens == t + 1)
            out[last] = h[last]
    return out.numpy()


@pytest.mark.parametrize("tag", CASES)
def test_fixture_agrees_with_torch_lstm_cell(tag):
    g = load_golden("seq")
    selfv, neigh, agg, concat, act = so.golden_case(g, tag)
    h = _torch_lstm_last(neigh, agg["kernel"], agg["bias"])
    fs, fn = selfv.astype(np.float64) @ agg["self_weights"], h @ agg["neigh_weights"]
    y = act(np.concatenate([fs, fn], axis=1) if concat else fs + fn)
    assert rel_err(g[tag + "_out"], y) < 1e-5


# ---------------------------------------------------------------- torch stand-ins for the kernels (TEST mocks)
def _fake_sage_gemm(parts, combine=ops.COMBINE_ADD, bias=None, act=ops.ACT_NONE, math=None, out=None, packed=None):
    ys = [a[:, :k] @ w for (a, k, w) in parts]
    y = torch.cat(ys, dim=1) if combine == ops.COMBINE_CONCAT else sum(ys[1:], ys[0])
    if bias is not None:
        y = y + bias
    return torch.relu(y) if act == ops.ACT_RELU else y


def _fake_gather_rows(feats, ids, out=None):
    r = feats[ids.long()].float()
    if out is not None:
        out.copy_(r)
        return out
    return r


def _fake_gather_rows_f32(feats, ids=None, row0=0, n=None, out=None):
    r = feats[ids.long()] if ids is not None else feats[row0:row0 + n]
    out.copy_(r.float())
    return out


def _fake_lstm_seq(P, Wh, used, n, k, row_ids=None, row0=0, out=None, keep=False):
    H = Wh.shape[0]
    idx = row_ids.long() if row_ids is not None else torch.arange(row0, row0 + n * k)
    lens = used[idx].reshape(n, k).long().sum(dim=1).clamp(min=1)
    h = torch.zeros(n, H)
    c = torch.zeros(n, H)
    kh, kc = torch.zeros(n, k, H), torch.zeros(n, k, H)
    res = torch.zeros(n, H)
    for t in range(k):
        G = P.reshape(n, k, -1)[:, t, :4 * H] + h @ Wh
        i, j, f, o = G.split(H, dim=1)
        c = c * torch.sigmoid(f + 1.0) + torch.sigmoid(i) * torch.tanh(j)
        h = torch.tanh(c) * torch.sigmoid(o)
        kh[:, t], kc[:, t] = h, c
        res[lens == t + 1] = h[lens == t + 1]
    kh[torch.arange(k).unsqueeze(0) >= lens.unsqueeze(1)] = float("nan")      # the kernel leaves these unwritten
    if out is not None:
        out.copy_(res)
        res = out
    return (res, kh, kc, lens.int()) if keep else res


@pytest.fixture()
def cpu_kernels(monkeypatch):
    monkeypatch.setattr(ops, "sage_gemm", _fake_sage_gemm)
    monkeypatch.setattr(ops, "gather_rows", _fake_gather_rows)
    monkeypatch.setattr(ops, "gather_rows_f32", _fake_gather_rows_f32)
    monkeypatch.setattr(ops, "row_used", lambda x, out=None: (x != 0).any(dim=1).to(torch.uint8))
    monkeypatch.setattr(ops, "lstm_seq", _fake_lstm_seq)


def _ref_layer(selfv, neigh, k, a, concat, last):
    """The oracle's op sequence as differentiable torch: an unrolled LSTM masked at t < len."""
    n = selfv.shape[0]
    x = neigh.reshape(n, k, -1)
    kern, b = a["kernel"], a["cbias"]
    d = x.shape[2]
    H = kern.shape[1] // 4
    lens = (x.detach() != 0).any(dim=2).sum(dim=1).clamp(min=1)
    h = torch.zeros(n, H)
    c = torch.zeros(n, H)
    outs = []
    for t in range(k):
        G = x[:, t] @ kern[:d] + h @ kern[d:] + b
        i, j, f, o = G.split(H, dim=1)
        c = c * torch.sigmoid(f + 1.0) + torch.sigmoid(i) * torch.tanh(j)
        h = torch.tanh(c) * torch.sigmoid(o)
        outs.append(h)
    hs = torch.stack(outs, dim=1)
    neigh_h = hs[torch.arange(n), lens - 1]
    fs, fn = selfv @ a["self_weights"], neigh_h @ a["neigh_weights"]
    y = torch.cat([fs, fn], dim=1) if concat else fs + fn
    return y if last else torch.relu(y)


@pytest.mark.parametrize("concat", [True, False])
def test_two_layer_seq_chain_gradients_match_autograd(cpu_kernels, concat):
    r = np.random.RandomState(4)
    N, F, D, B, k1, k2 = 40, 10, 6, 5, 3, 4
    feats = torch.from_numpy(r.randn(N, F).astype(np.float32))
    feats[7] = 0.0
    s0 = torch.from_numpy(r.randint(0, N, size=B).astype(np.int32))
    s1 = torch.from_numpy(r.randint(0, N, size=B * k1).astype(np.int32))
    s2 = torch.from_numpy(r.randint(0, N, size=B * k1 * k2).astype(np.int32))
    s2[1] = s2[5] = s2[k2 * 3] = s2[k2 * 3 + 1] = 7        # zero rows: in the middle, at the start, a shortened set
    s1[2] = 7
    dim_mult = 2 if concat else 1
    a0 = gs.SeqAggregator(F, D, act=gs.relu, concat=concat, device="cpu")
    a1 = gs.SeqAggregator(dim_mult * D, D, act=gs.identity, concat=concat, device="cpu")
    params = []
    for a in (a0, a1):
        a.cell_vars["bias"] = torch.from_numpy(r.randn(4 * a.hidden_dim).astype(np.float32) * 0.1)
        for dct in (a.vars, a.cell_vars):
            for key in dct:
                dct[key] = dct[key].detach().clone().requires_grad_(True)
                params.append(dct[key])
    seg0 = [ops.Seg(B, k1, self_ids=s0, neigh_ids=s1, out_row0=0), ops.Seg(B * k1, k2, self_ids=s1, neigh_ids=s2, out_row0=B)]
    h1 = sm._SeqAggregateRowsFn.apply(a0, feats, seg0, a0.vars["self_weights"], a0.vars["neigh_weights"],
                                      a0.cell_vars["kernel"], a0.cell_vars["bias"])
    seg1 = [ops.Seg(B, k1, self_row0=0, neigh_row0=B, out_row0=0)]
    out = sm._SeqAggregateRowsFn.apply(a1, h1, seg1, a1.vars["self_weights"], a1.vars["neigh_weights"],
                                       a1.cell_vars["kernel"], a1.cell_vars["bias"])
    R = torch.from_numpy(r.randn(*out.shape).astype(np.float32))
    (out * R).sum().backward()
    got = [p.grad.clone() for p in params]
    for p in params:
        p.grad = None
    w0 = dict(a0.vars, kernel=a0.cell_vars["kernel"], cbias=a0.cell_vars["bias"])
    w1 = dict(a1.vars, kernel=a1.cell_vars["kernel"], cbias=a1.cell_vars["bias"])
    x0, x1, x2 = feats[s0.long()], feats[s1.long()], feats[s2.long()]
    r_hop0 = _ref_layer(x0, x1, k1, w0, concat, last=False)
    r_hop1 = _ref_layer(x1, x2, k2, w0, concat, last=False)
    ref = _ref_layer(r_hop0, r_hop1, k1, w1, concat, last=True)
    assert torch.allclose(out.detach(), ref.detach(), rtol=1e-5, atol=1e-5)
    (ref * R).sum().backward()
    for p, gr in zip(params, got):
        assert p.grad is not None and torch.allclose(gr, p.grad, rtol=2e-4, atol=2e-5), float((gr - p.grad).abs().max())


def test_dense_call_ignores_dropout(cpu_kernels):
    """The reference stores dropout but never applies it in SeqAggregator._call."""
    g = load_golden("seq")
    selfv, neigh, agg, concat, act = so.golden_case(g, "c1")
    a = gs.SeqAggregator(selfv.shape[1], 16, dropout=0.5, concat=True, device="cpu")
    a.vars["self_weights"], a.vars["neigh_weights"] = torch.from_numpy(agg["self_weights"]), torch.from_numpy(agg["neigh_weights"])
    a.cell_vars["kernel"], a.cell_vars["bias"] = torch.from_numpy(agg["kernel"]), torch.from_numpy(agg["bias"])
    y1 = a((torch.from_numpy(selfv), torch.from_numpy(neigh)))
    y2 = a((torch.from_numpy(selfv), torch.from_numpy(neigh)))
    assert torch.equal(y1, y2)
    assert rel_err(y1.numpy(), g["c1_out"]) < 1e-5


def test_parameter_lists_train_the_cell_but_decay_only_aggregator_vars():
    a = gs.SeqAggregator(8, 4, concat=True, device="cpu")
    m = gs.MeanAggregator(8, 4, concat=True, device="cpu")
    every, decayed = sm.aggregator_parameters([a, m])
    assert len(every) == 2 + 2 + 2 and len(decayed) == 4
    ids = {id(t) for t in decayed}
    assert id(a.cell_vars["kernel"]) not in ids and id(a.cell_vars["bias"]) not in ids and id(a.vars["neigh_weights"]) in ids
    assert {id(t) for t in every} >= {id(a.cell_vars["kernel"]), id(a.cell_vars["bias"])}


@pytest.mark.parametrize("size,H", [("small", 128), ("big", 256)])
def test_shapes_and_model_size(size, H):
    a = gs.SeqAggregator(10, 6, model_size=size, neigh_input_dim=14, device="cpu")
    assert a.hidden_dim == H and "kernel" not in a.vars
    assert tuple(a.cell_vars["kernel"].shape) == (14 + H, 4 * H) and not a.cell_vars["bias"].any()
    assert tuple(a.vars["neigh_weights"].shape) == (H, 6) and tuple(a.vars["self_weights"].shape) == (10, 6)
    r = np.sqrt(6.0 / (14 + H + 4 * H))
    assert float(a.cell_vars["kernel"].abs().max()) <= r
    with pytest.raises(ValueError):
        gs.SeqAggregator(10, 6, model_size="huge", device="cpu")


@pytest.mark.parametrize("size", ["small", "big"])
def test_models_accept_seq(size):
    feats = np.zeros((11, 5), np.float32)
    adj = torch.zeros((11, 4), dtype=torch.int32)
    infos = [gs.SAGEInfo("node", None, 3, 8), gs.SAGEInfo("node", None, 2, 8)]
    m = gs.SampleAndAggregate({"batch_size": 4}, feats, adj, None, infos, aggregator_type="seq", model_size=size,
                              device="cpu")
    assert m.aggregator_cls is gs.SeqAggregator
    sup = gs.SupervisedGraphsage(3, {"batch_size": 4, "dropout": 0.}, feats, adj, None, infos, aggregator_type="seq",
                                 model_size=size, device="cpu")
    H = 128 if size == "small" else 256
    assert all(a.hidden_dim == H for a in sup.aggregators)
    assert tuple(sup.aggregators[1].cell_vars["kernel"].shape) == (16 + H, 4 * H)      # concat: layer-1 input is 2 x 8
    assert len(sup.parameters()) == 2 * 4 + 2 and len(sup.decayed_parameters()) == 2 * 2 + 2
    uns = gs.UnsupervisedGraphsage({"batch_size": 4, "dropout": 0.}, feats, adj, np.ones(10), infos,
                                   aggregator_type="seq", model_size=size, device="cpu")
    assert len(uns.parameters()) == 2 * 4


def test_sharded_table_is_refused():
    class _Sharded(object):
        shape = (11, 5)

        def c_table(self):
            raise AssertionError("not reached")

    infos = [gs.SAGEInfo("node", None, 3, 8)]
    with pytest.raises(NotImplementedError, match="sharded"):
        gs.SampleAndAggregate({"batch_size": 4}, _Sharded(), None, None, infos, aggregator_type="seq", device="cpu")
    with pytest.raises(NotImplementedError, match="sharded"):
        gs.SeqAggregator(5, 8, device="cpu").aggregate_rows(_Sharded(), [ops.Seg(1, 3)])
