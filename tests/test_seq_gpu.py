"""GPU: the LSTM neighbour aggregator (reference graphsage/aggregators.py:363-449) - gs_row_used and gs_lstm_seq against
numpy, SeqAggregator against the reference's own output (tests/golden/seq.npz), the full-size forward against the
oracle, CUDA-graph and pipelined replays, the launch list, and supervised / unsupervised training against torch-CPU
autograd."""
import numpy as np
import pytest
import torch

import seq_oracle as so
from conftest import bf16_round, load_golden, rel_err
from oracle import torch_ref

pytestmark = pytest.mark.gpu

TOL = 1e-4
BF16_TOL = 2e-2          # the max-pool bf16 tests' tolerance (bf16 operands, fp32 accumulate)


@pytest.fixture(scope="module")
def gs():
    assert torch.cuda.is_available(), "gpu tests need a CUDA device"
    import graphsage_b200
    graphsage_b200._lib.lib()
    yield graphsage_b200
    graphsage_b200.set_default_math("fp32")


def dev(x):
    return torch.as_tensor(np.ascontiguousarray(x)).cuda()


# ---------------------------------------------------------------- kernels
@pytest.mark.parametrize("dtype", ["f32", "bf16"])
def test_row_used_exact(gs, dtype):
    rs = np.random.RandomState(1)
    n, F, pitch = 1003, 37, 48
    x = rs.randn(n, pitch).astype(np.float32)
    x[rs.rand(n) < 0.3, :F] = 0.0
    x[5, :F] = -0.0                                   # negative zeros are zero
    x[6, :F] = 0.0
    x[6, F - 1] = 1e-30 if dtype == "f32" else 1e-3   # one tiny non-zero in the last column
    x[:, F:] = 1.0                                    # columns past F are not looked at
    t = dev(x)
    if dtype == "bf16":
        t = t.to(torch.bfloat16)
    used = gs.ops.row_used(t[:, :F]).cpu().numpy()
    ref = (t[:, :F].float().cpu().numpy() != 0).any(axis=1).astype(np.uint8)
    np.testing.assert_array_equal(used, ref)
    assert used[5] == 0 and used[6] == 1


def _lstm_from_P(P, Wh, used_rows, n, k):
    """numpy recurrence on a given input projection: (out, h[n, k, H], c[n, k, H], len)."""
    H = Wh.shape[0]
    lens = np.maximum(used_rows.reshape(n, k).sum(axis=1), 1)
    h = np.zeros((n, H), np.float32)
    c = np.zeros((n, H), np.float32)
    hs, cs = np.zeros((n, k, H), np.float32), np.zeros((n, k, H), np.float32)
    out = np.zeros((n, H), np.float32)
    sig = lambda v: 1.0 / (1.0 + np.exp(-v))                               # noqa: E731
    for t in range(k):
        G = P.reshape(n, k, -1)[:, t, :4 * H] + h @ Wh
        i, j, f, o = np.split(G, 4, axis=1)
        c = c * sig(f + 1.0) + sig(i) * np.tanh(j)
        h = np.tanh(c) * sig(o)
        hs[:, t], cs[:, t] = h, c
        out[lens == t + 1] = h[lens == t + 1]
    return out, hs, cs, lens


@pytest.mark.parametrize("H", [128, 256])
@pytest.mark.parametrize("k", [1, 10, 25, 64])
@pytest.mark.parametrize("by_ids", [True, False])
def test_lstm_seq_matches_numpy(gs, H, k, by_ids):
    rs = np.random.RandomState(H + k)
    n, N = 77, 500                                    # 77 sequences: a ragged last tile
    r = 1.0 / np.sqrt(H)
    P = (rs.randn(n * k, 4 * H + 8) * 0.7).astype(np.float32)         # row stride 4H + 8
    Wh = rs.uniform(-r, r, size=(H, 4 * H)).astype(np.float32)
    used_tab = (rs.rand(N) < 0.8).astype(np.uint8)
    if by_ids:
        ids = rs.randint(0, N, size=n * k).astype(np.int32)
        used_rows = used_tab[ids]
        kw = dict(row_ids=dev(ids))
    else:
        row0 = 7
        used_tab = (rs.rand(row0 + n * k) < 0.8).astype(np.uint8)
        used_rows = used_tab[row0:row0 + n * k]
        kw = dict(row0=row0)
    out, kh, kc, lens = gs.ops.lstm_seq(dev(P), dev(Wh), dev(used_tab), n, k, keep=True, **kw)
    ref, rh, rc, rl = _lstm_from_P(P, Wh, used_rows, n, k)
    np.testing.assert_array_equal(lens.cpu().numpy(), rl)
    assert rel_err(out.cpu().numpy(), ref) < TOL
    live = np.arange(k)[None, :] < rl[:, None]
    assert rel_err(kh.cpu().numpy()[live], rh[live]) < TOL
    assert rel_err(kc.cpu().numpy()[live], rc[live]) < TOL
    out2 = gs.ops.lstm_seq(dev(P), dev(Wh), dev(used_tab), n, k, **kw)        # inference form: no keep buffers
    assert torch.equal(out2, out)


def test_lstm_seq_refuses_unsupported_widths(gs):
    P = torch.zeros((4, 4 * 48), device="cuda")
    with pytest.raises(RuntimeError, match="-3"):
        gs.ops.lstm_seq(P, torch.zeros((48, 192), device="cuda"), torch.ones(4, dtype=torch.uint8, device="cuda"), 2, 2)


# ---------------------------------------------------------------- the aggregator
def _agg_from_case(gs, g, tag, math):
    selfv, neigh, ref_agg, concat, act = so.golden_case(g, tag)
    gs.set_default_math(math)
    H = ref_agg["neigh_weights"].shape[0]
    a = gs.SeqAggregator(selfv.shape[1], ref_agg["self_weights"].shape[1], model_size="big" if H == 256 else "small",
                         neigh_input_dim=neigh.shape[2], act=gs.identity if act is so.identity else gs.relu,
                         concat=concat)
    a.vars["self_weights"], a.vars["neigh_weights"] = dev(ref_agg["self_weights"]), dev(ref_agg["neigh_weights"])
    a.cell_vars["kernel"], a.cell_vars["bias"] = dev(ref_agg["kernel"]), dev(ref_agg["bias"])
    return a, selfv, neigh, ref_agg, concat, act


@pytest.mark.parametrize("math", ["fp32", "tf32x3", "bf16"])
@pytest.mark.parametrize("tag", ["c0", "c1", "id", "big", "cb", "k1"])
def test_seq_aggregator_golden(gs, tag, math):
    g = load_golden("seq")
    a, selfv, neigh, ref_agg, concat, act = _agg_from_case(gs, g, tag, math)
    y = a((dev(selfv), dev(neigh))).cpu().numpy()
    if math == "bf16":       # against the oracle on bf16-rounded operands of every GEMM
        assert rel_err(y, g[tag + "_out"]) < BF16_TOL
    else:
        assert rel_err(y, g[tag + "_out"]) < TOL


def _golden_khop_model(gs, g, math, counter=40):
    gs.set_default_math(math)
    adj, feats = g["khop_adj"], g["khop_feats"]
    fan, dims = [int(x) for x in g["khop_fanout"]], [int(x) for x in g["khop_dims"]]
    sampler = gs.UniformNeighborSampler(dev(adj), seed=123)
    sampler.counter = counter
    infos = [gs.SAGEInfo("node", sampler, fan[i], dims[i + 1]) for i in range(len(fan))]
    m = gs.SampleAndAggregate({"batch_size": len(g["khop_seeds"]), "dropout": 0.}, dev(feats), dev(adj), None, infos,
                              concat=True, aggregator_type="seq")
    return m, infos, fan, dims


def _inject_khop(gs, m, g):
    for li, (a, ra) in enumerate(zip(m.aggregators, so.golden_khop_aggs(g))):
        a.vars["self_weights"].copy_(dev(ra["self_weights"]))
        a.vars["neigh_weights"].copy_(dev(ra["neigh_weights"]))
        a.cell_vars["kernel"].copy_(dev(ra["kernel"]))
        a.cell_vars["bias"].copy_(dev(ra["bias"]))


@pytest.mark.parametrize("math", ["fp32", "tf32x3"])
def test_seq_khop_golden(gs, math):
    g = load_golden("seq")
    m, infos, fan, dims = _golden_khop_model(gs, g, math)
    samples, support = m.sample(dev(g["khop_seeds"]), infos)
    for h, s in enumerate(samples):
        np.testing.assert_array_equal(s.cpu().numpy(), g["khop_samples%d" % h])
    _, aggs = m.aggregate(samples, [m.features], dims, fan, support, concat=True)
    m.aggregators = aggs
    _inject_khop(gs, m, g)
    out, _ = m.aggregate(samples, [m.features], dims, fan, support, aggregators=aggs, concat=True)
    assert rel_err(out.cpu().numpy(), g["khop_out"]) < TOL
    lit = m._aggregate_materialised(samples, m.features, dims, fan, support, len(g["khop_seeds"]), aggs, True)
    assert rel_err(lit.cpu().numpy(), g["khop_out"]) < TOL


# ---------------------------------------------------------------- full size (configs[1] graph, fanout 25 x 10, batch 512)
@pytest.fixture(scope="module")
def reddit(gs):
    from graphsage_b200.synthetic import reddit_like
    g = reddit_like(n=232965, f=602, max_degree=128, seed=123)
    table = torch.zeros((g["n"] + 1, gs.ops.pad_cols(602)), dtype=torch.float32, device="cuda")
    table[:, :602] = torch.from_numpy(g["features"]).cuda()
    g["table"], g["adj_dev"] = table, torch.from_numpy(g["adj"]).cuda()
    return g


def _oracle_on_sample(m, g, seeds, samples, feats, n_check, round_weights=False):
    """The oracle on the first n_check seeds of a batch (hop h's ids are row-major nested, so they are a prefix)."""
    fan = [25, 10]
    sub = [samples[0][:n_check], samples[1][:n_check * 10], samples[2][:n_check * 250]]
    rnd = bf16_round if round_weights else (lambda x: x)
    aggs = [{"type": "seq", "kernel": rnd(a.cell_vars["kernel"].cpu().numpy()), "bias": a.cell_vars["bias"].cpu().numpy(),
             "neigh_weights": rnd(a.vars["neigh_weights"].cpu().numpy()),
             "self_weights": rnd(a.vars["self_weights"].cpu().numpy())} for a in m.aggregators]
    out = so.aggregate_khop(sub, feats, fan, [1, 10, 250], n_check, aggs, True)
    return so.l2_normalize(out)


@pytest.mark.parametrize("math", ["fp32", "tf32x3"])
def test_full_size_seq_forward_vs_oracle(gs, reddit, math):
    gs.set_default_math(math)
    g = reddit
    rs = np.random.RandomState(1)
    B = 512
    seeds = rs.randint(0, g["n"], size=B).astype(np.int32)
    sampler = gs.UniformNeighborSampler(g["adj_dev"], seed=123)
    infos = [gs.SAGEInfo("node", sampler, 25, 128), gs.SAGEInfo("node", sampler, 10, 128)]
    m = gs.SampleAndAggregate({"batch_size": B, "dropout": 0.}, g["table"][:, :602], g["adj_dev"], None, infos,
                              concat=True, aggregator_type="seq")
    out = m.forward(torch.from_numpy(seeds), normalize=True).cpu().numpy()
    assert out.shape == (B, 256)
    sampler.counter = 0
    samples, _ = m.sample(torch.from_numpy(seeds).cuda(), infos)
    samples = [s.cpu().numpy() for s in samples]
    n_check = 24
    ref = _oracle_on_sample(m, g, seeds, samples, g["features"], n_check)
    assert rel_err(out[:n_check], ref) < TOL


def test_full_size_seq_bf16_table_vs_oracle(gs, reddit):
    g = reddit
    gs.set_default_math("bf16")
    rs = np.random.RandomState(2)
    B = 512
    seeds = rs.randint(0, g["n"], size=B).astype(np.int32)
    sampler = gs.UniformNeighborSampler(g["adj_dev"], seed=123)
    infos = [gs.SAGEInfo("node", sampler, 25, 128), gs.SAGEInfo("node", sampler, 10, 128)]
    tb = g["table"].to(torch.bfloat16)
    m = gs.SampleAndAggregate({"batch_size": B, "dropout": 0.}, tb[:, :602], g["adj_dev"], None, infos, concat=True,
                              aggregator_type="seq")
    out = m.forward(torch.from_numpy(seeds), normalize=True).cpu().numpy()
    sampler.counter = 0
    samples = [s.cpu().numpy() for s in m.sample(torch.from_numpy(seeds).cuda(), infos)[0]]
    n_check = 16
    ref = _oracle_on_sample(m, g, seeds, samples, bf16_round(g["features"]), n_check, round_weights=True)
    assert rel_err(out[:n_check], ref) < BF16_TOL


# ---------------------------------------------------------------- graphs, pipelining, launches
def _small_model(gs, math="fp32", B=48, bf16=False):
    rs = np.random.RandomState(6)
    n, f = 400, 50
    adj = rs.randint(0, n, size=(n + 1, 32)).astype(np.int32)
    adj[n] = n
    adj[rs.rand(n + 1, 32) < 0.1] = n
    feats = np.vstack([rs.randn(n, f).astype(np.float32), np.zeros((1, f), np.float32)])
    gs.set_default_math(math)
    table = dev(feats)
    if bf16:
        table = torch.zeros((n + 1, gs.ops.pad_cols(f)), dtype=torch.bfloat16, device="cuda")
        table[:, :f] = dev(feats).to(torch.bfloat16)
        table = table[:, :f]
    sampler = gs.UniformNeighborSampler(dev(adj), seed=5)
    infos = [gs.SAGEInfo("node", sampler, 25, 64), gs.SAGEInfo("node", sampler, 10, 64)]
    m = gs.SampleAndAggregate({"batch_size": B, "dropout": 0.}, table, dev(adj), None, infos, concat=True,
                              aggregator_type="seq")
    seeds = [dev(rs.randint(0, n, size=B).astype(np.int32)) for _ in range(4)]
    return m, infos, seeds


@pytest.mark.parametrize("math", ["tf32x3", "bf16"])
def test_graphed_and_pipelined_match_eager(gs, math):
    m, infos, seeds = _small_model(gs, math, bf16=(math == "bf16"))
    eager = [m.forward(s, normalize=True).clone() for s in seeds]
    infos[0].neigh_sampler.counter = 0
    runner = m.graphed(len(seeds[0]), normalize=True)
    for i, s in enumerate(seeds):
        assert torch.equal(runner(s), eager[i]), "graphed replay %d differs from eager step %d" % (i, i)
    runner.close()
    infos[0].neigh_sampler.counter = 0
    pipe = m.pipelined(len(seeds[0]))
    outs = [torch.empty(eager[0].shape, dtype=torch.float32).pin_memory() for _ in seeds]
    for s, o in zip(seeds, outs):
        pipe.submit(s.cpu(), o)
    pipe.synchronize()
    pipe.close()
    for i in range(len(seeds)):
        assert torch.equal(outs[i], eager[i].cpu()), "pipelined step %d differs from eager step %d" % (i, i)


@pytest.mark.parametrize("math", ["tf32x3", "bf16"])
def test_seq_step_launches_only_library_kernels(gs, math):
    m, infos, seeds = _small_model(gs, math, bf16=(math == "bf16"))
    m.forward(seeds[0], normalize=True)
    torch.cuda.synchronize()
    from torch.autograd import DeviceType
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        m.forward(seeds[1], normalize=True)
        torch.cuda.synchronize()
    names = [e.name for e in prof.events() if e.device_type == DeviceType.CUDA]
    if not names:
        pytest.skip("the profiler recorded no device activity here (CUPTI unavailable)")
    foreign = [nm for nm in names if "gs::" not in nm and "memcpy" not in nm.lower() and "memset" not in nm.lower()]
    assert any("lstm_seq" in nm for nm in names) and any("row_used" in nm for nm in names), names
    assert not foreign, "non-library kernels in the seq step: %r" % foreign


# ---------------------------------------------------------------- training
def _cpu_seq_outputs(adj, feats, seeds, fan, aggs, concat, seed, counter):
    """The oracle's op sequence in differentiable torch on the CPU (an unrolled LSTM masked at t < len)."""
    A, Fe = torch.from_numpy(adj), torch.from_numpy(feats)
    L = len(fan)
    samples, sup = [torch.from_numpy(seeds)], 1
    support = [1]
    for k in range(L):
        t = L - k - 1
        sup *= fan[t]
        samples.append(torch_ref.sample_padded(A, samples[k], fan[t], seed, counter + k).reshape(-1))
        support.append(sup)
    hidden = [Fe.index_select(0, s.long()) for s in samples]
    for layer in range(L):
        a, last, nxt = aggs[layer], layer == L - 1, []
        for hop in range(L - layer):
            k = fan[L - hop - 1]
            selfv = hidden[hop]
            n = selfv.shape[0]
            x = hidden[hop + 1].reshape(n, k, -1)
            d = x.shape[2]
            H = a["kernel"].shape[1] // 4
            lens = (x.detach() != 0).any(dim=2).sum(dim=1).clamp(min=1)
            h, c, outs = torch.zeros(n, H), torch.zeros(n, H), []
            for t in range(k):
                G = x[:, t] @ a["kernel"][:d] + h @ a["kernel"][d:] + a["cbias"]
                i, j, f, o = G.split(H, dim=1)
                c = c * torch.sigmoid(f + 1.0) + torch.sigmoid(i) * torch.tanh(j)
                h = torch.tanh(c) * torch.sigmoid(o)
                outs.append(h)
            neigh_h = torch.stack(outs, dim=1)[torch.arange(n), lens - 1]
            fs, fn = selfv @ a["self_weights"], neigh_h @ a["neigh_weights"]
            y = torch.cat([fs, fn], dim=1) if concat else fs + fn
            nxt.append(y if last else torch.relu(y))
        hidden = nxt
    out = hidden[0]
    return out / torch.sqrt(torch.clamp((out * out).sum(dim=1, keepdim=True), min=1e-12))


def _cpu_params(m):
    aggs = []
    for a in m.aggregators:
        d = {k: v.detach().cpu().clone().requires_grad_(True) for k, v in a.vars.items()}
        d["kernel"] = a.cell_vars["kernel"].detach().cpu().clone().requires_grad_(True)
        d["cbias"] = a.cell_vars["bias"].detach().cpu().clone().requires_grad_(True)
        aggs.append(d)
    return aggs


def _seq_train_model(gs, g, B, C, wd, concat=True, seed=123):
    gs.set_default_math("fp32")
    adj, feats = g["khop_adj"], g["khop_feats"]
    sampler = gs.UniformNeighborSampler(dev(adj), seed=seed)
    infos = [gs.SAGEInfo("node", sampler, 5, 8), gs.SAGEInfo("node", sampler, 3, 8)]
    m = gs.SupervisedGraphsage(C, {"batch_size": B, "dropout": 0.}, dev(feats), dev(adj), None, infos, concat=concat,
                               aggregator_type="seq", sigmoid_loss=True, learning_rate=0.01, weight_decay=wd)
    for a in m.aggregators:                          # a non-zero cell bias so its gradient path is exercised
        a.cell_vars["bias"].data.add_(torch.randn_like(a.cell_vars["bias"]) * 0.1)
    return m, sampler


@pytest.mark.parametrize("concat", [True, False])
def test_seq_loss_and_gradients_match_cpu_autograd(gs, concat):
    g = load_golden("seq")
    rs = np.random.RandomState(5)
    adj, feats = g["khop_adj"], g["khop_feats"]
    n, B, C, wd = adj.shape[0] - 1, 16, 5, 1e-3
    seeds = rs.randint(0, n, size=B).astype(np.int32)
    seeds[0] = 3                                      # an isolated node: all its neighbour rows are the zero row
    labels = (rs.rand(B, C) < 0.3).astype(np.float32)
    m, _ = _seq_train_model(gs, g, B, C, wd, concat)
    aggs = _cpu_params(m)
    head = {k: v.detach().cpu().clone().requires_grad_(True) for k, v in m.node_pred_vars.items()}
    out = _cpu_seq_outputs(adj, feats, seeds, [5, 3], aggs, concat, 123, 0)
    ref = torch.nn.functional.binary_cross_entropy_with_logits(out @ head["weights"] + head["bias"],
                                                               torch.from_numpy(labels))
    for a in aggs:                                    # the reference decays aggregator.vars only, not the cell
        for k in ("neigh_weights", "self_weights"):
            ref = ref + wd * 0.5 * (a[k] * a[k]).sum()
    for v in head.values():
        ref = ref + wd * 0.5 * (v * v).sum()
    ref.backward()
    loss = m.loss(torch.from_numpy(seeds), torch.from_numpy(labels))
    loss.backward()
    assert abs(float(loss) - float(ref)) < 1e-5 * max(1.0, abs(float(ref)))
    for a, ra in zip(m.aggregators, aggs):
        for k in a.vars:
            assert rel_err(a.vars[k].grad.cpu().numpy(), ra[k].grad.numpy(), floor=1e-8) < 2e-4, k
        assert rel_err(a.cell_vars["kernel"].grad.cpu().numpy(), ra["kernel"].grad.numpy(), floor=1e-8) < 2e-4
        assert rel_err(a.cell_vars["bias"].grad.cpu().numpy().reshape(1, -1), ra["cbias"].grad.numpy().reshape(1, -1),
                       floor=1e-8) < 2e-4


def test_seq_training_steps_track_cpu_adam(gs):
    g = load_golden("seq")
    rs = np.random.RandomState(9)
    adj, feats = g["khop_adj"], g["khop_feats"]
    n, B, C = adj.shape[0] - 1, 32, 5
    m, _ = _seq_train_model(gs, g, B, C, 0.0)
    aggs = _cpu_params(m)
    head = {k: v.detach().cpu().clone().requires_grad_(True) for k, v in m.node_pred_vars.items()}
    params = [v for a in aggs for v in a.values()] + list(head.values())
    opt = torch.optim.Adam(params, lr=0.01)
    gpu_losses, cpu_losses = [], []
    for step in range(5):
        seeds = rs.randint(0, n, size=B).astype(np.int32)
        labels = (rs.rand(B, C) < 0.3).astype(np.float32)
        gpu_losses.append(float(m.train_step(torch.from_numpy(seeds), torch.from_numpy(labels))))
        opt.zero_grad()
        out = _cpu_seq_outputs(adj, feats, seeds, [5, 3], aggs, True, 123, 2 * step)
        ref = torch.nn.functional.binary_cross_entropy_with_logits(out @ head["weights"] + head["bias"],
                                                                   torch.from_numpy(labels))
        ref.backward()
        for p in params:
            p.grad.clamp_(-5.0, 5.0)
        opt.step()
        cpu_losses.append(float(ref))
    assert np.allclose(gpu_losses, cpu_losses, rtol=2e-3), (gpu_losses, cpu_losses)
    for a, ra in zip(m.aggregators, aggs):
        assert rel_err(a.cell_vars["kernel"].detach().cpu().numpy(), ra["kernel"].detach().numpy()) < 5e-3
        for k in a.vars:
            assert rel_err(a.vars[k].detach().cpu().numpy(), ra[k].detach().numpy()) < 5e-3


def test_seq_unsupervised_step_matches_cpu(gs):
    import oracle
    g = load_golden("seq")
    rs = np.random.RandomState(11)
    adj, feats = g["khop_adj"], g["khop_feats"]
    n, B, NEG = adj.shape[0] - 1, 16, 20
    deg = rs.randint(1, 40, size=n).astype(np.float64)
    b1 = rs.randint(0, n, size=B).astype(np.int32)
    b2 = rs.randint(0, n, size=B).astype(np.int32)
    gs.set_default_math("fp32")
    sampler = gs.UniformNeighborSampler(dev(adj), seed=123)
    infos = [gs.SAGEInfo("node", sampler, 5, 8), gs.SAGEInfo("node", sampler, 3, 8)]
    m = gs.UnsupervisedGraphsage({"batch_size": B, "dropout": 0.}, dev(feats), dev(adj), deg, infos, concat=True,
                                 aggregator_type="seq", neg_sample_size=NEG, learning_rate=0.01, weight_decay=1e-3,
                                 seed=77)
    aggs = _cpu_params(m)
    neg = oracle.sample_unigram(deg, NEG, 77, 0)
    o1 = _cpu_seq_outputs(adj, feats, b1, [5, 3], aggs, True, 123, 0)
    o2 = _cpu_seq_outputs(adj, feats, b2, [5, 3], aggs, True, 123, 2)
    on = _cpu_seq_outputs(adj, feats, neg, [5, 3], aggs, True, 123, 4)
    aff, neg_aff = (o1 * o2).sum(1), o1 @ on.t()
    ref = torch.nn.functional.softplus(-aff).sum() + torch.nn.functional.softplus(neg_aff).sum()
    for a in aggs:
        for k in ("neigh_weights", "self_weights"):
            ref = ref + 1e-3 * 0.5 * (a[k] * a[k]).sum()
    ref = ref / B
    loss = m.train_step(torch.from_numpy(b1), torch.from_numpy(b2))
    assert abs(float(loss) - float(ref.detach())) < 1e-5 * max(1.0, abs(float(ref.detach())))
