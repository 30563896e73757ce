"""SupervisedGraphsage - the training step around the hot path (SURVEY section 8f row 1; reference
graphsage/supervised_models.py:10-126).

Forward: the B200 kernels (sample -> fused gather+mean -> tcgen05 / fp32 GEMM), wrapped in
torch.autograd.Function so the step is differentiable.  Backward: the gradient formulas of the mean / GCN
aggregators, with the weight-gradient GEMMs (X^T dZ) as plain library matmuls (torch / cuBLAS fp32) - features
are not trainable (identity_dim = 0), so nothing is scattered into the table.  Head (l2_normalize -> Dense ->
sigmoid / softmax cross-entropy + weight decay), gradient clipping to +-5 and Adam follow
supervised_models.py:85-126.
"""
import torch

from . import ops
from .aggregators import MaxPoolingAggregator, SeqAggregator
from .layers import act_code, identity, relu  # noqa: F401
from .models import SampleAndAggregate


class _AggregateRowsFn(torch.autograd.Function):
    """y = agg.aggregate_rows(src, segments) for MeanAggregator / GCNAggregator, differentiable w.r.t. the
    aggregator weights and (for layers >= 1, where rows are addressed by ranges) w.r.t. src."""

    @staticmethod
    def forward(ctx, agg, src, segments, *weights):
        kind = "gcn" if "weights" in agg.vars else "mean"
        code, post = act_code(agg.act)
        if post is not None:
            raise NotImplementedError("training supports act=relu or identity")
        with torch.no_grad():
            if kind == "mean":
                xs, xm = ops.gather_mean(src, segments, want_self=True)
            else:
                xs, xm = None, ops.gather_mean(src, segments, include_self=True, want_self=False)[1]
            F_in = src.shape[1]
            if kind == "mean":
                parts = [(xs, F_in, weights[0]), (xm, F_in, weights[1])]
                combine = ops.COMBINE_CONCAT if agg.concat else ops.COMBINE_ADD
            else:
                parts, combine = [(xm, F_in, weights[0])], ops.COMBINE_ADD
            y = ops.sage_gemm(parts, combine=combine, bias=agg.vars.get("bias"), act=code, math=agg.math)
        ctx.kind, ctx.relu, ctx.concat = kind, code == ops.ACT_RELU, bool(agg.concat)
        ctx.segments, ctx.src_shape, ctx.F_in = segments, tuple(src.shape), F_in
        ctx.src_needs_grad = bool(torch.is_tensor(src) and src.requires_grad)
        ctx.has_bias = "bias" in agg.vars
        ctx.save_for_backward(xm if xs is None else xs, xm, y, *weights)
        return y

    @staticmethod
    def backward(ctx, dy):
        xs, xm, y = ctx.saved_tensors[:3]
        weights = ctx.saved_tensors[3:]
        F_in = ctx.F_in
        dz = dy * (y > 0).to(dy.dtype) if ctx.relu else dy
        grads_w, dsrc = [], None
        if ctx.kind == "mean":
            Ws, Wn = weights
            D = Ws.shape[1]
            dz_s, dz_n = (dz[:, :D], dz[:, D:]) if ctx.concat else (dz, dz)
            grads_w = [xs[:, :F_in].t() @ dz_s, xm[:, :F_in].t() @ dz_n]         # dW = X^T dZ  (library GEMM)
            if ctx.src_needs_grad:
                dxs, dxm = dz_s @ Ws.t(), dz_n @ Wn.t()
        else:
            (W,) = weights
            grads_w = [xm[:, :F_in].t() @ dz]
            if ctx.src_needs_grad:
                dxm = dz @ W.t()
                dxs = None
        if ctx.src_needs_grad:
            dsrc = torch.zeros(ctx.src_shape, dtype=dy.dtype, device=dy.device)
            for s in ctx.segments:
                if s.self_ids is not None or s.neigh_ids is not None:
                    raise NotImplementedError("gradient w.r.t. an id-addressed source (trainable features) is out of scope")
                n, k = s.n, s.k
                rows = slice(s.out_row0, s.out_row0 + n)
                div = float(k + (1 if ctx.kind == "gcn" else 0))
                dsrc[s.neigh_row0:s.neigh_row0 + n * k].view(n, k, -1).add_((dxm[rows] / div).unsqueeze(1))
                if ctx.kind == "gcn":
                    dsrc[s.self_row0:s.self_row0 + n].add_(dxm[rows] / div)
                else:
                    dsrc[s.self_row0:s.self_row0 + n].add_(dxs[rows])
        return (None, dsrc, None) + tuple(grads_w)


def pool_branch_backward(pool, xn, h, hp, dhp, Wm, k, need_dx):
    """Gradients through hp = pool_k(h), h = relu(xn @ Wm + bm) for one hop (reference aggregators.py:176-182 /
    :256-262 backwards).  xn [n*k, F], h [n*k, hid] (post-ReLU), hp / dhp [n, hid].
    max: the gradient of a maximum goes to the positions that attain it, split evenly among ties (TensorFlow's
    reduce_max gradient); mean: dhp / k to every position.  Returns (dWm, dbm, dxn or None)."""
    n, hid = hp.shape
    h3 = h.reshape(n, k, hid)
    if pool == "max":
        sel = h3 == hp.unsqueeze(1)
        share = dhp / sel.sum(dim=1).to(dhp.dtype)
        dh = sel.to(dhp.dtype) * share.unsqueeze(1)
    else:
        dh = (dhp / float(k)).unsqueeze(1).expand(n, k, hid)
    dpre = (dh * (h3 > 0).to(dhp.dtype)).reshape(n * k, hid)             # ReLU of the Dense layer
    dWm = xn.t() @ dpre
    dbm = dpre.sum(dim=0)
    return dWm, dbm, (dpre @ Wm.t() if need_dx else None)


class _PoolAggregateRowsFn(torch.autograd.Function):
    """y = agg.aggregate_rows(src, segments) for MaxPoolingAggregator / MeanPoolingAggregator on the unfused fp32 path
    (gather -> Dense(relu, bias) -> pool over the fanout -> both matmuls), differentiable w.r.t. the four weight tensors
    and (layers >= 1) src.  The gathered neighbour rows and the MLP activations are kept for the backward pass."""

    @staticmethod
    def forward(ctx, agg, src, segments, Ws, Wn, Wm, bm):
        code, post = act_code(agg.act)
        if post is not None:
            raise NotImplementedError("training supports act=relu or identity")
        if len(agg.mlp_layers) != 1 or agg.dropout:
            raise NotImplementedError("training supports one MLP layer and dropout = 0")
        F_in, hid = src.shape[1], agg.hidden_dim
        rows = max(s.out_row0 + s.n for s in segments)
        with torch.no_grad():
            xs = torch.empty((rows, ops.pad_cols(F_in)), dtype=torch.float32, device=src.device)[:, :F_in]
            hp = torch.empty((rows, hid), dtype=torch.float32, device=src.device)
            kept = []
            for s in segments:
                n, k = s.n, s.k
                xn = ops.gather_rows(src, s.neigh_ids[:n * k]) if s.neigh_ids is not None else \
                    src[s.neigh_row0:s.neigh_row0 + n * k]
                mlp = agg.mlp_layers[0]
                mlp.math = agg.math
                h = mlp(xn)
                if agg.pool == "mean":
                    hp[s.out_row0:s.out_row0 + n] = ops.gather_mean(h, [ops.Seg(n, k)], want_self=False, out_pitch=hid)[1]
                else:
                    hp[s.out_row0:s.out_row0 + n] = ops.segment_max(h, n, k)
                if s.self_ids is not None:
                    ops.gather_rows(src, s.self_ids[:n], out=xs[s.out_row0:s.out_row0 + n])
                else:
                    xs[s.out_row0:s.out_row0 + n] = src[s.self_row0:s.self_row0 + n]
                kept.extend([xn, h])
            y = agg._finish([(xs, agg.input_dim, Ws), (hp, hid, Wn)], agg._combine())
        ctx.pool, ctx.relu, ctx.concat = agg.pool, code == ops.ACT_RELU, bool(agg.concat)
        ctx.segments, ctx.src_shape, ctx.F_in = segments, tuple(src.shape), F_in
        ctx.src_needs_grad = bool(torch.is_tensor(src) and src.requires_grad)
        ctx.save_for_backward(xs, hp, y, Ws, Wn, Wm, *kept)
        return y

    @staticmethod
    def backward(ctx, dy):
        xs, hp, y, Ws, Wn, Wm = ctx.saved_tensors[:6]
        kept = ctx.saved_tensors[6:]
        F_in = ctx.F_in
        dz = dy * (y > 0).to(dy.dtype) if ctx.relu else dy
        D = Ws.shape[1]
        dz_s, dz_n = (dz[:, :D], dz[:, D:]) if ctx.concat else (dz, dz)
        dWs, dWn = xs.t() @ dz_s, hp.t() @ dz_n
        dhp = dz_n @ Wn.t()
        dWm, dbm = torch.zeros_like(Wm), torch.zeros(Wm.shape[1], dtype=dy.dtype, device=dy.device)
        dsrc = torch.zeros(ctx.src_shape, dtype=dy.dtype, device=dy.device) if ctx.src_needs_grad else None
        dxs = dz_s @ Ws.t() if ctx.src_needs_grad else None
        for i, s in enumerate(ctx.segments):
            n, k = s.n, s.k
            rows = slice(s.out_row0, s.out_row0 + n)
            xn, h = kept[2 * i][:, :F_in], kept[2 * i + 1]
            g_wm, g_bm, dxn = pool_branch_backward(ctx.pool, xn, h, hp[rows], dhp[rows], Wm, k, ctx.src_needs_grad)
            dWm += g_wm
            dbm += g_bm
            if ctx.src_needs_grad:
                if s.self_ids is not None or s.neigh_ids is not None:
                    raise NotImplementedError("gradient w.r.t. an id-addressed source (trainable features) is out of scope")
                dsrc[s.neigh_row0:s.neigh_row0 + n * k] += dxn
                dsrc[s.self_row0:s.self_row0 + n] += dxs[rows]
        return None, dsrc, None, dWs, dWn, dWm, dbm


def lstm_seq_backward(P, X, Wx, Wh, keep_h, keep_c, lengths, dout, need_dx):
    """BPTT through out = h_{len-1} of BasicLSTMCell over one hop's n sequences of k steps (reference
    aggregators.py:408-433 backwards).  P [n*k, 4H] is the input projection, X [n*k, in] its input, keep_h / keep_c
    [n, k, H] the states the forward kept (steps t >= len unspecified) and dout [n, H] the gradient of the outputs.
    Gate activations are recomputed from P + h_{t-1} @ Wh; steps t >= len carry no gradient, and len none at all.
    Returns (dWx, dWh, db, dX or None)."""
    n, k, H = keep_h.shape
    live = (torch.arange(k, device=P.device).unsqueeze(0) < lengths.long().unsqueeze(1)).unsqueeze(2)   # [n, k, 1]
    hs = torch.where(live, keep_h, torch.zeros((), dtype=keep_h.dtype, device=keep_h.device))
    cs = torch.where(live, keep_c, torch.zeros((), dtype=keep_c.dtype, device=keep_c.device))
    h_prev = torch.cat([torch.zeros_like(hs[:, :1]), hs[:, :-1]], dim=1)
    c_prev = torch.cat([torch.zeros_like(cs[:, :1]), cs[:, :-1]], dim=1)
    G = P[:, :4 * H].reshape(n, k, 4 * H) + (h_prev.reshape(n * k, H) @ Wh).reshape(n, k, 4 * H)
    gi, gj, gf, go = G.split(H, dim=2)
    si, tj, sf, so = torch.sigmoid(gi), torch.tanh(gj), torch.sigmoid(gf + 1.0), torch.sigmoid(go)
    tc = torch.tanh(cs)
    last = lengths.long() - 1
    dG = torch.zeros_like(G)
    dh = torch.zeros((n, H), dtype=dout.dtype, device=dout.device)
    dc = torch.zeros_like(dh)
    for t in range(k - 1, -1, -1):
        dh = dh + torch.where((last == t).unsqueeze(1), dout, torch.zeros((), dtype=dout.dtype, device=dout.device))
        m = live[:, t].to(dout.dtype)
        dh = dh * m
        dc = (dc + dh * so[:, t] * (1.0 - tc[:, t] * tc[:, t])) * m
        d_o = dh * tc[:, t] * so[:, t] * (1.0 - so[:, t])
        d_i = dc * tj[:, t] * si[:, t] * (1.0 - si[:, t])
        d_j = dc * si[:, t] * (1.0 - tj[:, t] * tj[:, t])
        d_f = dc * c_prev[:, t] * sf[:, t] * (1.0 - sf[:, t])
        dG[:, t] = torch.cat([d_i, d_j, d_f, d_o], dim=1)
        dh = dG[:, t] @ Wh.t()
        dc = dc * sf[:, t]
    dP = dG.reshape(n * k, 4 * H)
    dWh = h_prev.reshape(n * k, H).t() @ dP
    return X.t() @ dP, dWh, dP.sum(dim=0), (dP @ Wx.t() if need_dx else None)


class _SeqAggregateRowsFn(torch.autograd.Function):
    """y = agg.aggregate_rows(src, segments) for SeqAggregator, differentiable w.r.t. self / neigh weights, the cell's
    kernel and bias, and (layers >= 1) src.  The forward runs the inference kernels (gather, projection GEMM,
    gs_lstm_seq, final GEMM) and keeps X, P, h_t, c_t and the lengths of every hop for the BPTT backward."""

    @staticmethod
    def forward(ctx, agg, src, segments, Ws, Wn, kernel, cbias):
        code, post = act_code(agg.act)
        if post is not None:
            raise NotImplementedError("training supports act=relu or identity")
        rows = max(s.out_row0 + s.n for s in segments)
        H = agg.hidden_dim
        with torch.no_grad():
            used = agg._used_table(src, False)
            Wh = kernel[agg.neigh_input_dim:]
            neigh_h = torch.empty((rows, H), dtype=torch.float32, device=src.device)
            kept = []
            for s in segments:
                X = agg.neighbour_rows(src, s)
                P = agg._project(X)
                _, kh, kc, lens = ops.lstm_seq(P, Wh, used, s.n, s.k,
                                               row_ids=None if s.neigh_ids is None else s.neigh_ids[:s.n * s.k],
                                               row0=s.neigh_row0, out=neigh_h[s.out_row0:s.out_row0 + s.n], keep=True)
                kept.extend([X, P, kh, kc, lens])
            xs = agg.self_rows(src, segments, rows)
            y = agg._finish([(xs, agg.input_dim, Ws), (neigh_h, H, Wn)], agg._combine())
        ctx.relu, ctx.concat, ctx.F_in = code == ops.ACT_RELU, bool(agg.concat), agg.neigh_input_dim
        ctx.segments, ctx.src_shape = segments, tuple(src.shape)
        ctx.src_needs_grad = bool(torch.is_tensor(src) and src.requires_grad)
        ctx.save_for_backward(xs, neigh_h, y, Ws, Wn, kernel, *kept)
        return y

    @staticmethod
    def backward(ctx, dy):
        xs, neigh_h, y, Ws, Wn, kernel = ctx.saved_tensors[:6]
        kept = ctx.saved_tensors[6:]
        dz = dy * (y > 0).to(dy.dtype) if ctx.relu else dy
        D = Ws.shape[1]
        dz_s, dz_n = (dz[:, :D], dz[:, D:]) if ctx.concat else (dz, dz)
        dWs, dWn = xs.t() @ dz_s, neigh_h.t() @ dz_n
        dneigh = dz_n @ Wn.t()
        Wx, Wh = kernel[:ctx.F_in], kernel[ctx.F_in:]
        dWx, dWh = torch.zeros_like(Wx), torch.zeros_like(Wh)
        db = torch.zeros(kernel.shape[1], dtype=dy.dtype, device=dy.device)
        dsrc = torch.zeros(ctx.src_shape, dtype=dy.dtype, device=dy.device) if ctx.src_needs_grad else None
        dxs = dz_s @ Ws.t() if ctx.src_needs_grad else None
        for i, s in enumerate(ctx.segments):
            X, P, kh, kc, lens = kept[5 * i:5 * i + 5]
            rows = slice(s.out_row0, s.out_row0 + s.n)
            g_wx, g_wh, g_b, dX = lstm_seq_backward(P, X, Wx, Wh, kh, kc, lens, dneigh[rows], ctx.src_needs_grad)
            dWx += g_wx
            dWh += g_wh
            db += g_b
            if ctx.src_needs_grad:
                if s.self_ids is not None or s.neigh_ids is not None:
                    raise NotImplementedError("gradient w.r.t. an id-addressed source (trainable features) is out of scope")
                dsrc[s.neigh_row0:s.neigh_row0 + s.n * s.k] += dX
                dsrc[s.self_row0:s.self_row0 + s.n] += dxs[rows]
        return None, dsrc, None, dWs, dWn, torch.cat([dWx, dWh], dim=0), db


def differentiable_outputs(model, batch, normalize=True):
    """sample -> aggregate (-> l2_normalize) with an autograd graph over the aggregator weights; `model` is a
    SampleAndAggregate whose .aggregators exist (reference models.py:347-350 / supervised_models.py:79-85)."""
    batch = batch.to(device=model.device, dtype=torch.int32).reshape(-1)
    n = batch.numel()
    with torch.no_grad():
        samples, support = model.sample(batch, model.layer_infos, batch_size=n)
    num_samples = [info.num_samples for info in model.layer_infos]
    L = len(num_samples)
    counts = [n * support[h] for h in range(L + 1)]
    src = model.features
    for layer in range(L):
        hops = L - layer
        row0 = [sum(counts[:h]) for h in range(hops + 1)]
        segs = []
        for hop in range(hops):
            k = num_samples[L - hop - 1]
            if layer == 0:
                segs.append(ops.Seg(counts[hop], k, self_ids=samples[hop], neigh_ids=samples[hop + 1],
                                    out_row0=row0[hop]))
            else:
                segs.append(ops.Seg(counts[hop], k, self_row0=row0[hop], neigh_row0=row0[hop + 1],
                                    out_row0=row0[hop]))
        agg = model.aggregators[layer]
        if isinstance(agg, SeqAggregator):                  # LSTM
            src = _SeqAggregateRowsFn.apply(agg, src, segs, agg.vars["self_weights"], agg.vars["neigh_weights"],
                                            agg.cell_vars["kernel"], agg.cell_vars["bias"])
        elif hasattr(agg, "mlp_layers"):                      # max-pool / mean-pool
            mlp = agg.mlp_layers[0].vars
            src = _PoolAggregateRowsFn.apply(agg, src, segs, agg.vars["self_weights"], agg.vars["neigh_weights"],
                                             mlp["weights"], mlp["bias"])
        else:
            ws = (agg.vars["weights"],) if "weights" in agg.vars else (agg.vars["self_weights"], agg.vars["neigh_weights"])
            src = _AggregateRowsFn.apply(agg, src, segs, *ws)
    out = src[:counts[0]]
    if normalize:
        out = out / torch.sqrt(torch.clamp((out * out).sum(dim=1, keepdim=True), min=1e-12))   # tf.nn.l2_normalize
    return out


def build_aggregators(model):
    """One aggregator per layer, as SampleAndAggregate.aggregate creates them (reference models.py:303-315)."""
    if float(model.placeholders.get("dropout", 0.) or 0.) != 0.:
        # the reference applies dropout inside the aggregators and in the prediction Dense (supervised_models.py:88-90);
        # the differentiable path here has no dropout, so refuse rather than silently train a different model
        raise NotImplementedError("training with placeholders['dropout'] > 0 is not implemented (forward-only "
                                  "dropout runs through SampleAndAggregate.aggregate's materialised path)")
    L = len(model.layer_infos)
    aggs = []
    for layer in range(L):
        dim_mult = 2 if model.concat and layer != 0 else 1
        act = identity if layer == L - 1 else relu
        extra = {"model_size": model.model_size} if issubclass(model.aggregator_cls, (MaxPoolingAggregator, SeqAggregator)) \
            else {}
        aggs.append(model.aggregator_cls(dim_mult * model.dims[layer], model.dims[layer + 1], act=act, dropout=0.,
                                         concat=model.concat, device=model.device, **extra))
    return aggs


def aggregator_parameters(aggregators):
    """(all trainable tensors, the subset the reference applies weight decay to).  The reference decays
    `aggregator.vars` only (supervised_models.py:103-105, models.py:385-387) - the pooling aggregators' Dense variables
    live in `mlp_layers[0].vars`, the seq aggregator's LSTM variables in `cell_vars` (the reference keeps them in the
    cell); both are trained but not decayed."""
    decayed = [v for a in aggregators for v in a.vars.values()]
    extra = [v for a in aggregators for layer in getattr(a, "mlp_layers", []) for v in layer.vars.values()]
    extra += [v for a in aggregators for v in getattr(a, "cell_vars", {}).values()]
    return decayed + extra, decayed


def classification_loss(logits, labels, sigmoid_loss):
    """reference supervised_models.py:109-117: mean over ALL elements of the sigmoid cross-entropy (multi-label), or the
    mean over nodes of the softmax cross-entropy."""
    if sigmoid_loss:
        return torch.nn.functional.binary_cross_entropy_with_logits(logits, labels, reduction="mean")
    return (-(labels * torch.log_softmax(logits, dim=1)).sum(dim=1)).mean()


def weight_decay_term(params, weight_decay):
    """weight_decay * tf.nn.l2_loss(var) = weight_decay * sum(var^2) / 2 over every variable (supervised_models.py:103-107)."""
    total = None
    for p in params:
        t = weight_decay * 0.5 * (p * p).sum()
        total = t if total is None else total + t
    return total


class SupervisedGraphsage(SampleAndAggregate):
    """Supervised GraphSAGE (reference graphsage/supervised_models.py:10-126): the hot path, then
    l2_normalize -> Dense(-> num_classes) -> sigmoid / softmax cross-entropy (+ weight decay), gradients clipped to
    [-5, 5], Adam.  TF FLAGS become constructor arguments (learning_rate, weight_decay)."""

    def __init__(self, num_classes, placeholders, features, adj, degrees, layer_infos, concat=True,
                 aggregator_type="mean", model_size="small", sigmoid_loss=False, identity_dim=0, learning_rate=0.01,
                 weight_decay=0.0, device="cuda", distributed=False, group=None, **kwargs):
        super(SupervisedGraphsage, self).__init__(placeholders, features, adj, degrees, layer_infos, concat=concat,
                                                  aggregator_type=aggregator_type, model_size=model_size,
                                                  identity_dim=identity_dim, device=device, **kwargs)
        if aggregator_type not in ("mean", "gcn", "maxpool", "meanpool", "seq"):
            raise NotImplementedError("training is implemented for the mean, gcn, maxpool, meanpool and seq aggregators")
        self.num_classes = num_classes
        self.sigmoid_loss = sigmoid_loss
        self.learning_rate, self.weight_decay = learning_rate, weight_decay
        self.distributed, self.group, self.last_allreduce_bytes = bool(distributed), group, 0
        self.build()

    def build(self):
        from .inits import glorot, zeros
        self.aggregators = build_aggregators(self)
        dim_mult = 2 if self.concat else 1
        self.node_pred_vars = {"weights": glorot([dim_mult * self.dims[-1], self.num_classes], device=self.device),
                               "bias": zeros([self.num_classes], device=self.device)}   # supervised_models.py:88-90
        if self.distributed:                                                     # every rank starts from rank 0's weights
            from .parallel import broadcast_parameters
            broadcast_parameters(self.parameters(), 0, self.group)
        for p in self.parameters():
            p.requires_grad_(True)
        self.optimizer = torch.optim.Adam(self.parameters(), lr=self.learning_rate)      # TF AdamOptimizer defaults

    def parameters(self):
        return aggregator_parameters(self.aggregators)[0] + list(self.node_pred_vars.values())

    def decayed_parameters(self):
        return aggregator_parameters(self.aggregators)[1] + list(self.node_pred_vars.values())

    def outputs(self, batch):
        """l2-normalised node representations, differentiable (supervised_models.py:79-85)."""
        return differentiable_outputs(self, batch)

    def logits(self, batch):
        return self.outputs(batch) @ self.node_pred_vars["weights"] + self.node_pred_vars["bias"]

    def loss(self, batch, labels):
        """supervised_models.py:101-118: weight decay * l2_loss(var) over aggregator + head variables, then the
        mean of the per-element sigmoid xent (multi-label) or the mean of the per-node softmax xent."""
        logits = self.logits(batch)
        labels = labels.to(device=logits.device, dtype=torch.float32)
        loss = classification_loss(logits, labels, self.sigmoid_loss)
        if self.weight_decay:
            loss = loss + weight_decay_term(self.decayed_parameters(), self.weight_decay)
        return loss

    def train_step(self, batch, labels):
        self.optimizer.zero_grad(set_to_none=True)
        loss = self.loss(batch, labels)
        loss.backward()
        if self.distributed:                                                     # data parallel: mean gradient over ranks
            from .parallel import allreduce_gradients
            self.last_allreduce_bytes = allreduce_gradients(self.parameters(), self.group)
        for p in self.parameters():                                              # clip_by_value(grad, -5, 5)  :93-94
            if p.grad is not None:
                p.grad.clamp_(-5.0, 5.0)
        self.optimizer.step()
        return loss.detach()

    def predict(self, batch):
        with torch.no_grad():
            lg = self.logits(batch)
            return torch.sigmoid(lg) if self.sigmoid_loss else torch.softmax(lg, dim=1)
