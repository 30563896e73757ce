"""SAGEInfo and SampleAndAggregate.sample / .aggregate - the surface of reference
graphsage/models.py:178-330 over the B200 kernels.

The TF placeholders / FLAGS the reference threads through become explicit arguments:
`placeholders` is a plain dict ({"batch_size": int, "dropout": float, ...}).
"""
from collections import namedtuple

import torch

from . import ops
from .aggregators import GCNAggregator, MaxPoolingAggregator, MeanAggregator, MeanPoolingAggregator, SeqAggregator
from .layers import identity, relu  # noqa: F401

# reference graphsage/models.py:180-185
SAGEInfo = namedtuple("SAGEInfo",
                      ["layer_name",      # name of the layer (always "node"; unused)
                       "neigh_sampler",   # callable neigh_sampler
                       "num_samples",
                       "output_dim"])     # the output (i.e., hidden) dimension

_AGGREGATORS = {"mean": MeanAggregator, "maxpool": MaxPoolingAggregator, "gcn": GCNAggregator,
                "meanpool": MeanPoolingAggregator, "seq": SeqAggregator}


class SampleAndAggregate(object):
    """The sample -> K-hop gather -> aggregate recursion of GraphSAGE (reference models.py:187-330).

    features : float32 CUDA tensor [N+1, F] whose LAST row is the all-zero dummy row
               (reference supervised_train.py:133-135), or a numpy array (uploaded, dummy row NOT added).
    adj      : int32 CUDA tensor [N+1, max_degree] padded adjacency (reference minibatch.py:227-245).
    """

    def __init__(self, placeholders, features, adj, degrees, layer_infos, concat=True, aggregator_type="mean",
                 model_size="small", identity_dim=0, device="cuda", **kwargs):
        allowed_kwargs = {"name", "logging", "model_size"}
        for kwarg in kwargs.keys():
            assert kwarg in allowed_kwargs, "Invalid keyword argument: " + kwarg   # reference models.py:22-24
        if aggregator_type not in _AGGREGATORS:
            raise ValueError("Unknown aggregator: %r" % (aggregator_type,))
        self.aggregator_cls = _AGGREGATORS[aggregator_type]
        if identity_dim > 0:
            raise NotImplementedError("identity_dim > 0 (trainable node embeddings) is out of scope (SURVEY appendix A)")
        if features is None:
            raise ValueError("Must have a positive value for identity feature dimension if no input features given.")
        self.placeholders = placeholders if placeholders is not None else {}
        self.inputs1 = self.placeholders.get("batch1")
        self.inputs2 = self.placeholders.get("batch2")
        self.model_size = model_size
        self.adj_info = adj
        if hasattr(features, "c_table"):                 # parallel.ShardedFeatures: node-partitioned table
            if aggregator_type == "seq":
                raise NotImplementedError("the seq aggregator does not read node-partitioned (sharded) feature tables")
            self.features = features
            self._finish_init(placeholders, adj, degrees, layer_infos, concat, model_size, identity_dim, device)
            return
        if not torch.is_tensor(features):
            features = torch.as_tensor(features, dtype=torch.float32)
        dt = torch.bfloat16 if features.dtype == torch.bfloat16 else torch.float32   # bf16 tables are kept (config 3)
        features = features.to(device=device, dtype=dt)
        F_ = features.shape[1]
        if features.stride(1) != 1 or features.stride(0) % 8 != 0 or features.data_ptr() % 16 != 0 \
                or features.stride(0) < ops.pad_cols(F_):
            # re-pitch once so rows are 16-byte multiples (TMA bulk copies / 128-bit loads); keep the [N+1, F] view
            table = torch.zeros((features.shape[0], ops.pad_cols(F_)), dtype=dt, device=features.device)
            table[:, :F_] = features
            features = table[:, :F_]
        self.features = features
        self._finish_init(placeholders, adj, degrees, layer_infos, concat, model_size, identity_dim, device)

    def _finish_init(self, placeholders, adj, degrees, layer_infos, concat, model_size, identity_dim, device):
        self.degrees = degrees
        self.concat = concat
        self.dims = [self.features.shape[1] + identity_dim]
        self.dims.extend([layer_infos[i].output_dim for i in range(len(layer_infos))])   # models.py:244-245
        self.batch_size = self.placeholders.get("batch_size")
        self.layer_infos = layer_infos
        self.device = torch.device(device)
        self.aggregators = None

    # ------------------------------------------------------------------ models.py:254-275
    def sample(self, inputs, layer_infos, batch_size=None):
        """Sample neighbours to be the supportive fields for multi-layer convolutions.
        Returns (samples, support_sizes); samples[h] is a flat int32 vector of batch*support[h] ids,
        row-major nested: samples[h+1][i*k + j] is neighbour j of samples[h][i]."""
        if batch_size is None:
            batch_size = self.batch_size if self.batch_size is not None else inputs.numel()
        samples = [inputs.reshape(-1)]
        support_size = 1
        support_sizes = [support_size]
        L = len(layer_infos)
        fan = [layer_infos[L - k - 1].num_samples for k in range(L)]          # hop order (models.py:268-272)
        s0 = layer_infos[0].neigh_sampler
        if (L <= 4 and hasattr(s0, "sample_khop") and all(i.neigh_sampler is s0 for i in layer_infos)
                and max(fan) <= 64 and samples[0].numel() == batch_size):
            for k, ids in enumerate(s0.sample_khop(samples[0], fan)):          # one launch for all hops
                support_size *= fan[k]
                samples.append(ids)
                support_sizes.append(support_size)
            return samples, support_sizes
        for k in range(len(layer_infos)):
            t = len(layer_infos) - k - 1
            support_size *= layer_infos[t].num_samples
            sampler = layer_infos[t].neigh_sampler
            node = sampler((samples[k], layer_infos[t].num_samples))
            samples.append(node.reshape(support_size * batch_size))
            support_sizes.append(support_size)
        return samples, support_sizes

    # ------------------------------------------------------------------ models.py:278-330
    def aggregate(self, samples, input_features, dims, num_samples, support_sizes, batch_size=None,
                  aggregators=None, name=None, concat=False, model_size="small", _final=None):
        """At each layer, aggregate hidden representations of neighbours to compute the hidden
        representations at the next layer.  `input_features` is the feature table [N+1, F] (the
        reference passes `[self.features]` - a 1-element list - and indexes it implicitly; both forms
        are accepted).  Returns (hidden[0] of shape [batch, out_w], aggregators)."""
        if batch_size is None:
            batch_size = self.batch_size if self.batch_size is not None else samples[0].numel()
        feats = input_features[0] if isinstance(input_features, (list, tuple)) else input_features
        L = len(num_samples)
        new_agg = aggregators is None
        if new_agg:
            aggregators = []
            for layer in range(L):
                dim_mult = 2 if concat and (layer != 0) else 1
                act = identity if layer == L - 1 else relu                      # models.py:307-310
                kw = dict(act=act, dropout=self.placeholders.get("dropout", 0.), name=name, concat=concat,
                          device=self.device)
                if issubclass(self.aggregator_cls, (MaxPoolingAggregator, SeqAggregator)):
                    kw["model_size"] = model_size
                aggregators.append(self.aggregator_cls(dim_mult * dims[layer], dims[layer + 1], **kw))
        if any(getattr(a, "dropout", 0.) for a in aggregators):
            return self._aggregate_materialised(samples, feats, dims, num_samples, support_sizes, batch_size,
                                                aggregators, concat), aggregators
        # gather-fused recursion: hop h of a layer occupies rows [row0[h], row0[h] + batch*support[h])
        counts = [batch_size * support_sizes[h] for h in range(L + 1)]
        src = feats
        for layer in range(L):
            hops = L - layer
            row0 = [sum(counts[:h]) for h in range(hops + 1)]
            segs = []
            for hop in range(hops):
                k = num_samples[L - hop - 1]                                     # models.py:324
                if layer == 0:
                    segs.append(ops.Seg(counts[hop], k, self_ids=samples[hop], neigh_ids=samples[hop + 1],
                                        out_row0=row0[hop]))
                else:
                    segs.append(ops.Seg(counts[hop], k, self_row0=row0[hop], neigh_row0=row0[hop + 1],
                                        out_row0=row0[hop]))
            src = aggregators[layer].aggregate_rows(src, segs, final=_final if layer == L - 1 else None,
                                                    src_persistent=(layer == 0))
        return src[:counts[0]], aggregators

    def _aggregate_materialised(self, samples, feats, dims, num_samples, support_sizes, batch_size, aggregators,
                                concat):
        """The reference's literal recursion (hidden[h] materialised); used when dropout > 0."""
        hidden = [ops.gather_rows(feats, s) for s in samples]                    # models.py:299
        L = len(num_samples)
        for layer in range(L):
            nxt = []
            for hop in range(L - layer):
                d = hidden[hop + 1].shape[1]
                neigh = hidden[hop + 1].reshape(batch_size * support_sizes[hop], num_samples[L - hop - 1], d)
                nxt.append(aggregators[layer]((hidden[hop], neigh)))
            hidden = nxt
        return hidden[0]

    # ------------------------------------------------------------------ convenience: the whole path
    def graphed(self, batch_size, normalize=True, probe=None):
        """CUDA-graph runner of forward() for a fixed batch size (see GraphedForward)."""
        return GraphedForward(self, batch_size, normalize, probe)

    def pipelined(self, batch_size, normalize=True, depth=2):
        """Host-buffer, copy/compute-overlapped front end (see PipelinedForward)."""
        return PipelinedForward(self, batch_size, normalize, depth)

    def export_embeddings(self, node_ids, batch_size=512, out_prefix=None):
        """Embedding export (reference graphsage/unsupervised_train.py:94-117): forward every given node in batches,
        return float32 [n, out_w]; with out_prefix also write `<prefix>.npy` and `<prefix>.txt` (one id per line)."""
        import numpy as np
        ids = torch.as_tensor(node_ids, dtype=torch.int32).reshape(-1)
        outs = []
        for i in range(0, ids.numel(), batch_size):
            outs.append(self.forward(ids[i:i + batch_size], normalize=True).cpu())
        emb = torch.cat(outs).numpy() if outs else np.zeros((0, 0), np.float32)
        if out_prefix is not None:
            np.save(out_prefix + ".npy", emb)
            with open(out_prefix + ".txt", "w") as fp:
                fp.write("\n".join(str(int(x)) for x in ids.tolist()))
        return emb

    def forward(self, batch, normalize=True):
        """sample -> aggregate -> l2_normalize (reference models.py:347-350, 368) for one id batch."""
        batch = batch.to(device=self.device, dtype=torch.int32).reshape(-1)
        n = batch.numel()
        samples, support = self.sample(batch, self.layer_infos, batch_size=n)
        num_samples = [info.num_samples for info in self.layer_infos]
        final = {"l2_normalize": bool(normalize), "bump": getattr(self, "_graph_bump", None)}
        out, self.aggregators = self.aggregate(samples, [self.features], self.dims, num_samples, support,
                                               batch_size=n, aggregators=self.aggregators, concat=self.concat,
                                               model_size=self.model_size, _final=final)
        if normalize and not final.get("normalized"):
            out = ops.l2_normalize_rows_(out.contiguous())
        if final["bump"] is not None and not final.get("bumped"):
            ops.check(ops.lib().gs_bump_counter(final["bump"][0].data_ptr(), int(final["bump"][1]), ops.stream_ptr()))
            ops._launched(1)
        return out


class GraphedForward(object):
    """SampleAndAggregate.forward for a fixed batch size captured into CUDA graph(s): one replay =
    one batch through sample -> gather -> aggregate (-> l2_normalize) with no per-kernel host work.

    The samplers' RNG call counter lives on the device (`self.counter`) and is advanced by the graph
    itself, so replay r draws exactly what the r-th eager forward would draw (counter0 + n_calls*r + j).
    `probe` (an ops probe name such as "gather_mean/5632") isolates that launch in its own graph so
    bench.py can bracket it with CUDA events inside the timed region.
    """

    def __init__(self, model, batch_size, normalize=True, probe=None, first_step=0, step_stride=1):
        """first_step / step_stride: this runner replays eager steps first_step, first_step + step_stride, ...
        (several runners can interleave - PipelinedForward uses two - and still reproduce the eager RNG sequence)."""
        self.model, self.batch_size, self.normalize = model, int(batch_size), normalize
        dev = model.device
        self.ids = torch.zeros(self.batch_size, dtype=torch.int32, device=dev)
        self.first_step, self.step_stride = int(first_step), int(step_stride)
        self.counter = torch.full((1,), len(model.layer_infos) * self.first_step, dtype=torch.int64, device=dev)
        samplers = []
        for info in model.layer_infos:
            if all(info.neigh_sampler is not s for s in samplers):
                samplers.append(info.neigh_sampler)
        if len(samplers) != 1:
            # every sampler object would need its own device-side call counter advanced by ITS calls per step; with one
            # shared counter replay r would not draw what eager step r draws.  The reference shares one sampler
            # (supervised_train.py:152-159), so refuse the other case instead of mis-counting silently.
            raise NotImplementedError("GraphedForward needs all layer_infos to share one neigh_sampler object")
        self.samplers = samplers
        self.base_counters = [s.counter for s in samplers]
        self.n_calls = len(model.layer_infos)
        self.graphs, self.probe_index = [], None
        self.stream = torch.cuda.Stream(device=dev)
        self.stream.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(self.stream):
            for _ in range(2):                                 # warm-up: lazy inits, aggregator creation
                model.forward(self.ids, normalize)
            self._reset_python_counters()
            for s in samplers:
                s.counter_dev = self.counter
            pool = torch.cuda.graph_pool_handle()
            state = {"g": torch.cuda.CUDAGraph()}
            state["g"].capture_begin(pool=pool)

            def hook(name, phase):
                if probe is None or name != probe:
                    return
                state["g"].capture_end()
                self.graphs.append(state["g"])
                if phase == "pre":
                    self.probe_index = len(self.graphs)
                state["g"] = torch.cuda.CUDAGraph()
                state["g"].capture_begin(pool=pool)

            ops.STAGE_HOOK = hook
            try:
                launches0 = ops.LAUNCHES
                model._graph_bump = (self.counter, self.n_calls * self.step_stride)   # the step advances the device RNG counter
                try:
                    self.out = model.forward(self.ids, normalize)
                finally:
                    model._graph_bump = None
                self.launches_per_replay = ops.LAUNCHES - launches0
            finally:
                ops.STAGE_HOOK = None
                state["g"].capture_end()
                self.graphs.append(state["g"])
            self._reset_python_counters()
            for s in samplers:
                s.counter_dev = None          # the counter's address is baked into the graph; eager calls made while this
                                              # runner is alive keep the documented host-side sequence
        torch.cuda.current_stream(dev).wait_stream(self.stream)
        self.replays = 0
        # the warm-up forwards and the capture pass advanced the device counter through the fused bump; rewind
        self.counter.fill_(self.n_calls * self.first_step)

    def _reset_python_counters(self):
        for s, c in zip(self.samplers, self.base_counters):
            s.counter = c

    def reset(self, replays=0):
        """Next replay behaves like this runner's replay number `replays` (eager step first_step + replays*step_stride)."""
        self.counter.fill_(self.n_calls * (self.first_step + replays * self.step_stride))
        self.replays = replays

    def __call__(self, ids=None, probe_events=None):
        if ids is not None:
            self.ids.copy_(ids.reshape(-1), non_blocking=True)
        for gi, g in enumerate(self.graphs):
            if probe_events is not None and gi == self.probe_index:
                probe_events[0].record()
                g.replay()
                probe_events[1].record()
            else:
                g.replay()
        self.replays += 1
        return self.out

    def close(self):
        for s in self.samplers:
            s.counter_dev = None


class PipelinedForward(object):
    """Host-buffer front end of the hot path: ids come from (pinned) host memory, the result lands in (pinned) host
    memory, and consecutive steps overlap - two CUDA-graph runners alternate on the compute stream while a copy
    stream drains the previous step's result, so the device->host transfer hides behind the next step's kernels.
    Step i reproduces eager forward number i (same RNG counters).

        pipe = model.pipelined(batch_size)
        for i in range(n): pipe.submit(ids_host[i], out_host[i])
        pipe.synchronize()
    """

    def __init__(self, model, batch_size, normalize=True, depth=2):
        dev = model.device
        self.model, self.depth = model, int(depth)
        self.runners = [GraphedForward(model, batch_size, normalize, first_step=r, step_stride=self.depth)
                        for r in range(self.depth)]
        # one compute stream per runner: consecutive steps are independent (own ids / outputs / RNG counter), so the
        # sampler + gather of step i+1 may overlap the GEMM / last layer of step i on SMs the latter leaves idle
        self.computes = [torch.cuda.Stream(device=dev) for _ in range(self.depth)]
        self.compute = self.computes[0]
        self.copy = torch.cuda.Stream(device=dev)
        self.h2d = torch.cuda.Stream(device=dev)
        self.ids_ready = [torch.cuda.Event() for _ in range(self.depth)]
        self.done = [torch.cuda.Event() for _ in range(self.depth)]
        self.drained = [torch.cuda.Event() for _ in range(self.depth)]
        self.step = 0
        import os
        self.use_c_step = os.environ.get("GS_PIPELINE_PY", "0") != "1"     # GS_PIPELINE_PY=1: torch-API path (debug)
        for c in self.computes:
            c.wait_stream(torch.cuda.current_stream(dev))
        for e in self.drained + self.done + self.ids_ready:   # also creates the underlying CUDA events
            e.record(self.compute)

    def _fast_handles(self):
        """Raw CUDA handles for gs_pipeline_step (one C call per step); None if torch does not expose them."""
        if getattr(self, "_handles", None) is None:
            try:
                from ._lib import c_vp
                hs = []
                for r, run in enumerate(self.runners):
                    execs = (c_vp * len(run.graphs))(*[g.raw_cuda_graph_exec() for g in run.graphs])
                    hs.append((execs, len(run.graphs), run.ids.data_ptr(), run.ids.numel() * 4, run.out.data_ptr(),
                               run.out.numel() * 4, self.ids_ready[r].cuda_event, self.done[r].cuda_event,
                               self.drained[r].cuda_event))
                self._handles = hs
            except Exception:
                self._handles = False
        return self._handles

    def submit(self, ids_host, out_host):
        r = self.step % self.depth
        run = self.runners[r]
        hs = self._fast_handles() if self.use_c_step else None
        if ids_host.numel() != run.ids.numel():
            raise ValueError("PipelinedForward.submit: %d ids for a runner captured at batch size %d (pad the last "
                             "batch or build another runner)" % (ids_host.numel(), run.ids.numel()))
        if out_host.numel() != run.out.numel() or out_host.dtype != torch.float32:
            raise ValueError("PipelinedForward.submit: out_host must be float32 with %d elements" % run.out.numel())
        if hs and ids_host.dtype == torch.int32 and not ids_host.is_cuda and ids_host.is_contiguous() \
                and not out_host.is_cuda and out_host.is_contiguous():
            execs, n, ids_dev, ids_bytes, out_dev, out_bytes, ev_ids, ev_done, ev_drained = hs[r]
            ops.check(ops.lib().gs_pipeline_step(ids_host.data_ptr(), ids_dev, ids_bytes, execs, n, out_dev,
                                                 out_host.data_ptr(), out_bytes, self.h2d.cuda_stream,
                                                 self.computes[r].cuda_stream, self.copy.cuda_stream, ev_ids, ev_done,
                                                 ev_drained))
            run.replays += 1
            self.step += 1
            return
        with torch.cuda.stream(self.computes[r]):
            self.computes[r].wait_event(self.drained[r])      # this runner's previous result has left the device
            out = run(ids_host)                               # async H2D of the ids + graph replay
            self.done[r].record(self.computes[r])
        with torch.cuda.stream(self.copy):
            self.copy.wait_event(self.done[r])
            out_host.copy_(out, non_blocking=True)
            self.drained[r].record(self.copy)
        self.step += 1

    def submit_device(self, ids_dev):
        """Device-resident variant: ids already in HBM, result stays in the runner's output buffer (returned)."""
        r = self.step % self.depth
        with torch.cuda.stream(self.computes[r]):
            out = self.runners[r](ids_dev)
        self.step += 1
        return out

    def synchronize(self):
        self.h2d.synchronize()
        for c in self.computes:
            c.synchronize()
        self.copy.synchronize()

    def close(self):
        self.synchronize()
        for run in self.runners:
            run.close()
