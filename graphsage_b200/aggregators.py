"""MeanAggregator / GCNAggregator / MaxPoolingAggregator / MeanPoolingAggregator / SeqAggregator - the surface of
reference graphsage/aggregators.py over the B200 kernels.

Two entry points per aggregator:
  agg((self_vecs[n, in], neigh_vecs[n, k, neigh_in])) -> [n, out * (2 if concat else 1)]
      the reference call convention (dense, already-gathered inputs);
  agg.aggregate_rows(src, segments) -> [rows, out_w]
      the gather-fused form used by SampleAndAggregate.aggregate: neighbours are addressed by
      id lists (or row ranges) into `src`, the [n*k, F] neighbour tensor is never materialised.
"""
import torch

from . import ops
from .inits import glorot, zeros
from .layers import Dense, Layer, act_code, identity, relu  # noqa: F401  (relu/identity re-exported as `act` values)

_DEFAULT_MATH = [ops.MATH_FP32_SIMT]
_MATH_NAMES = {"fp32": ops.MATH_FP32_SIMT, "simt": ops.MATH_FP32_SIMT, "tf32x3": ops.MATH_TF32X3,
               "tf32": ops.MATH_TF32, "bf16": ops.MATH_BF16}


def set_default_math(mode):
    """Arithmetic of the dense contraction for aggregators created afterwards: 'fp32' (CUDA cores),
    'tf32x3' (tcgen05, fp32-accurate), 'tf32', 'bf16'."""
    _DEFAULT_MATH[0] = _MATH_NAMES[mode] if isinstance(mode, str) else int(mode)


def _dropout(x, p):
    return torch.nn.functional.dropout(x, p=float(p), training=True) if p else x


def _dense_segment(n, k):
    return [ops.make_segment(n, k)]


USE_GEMM_IMAGES = [False]     # opt-in: tf32x3 layers hand the gathered rows to the GEMM as tensor-core tile images
                              # (ops.gather_mean_images + ops.sage_gemm_img; bit-identical results).  Measured on the bench step:
                              # the GEMM's A side becomes one bulk copy per K-block, but the gather - the critical kernel -
                              # writes hi + lo images of both parts (55 MB instead of 27 MB): 59.3 us instead of 55.4, and the
                              # pipelined step went from 74.1 to 76.3 us.  Kept off.


class _SageAggregator(Layer):
    def _image_layer(self, src, segments, parts, combine, include_self, want_self):
        """gather + mean -> tile images -> tcgen05 GEMM (tf32x3); None when the image form does not apply."""
        code, post = act_code(self.act)
        if not USE_GEMM_IMAGES[0] or self.math != ops.MATH_TF32X3 or post is not None or self.dropout \
                or any(K != src.shape[1] for (_, K, _) in parts):
            return None
        res = ops.gather_mean_images(src, segments, include_self=include_self, want_self=want_self)
        if res is None:
            return None
        images, rows = res
        if getattr(self, "_packed", None) is None:
            self._packed = ops.PackedWeights()
        return ops.sage_gemm_img(rows, images, parts, combine=combine, bias=self.vars.get("bias"), act=code,
                                 packed=self._packed)

    def _finish(self, parts, combine):
        code, post = act_code(self.act)
        if getattr(self, "_packed", None) is None:
            self._packed = ops.PackedWeights()
        y = ops.sage_gemm(parts, combine=combine, bias=self.vars.get("bias"), act=code, math=self.math,
                          packed=self._packed)
        return post(y) if post else y

    def _small_layer(self, src, segments, parts, combine, include_self, final):
        """Whole layer in one launch when it is small (last layers: B rows).  Returns None if not applicable."""
        code, post = act_code(self.act)
        if (len(segments) != 1 or not torch.is_tensor(src) or post is not None or self.dropout
                or segments[0].out_row0 + segments[0].n > ops.SMALL_LAYER_MAX_ROWS or src.shape[1] > 2048
                or any(K != src.shape[1] for (_, K, _) in parts)
                or (sum(B.shape[1] for (_, _, B) in parts) if combine == ops.COMBINE_CONCAT else parts[0][2].shape[1]) > 1024):
            return None       # gs_sage_layer_small limits: rows, K <= 2048, total output width <= 1024
        l2 = bool(final and final.get("l2_normalize"))
        bump = final.get("bump") if final else None
        y = ops.sage_layer_small(src, segments[0], parts, combine=combine, include_self=include_self,
                                 bias=self.vars.get("bias"), act=code, l2_normalize=l2,
                                 counter_dev=None if bump is None else bump[0], counter_inc=0 if bump is None else bump[1])
        if final is not None:
            final["normalized"] = l2
            final["bumped"] = bump is not None
        return y

    @property
    def output_width(self):
        return self.output_dim * (2 if (self.concat and "self_weights" in self.vars) else 1)


class MeanAggregator(_SageAggregator):
    """act(concat_or_add(self @ self_weights, mean_k(neigh) @ neigh_weights)) - aggregators.py:43-64."""

    def __init__(self, input_dim, output_dim, neigh_input_dim=None, dropout=0., bias=False, act=relu, name=None,
                 concat=False, device="cuda", **kwargs):
        super(MeanAggregator, self).__init__(**kwargs)
        self.dropout = dropout
        self.bias = bias
        self.act = act
        self.concat = concat
        if neigh_input_dim is None:
            neigh_input_dim = input_dim
        self.vars["neigh_weights"] = glorot([neigh_input_dim, output_dim], name="neigh_weights", device=device)
        self.vars["self_weights"] = glorot([input_dim, output_dim], name="self_weights", device=device)
        if self.bias:   # the reference dereferences self.output_dim too early here (aggregators.py:34-35); fixed, not replicated
            self.vars["bias"] = zeros([output_dim * (2 if concat else 1)], name="bias", device=device)
        self.input_dim = input_dim
        self.output_dim = output_dim
        self.neigh_input_dim = neigh_input_dim
        self.math = _DEFAULT_MATH[0]

    def _combine(self):
        return ops.COMBINE_CONCAT if self.concat else ops.COMBINE_ADD

    def _call(self, inputs):
        self_vecs, neigh_vecs = inputs
        n, k, d = neigh_vecs.shape
        neigh_vecs = _dropout(neigh_vecs, self.dropout)
        self_vecs = _dropout(self_vecs, self.dropout)
        _, means = ops.gather_mean(neigh_vecs.reshape(n * k, d), _dense_segment(n, k), want_self=False)
        return self._finish([(self_vecs, self.input_dim, self.vars["self_weights"]),
                             (means, self.neigh_input_dim, self.vars["neigh_weights"])], self._combine())

    def aggregate_rows(self, src, segments, final=None, src_persistent=False):
        if self.dropout:
            raise NotImplementedError("dropout > 0 uses the dense call path")
        y = self._small_layer(src, segments, [(None, self.input_dim, self.vars["self_weights"]),
                                              (None, self.neigh_input_dim, self.vars["neigh_weights"])],
                              self._combine(), False, final)
        if y is not None:
            return y
        y = self._image_layer(src, segments, [(None, self.input_dim, self.vars["self_weights"]),
                                              (None, self.neigh_input_dim, self.vars["neigh_weights"])],
                              self._combine(), False, True)
        if y is not None:
            return y
        xs, xm = ops.gather_mean(src, segments, want_self=True)
        return self._finish([(xs, self.input_dim, self.vars["self_weights"]),
                             (xm, self.neigh_input_dim, self.vars["neigh_weights"])], self._combine())


class GCNAggregator(_SageAggregator):
    """act(mean_{k+1}(neigh U self) @ weights) - aggregators.py:101-116 (single weight, concat ignored)."""

    def __init__(self, input_dim, output_dim, neigh_input_dim=None, dropout=0., bias=False, act=relu, name=None,
                 concat=False, device="cuda", **kwargs):
        super(GCNAggregator, self).__init__(**kwargs)
        self.dropout = dropout
        self.bias = bias
        self.act = act
        self.concat = concat
        if neigh_input_dim is None:
            neigh_input_dim = input_dim
        self.vars["weights"] = glorot([neigh_input_dim, output_dim], name="neigh_weights", device=device)
        if self.bias:
            self.vars["bias"] = zeros([output_dim], name="bias", device=device)
        self.input_dim = input_dim
        self.output_dim = output_dim
        self.neigh_input_dim = neigh_input_dim
        self.math = _DEFAULT_MATH[0]

    def _call(self, inputs):
        self_vecs, neigh_vecs = inputs
        n, k, d = neigh_vecs.shape
        if self_vecs.shape[1] != d:
            raise ValueError("GCNAggregator needs self and neighbour vectors of equal width")
        neigh_vecs = _dropout(neigh_vecs, self.dropout)
        self_vecs = _dropout(self_vecs, self.dropout)
        # one source matrix: neighbours first, then the self rows
        src = torch.cat([neigh_vecs.reshape(n * k, d), self_vecs], dim=0)
        seg = [ops.make_segment(n, k, self_row0=n * k, neigh_row0=0)]
        _, means = ops.gather_mean(src, seg, include_self=True, want_self=False)
        return self._finish([(means, self.neigh_input_dim, self.vars["weights"])], ops.COMBINE_ADD)

    def aggregate_rows(self, src, segments, final=None, src_persistent=False):
        if self.dropout:
            raise NotImplementedError("dropout > 0 uses the dense call path")
        y = self._small_layer(src, segments, [(None, self.neigh_input_dim, self.vars["weights"])], ops.COMBINE_ADD, True,
                              final)
        if y is not None:
            return y
        y = self._image_layer(src, segments, [(None, self.neigh_input_dim, self.vars["weights"])], ops.COMBINE_ADD, True, False)
        if y is not None:
            return y
        _, means = ops.gather_mean(src, segments, include_self=True, want_self=False)
        return self._finish([(means, self.neigh_input_dim, self.vars["weights"])], ops.COMBINE_ADD)


class MaxPoolingAggregator(_SageAggregator):
    """act(concat_or_add(self @ Ws, max_k(relu(neigh @ Wm + bm)) @ Wn)) - aggregators.py:119-195,
    with Dense (layers.py:73-116) as the single MLP layer; hidden 512 ("small") / 1024 ("big")."""

    def __init__(self, input_dim, output_dim, model_size="small", neigh_input_dim=None, dropout=0., bias=False,
                 act=relu, name=None, concat=False, device="cuda", **kwargs):
        super(MaxPoolingAggregator, self).__init__(**kwargs)
        self.dropout = dropout
        self.bias = bias
        self.act = act
        self.concat = concat
        if neigh_input_dim is None:
            neigh_input_dim = input_dim
        if model_size == "small":
            hidden_dim = self.hidden_dim = 512
        elif model_size == "big":
            hidden_dim = self.hidden_dim = 1024
        else:
            raise ValueError("model_size must be 'small' or 'big'")
        self.math = _DEFAULT_MATH[0]
        self.mlp_layers = [Dense(input_dim=neigh_input_dim, output_dim=hidden_dim, act=relu, dropout=dropout,
                                 sparse_inputs=False, logging=self.logging, device=device, math=self.math)]
        self.vars["neigh_weights"] = glorot([hidden_dim, output_dim], name="neigh_weights", device=device)
        self.vars["self_weights"] = glorot([input_dim, output_dim], name="self_weights", device=device)
        if self.bias:
            self.vars["bias"] = zeros([output_dim * (2 if concat else 1)], name="bias", device=device)
        self.input_dim = input_dim
        self.output_dim = output_dim
        self.neigh_input_dim = neigh_input_dim

    def _combine(self):
        return ops.COMBINE_CONCAT if self.concat else ops.COMBINE_ADD

    pool = "max"

    def _pool(self, rows, n, k):
        h = rows
        for layer in self.mlp_layers:
            layer.math = self.math
            h = layer(h)
        if self.pool == "mean":
            return ops.gather_mean(h, [ops.Seg(n, k)], want_self=False, out_pitch=h.shape[1])[1]
        return ops.segment_max(h, n, k)

    def _call(self, inputs):
        self_vecs, neigh_vecs = inputs
        n, k, d = neigh_vecs.shape
        hmax = self._pool(neigh_vecs.reshape(n * k, d), n, k)
        return self._finish([(self_vecs, self.input_dim, self.vars["self_weights"]),
                             (hmax, self.hidden_dim, self.vars["neigh_weights"])], self._combine())

    def _bf16_table(self, src, persistent):
        """K4's operand table: bf16 rows with a 16-byte-multiple pitch.  A bf16 source is used as is.  An fp32 source is
        cast by gs_cast_rows_bf16 - once per tensor version when the caller says it is the persistent feature table
        (layer 0), on EVERY call otherwise: intermediate activations are fresh torch.empty buffers the C library
        fills, so neither their address nor their _version tells one step's values from the next."""
        if src.dtype == torch.bfloat16:
            if src.stride(0) % 8 != 0 or src.data_ptr() % 16 != 0:
                raise ValueError("bfloat16 source rows must be 16-byte aligned multiples (pitch % 8 == 0)")
            return src
        if not persistent:
            return ops.cast_rows_bf16(src)
        key = (src.data_ptr(), src._version, tuple(src.shape))
        if getattr(self, "_bf16_ref", None) is not src or getattr(self, "_bf16_key", None) != key:
            self._bf16_src, self._bf16_ref, self._bf16_key = ops.cast_rows_bf16(src), src, key
        return self._bf16_src

    def _fused_ok(self, src, segments):
        return (self.math == ops.MATH_BF16 and torch.is_tensor(src) and not self.dropout and len(self.mlp_layers) == 1
                and self.neigh_input_dim <= 640 and self.hidden_dim % 128 == 0 and all(s.k <= 128 for s in segments)
                and self.mlp_layers[0].act is relu and "bias" in self.mlp_layers[0].vars)

    def aggregate_rows(self, src, segments, final=None, src_persistent=False):
        rows = max(s.out_row0 + s.n for s in segments)
        dev = src.device
        if self._fused_ok(src, segments):
            # K4: gather -> MLP -> ReLU -> max over the fanout in one tcgen05 kernel per hop (bf16 operands).
            # Every launch of this branch is one of the library's kernels (no torch copy / convert kernels in the step).
            table = self._bf16_table(src, src_persistent)
            if getattr(self, "_packed_mlp", None) is None:
                self._packed_mlp = ops.PackedMlpWeights()
            mlp = self.mlp_layers[0]
            F_in = src.shape[1]
            hmax = torch.empty((rows, self.hidden_dim), dtype=torch.float32, device=dev)
            for s in segments:
                ops.maxpool_mlp_fused(table, s.n, s.k, mlp.vars["weights"], mlp.vars["bias"], self._packed_mlp,
                                      row_ids=s.neigh_ids, row0=s.neigh_row0, K=self.neigh_input_dim,
                                      out=hmax[s.out_row0:s.out_row0 + s.n], pool=self.pool)
            s0 = segments[0]
            if len(segments) == 1 and s0.self_ids is None and s0.out_row0 == 0 and src.dtype == torch.float32:
                xs = src[s0.self_row0:s0.self_row0 + s0.n]         # the self rows are already a dense fp32 row range
            else:
                xs = torch.empty((rows, ops.pad_cols(F_in)), dtype=torch.float32, device=dev)[:, :F_in]
                for s in segments:
                    ops.gather_rows_f32(src, ids=None if s.self_ids is None else s.self_ids[:s.n], row0=s.self_row0,
                                        n=s.n, out=xs[s.out_row0:s.out_row0 + s.n])
            return self._finish([(xs, self.input_dim, self.vars["self_weights"]),
                                 (hmax, self.hidden_dim, self.vars["neigh_weights"])], self._combine())
        # materialised form (fp32 / tf32 arithmetic, fanout > 128, wide inputs, sharded tables): the MLP is a plain GEMM over
        # the gathered neighbour rows (widened to fp32 when the table is bf16), then the pooling kernel
        xs = torch.empty((rows, ops.pad_cols(src.shape[1])), dtype=torch.float32, device=dev)[:, :src.shape[1]]
        hmax = torch.empty((rows, self.hidden_dim), dtype=torch.float32, device=dev)
        widen = torch.is_tensor(src) and src.dtype != torch.float32
        for s in segments:
            n, k = s.n, s.k
            if widen:
                nrows = ops.gather_rows_f32(src, ids=None if s.neigh_ids is None else s.neigh_ids[:n * k],
                                            row0=s.neigh_row0, n=n * k)
                ops.gather_rows_f32(src, ids=None if s.self_ids is None else s.self_ids[:n], row0=s.self_row0, n=n,
                                    out=xs[s.out_row0:s.out_row0 + n])
                hmax[s.out_row0:s.out_row0 + n] = self._pool(nrows, n, k)
                continue
            if s.neigh_ids is not None:
                nrows = ops.gather_rows(src, s.neigh_ids[:n * k])
            else:
                nrows = src[s.neigh_row0:s.neigh_row0 + n * k]
            hmax[s.out_row0:s.out_row0 + n] = self._pool(nrows, n, k)
            if s.self_ids is not None:
                ops.gather_rows(src, s.self_ids[:n], out=xs[s.out_row0:s.out_row0 + n])
            else:
                xs[s.out_row0:s.out_row0 + n] = src[s.self_row0:s.self_row0 + n]
        return self._finish([(xs, self.input_dim, self.vars["self_weights"]),
                             (hmax, self.hidden_dim, self.vars["neigh_weights"])], self._combine())


class SeqAggregator(_SageAggregator):
    """act(concat_or_add(self @ Ws, h_{len-1} @ Wn)) with h the outputs of an LSTM run over the neighbour rows in sampled
    order - reference graphsage/aggregators.py:363-449.  BasicLSTMCell(H), H = 128 ("small") / 256 ("big"); len = the
    number of non-zero neighbour rows (at least 1), and the LSTM consumes the FIRST len rows (dynamic_rnn's
    sequence_length), zero rows included.

    The cell's kernel [neigh_in + H, 4H] (gate columns i, j, f, o) and bias [4H] live in `cell_vars`, not in `vars`: the
    reference keeps them in the cell, so they are trained but not weight-decayed.  Like the reference, the aggregator
    stores `dropout` but never applies it.  Kernels per hop: gather of the neighbour rows (layer 0), the input projection
    on gs_sage_gemm, gs_lstm_seq for the recurrence, then gs_sage_gemm for the two matmuls, combine, bias and act."""

    def __init__(self, input_dim, output_dim, model_size="small", neigh_input_dim=None, dropout=0., bias=False,
                 act=relu, name=None, concat=False, device="cuda", **kwargs):
        super(SeqAggregator, self).__init__(**kwargs)
        self.dropout = dropout
        self.bias = bias
        self.act = act
        self.concat = concat
        if neigh_input_dim is None:
            neigh_input_dim = input_dim
        if model_size == "small":
            hidden_dim = self.hidden_dim = 128
        elif model_size == "big":
            hidden_dim = self.hidden_dim = 256
        else:
            raise ValueError("model_size must be 'small' or 'big'")
        self.vars["neigh_weights"] = glorot([hidden_dim, output_dim], name="neigh_weights", device=device)
        self.vars["self_weights"] = glorot([input_dim, output_dim], name="self_weights", device=device)
        if self.bias:   # the reference reads self.output_dim before setting it here (aggregators.py:394-395); fixed
            self.vars["bias"] = zeros([output_dim * (2 if concat else 1)], name="bias", device=device)
        # BasicLSTMCell variables: TF's get_variable default (glorot uniform over the full shape), zero bias
        self.cell_vars = {"kernel": glorot([neigh_input_dim + hidden_dim, 4 * hidden_dim], name="kernel", device=device),
                          "bias": zeros([4 * hidden_dim], name="bias", device=device)}
        self.input_dim = input_dim
        self.output_dim = output_dim
        self.neigh_input_dim = neigh_input_dim
        self.math = _DEFAULT_MATH[0]

    def parameters(self):
        return list(self.vars.values()) + list(self.cell_vars.values())

    def _combine(self):
        return ops.COMBINE_CONCAT if self.concat else ops.COMBINE_ADD

    def _cell_weights(self):
        kernel = self.cell_vars["kernel"]
        return kernel[:self.neigh_input_dim], kernel[self.neigh_input_dim:]

    def _project(self, x):
        """P = x @ kernel[:neigh_in] + cell bias: the input half of every gate pre-activation, for all steps at once."""
        if getattr(self, "_packed_cell", None) is None:
            self._packed_cell = ops.PackedWeights()
        Wx, _ = self._cell_weights()
        return ops.sage_gemm([(x, self.neigh_input_dim, Wx)], bias=self.cell_vars["bias"], act=ops.ACT_NONE,
                             math=self.math, packed=self._packed_cell)

    def _call(self, inputs):
        self_vecs, neigh_vecs = inputs                      # dropout is stored but not applied (aggregators.py:405-449)
        n, k, d = neigh_vecs.shape
        x = neigh_vecs.reshape(n * k, d)
        if x.stride(1) != 1:
            x = x.contiguous()
        used = ops.row_used(x)
        neigh_h = ops.lstm_seq(self._project(x), self._cell_weights()[1], used, n, k)
        return self._finish([(self_vecs, self.input_dim, self.vars["self_weights"]),
                             (neigh_h, self.hidden_dim, self.vars["neigh_weights"])], self._combine())

    def _used_table(self, src, persistent):
        """used[] over the source rows.  The feature table (layer 0) is scanned once per tensor version, as
        MaxPoolingAggregator._bf16_table casts it; intermediate activations are fresh buffers, scanned on every call."""
        if not persistent:
            return ops.row_used(src)
        key = (src.data_ptr(), src._version, tuple(src.shape))
        if getattr(self, "_used_ref", None) is not src or getattr(self, "_used_key", None) != key:
            self._used, self._used_ref, self._used_key = ops.row_used(src), src, key
        return self._used

    def neighbour_rows(self, src, s):
        """The n*k neighbour rows of segment s as an fp32 matrix (a view of src for range-addressed rows)."""
        n, k = s.n, s.k
        if s.neigh_ids is None and src.dtype == torch.float32:
            return src[s.neigh_row0:s.neigh_row0 + n * k]
        F = src.shape[1]
        x = torch.empty((n * k, ops.pad_cols(F)), dtype=torch.float32, device=src.device)[:, :F]
        if src.dtype == torch.float32:
            return ops.gather_rows(src, s.neigh_ids[:n * k], out=x)
        return ops.gather_rows_f32(src, ids=None if s.neigh_ids is None else s.neigh_ids[:n * k], row0=s.neigh_row0,
                                   n=n * k, out=x)

    def self_rows(self, src, segments, rows):
        s0 = segments[0]
        if len(segments) == 1 and s0.self_ids is None and s0.out_row0 == 0 and src.dtype == torch.float32:
            return src[s0.self_row0:s0.self_row0 + s0.n]         # the self rows are already a dense fp32 row range
        F = src.shape[1]
        xs = torch.empty((rows, ops.pad_cols(F)), dtype=torch.float32, device=src.device)[:, :F]
        for s in segments:
            ops.gather_rows_f32(src, ids=None if s.self_ids is None else s.self_ids[:s.n], row0=s.self_row0, n=s.n,
                                out=xs[s.out_row0:s.out_row0 + s.n])
        return xs

    def aggregate_rows(self, src, segments, final=None, src_persistent=False):
        if hasattr(src, "c_table"):
            raise NotImplementedError("the seq aggregator does not read node-partitioned (sharded) feature tables")
        rows = max(s.out_row0 + s.n for s in segments)
        used = self._used_table(src, src_persistent)
        Wh = self._cell_weights()[1]
        neigh_h = torch.empty((rows, self.hidden_dim), dtype=torch.float32, device=src.device)
        for s in segments:
            P = self._project(self.neighbour_rows(src, s))
            ops.lstm_seq(P, Wh, used, s.n, s.k, row_ids=None if s.neigh_ids is None else s.neigh_ids[:s.n * s.k],
                         row0=s.neigh_row0,
                         out=neigh_h[s.out_row0:s.out_row0 + s.n])
        return self._finish([(self.self_rows(src, segments, rows), self.input_dim, self.vars["self_weights"]),
                             (neigh_h, self.hidden_dim, self.vars["neigh_weights"])], self._combine())


class MeanPoolingAggregator(MaxPoolingAggregator):
    """act(concat_or_add(self @ Ws, mean_k(relu(neigh @ Wm + bm)) @ Wn)) - reference graphsage/aggregators.py:197-273.
    Same kernels as the max-pool aggregator with the pooling operator swapped (SURVEY section 8f row 4)."""
    pool = "mean"
