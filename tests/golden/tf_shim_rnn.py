"""The recurrent part of the numpy TensorFlow stand-in (tf_shim.py): what the reference's SeqAggregator._call touches
(graphsage/aggregators.py:363-449) on top of the symbols tf_shim.install() provides - tf.contrib.rnn.BasicLSTMCell,
tf.nn.dynamic_rnn with sequence_length, tf.sign / abs / maximum / range / gather.  Each op restates the documented TF
semantics in numpy fp32.

Used ONLY by tests/golden/make_golden_seq.py.  Not product code, not oracle code.
"""
import types

import numpy as np

LSTM_SEED0 = 5000
LSTM_BUILT = 0


def lstm_kernel(seed, shape):
    """glorot-uniform [rows, cols] float32 from RandomState(seed): U(-r, r), r = sqrt(6 / (rows + cols))."""
    r = np.sqrt(6.0 / (shape[0] + shape[1]))
    return np.random.RandomState(seed).uniform(-r, r, size=shape).astype(np.float32)


class BasicLSTMCell(object):
    """tf.contrib.rnn.BasicLSTMCell(num_units), forget_bias 1.0, state (c, h).  The kernel [depth + H, 4H] (gate columns
    i, j, f, o) is drawn glorot-uniform over its full shape when the cell first sees its input depth (get_variable's
    default initialiser); the bias starts at zero.  Both stay readable as .kernel / .bias.  Each kernel comes from its own
    stream, lstm_kernel(seed, shape) with seed = LSTM_SEED0 + the number of cells built before it (kept as .kernel_seed),
    so a fixture can store the seed instead of the [depth + H, 4H] values."""

    def __init__(self, num_units, forget_bias=1.0, **k):
        self.num_units, self.forget_bias = int(num_units), float(forget_bias)
        self.kernel = self.bias = None

    def build(self, depth):
        global LSTM_BUILT
        if self.kernel is None:
            self.kernel_seed = LSTM_SEED0 + LSTM_BUILT
            LSTM_BUILT += 1
            self.kernel = lstm_kernel(self.kernel_seed, (int(depth) + self.num_units, 4 * self.num_units))
            self.bias = np.zeros((4 * self.num_units,), np.float32)

    def zero_state(self, batch_size, dtype):
        z = np.zeros((int(batch_size), self.num_units), dtype=dtype)
        return (z, z.copy())

    def __call__(self, x, state):
        c, h = state
        self.build(x.shape[1])
        gates = np.concatenate([x, h], axis=1) @ self.kernel + self.bias
        i, j, f, o = np.split(gates, 4, axis=1)
        sig = lambda v: (1.0 / (1.0 + np.exp(-v))).astype(np.float32)  # noqa: E731
        c = c * sig(f + np.float32(self.forget_bias)) + sig(i) * np.tanh(j)
        h = np.tanh(c) * sig(o)
        return h, (c, h)


class _Shaped(np.ndarray):
    """an ndarray that also answers get_shape() like a tf.Tensor"""

    def get_shape(self):
        return self.shape


def dynamic_rnn(cell, inputs, sequence_length=None, initial_state=None, dtype=None, time_major=False, **k):
    """batch-major dynamic_rnn: for t >= sequence_length[b] the output is zero and the state is carried unchanged."""
    x = np.asarray(inputs).astype(np.float32)
    B, T = x.shape[0], x.shape[1]
    state = initial_state if initial_state is not None else cell.zero_state(B, np.float32)
    lens = np.full((B,), T) if sequence_length is None else np.asarray(sequence_length).astype(np.int64)
    outs = np.zeros((B, T, cell.num_units), np.float32)
    for t in range(T):
        h, (c2, h2) = cell(x[:, t], state)
        live = (t < lens)[:, None]
        outs[:, t] = np.where(live, h, 0.0)
        state = (np.where(live, c2, state[0]), np.where(live, h2, state[1]))
    return outs.view(_Shaped), state


def install(tf):
    """Add the recurrent symbols to the module tf_shim.install() returned."""
    tf.contrib.rnn = types.SimpleNamespace(BasicLSTMCell=BasicLSTMCell)
    tf.nn.dynamic_rnn = dynamic_rnn
    tf.sign = lambda x: np.sign(np.asarray(x))
    tf.abs = lambda x: np.abs(np.asarray(x))
    tf.maximum = lambda a, b: np.maximum(np.asarray(a), np.asarray(b))
    tf.range = lambda start, limit=None, delta=1: np.arange(start, limit, delta, dtype=np.int32)
    tf.gather = lambda params, indices: np.asarray(params)[np.asarray(indices).astype(np.int64)]
    return tf
