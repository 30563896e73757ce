"""Unsupervised GraphSAGE head around the hot path (SURVEY section 8f row 2; reference
graphsage/models.py:332-405 `_build` / `_loss` / `_accuracy`, graphsage/prediction.py:68-110).

Three passes of the hot path share one set of aggregators (batch1, batch2, and neg_sample_size negatives drawn with
probability ~ degree^0.75 and shared by the whole batch); skip-gram style cross-entropy on the l2-normalised
outputs; MRR of the true pair among the negatives.  Forward through the B200 kernels, backward as in
supervised_models.py.
"""
import numpy as np
import torch

from . import ops
from .models import SampleAndAggregate
from .prediction import BipartiteEdgePredLayer, mrr_from_affinities
from .supervised_models import aggregator_parameters, build_aggregators, differentiable_outputs, weight_decay_term


class UnigramNegativeSampler(object):
    """tf.nn.fixed_unigram_candidate_sampler(unique=False, distortion=0.75, unigrams=degrees) -
    reference graphsage/models.py:336-343.  One Philox call counter per sampler object."""

    def __init__(self, degrees, distortion=0.75, seed=123, device="cuda"):
        w = np.asarray(degrees, dtype=np.float64) ** distortion
        self.cdf = torch.from_numpy(np.cumsum(w)).to(device)
        self.seed, self.counter, self.counter_dev = int(seed), 0, None

    def __call__(self, num_sampled):
        out = ops.sample_unigram(self.cdf, int(num_sampled), self.seed, self.counter, counter_dev=self.counter_dev)
        self.counter += 1
        return out


class UnsupervisedGraphsage(SampleAndAggregate):
    """reference graphsage/models.py:187-405 (SampleAndAggregate with its unsupervised `_build`)."""

    def __init__(self, placeholders, features, adj, degrees, layer_infos, concat=True, aggregator_type="mean",
                 model_size="small", identity_dim=0, neg_sample_size=20, neg_sample_weights=1.0, learning_rate=0.00001,
                 weight_decay=0.0, seed=123, device="cuda", distributed=False, group=None, **kwargs):
        super(UnsupervisedGraphsage, self).__init__(placeholders, features, adj, degrees, layer_infos, concat=concat,
                                                    aggregator_type=aggregator_type, model_size=model_size,
                                                    identity_dim=identity_dim, device=device, **kwargs)
        if aggregator_type not in ("mean", "gcn", "maxpool", "meanpool", "seq"):
            raise NotImplementedError("training is implemented for the mean, gcn, maxpool, meanpool and seq aggregators")
        self.neg_sample_size, self.neg_sample_weights = int(neg_sample_size), float(neg_sample_weights)
        self.learning_rate, self.weight_decay = learning_rate, weight_decay
        self.neg_sampler = UnigramNegativeSampler(degrees, 0.75, seed, device)      # models.py:336-343
        self.aggregators = build_aggregators(self)
        dim_mult = 2 if self.concat else 1
        self.link_pred_layer = BipartiteEdgePredLayer(dim_mult * self.dims[-1], dim_mult * self.dims[-1], placeholders,
                                                      neg_sample_weights=self.neg_sample_weights, bilinear_weights=False,
                                                      device=device, name="edge_predict")      # models.py:362-365
        self.distributed, self.group, self.last_allreduce_bytes = bool(distributed), group, 0
        if self.distributed:                                                         # every rank starts from rank 0's weights
            from .parallel import broadcast_parameters
            broadcast_parameters(self.parameters(), 0, group)
        for p in self.parameters():
            p.requires_grad_(True)
        self.optimizer = torch.optim.Adam(self.parameters(), lr=self.learning_rate)

    def parameters(self):
        return aggregator_parameters(self.aggregators)[0]

    def decayed_parameters(self):
        return aggregator_parameters(self.aggregators)[1]

    def embed(self, batch):
        return differentiable_outputs(self, batch)                                   # models.py:347-370

    def _passes(self, batch1, batch2):
        neg = self.neg_sampler(self.neg_sample_size)
        o1, o2 = self.embed(batch1), self.embed(batch2)
        on = self.embed(neg)                                                         # batch_size = neg_sample_size (:356-360)
        return o1, o2, on, neg

    def loss(self, batch1, batch2):
        """weight decay + BipartiteEdgePredLayer._xent_loss (prediction.py:102-110), divided by the batch size
        (models.py:378)."""
        o1, o2, on, _ = self._passes(batch1, batch2)
        loss = self.link_pred_layer.loss(o1, o2, on)
        if self.weight_decay:
            loss = loss + weight_decay_term(self.decayed_parameters(), self.weight_decay)       # models.py:385-387
        with torch.no_grad():
            self._last = (self.link_pred_layer.affinity(o1, o2), self.link_pred_layer.neg_cost(o1, on))
        return loss / float(o1.shape[0])

    def mrr(self):
        """models.py:393-405 on the affinities of the last loss() call."""
        return mrr_from_affinities(*self._last)

    def train_step(self, batch1, batch2):
        self.optimizer.zero_grad(set_to_none=True)
        loss = self.loss(batch1, batch2)
        loss.backward()
        if self.distributed:                                                         # data parallel: mean gradient over ranks
            from .parallel import allreduce_gradients
            self.last_allreduce_bytes = allreduce_gradients(self.parameters(), self.group)
        for p in self.parameters():
            if p.grad is not None:
                p.grad.clamp_(-5.0, 5.0)                                             # models.py:380-381
        self.optimizer.step()
        return loss.detach()
