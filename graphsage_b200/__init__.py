"""graphsage_b200 - a B200-native (sm_100a) sample-and-aggregate engine behind the
graphsage.neigh_samplers / graphsage.aggregators / graphsage.models.SampleAndAggregate surface of
williamleif/GraphSAGE.  `import graphsage_b200 as graphsage` is the intended drop-in for that path.

All compute goes through libgraphsage_b200.so (include/graphsage_b200.h); there is no CPU fallback.
"""
from . import _lib, aggregators, graph, inits, layers, minibatch, models, neigh_samplers, ops, prediction, utils  # noqa: F401
from .aggregators import (GCNAggregator, MaxPoolingAggregator, MeanAggregator, MeanPoolingAggregator,  # noqa: F401
                          SeqAggregator, set_default_math)
from .layers import Dense, Layer, identity, relu  # noqa: F401
from .models import SAGEInfo, SampleAndAggregate  # noqa: F401
from .neigh_samplers import CSRNeighborSampler, UniformNeighborSampler  # noqa: F401
from .prediction import BipartiteEdgePredLayer  # noqa: F401
from .supervised_models import SupervisedGraphsage  # noqa: F401
from .unsupervised_models import UnigramNegativeSampler, UnsupervisedGraphsage  # noqa: F401

__version__ = "0.1.0"
