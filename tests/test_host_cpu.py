"""CPU: host-side logic and the C-ABI surface (no compute kernels are launched)."""
import os
import re

import numpy as np
import pytest

import oracle
from conftest import ROOT, load_golden


@pytest.fixture(scope="module")
def built_lib():
    from graphsage_b200.build import build_library
    return build_library()


def test_library_exports_every_declared_symbol(built_lib):
    import ctypes
    header = open(os.path.join(ROOT, "include", "graphsage_b200.h")).read()
    declared = set(re.findall(r"\b(gs_[a-z0-9_]+)\s*\(", header))
    declared -= {"gs_status", "gs_dtype"}
    assert len(declared) >= 12
    lib = ctypes.CDLL(built_lib)
    for name in sorted(declared):
        assert hasattr(lib, name), "symbol %s declared in the header but not exported" % name
    from graphsage_b200 import _lib
    assert set(_lib.exported_symbols()) == declared
    assert _lib.lib().gs_version() == 2


def test_perm_prefix_host_matches_oracle(built_lib):
    from graphsage_b200 import _lib
    for seed, counter, md, k in [(123, 0, 128, 10), (123, 1, 128, 25), (5, 2**40 + 3, 100, 100), (2**63 + 9, 7, 8, 8),
                                 (1, 1, 1, 1), (3, 3, 16, 0)]:
        assert _lib.perm_prefix_host(seed, counter, md, k) == [int(x) for x in oracle.perm_prefix(seed, counter, md, k)]
    with pytest.raises(RuntimeError, match="max_deg"):
        _lib.perm_prefix_host(1, 1, 8, 9)


def test_no_cpu_fallback(built_lib):
    import torch
    import graphsage_b200 as gs
    adj = torch.zeros((4, 4), dtype=torch.int32)
    with pytest.raises(RuntimeError, match="CUDA-only"):     # host tensors are refused with or without a GPU
        gs.ops.sample_padded(adj, torch.zeros(2, dtype=torch.int32), 2, 1, 0)
    if not torch.cuda.is_available():
        with pytest.raises((RuntimeError, AssertionError)):
            gs.MeanAggregator(4, 4, device="cuda")  # weights live on the GPU; no CPU construction path


def test_layer_kwarg_whitelist_and_names(built_lib):
    from graphsage_b200.layers import Layer
    a, b = Layer(), Layer()
    assert a.name.startswith("layer_") and a.name != b.name and a.vars == {}
    assert Layer(name="x", logging=True, model_size="big").name == "x"
    with pytest.raises(AssertionError, match="Invalid keyword argument"):
        Layer(bogus=1)


def test_construct_adj_matches_reference_under_shim():
    from graphsage_b200.minibatch import construct_adj, construct_test_adj
    g = load_golden("adjacency")
    order = [int(x) for x in g["node_order"]]
    n = len(order)
    ptr = g["nb_ptr"]
    # CSR over node index, in each node's neighbour iteration order
    indptr = np.zeros(n + 1, dtype=np.int64)
    rows = {}
    for pos, u in enumerate(order):
        rows[u] = (g["nb_idx"][ptr[pos]:ptr[pos + 1]], g["nb_removed"][ptr[pos]:ptr[pos + 1]], bool(g["val_or_test"][pos]))
    idx, rem, skip = [], [], np.zeros(n, bool)
    for u in range(n):
        indptr[u + 1] = indptr[u] + len(rows[u][0])
        idx.append(rows[u][0]); rem.append(rows[u][1]); skip[u] = rows[u][2]
    idx, rem = np.concatenate(idx), np.concatenate(rem)
    rng = np.random.RandomState(123)
    adj, deg = construct_adj(indptr, idx, int(g["max_degree"]), skip, rem, order, rng)
    test_adj = construct_test_adj(indptr, idx, int(g["max_degree"]), order, rng)
    np.testing.assert_array_equal(adj, g["adj"])
    np.testing.assert_array_equal(deg, g["deg"])
    np.testing.assert_array_equal(test_adj, g["test_adj"])


def test_padded_from_csr_fast_properties():
    from graphsage_b200.minibatch import padded_from_csr_fast
    from graphsage_b200.synthetic import community_graph_csr
    indptr, indices, comm = community_graph_csr(3000, n_comm=5, mean_deg=20, seed=1)
    md = 16
    adj, deg = padded_from_csr_fast(indptr, indices, md, seed=2)
    n = 3000
    assert adj.shape == (n + 1, md) and adj.dtype == np.int32 and (adj[n] == n).all()
    for u in range(0, n, 37):
        nb = set(indices[indptr[u]:indptr[u + 1]].tolist())
        if not nb:
            assert (adj[u] == n).all()
            continue
        assert set(adj[u].tolist()) <= nb
        if len(nb) >= md:
            assert len(set(adj[u].tolist())) == md
    # symmetric, no self loops
    a = np.repeat(np.arange(n), np.diff(indptr))
    assert (a != indices).all()
    fwd = set(zip(a[:2000].tolist(), indices[:2000].tolist()))
    allp = set(zip(a.tolist(), indices.tolist()))
    assert all((v, u) in allp for (u, v) in fwd)


def test_rmat_generator_properties():
    from graphsage_b200.synthetic import rmat_csr
    indptr, indices = rmat_csr(12, edge_factor=8, seed=5)
    n = 1 << 12
    assert indptr.shape == (n + 1,) and indptr[0] == 0 and indptr[-1] == len(indices) and indices.dtype == np.int32
    deg = np.diff(indptr)
    assert 0.5 * 8 * n < len(indices) <= 8 * n                    # duplicates and self loops removed
    for u in (0, 1, 17, n - 1):                                   # sorted, unique, no self loop
        row = indices[indptr[u]:indptr[u + 1]]
        assert np.all(np.diff(row) > 0) and u not in row
    assert deg.max() > 20 * deg.mean()                            # the skew R-MAT is used for
    assert deg[:n // 2].sum() > 2.5 * deg[n // 2:].sum()          # a + b = 0.76 of the mass on the low half of the sources
    again = rmat_csr(12, edge_factor=8, seed=5)
    assert np.array_equal(again[0], indptr) and np.array_equal(again[1], indices)
    ip2, ix2 = rmat_csr(12, edge_factor=8, seed=5, n_nodes=3000, undirected=True, chunk=5000)
    assert ip2.shape == (3001,) and ix2.max() < 3000
    und = set(zip(np.repeat(np.arange(3000), np.diff(ip2)).tolist(), ix2.tolist()))
    assert all((v, u) in und for (u, v) in list(und)[:2000])      # symmetric


def test_rmat_oracle_properties():
    """the R-MAT oracle (config 5's graph): mean degree = edge_factor, no self loops, ids in range, hubs scrambled, and the
    row marginal it is built from: a node's expected degree follows (a+b)^zeros (c+d)^ones of its R-MAT id"""
    import oracle
    n = 1 << 12
    indptr, indices = oracle.rmat.rmat_csr(12, n, 16.0, seed=5)
    deg = np.diff(indptr)
    assert abs(indptr[-1] / float(n) - 16.0) < 0.2
    assert indices.min() >= 0 and indices.max() < n
    assert not (np.repeat(np.arange(n), deg) == indices).any()
    mul, mul_inv, add = oracle.rmat.scramble_constants(n)
    assert (mul * mul_inv) % n == 1
    r = ((np.arange(n) - add) % n) * mul_inv % n                     # R-MAT id behind every output row
    ones = np.array([bin(int(x)).count("1") for x in r])
    lam = 16.0 * n * (0.76 ** (12 - ones)) * (0.24 ** ones)
    assert np.all(np.abs(deg - lam) < 1.0 + 1e-9)                     # stochastic rounding of the expectation
    indeg = np.bincount(indices, minlength=n)
    assert np.corrcoef(np.log1p(indeg), np.log1p(deg))[0, 1] > 0.8    # b == c: the column marginal mirrors the row marginal
