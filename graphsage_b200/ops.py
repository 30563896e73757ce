"""Functional wrappers: torch CUDA tensors in, torch CUDA tensors out, all work done by
libgraphsage_b200.so on the current CUDA stream.  torch only owns memory and streams here."""
import torch

from . import _lib
from ._lib import (ACT_NONE, ACT_RELU, COMBINE_ADD, COMBINE_CONCAT, MATH_FP32_SIMT, MATH_TF32X3, MATH_TF32,
                   MATH_BF16, GemmPart, Segment, check, lib, ptr, require_cuda, stream_ptr)

_U64 = 2**64 - 1

# optional per-kernel timing (bench.py): name -> list of (start_event, end_event) on the current stream
PROBE = None
LAUNCHES = 0          # kernels of ours launched through this module (bench.py reports it as gpu_launches)
STAGE_HOOK = None     # callable(name, "pre"|"post") around probe-able launches (models.GraphedForward splits graphs here)


def _probe(name):
    if STAGE_HOOK is not None:
        STAGE_HOOK(name, "pre")
    if PROBE is None:
        return _PostHook(name) if STAGE_HOOK is not None else None
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    PROBE.setdefault(name, []).append((e0, e1))
    e0.record()
    return e1


class _PostHook(object):
    def __init__(self, name):
        self.name = name

    def record(self):
        if STAGE_HOOK is not None:
            STAGE_HOOK(self.name, "post")


def _launched(n=1, ev=None):
    global LAUNCHES
    LAUNCHES += n
    if ev is not None:
        ev.record()


def pad_cols(f):
    return (int(f) + 7) // 8 * 8


def _i32(t, name):
    if t.dtype != torch.int32:
        raise TypeError("%s must be int32 (got %s)" % (name, t.dtype))
    return t.contiguous()


def sample_padded(adj, ids, k, seed, counter, col_perm=None, counter_dev=None, out=None):
    """UniformNeighborSampler._call - reference graphsage/neigh_samplers.py:24-29."""
    require_cuda(adj, ids, col_perm, counter_dev)
    adj, ids = _i32(adj, "adj"), _i32(ids.reshape(-1), "ids")
    n = ids.numel()
    if out is None:
        out = torch.empty((n, k), dtype=torch.int32, device=adj.device)
    ev = _probe("sample_padded")
    check(lib().gs_sample_padded(ptr(adj), adj.shape[0], adj.shape[1], ptr(ids), n, k, ptr(col_perm), seed & _U64,
                                 counter & _U64, ptr(counter_dev), ptr(out), stream_ptr()))
    _launched(1 if n * k else 0, ev)
    return out


def sample_padded_khop(adj, seeds, fanouts, seed, counter, counter_dev=None):
    """SampleAndAggregate.sample's whole frontier expansion (reference models.py:254-275) in one launch.
    fanouts in HOP order ([10, 25]); returns [hop1 ids, hop2 ids, ...] (flat int32), bit-identical to successive
    sample_padded calls with counters counter, counter+1, ..."""
    require_cuda(adj, seeds, counter_dev)
    adj, seeds = _i32(adj, "adj"), _i32(seeds.reshape(-1), "seeds")
    n = seeds.numel()
    outs, cnt = [], n
    for k in fanouts:
        cnt *= int(k)
        outs.append(torch.empty((cnt,), dtype=torch.int32, device=adj.device))
    fan = (_lib.c_i32 * len(fanouts))(*[int(k) for k in fanouts])
    optr = (_lib.c_vp * len(fanouts))(*[ptr(o) for o in outs])
    ev = _probe("sample_padded_khop")
    check(lib().gs_sample_padded_khop(ptr(adj), adj.shape[0], adj.shape[1], ptr(seeds), n, fan, len(fanouts),
                                      seed & _U64, counter & _U64, ptr(counter_dev), optr, stream_ptr()))
    _launched(1 if n else 0, ev)
    return outs


def build_padded_adj(indptr, indices, max_degree, seed=123, counter=0, skip=None):
    """Padded adjacency [N+1, max_degree] (+ degree vector) from CSR on the device - the sampler's input contract,
    reference graphsage/minibatch.py:227-259.  skip: optional bool/uint8 [N] (val/test nodes keep all-N rows)."""
    require_cuda(indptr, indices, skip)
    if indptr.dtype != torch.int64:
        raise TypeError("indptr must be int64")
    indices = _i32(indices, "indices")
    n = indptr.numel() - 1
    adj = torch.empty((n + 1, max_degree), dtype=torch.int32, device=indptr.device)
    deg = torch.empty((n,), dtype=torch.float32, device=indptr.device)
    sk = None if skip is None else skip.to(torch.uint8).contiguous()
    check(lib().gs_build_padded_adj(ptr(indptr), ptr(indices), n, max_degree, ptr(sk), seed & _U64, counter & _U64,
                                    ptr(adj), ptr(deg), stream_ptr()))
    _launched(1)
    return adj, deg


def sample_unigram(cdf, num_sampled, seed, counter, counter_dev=None):
    """tf.nn.fixed_unigram_candidate_sampler(unique=False) - reference graphsage/models.py:336-343.
    cdf: float64 CUDA tensor, inclusive prefix sum of the (distorted) unigram weights."""
    require_cuda(cdf, counter_dev)
    if cdf.dtype != torch.float64:
        raise TypeError("cdf must be float64")
    out = torch.empty((num_sampled,), dtype=torch.int32, device=cdf.device)
    check(lib().gs_sample_unigram(ptr(cdf), cdf.numel(), num_sampled, seed & _U64, counter & _U64, ptr(counter_dev),
                                  ptr(out), stream_ptr()))
    _launched(1 if num_sampled else 0)
    return out


def sample_csr(indptr, indices, ids, k, seed, counter, replace_if_short=True, pad_id=-1, counter_dev=None):
    require_cuda(indptr, indices, ids)
    if indptr.dtype != torch.int64:
        raise TypeError("indptr must be int64")
    indices, ids = _i32(indices, "indices"), _i32(ids.reshape(-1), "ids")
    n = ids.numel()
    out = torch.empty((n, k), dtype=torch.int32, device=ids.device)
    check(lib().gs_sample_csr(ptr(indptr), ptr(indices), indptr.numel() - 1, ptr(ids), n, k, int(bool(replace_if_short)),
                              seed & _U64, counter & _U64, ptr(counter_dev), pad_id, ptr(out), stream_ptr()))
    _launched(1 if n * k else 0)
    return out


def _dtype_code(t):
    if t.dtype == torch.float32:
        return _lib.GS_F32
    if t.dtype == torch.bfloat16:
        return _lib.GS_BF16
    raise TypeError("features must be float32 or bfloat16 (got %s)" % t.dtype)


def gather_rows(feats, ids, out=None):
    """tf.nn.embedding_lookup(features, ids) - reference graphsage/models.py:299."""
    if hasattr(feats, "c_table"):
        ids = _i32(ids.reshape(-1), "ids")
        n, F = ids.numel(), feats.shape[1]
        if out is None:
            out = torch.empty((n, pad_cols(F)), dtype=torch.float32, device=feats.device)[:, :F]
        check(lib().gs_gather_rows_sharded(feats.c_table(), _lib.GS_F32, F, feats.pitch, ptr(ids), n, ptr(out),
                                           out.stride(0), stream_ptr()))
        _launched(1 if n else 0)
        return out
    require_cuda(feats, ids)
    if feats.dim() != 2 or feats.stride(1) != 1:
        raise ValueError("features must be a row-major 2-D tensor")
    ids = _i32(ids.reshape(-1), "ids")
    n, F = ids.numel(), feats.shape[1]
    if out is None:
        out = torch.empty((n, F), dtype=feats.dtype, device=feats.device)
    check(lib().gs_gather_rows(ptr(feats), _dtype_code(feats), feats.shape[0], F, feats.stride(0), ptr(ids), n,
                               ptr(out), out.stride(0), stream_ptr()))
    _launched(1 if n * F else 0)
    return out


def gather_rows_f32(feats, ids=None, row0=0, n=None, out=None):
    """embedding_lookup widened to fp32 (reference graphsage/models.py:299): rows ids[i] (or row0 + i) of a bf16 / fp32
    table into an fp32 [n, pad_cols(F)] buffer (returned as its [:, :F] view); pad columns are zeroed."""
    require_cuda(feats, ids, out)
    if feats.dim() != 2 or feats.stride(1) != 1:
        raise ValueError("features must be a row-major 2-D tensor")
    F = feats.shape[1]
    if ids is not None:
        ids = _i32(ids.reshape(-1), "ids")
        n = ids.numel() if n is None else int(n)
    if n is None:
        raise ValueError("n is required without ids")
    if out is None:
        out = torch.empty((n, pad_cols(F)), dtype=torch.float32, device=feats.device)[:, :F]
    if out.dtype != torch.float32 or out.stride(1) != 1 or out.shape[0] < n:
        raise ValueError("out must be a row-major float32 matrix with >= n rows")
    check(lib().gs_gather_rows_f32(ptr(feats), _dtype_code(feats), feats.shape[0], F, feats.stride(0), ptr(ids), int(row0), n,
                                   ptr(out), out.stride(0), stream_ptr()))
    _launched(1 if n else 0)
    return out


def cast_rows_bf16(x, out=None):
    """fp32 [n, F] -> bf16 [n, pad_cols(F)] (round to nearest even, pad columns zeroed); returns the [:, :F] view."""
    require_cuda(x, out)
    if x.dtype != torch.float32 or x.dim() != 2 or x.stride(1) != 1:
        raise ValueError("x must be a row-major float32 matrix")
    n, F = x.shape
    if out is None:
        out = torch.empty((n, pad_cols(F)), dtype=torch.bfloat16, device=x.device)[:, :F]
    if out.dtype != torch.bfloat16 or out.stride(1) != 1 or out.shape[0] < n or out.stride(0) < F:
        raise ValueError("out must be a row-major bfloat16 matrix with >= n rows")
    check(lib().gs_cast_rows_bf16(ptr(x), n, F, x.stride(0), ptr(out), out.stride(0), stream_ptr()))
    _launched(1 if n else 0)
    return out


class Seg(object):
    """One hop's rows for gather_mean: n output rows with fanout k.  Neighbour j of row i is
    src[neigh_ids[i*k + j]] (or src[neigh_row0 + i*k + j] when neigh_ids is None); the self row is
    src[self_ids[i]] (or src[self_row0 + i]).  Output row = out_row0 + i."""
    __slots__ = ("n", "k", "self_ids", "neigh_ids", "self_row0", "neigh_row0", "out_row0")

    def __init__(self, n, k, self_ids=None, neigh_ids=None, self_row0=0, neigh_row0=0, out_row0=0):
        self.n, self.k = int(n), int(k)
        self.self_ids = None if self_ids is None else _i32(self_ids.reshape(-1), "self_ids")
        self.neigh_ids = None if neigh_ids is None else _i32(neigh_ids.reshape(-1), "neigh_ids")
        self.self_row0, self.neigh_row0, self.out_row0 = int(self_row0), int(neigh_row0), int(out_row0)
        if self.self_ids is not None and self.self_ids.numel() < self.n:
            raise ValueError("self_ids shorter than n")
        if self.neigh_ids is not None and self.neigh_ids.numel() < self.n * self.k:
            raise ValueError("neigh_ids shorter than n*k")

    def c_struct(self):
        require_cuda(self.self_ids, self.neigh_ids)
        return Segment(ptr(self.self_ids), ptr(self.neigh_ids), self.self_row0, self.neigh_row0, self.n, self.k, 0,
                       self.out_row0)


def make_segment(n, k, self_ids=None, neigh_ids=None, self_row0=0, neigh_row0=0, out_row0=0):
    return Seg(n, k, self_ids, neigh_ids, self_row0, neigh_row0, out_row0)



def _check_out(t, rows, out_pitch, name):
    """A caller-provided output of gather_mean: the library writes rows x out_pitch floats at row stride out_pitch."""
    if t is None:
        return
    require_cuda(t)
    if t.dtype != torch.float32 or t.dim() != 2 or t.stride(1) != 1 or t.stride(0) != out_pitch or t.shape[0] < rows:
        raise ValueError("%s must be a float32 [>= %d, .] CUDA matrix with row stride out_pitch = %d" % (name, rows, out_pitch))


def gather_mean(src, segments, include_self=False, want_self=True, out_pitch=None, out_mean=None, out_self=None):
    """Fused embedding_lookup + reduce_mean over the fanout (models.py:299 + aggregators.py:48 / :106-107).
    segments: list of Seg; returns (out_self or None, out_mean), each [rows, out_pitch].
    `src` is a float32 [rows, F] CUDA tensor, or a parallel.ShardedFeatures (node-partitioned table)."""
    if hasattr(src, "c_table"):
        return _gather_mean_sharded(src, segments, include_self, want_self, out_pitch, out_mean, out_self)
    require_cuda(src)
    if src.dtype not in (torch.float32, torch.bfloat16) or src.dim() != 2 or src.stride(1) != 1:
        raise ValueError("src must be a row-major float32 (or bfloat16) 2-D tensor")
    F = src.shape[1]
    if out_pitch is None:
        out_pitch = pad_cols(F)
    rows = max([s.out_row0 + s.n for s in segments] + [0])
    _check_out(out_mean, rows, out_pitch, "out_mean")
    _check_out(out_self if want_self else None, rows, out_pitch, "out_self")
    if out_mean is None:
        out_mean = torch.empty((rows, out_pitch), dtype=torch.float32, device=src.device)
    if want_self and out_self is None:
        out_self = torch.empty((rows, out_pitch), dtype=torch.float32, device=src.device)
    arr = (Segment * max(len(segments), 1))(*[s.c_struct() for s in segments])
    ev = _probe("gather_mean/%d" % rows)
    check(lib().gs_gather_mean(ptr(src), _dtype_code(src), src.shape[0], F, src.stride(0), arr, len(segments),
                               int(bool(include_self)), ptr(out_self) if want_self else 0, ptr(out_mean), out_pitch,
                               stream_ptr()))
    _launched(1 if rows else 0, ev)
    return (out_self if want_self else None), out_mean


def translate_ids(table, ids):
    """ids -> locators of a parallel.ShardedFeatures with replicas (gs_translate_ids): >= 0 a row of this GPU's own buffer,
    < 0 -> -(global id) - 1 (the row has to come from its owner)."""
    ids = _i32(ids.reshape(-1), "ids")
    out = torch.empty_like(ids)
    check(lib().gs_translate_ids(table.c_table(), ptr(ids), ids.numel(), ptr(out), stream_ptr()))
    _launched(1 if ids.numel() else 0)
    return out


def _shard_prepare(src, segments):
    """Row addressing for a gather over a parallel.ShardedFeatures: returns (segments, ids_are_locators, staging)."""
    F = src.shape[1]
    locators, staging = 0, None
    by_ids = any(s.self_ids is not None or s.neigh_ids is not None for s in segments)
    if by_ids and src.world > 1 and getattr(src, "stage_halo", True):
        # halo staging: every remote row of the step crosses NVLink once (claim -> fetch -> translate), then the gather
        # reads local memory only.  All buffers are per call: under CUDA-graph capture they live in the graph's pool.
        lists, order = {}, []
        for s in segments:
            if (s.self_ids is None) != (s.neigh_ids is None):
                raise ValueError("a segment over a sharded table must address self and neighbours the same way")
            for t in (s.self_ids, s.neigh_ids):
                key = (t.data_ptr(), t.numel())
                if key not in lists:
                    lists[key] = t
                    order.append(key)
        capacity = sum(lists[k].numel() for k in order)
        dev = src.device
        claim = torch.empty((src.shape[0],), dtype=torch.int32, device=dev)
        count = torch.empty((1,), dtype=torch.int32, device=dev)
        stage_ids = torch.empty((capacity,), dtype=torch.int32, device=dev)
        staging = torch.empty((capacity, src.pitch), dtype=torch.float32, device=dev)
        check(lib().gs_halo_begin(ptr(claim), src.shape[0], ptr(count), stream_ptr()))
        for k in order:
            check(lib().gs_halo_claim(src.c_table(), ptr(lists[k]), lists[k].numel(), ptr(claim), ptr(count), ptr(stage_ids),
                                      capacity, stream_ptr()))
        check(lib().gs_halo_fetch(src.c_table(), F, src.pitch, ptr(stage_ids), ptr(count), capacity, ptr(staging), src.pitch,
                                  stream_ptr()))
        locs = {}
        for k in order:
            locs[k] = torch.empty_like(lists[k])
            check(lib().gs_halo_translate(src.c_table(), ptr(lists[k]), lists[k].numel(), ptr(claim), ptr(locs[k]), stream_ptr()))
        _launched(2 * len(order) + 1)
        segments = [Seg(s.n, s.k, locs[(s.self_ids.data_ptr(), s.self_ids.numel())],
                        locs[(s.neigh_ids.data_ptr(), s.neigh_ids.numel())], s.self_row0, s.neigh_row0, s.out_row0)
                    for s in segments]
        locators = 2
    elif by_ids and getattr(src, "remap", None) is not None:
        # replicas, no staging: resolve every id list once (one pass per distinct tensor; hop-1 ids are self ids of one
        # segment and neighbour ids of another) so the gather kernel's issue path has no table lookup
        done, segs = {}, []

        def tr(t):
            if t is None:
                return None
            key = (t.data_ptr(), t.numel())
            if key not in done:
                done[key] = translate_ids(src, t)
            return done[key]

        for s in segments:
            if (s.self_ids is None) != (s.neigh_ids is None):
                raise ValueError("a segment over a replicated sharded table must address self and neighbours the same way")
            segs.append(Seg(s.n, s.k, tr(s.self_ids), tr(s.neigh_ids), s.self_row0, s.neigh_row0, s.out_row0))
        segments, locators = segs, 1
    return segments, locators, staging


def _gather_mean_sharded(src, segments, include_self, want_self, out_pitch, out_mean, out_self):
    F = src.shape[1]
    if out_pitch is None:
        out_pitch = pad_cols(F)
    rows = max([s.out_row0 + s.n for s in segments] + [0])
    _check_out(out_mean, rows, out_pitch, "out_mean")
    _check_out(out_self if want_self else None, rows, out_pitch, "out_self")
    if out_mean is None:
        out_mean = torch.empty((rows, out_pitch), dtype=torch.float32, device=src.device)
    if want_self and out_self is None:
        out_self = torch.empty((rows, out_pitch), dtype=torch.float32, device=src.device)
    segments, locators, staging = _shard_prepare(src, segments)
    arr = (Segment * max(len(segments), 1))(*[s.c_struct() for s in segments])
    ev = _probe("gather_mean/%d" % rows)
    check(lib().gs_gather_mean_sharded(src.c_table(), _lib.GS_F32, F, src.pitch, arr, len(segments),
                                       int(bool(include_self)), locators, ptr(staging), ptr(out_self) if want_self else 0,
                                       ptr(out_mean), out_pitch, stream_ptr()))
    _launched(1 if rows else 0, ev)
    return (out_self if want_self else None), out_mean


def gather_mean_images(src, segments, include_self=False, want_self=True):
    """gs_gather_mean_img: the fused gather + fanout mean whose result is written as tf32 hi/lo UMMA tile images (the A
    operand of sage_gemm_img).  Returns (images uint8 tensor, rows) or None when the image form does not apply."""
    sharded = hasattr(src, "c_table")
    if not sharded:
        require_cuda(src)
        if src.dtype != torch.float32 or src.dim() != 2 or src.stride(1) != 1:
            return None
    F = src.shape[1]
    pitch = src.pitch if sharded else src.stride(0)
    if F > 1280 or pitch % 4 != 0 or (not sharded and src.data_ptr() % 16 != 0):
        return None
    rows = max([s.out_row0 + s.n for s in segments] + [0])
    if rows == 0:
        return None
    nbytes = lib().gs_gather_mean_img_bytes(rows, F, int(bool(want_self)))
    dev = src.device
    buf = torch.empty((nbytes + 1024,), dtype=torch.uint8, device=dev)
    off = (-buf.data_ptr()) % 1024
    images = buf[off:off + nbytes]
    locators, staging = 0, None
    if sharded:
        segments, locators, staging = _shard_prepare(src, segments)
    arr = (Segment * max(len(segments), 1))(*[s.c_struct() for s in segments])
    ev = _probe("gather_mean/%d" % rows)
    rc = lib().gs_gather_mean_img(0 if sharded else ptr(src), 0 if sharded else src.shape[0], src.c_table() if sharded else None,
                                  locators, ptr(staging), F, pitch, arr, len(segments), int(bool(include_self)),
                                  int(bool(want_self)), ptr(images), stream_ptr())
    if rc == -3:                       # GS_ERR_UNSUPPORTED: the caller uses the fp32 pair
        return None
    check(rc)
    _launched(1, ev)
    return images, rows


def sage_gemm_img(M, images, parts, combine=COMBINE_ADD, bias=None, act=ACT_NONE, packed=None, a_part0=0, out=None):
    """gs_sage_gemm_img: act(concat_or_add(A_p @ B_p) + bias) in tf32x3 arithmetic with the A operands taken from the tile
    images gather_mean_images wrote (part p reads image part a_part0 + p).  parts: [(None, K, B[K, N])]."""
    _, arr, keep = _gemm_parts([(None, K, B) for (_, K, B) in parts])
    ntot = sum(p[2].shape[1] for p in parts) if (combine == COMBINE_CONCAT) else parts[0][2].shape[1]
    dev = images.device
    if out is None:
        out = torch.empty((M, ntot), dtype=torch.float32, device=dev)
    if packed is None:
        packed = PackedWeights()
    ws = packed.get(parts, arr, MATH_TF32X3, dev)
    ev = _probe("sage_gemm/%d" % M)
    check(lib().gs_sage_gemm_img(M, arr, len(parts), combine, ptr(bias), act, ptr(out), out.stride(0), ptr(ws), ptr(images),
                                 int(a_part0), stream_ptr()))
    _launched(1 if M else 0, ev)
    return out


def segment_max(x, n, k):
    require_cuda(x)
    C = x.shape[1]
    out = torch.empty((n, C), dtype=torch.float32, device=x.device)
    check(lib().gs_segment_max(ptr(x), n, k, C, x.stride(0), ptr(out), out.stride(0), stream_ptr()))
    _launched(1 if n * C else 0)
    return out


def _gemm_parts(parts):
    M = parts[0][0].shape[0] if parts[0][0] is not None else 0
    arr = (GemmPart * len(parts))()
    keep = []
    for i, (A, K, B) in enumerate(parts):
        require_cuda(A, B)
        if (A is not None and A.dtype != torch.float32) or B.dtype != torch.float32:
            raise TypeError("sage_gemm operands must be float32")
        if A is not None and (A.stride(1) != 1 or A.shape[0] != M or A.shape[1] < K):
            raise ValueError("bad A operand for part %d" % i)
        B = B.contiguous()
        if B.shape[0] != K:
            raise ValueError("part %d: B has %d rows, expected K=%d" % (i, B.shape[0], K))
        keep.append(B)
        arr[i] = GemmPart(ptr(A), A.stride(0) if A is not None else K, K, ptr(B), B.stride(0), B.shape[1])
    return M, arr, keep


class PackedWeights(object):
    """Tensor-core weight images cached across calls (inference: the weights do not change between steps).
    Re-packed automatically when a weight tensor is replaced or modified in place."""

    def __init__(self):
        self.key, self.ws = None, None

    def get(self, parts, arr, math, dev):
        key = (math,) + tuple((p[2].data_ptr(), p[2]._version, tuple(p[2].shape)) for p in parts)
        if key != self.key:
            nbytes = lib().gs_sage_gemm_workspace_bytes(1, arr, len(parts), math)
            if nbytes < 0:
                check(-1)
            if self.ws is None or self.ws.numel() < nbytes:
                self.ws = torch.empty((max(nbytes, 1),), dtype=torch.uint8, device=dev)
            check(lib().gs_sage_gemm_pack(arr, len(parts), math, ptr(self.ws), stream_ptr()))
            _launched(1)
            self.key = key
        return self.ws


def sage_gemm(parts, combine=COMBINE_ADD, bias=None, act=ACT_NONE, math=MATH_FP32_SIMT, out=None, packed=None):
    """parts: [(A[M, >=K] (row stride used as lda), K, B[K, N])] (1 or 2).  act(concat_or_add(A_p[:, :K] @ B_p) + bias).
    packed: optional PackedWeights cache (tensor-core modes) so the weight images are built once, not per call."""
    M, arr, keep = _gemm_parts(parts)
    ntot = sum(p[2].shape[1] for p in parts) if (combine == COMBINE_CONCAT) else parts[0][2].shape[1]
    dev = parts[0][0].device
    if out is None:
        out = torch.empty((M, ntot), dtype=torch.float32, device=dev)
    if math == MATH_FP32_SIMT or packed is None:
        ws_bytes = lib().gs_sage_gemm_workspace_bytes(M, arr, len(parts), math)
        if ws_bytes < 0:
            check(-1)
        ws = torch.empty((ws_bytes,), dtype=torch.uint8, device=dev) if ws_bytes > 0 else None
        ev = _probe("sage_gemm/%d" % M)
        check(lib().gs_sage_gemm(M, arr, len(parts), combine, ptr(bias), act, math, ptr(out), out.stride(0), ptr(ws),
                                 stream_ptr()))
        _launched((2 if ws is not None else 1) if M else 0, ev)
        return out
    ws = packed.get(parts, arr, math, dev)
    ev = _probe("sage_gemm/%d" % M)
    check(lib().gs_sage_gemm_prepacked(M, arr, len(parts), combine, ptr(bias), act, math, ptr(out), out.stride(0),
                                       ptr(ws), stream_ptr()))
    _launched(1 if M else 0, ev)
    return out


SMALL_LAYER_MAX_ROWS = 2048


def sage_layer_small(src, seg, parts, combine=COMBINE_ADD, include_self=False, bias=None, act=ACT_NONE,
                     l2_normalize=False, counter_dev=None, counter_inc=0):
    """One whole aggregator layer (fanout mean -> matmuls -> add|concat -> bias -> act -> optional row
    l2-normalise) for a small number of rows in ONE launch, exact fp32.  parts: [(None, K, B)] with K == src width."""
    require_cuda(src, bias, counter_dev)
    if src.dtype != torch.float32 or src.stride(1) != 1:
        raise ValueError("src must be row-major float32")
    _, arr, keep = _gemm_parts([(None, K, B) for (_, K, B) in parts])
    ntot = sum(p[2].shape[1] for p in parts) if (combine == COMBINE_CONCAT) else parts[0][2].shape[1]
    rows = seg.out_row0 + seg.n
    out = torch.empty((rows, ntot), dtype=torch.float32, device=src.device)
    cseg = seg.c_struct()
    ev = _probe("sage_layer_small/%d" % rows)
    check(lib().gs_sage_layer_small(ptr(src), src.shape[0], src.shape[1], src.stride(0), cseg, int(bool(include_self)),
                                    arr, len(parts), combine, ptr(bias), act, int(bool(l2_normalize)), ptr(out),
                                    out.stride(0), ptr(counter_dev), int(counter_inc), stream_ptr()))
    _launched(1 if seg.n else 0, ev)
    return out


class PackedMlpWeights(object):
    """bf16 tile images of the max-pool MLP weight for gs_maxpool_mlp_fused, re-packed when the weight changes."""

    def __init__(self):
        self.key, self.ws = None, None

    def get(self, W):
        key = (W.data_ptr(), W._version, tuple(W.shape))
        if key != self.key:
            K, hidden = W.shape
            nbytes = lib().gs_maxpool_mlp_workspace_bytes(K, hidden)
            self.ws = torch.empty((nbytes,), dtype=torch.uint8, device=W.device)
            Wc = W.contiguous()
            check(lib().gs_maxpool_mlp_pack(ptr(Wc), Wc.stride(0), K, hidden, ptr(self.ws), stream_ptr()))
            _launched(1)
            self.key = key
        return self.ws


def maxpool_mlp_fused(table, n_groups, k, W, bias, packed, row_ids=None, row0=0, K=None, out=None, pool="max"):
    """out[g, :] = max_j relu(table[row(g, j), :K] @ W + bias) in one tcgen05 kernel (bf16 operands, fp32 accumulate).
    table: bfloat16 [rows, >=K] row-major with pitch % 8 == 0; W: float32 [K, hidden] (hidden % 128 == 0)."""
    require_cuda(table, W, bias, row_ids)
    if table.dtype != torch.bfloat16 or table.stride(1) != 1:
        raise TypeError("table must be row-major bfloat16")
    K = W.shape[0] if K is None else K
    hidden = W.shape[1]
    if out is None:
        out = torch.empty((n_groups, hidden), dtype=torch.float32, device=table.device)
    ws = packed.get(W)
    if row_ids is not None:
        row_ids = _i32(row_ids.reshape(-1), "row_ids")
    ev = _probe("maxpool_mlp/%d" % n_groups)
    fn = lib().gs_meanpool_mlp_fused if pool == "mean" else lib().gs_maxpool_mlp_fused
    check(fn(ptr(table), table.shape[0], K, table.stride(0), ptr(row_ids), row0, n_groups, k,
             ptr(ws), ptr(bias), hidden, ptr(out), out.stride(0), stream_ptr()))
    _launched(1 if n_groups else 0, ev)
    return out


def row_used(x, out=None):
    """tf.sign(tf.reduce_max(tf.abs(x), axis=-1)) per row (reference graphsage/aggregators.py:411) as uint8 [rows]:
    1 where the row has any non-zero element.  x: float32 or bfloat16, row-major [rows, F] (any row stride)."""
    require_cuda(x, out)
    if x.dim() != 2 or x.stride(1) != 1:
        raise ValueError("x must be a row-major 2-D tensor")
    n, F = x.shape
    if out is None:
        out = torch.empty((n,), dtype=torch.uint8, device=x.device)
    if out.dtype != torch.uint8 or out.numel() < n or not out.is_contiguous():
        raise ValueError("out must be a contiguous uint8 tensor with >= rows elements")
    ev = _probe("row_used/%d" % n)
    check(lib().gs_row_used(ptr(x), _dtype_code(x), n, F, x.stride(0), ptr(out), stream_ptr()))
    _launched(1 if n else 0, ev)
    return out


def lstm_seq(P, Wh, used, n, k, row_ids=None, row0=0, out=None, keep=False):
    """dynamic_rnn(BasicLSTMCell(H), sequence_length = max(1, sum(used))) and the gather of h_{len-1} (reference
    graphsage/aggregators.py:408-433) for n sequences of k steps, in one launch of gs_lstm_seq.
    P: float32 [n*k, >=4H] input projection (x @ kernel[:in] + bias); Wh: float32 [H, 4H] (kernel[in:]); used: uint8 rows
    addressed by row_ids[g*k + t] (or row0 + g*k + t).  Returns out [n, H], or (out, keep_h, keep_c, lengths) with keep
    (keep_h / keep_c [n, k, H] hold h_t / c_t for t < len; later steps are not written)."""
    require_cuda(P, Wh, used, row_ids, out)
    if P.dtype != torch.float32 or P.stride(1) != 1 or Wh.dtype != torch.float32:
        raise TypeError("P and Wh must be row-major float32")
    if used.dtype != torch.uint8:
        raise TypeError("used must be uint8")
    H = Wh.shape[0]
    if Wh.shape[1] != 4 * H:
        raise ValueError("Wh must be [H, 4H]")
    Wh = Wh.contiguous()
    n, k = int(n), int(k)
    if P.shape[0] < n * k or P.shape[1] < 4 * H:
        raise ValueError("P must be [>= n*k, >= 4H]")
    if row_ids is not None:
        row_ids = _i32(row_ids.reshape(-1), "row_ids")
        if row_ids.numel() < n * k:
            raise ValueError("row_ids shorter than n*k")
    dev = P.device
    if out is None:
        out = torch.empty((n, H), dtype=torch.float32, device=dev)
    if out.dtype != torch.float32 or out.stride(1) != 1 or out.shape[0] < n or out.shape[1] < H:
        raise ValueError("out must be a row-major float32 [>= n, >= H] matrix")
    keep_h = keep_c = lengths = None
    if keep:
        keep_h = torch.empty((n, k, H), dtype=torch.float32, device=dev)
        keep_c = torch.empty((n, k, H), dtype=torch.float32, device=dev)
        lengths = torch.empty((n,), dtype=torch.int32, device=dev)
    ev = _probe("lstm_seq/%d" % n)
    check(lib().gs_lstm_seq(ptr(P), P.stride(0), ptr(Wh), H, ptr(used), ptr(row_ids), int(row0), n, k, ptr(out),
                            out.stride(0), ptr(keep_h), ptr(keep_c), ptr(lengths), stream_ptr()))
    _launched(1 if n else 0, ev)
    return (out, keep_h, keep_c, lengths) if keep else out


def l2_normalize_rows_(x):
    """In-place tf.nn.l2_normalize(x, 1) - reference graphsage/models.py:368."""
    require_cuda(x)
    check(lib().gs_l2_normalize_rows(ptr(x), x.shape[0], x.shape[1], x.stride(0), stream_ptr()))
    _launched(1 if x.numel() else 0)
    return x
