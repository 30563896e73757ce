/*
 * graphsage_b200.h - C-ABI of libgraphsage_b200.so (sm_100a).
 *
 * The reference (williamleif/GraphSAGE) has NO FFI boundary: its hot path is python
 * classes composing TensorFlow library ops.  Each entry point below therefore names the
 * TF op sequence (reference file:line) it replaces; the python classes that keep the
 * reference's surface (graphsage_b200/{neigh_samplers,aggregators,models}.py) bind these
 * through ctypes (see INTEGRATION.md).
 *
 * Conventions
 *   - extern "C", plain pointers and sizes, no torch types.
 *   - Pointers are DEVICE pointers unless the name ends in _host.  Row-major.  "pitch"/"ld"
 *     are in ELEMENTS.  The library never synchronises: every call only enqueues work on `stream`
 *     (a cudaStream_t passed as void*).  It never allocates device memory either, with one exception:
 *     gs_shard_alloc/gs_shard_free (cudaMalloc'd buffers that can be exported through CUDA IPC).
 *   - Return value: 0 = OK, <0 = gs_status error; gs_last_error_string() (thread-local, host)
 *     describes the last failure.  No exceptions cross the boundary.
 *   - There is no CPU fallback: without a CUDA device every compute entry returns GS_ERR_CUDA.
 */
#ifndef GRAPHSAGE_B200_H_
#define GRAPHSAGE_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GS_ABI_VERSION 2

typedef enum {
  GS_OK = 0,
  GS_ERR_INVALID_ARG = -1,
  GS_ERR_CUDA = -2,
  GS_ERR_UNSUPPORTED = -3
} gs_status;

typedef enum { GS_F32 = 0, GS_BF16 = 1 } gs_dtype;
typedef enum { GS_ACT_NONE = 0, GS_ACT_RELU = 1 } gs_act;
/* how the neighbour part and the self part are combined */
typedef enum {
  GS_COMBINE_ADD = 0,    /* tf.add_n([from_self, from_neighs])      aggregators.py:55-56 */
  GS_COMBINE_CONCAT = 1  /* tf.concat([from_self, from_neighs], 1)  aggregators.py:57-58 */
} gs_combine;
/* arithmetic of the dense contraction */
typedef enum {
  GS_MATH_FP32_SIMT = 0,  /* fp32 FFMA on CUDA cores (bring-up / cross-check path)          */
  GS_MATH_TF32X3 = 1,     /* tcgen05 kind::tf32, 3-term hi/lo split, fp32 accumulate in TMEM */
  GS_MATH_TF32 = 2,       /* tcgen05 kind::tf32 single pass                                  */
  GS_MATH_BF16 = 3        /* tcgen05 kind::f16 (bf16 operands), fp32 accumulate              */
} gs_math;

int32_t gs_version(void);
const char* gs_last_error_string(void);
/* Tuning knobs for experiments; returns the previous value.  Keys (default):
 *   gather_variant (2)      gs_gather_mean / gs_gather_rows: 2 grouped double-buffered TMA, 1 whole-node TMA, 0 LDG
 *   gather_ctas_per_sm (8)  grid cap of the LDG / simple gather kernels
 *   gemm_async (0)          gs_sage_gemm tcgen05 producers: 1 = cp.async staging instead of register prefetch
 *   mma_issue (1)           tcgen05 issue form: 1 = whole warp + elect.sync (tensor-pipe floor), 0 = single thread
 *   k4_kernel (0)           gs_maxpool/meanpool_mlp_fused kernel family: 0 = weights in tensor memory, gathered rows = B
 *                           operand (default); 3 / 2 = weights resident in shared memory, 128- / 256-row tiles; 1 = the
 *                           round-1 form (gathered rows = A operand; k4_producer 0 cp.async, 1 gather4, 2 gather4 multicast)
 *   k4_cluster (2)          k4_kernel 0: thread-block cluster size (2, 4, 8; -1 = hidden / 128; 0 = no clusters) - the CTAs
 *                           of a cluster share one gathered tile through TMA gather4 multicast
 *   k4_tile (128)           k4_kernel 0: rows per tile (128; 256 = the wide tile, which runs without clusters)
 *   k4_pipes (1)            k4_kernel 0 without clusters: 2 = two half-ring pipelines / two accumulators
 *   k4_stages (0)           k4_kernel 0: cap on the operand ring depth (0 = as many as fit)
 *   k4_wide_producer (1)    k4_kernel 3: 1 = TMA gather4 producers, 0 = cp.async producers
 *   halo_fetch_ctas_per_sm (2)  grid of gs_halo_fetch
 * Every K4 variant is parity-tested (tests/test_gpu_parity.py: K4_VARIANTS); DESIGN.md section 4a has the measurements.
 * The Python host also reads them from the environment: GS_TUNING="key=value,key=value". */
int32_t gs_set_tuning(const char* key, int32_t value);

/* ---------------------------------------------------------------------------------------------
 * UniformNeighborSampler._call           reference graphsage/neigh_samplers.py:24-29
 *   out[i, j] = adj[ids[i], pi[j]], j < k, ONE column permutation pi per call.
 *   pi = col_perm (device int32[>=k]) if non-null, else the on-device Philox4x32-10 forward
 *   Fisher-Yates prefix of (seed, counter + (counter_dev ? *counter_dev : 0)) - bit-identical to
 *   oracle/sampler.py:perm_prefix.  ids outside [0, n_rows) read the dummy row n_rows-1.
 * --------------------------------------------------------------------------------------------- */
int32_t gs_sample_padded(const int32_t* adj, int64_t n_rows, int32_t max_deg,
                         const int32_t* ids, int64_t n, int32_t k,
                         const int32_t* col_perm, uint64_t seed, uint64_t counter,
                         const uint64_t* counter_dev, int32_t* out, void* stream);

/* SampleAndAggregate.sample - the whole frontier expansion (reference graphsage/models.py:254-275) in
 * ONE launch: hop t (t = 1..n_hops) is sample_padded(samples[t-1], fanout[t-1]) with RNG counter
 * counter + t - 1 (fanout[] is in HOP order, i.e. reversed layer order: {10, 25} for samples_1=25,
 * samples_2=10).  out[t-1] receives the B*fanout[0]*...*fanout[t-1] ids of hop t (row-major nested).
 * Bit-identical to n_hops successive gs_sample_padded calls.  n_hops <= GS_MAX_HOPS. */
#define GS_MAX_HOPS 4
int32_t gs_sample_padded_khop(const int32_t* adj, int64_t n_rows, int32_t max_deg,
                              const int32_t* seeds, int64_t n_seeds, const int32_t* fanout_host,
                              int32_t n_hops, uint64_t seed, uint64_t counter,
                              const uint64_t* counter_dev, int32_t* const* out_host, void* stream);

/* Per-node draws from a CSR adjacency (north_star's warp-per-node mode; no reference
 * counterpart).  Semantics: oracle/sampler.py:sample_csr.  k <= 32. */
int32_t gs_sample_csr(const int64_t* indptr, const int32_t* indices, int64_t n_nodes,
                      const int32_t* ids, int64_t n, int32_t k, int32_t replace_if_short,
                      uint64_t seed, uint64_t counter, const uint64_t* counter_dev,
                      int32_t pad_id, int32_t* out, void* stream);

/* tf.nn.fixed_unigram_candidate_sampler(unique=False)   reference graphsage/models.py:336-343
 *   num_sampled ids drawn with replacement with probability proportional to the weights behind `cdf`
 *   (cdf[i] = sum_{j<=i} deg[j]^0.75, float64, non-decreasing, length n).  Draw j uses word j&3 of
 *   Philox4x32-10 block (counter, c2 = 0, GS unigram stream tag + j>>2): u = (draw + 0.5) / 2^32 * cdf[n-1],
 *   out[j] = first index with cdf[index] > u (oracle/sampler.py:sample_unigram; TF's own stream is unobtainable). */
int32_t gs_sample_unigram(const double* cdf, int64_t n, int32_t num_sampled, uint64_t seed, uint64_t counter,
                          const uint64_t* counter_dev, int32_t* out, void* stream);

/* Device-side construction of the padded adjacency table from CSR (the sampler's input contract, reference
 * graphsage/minibatch.py:227-259; SURVEY section 8f row 3).  adj is [n_nodes + 1, max_deg] int32:
 *   row n_nodes (dummy) and rows of skipped nodes (skip[u] != 0: val/test nodes, minibatch.py:232-233) or of
 *   nodes without neighbours = n_nodes;  deg == max_deg: the neighbours in CSR order;
 *   deg <  max_deg: max_deg draws WITH replacement (minibatch.py:242-243);
 *   deg >  max_deg: max_deg distinct neighbours (Floyd's algorithm; minibatch.py:240-241).
 * Draw j of node u is word j&3 of Philox block (counter, c2 = u, build tag + j>>2)  (oracle/adjacency.py:
 * build_padded_adj; the reference's numpy RandomState stream is reproduced by the HOST builder
 * graphsage_b200/minibatch.py instead).  max_deg <= 1024.  deg (float32 [n_nodes], may be NULL) receives the
 * neighbour counts (minibatch.py:237). */
int32_t gs_build_padded_adj(const int64_t* indptr, const int32_t* indices, int64_t n_nodes, int32_t max_deg,
                            const uint8_t* skip, uint64_t seed, uint64_t counter, int32_t* adj, float* deg,
                            void* stream);

/* host helper: the first k entries of pi for (seed, counter) - what the kernel computes */
int32_t gs_perm_prefix_host(uint64_t seed, uint64_t counter, int32_t max_deg, int32_t k,
                            int32_t* out_host);

/* ---------------------------------------------------------------------------------------------
 * tf.nn.embedding_lookup(features, ids)   reference graphsage/models.py:299
 *   out[i, 0:F] = feats[ids[i], 0:F].  When row bytes are 16-B multiples and pointers 16-B
 *   aligned the copy is staged global->shared->global by the TMA bulk-copy engine.
 * --------------------------------------------------------------------------------------------- */
int32_t gs_gather_rows(const void* feats, int32_t dtype, int64_t n_rows, int32_t F,
                       int64_t pitch, const int32_t* ids, int64_t n, void* out,
                       int64_t out_pitch, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Fused K-hop gather + fixed-fanout segmented mean:
 *   tf.nn.embedding_lookup (models.py:299) + tf.reduce_mean(neigh_vecs, axis=1)
 *   (aggregators.py:48), or the GCN form mean(concat([neigh, self]))  (aggregators.py:106-107),
 *   without materialising the [n*k, F] neighbour tensor.
 * A call processes up to GS_MAX_SEGMENTS segments (one per hop) in one launch.  For segment s,
 * output row r = out_row0 + i (i < n):
 *   neigh row j of i = src[neigh_ids ? neigh_ids[i*k + j] : neigh_row0 + i*k + j]
 *   self  row   of i = src[self_ids  ? self_ids[i]        : self_row0 + i]
 *   out_mean[r] = (sum_j neigh_j (+ self if include_self)) / (k (+1 if include_self))
 *   out_self[r] = self row (only if out_self != NULL)
 * src is [n_src_rows, F] with `pitch`; F columns are produced, columns F..out_pitch-1 are zeroed.
 * dtype GS_F32, or GS_BF16: a bfloat16 table (rows 16-byte multiples: pitch % 8 == 0, out_pitch % 8 == 0) summed in fp32 -
 * the outputs stay fp32 and equal the fp32 kernel's on the bf16-rounded table (half the gathered bytes).
 * --------------------------------------------------------------------------------------------- */
#define GS_MAX_SEGMENTS 4
typedef struct {
  const int32_t* self_ids;   /* device, may be NULL */
  const int32_t* neigh_ids;  /* device, may be NULL */
  int64_t self_row0;
  int64_t neigh_row0;
  int64_t n;
  int32_t k;
  int32_t _pad;
  int64_t out_row0;
} gs_segment;

int32_t gs_gather_mean(const void* src, int32_t dtype, int64_t n_src_rows, int32_t F, int64_t pitch,
                       const gs_segment* segments_host, int32_t n_segments, int32_t include_self,
                       void* out_self, void* out_mean, int64_t out_pitch, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Node-partitioned feature table (multi-GPU, SURVEY 8e; no reference counterpart - the reference is
 * single-device).  Shard r owns the global ids [row_start[r], row_start[r+1]) (contiguous ranges - align them
 * with communities); every rank maps all shards into its address space (CUDA IPC over NVLink/NVSwitch), so the
 * gather kernel resolves
 *   row(id) = base[owner(id)] + (id - row_start[owner(id)]) * pitch
 * and pulls remote rows itself - one cp.async.bulk per row over NVLink into shared memory (or 128-bit loads with
 * gather_variant=0): the halo exchange is fused into the gather, no staging buffer, no collective on the data path.
 * A rank may also hold REPLICAS of the remote rows it reads most: remap (device int32 [n_global_rows], may be NULL)
 * gives, for every id, the row index inside this rank's OWN buffer (own rows, zero row, replicas) or -1 when the
 * row has to come from its owner.  Ids outside [0, n_global_rows-1) - including the dummy id N - read the caller's
 * local zero row (index zero_row of its own buffer).
 * gs_gather_mean_sharded has the semantics of gs_gather_mean with `src` replaced by the table.
 * --------------------------------------------------------------------------------------------- */
#define GS_MAX_SHARDS 16
typedef struct {
  const void* base[GS_MAX_SHARDS];       /* device pointers; shard r holds its own rows first */
  int64_t row_start[GS_MAX_SHARDS + 1];  /* row_start[0] = 0 ... row_start[n_shards] = N */
  int32_t n_shards;
  int32_t my_shard;
  int64_t n_global_rows;                 /* N + 1 (the dummy row is virtual: every shard carries its own zero row) */
  int64_t zero_row;                      /* index of the all-zero row inside base[my_shard] */
  const int32_t* remap;                  /* device, [n_global_rows] or NULL (see above) */
} gs_sharded_table;

/* ids_are_locators: 0 = global ids; 1 = gs_translate_ids locators; 2 = gs_halo_translate locators (negative values index
 * `staging`, this step's halo rows fetched by gs_halo_fetch; staging has the table's pitch) */
int32_t gs_gather_mean_sharded(const gs_sharded_table* table_host, int32_t dtype, int32_t F, int64_t pitch,
                               const gs_segment* segments_host, int32_t n_segments, int32_t include_self,
                               int32_t ids_are_locators, const void* staging, void* out_self, void* out_mean,
                               int64_t out_pitch, void* stream);
/* Halo staging - every remote row a step needs crosses NVLink ONCE (a frontier repeats remote nodes; peer reads bypass the
 * local L2).  Per step:  gs_halo_begin (claim[] = -1, *count = 0)  ->  gs_halo_claim for every id list (first sighting of a
 * remote id takes the next staging slot; stage_ids[slot] = id)  ->  gs_halo_fetch (rows of stage_ids[0 .. *count) from their
 * owners into staging[slot])  ->  gs_halo_translate for every id list (out = row of this GPU's own buffer when the row is
 * held locally, else -(slot) - 1)  ->  gs_gather_mean_sharded(..., ids_are_locators = 2, staging).
 * claim: int32 [n_global_rows]; count: int32 [1]; stage_ids: int32 [capacity]; staging: float [capacity, staging_pitch];
 * capacity >= the number of ids claimed (the sum of the lists' lengths always suffices). */
int32_t gs_halo_begin(int32_t* claim, int64_t n_global_rows, int32_t* count, void* stream);
int32_t gs_halo_claim(const gs_sharded_table* table_host, const int32_t* ids, int64_t n, int32_t* claim, int32_t* count,
                      int32_t* stage_ids, int64_t capacity, void* stream);
int32_t gs_halo_fetch(const gs_sharded_table* table_host, int32_t F, int64_t pitch, const int32_t* stage_ids,
                      const int32_t* count, int64_t capacity, float* staging, int64_t staging_pitch, void* stream);
int32_t gs_halo_translate(const gs_sharded_table* table_host, const int32_t* ids, int64_t n, const int32_t* claim,
                          int32_t* out, void* stream);
/* ids -> locators for a table with replicas (remap != NULL): out[i] = remap[ids[i]] (a row index inside this GPU's own
 * buffer) when the row is held locally - own rows, replicas, the zero row for ids outside [0, N) -, else -(ids[i]) - 1.
 * One cheap, fully parallel pass per id list; the gather kernel then needs no table lookup on its copy-issue path. */
int32_t gs_translate_ids(const gs_sharded_table* table_host, const int32_t* ids, int64_t n, int32_t* out, void* stream);
int32_t gs_gather_rows_sharded(const gs_sharded_table* table_host, int32_t dtype, int32_t F, int64_t pitch,
                               const int32_t* ids, int64_t n, void* out, int64_t out_pitch, void* stream);

/* Shard buffers are allocated by the library with cudaMalloc so that they can be exported through
 * CUDA IPC (the only allocation the library ever makes; freed by gs_shard_free). */
int32_t gs_shard_alloc(int64_t bytes, void** dev_ptr_out);
int32_t gs_shard_free(void* dev_ptr);
int32_t gs_ipc_export(const void* dev_ptr, uint8_t* handle64_out_host);
int32_t gs_ipc_import(const uint8_t* handle64_host, void** dev_ptr_out);
int32_t gs_ipc_close(void* dev_ptr);

/* embedding_lookup (models.py:299) with the result widened to fp32: out[i, 0:F] = (float)feats[ids ? ids[i] : row0 + i, 0:F],
 * columns F..out_pitch-1 zeroed.  feats is GS_BF16 or GS_F32.  The bf16 max-pool path uses it for the SELF rows, which
 * meet the fp32 self_weights contraction (aggregators.py:185). */
int32_t gs_gather_rows_f32(const void* feats, int32_t dtype, int64_t n_rows, int32_t F, int64_t pitch,
                           const int32_t* ids, int64_t row0, int64_t n, float* out, int64_t out_pitch,
                           void* stream);
/* fp32 [n, F] (row stride ldx) -> bf16 [n, out_pitch], round-to-nearest-even, pad columns zeroed: the next layer's
 * bf16 source table of the max-pool path (the hidden[hop] list of models.py:321-329 kept in the K4 operand type). */
int32_t gs_cast_rows_bf16(const float* x, int64_t n, int32_t F, int64_t ldx, void* out_bf16, int64_t out_pitch,
                          void* stream);

/* ---------------------------------------------------------------------------------------------
 * R-MAT graph written directly as CSR on the device (BASELINE.json configs[4]: scale 27 trimmed to 10^8 nodes, about 20
 * entries per node, a, b, c, d = 0.57, 0.19, 0.19, 0.05).  No reference counterpart - the reference reads graphs from
 * disk (graphsage/utils.py:19-75); this is the synthetic stand-in at that size.  Contract: oracle/rmat.py, csrc/rmat.cu.
 *   1. gs_rmat_degrees -> deg[n_nodes] (int32);  2. caller: indptr = exclusive prefix sum (int64 [n_nodes + 1]);
 *   3. gs_rmat_fill -> indices[indptr[n_nodes]] (int32 neighbour ids, unsorted, duplicates possible, no self loops).
 * Node ids are scrambled by y = (x * mul + add) mod n_nodes, which must be a bijection: (mul * mul_inv) mod n_nodes == 1.
 * --------------------------------------------------------------------------------------------- */
int32_t gs_rmat_degrees(int32_t scale, int64_t n_nodes, double edge_factor, double a, double b, double c, double d,
                        uint64_t seed, uint64_t mul, uint64_t mul_inv, uint64_t add, int32_t* deg_out, void* stream);
/* long_rows (device int64 [n_long], may be NULL with n_long = 0): the rows with more than long_threshold entries - R-MAT's
 * hubs (1.2 M entries in one row at scale 27); they are filled by a whole grid each instead of one warp.  n_long <= 65535. */
int32_t gs_rmat_fill(int32_t scale, int64_t n_nodes, double a, double b, double c, double d, uint64_t seed, uint64_t mul,
                     uint64_t mul_inv, uint64_t add, const int64_t* indptr, int32_t* indices, const int64_t* long_rows,
                     int64_t n_long, int64_t long_threshold, void* stream);

/* segmented max over fixed fanout: out[i, c] = max_j x[i*k + j, c]   (aggregators.py:182) */
int32_t gs_segment_max(const float* x, int64_t n, int32_t k, int32_t C, int64_t ldx,
                       float* out, int64_t ldo, void* stream);

/* ---------------------------------------------------------------------------------------------
 * The dense contraction of an aggregator (aggregators.py:51-64, 110-116, 184-195; Dense
 * layers.py:104-116):
 *   part p (p < n_parts <= 2):  P_p = A_p[M, K_p] @ B_p[K_p, N_p]      (B row-major, ldb)
 *   combine ADD   : out[:, 0:N]            = act(P_0 + P_1 + bias)      (N_0 == N_1)
 *   combine CONCAT: out[:, 0:N_0]          = act(P_0 + bias[0:N_0]),
 *                   out[:, N_0:N_0+N_1]    = act(P_1 + bias[N_0:])
 *   bias may be NULL.  fp32 in/out.  `math` selects the arithmetic (gs_math).
 *   workspace: device scratch of gs_sage_gemm_workspace_bytes(...) bytes (may be NULL if 0).
 * --------------------------------------------------------------------------------------------- */
typedef struct {
  const float* A; int64_t lda; int32_t K;
  const float* B; int64_t ldb; int32_t N;
} gs_gemm_part;

int64_t gs_sage_gemm_workspace_bytes(int64_t M, const gs_gemm_part* parts_host, int32_t n_parts,
                                     int32_t math);
int32_t gs_sage_gemm(int64_t M, const gs_gemm_part* parts_host, int32_t n_parts, int32_t combine,
                     const float* bias, int32_t act, int32_t math, float* out, int64_t ldo,
                     void* workspace, void* stream);

/* Weight packing for the tensor-core modes can be hoisted out of the step when the weights do not
 * change (inference): gs_sage_gemm_pack fills `workspace` (gs_sage_gemm_workspace_bytes) from the parts'
 * B matrices; gs_sage_gemm_prepacked then runs only the GEMM.  gs_sage_gemm == pack + prepacked. */
int32_t gs_sage_gemm_pack(const gs_gemm_part* parts_host, int32_t n_parts, int32_t math, void* workspace,
                          void* stream);
int32_t gs_sage_gemm_prepacked(int64_t M, const gs_gemm_part* parts_host, int32_t n_parts, int32_t combine,
                               const float* bias, int32_t act, int32_t math, float* out, int64_t ldo,
                               const void* workspace, void* stream);

/* ---------------------------------------------------------------------------------------------
 * The mean / GCN layer-0 pair with the A operand handed over as tensor-core tile images (tf32x3 arithmetic):
 *   gs_gather_mean_img : the fused gather + fanout mean of gs_gather_mean / gs_gather_mean_sharded (same segments, same
 *       table forms: pass `src` (dense fp32 [n_src_rows, pitch]) or `table_host` (node-partitioned; ids_are_locators /
 *       staging as in gs_gather_mean_sharded)), whose result rows are written ALREADY SPLIT into tf32 hi / lo and laid
 *       out as UMMA K-major SWIZZLE_128B tile images: part p (0 = self rows, 1 = mean rows when want_self; only the mean
 *       part when !want_self), 128-row tile mt, 32-column K-block kb at
 *       images + (((p * n_mtiles + mt) * kblocks + kb) * 2 + hl) * 16384, hl = 0 hi / 1 lo.  images: device buffer of
 *       gs_gather_mean_img_bytes(rows, F, want_self) bytes, 1024-byte aligned; rows = max(out_row0 + n).
 *       GS_ERR_UNSUPPORTED when the bulk-copy gather does not apply (F > 1280, unaligned pitch): use the fp32 pair.
 *   gs_sage_gemm_img : gs_sage_gemm_prepacked(math = GS_MATH_TF32X3) with part p's A operand = image part a_part0 + p
 *       (parts[].A / lda are ignored; every part's K = F).  Bit-identical results to the fp32-operand form.
 * Reference ops: tf.nn.embedding_lookup + reduce_mean + matmul + concat/add_n + relu (models.py:299,
 * aggregators.py:48-64 / 106-116).
 * --------------------------------------------------------------------------------------------- */
int64_t gs_gather_mean_img_bytes(int64_t rows, int32_t F, int32_t want_self);
int32_t gs_gather_mean_img(const void* src, int64_t n_src_rows, const gs_sharded_table* table_host, int32_t ids_are_locators,
                           const void* staging, int32_t F, int64_t pitch, const gs_segment* segments_host,
                           int32_t n_segments, int32_t include_self, int32_t want_self, void* images, void* stream);
int32_t gs_sage_gemm_img(int64_t M, const gs_gemm_part* parts_host, int32_t n_parts, int32_t combine, const float* bias,
                         int32_t act, float* out, int64_t ldo, const void* workspace, const void* a_images,
                         int32_t a_part0, void* stream);

/* ---------------------------------------------------------------------------------------------
 * One whole aggregator layer for a SMALL number of output rows (the last layers of the recursion:
 * 512 rows at batch 512) in one launch, exact fp32 FFMA:
 *   mean over the fanout (gs_gather_mean semantics, one segment) -> two (or one) matmuls ->
 *   add | concat -> + bias -> act -> optional row l2_normalize (reference aggregators.py:43-64 /
 *   101-116, models.py:368).  parts: part 0 multiplies the SELF rows, part 1 the MEAN rows; with
 *   n_parts == 1 the single part multiplies the mean rows (GCN form, include_self = 1).
 *   parts[i].A is ignored (the operands are produced in shared memory).
 *   If counter_dev != NULL, *counter_dev += counter_inc after the layer (advances the samplers'
 *   device-side call counter for the next CUDA-graph replay).
 * Limits: K_p <= 2048, total output width <= 1024.
 * --------------------------------------------------------------------------------------------- */
int32_t gs_sage_layer_small(const float* src, int64_t n_src_rows, int32_t F, int64_t pitch,
                            const gs_segment* segment_host, int32_t include_self,
                            const gs_gemm_part* parts_host, int32_t n_parts, int32_t combine,
                            const float* bias, int32_t act, int32_t l2_normalize,
                            float* out, int64_t ldo, uint64_t* counter_dev, uint64_t counter_inc,
                            void* stream);

/* ---------------------------------------------------------------------------------------------
 * K4 - the max-pool aggregator's neighbour branch fused end to end on tcgen05 (bf16 operands, fp32
 * accumulate):   out[g, h] = max_{j<k} relu( table[row(g,j), 0:K] . Wm[0:K, h] + bm[h] )
 *   reference graphsage/aggregators.py:176-182 (reshape -> Dense(relu,bias) -> reshape -> reduce_max),
 *   graphsage/layers.py:104-116, with the gather of graphsage/models.py:299 fused in front.
 *   row(g, j) = row_ids ? row_ids[g*k + j] : row0 + g*k + j;  table is bf16 [n_rows, pitch] (pitch % 8 == 0).
 *   packed_weights: gs_maxpool_mlp_pack(Wm fp32 [K, hidden] row-major) into gs_maxpool_mlp_workspace_bytes
 *   bytes (do it once per weight update).  Limits: K <= 640, k <= 128, hidden % 128 == 0 (else
 *   GS_ERR_UNSUPPORTED: use gs_gather_rows + gs_sage_gemm + gs_segment_max).
 * --------------------------------------------------------------------------------------------- */
int64_t gs_maxpool_mlp_workspace_bytes(int32_t K, int32_t hidden);
int32_t gs_maxpool_mlp_pack(const float* Wm, int64_t ldw, int32_t K, int32_t hidden, void* workspace,
                            void* stream);
int32_t gs_maxpool_mlp_fused(const void* table_bf16, int64_t n_rows, int32_t K, int64_t pitch,
                             const int32_t* row_ids, int64_t row0, int64_t n_groups, int32_t k,
                             const void* packed_weights, const float* bias, int32_t hidden,
                             float* out, int64_t ldo, void* stream);
/* MeanPoolingAggregator's neighbour branch (reference graphsage/aggregators.py:246-273): same kernel, the
 * epilogue averages relu(x + b) over the fanout instead of taking the max. */
int32_t gs_meanpool_mlp_fused(const void* table_bf16, int64_t n_rows, int32_t K, int64_t pitch,
                              const int32_t* row_ids, int64_t row0, int64_t n_groups, int32_t k,
                              const void* packed_weights, const float* bias, int32_t hidden,
                              float* out, int64_t ldo, void* stream);

/* ---------------------------------------------------------------------------------------------
 * SeqAggregator - the LSTM neighbour aggregator (reference graphsage/aggregators.py:363-449).
 *   gs_row_used : used[r] = 1 if any of x[r, 0:F] is non-zero, else 0 - tf.sign(tf.reduce_max(tf.abs(x), axis=-1))
 *       (aggregators.py:411).  dtype GS_F32 or GS_BF16; rows at stride `pitch`.
 *   gs_lstm_seq : tf.nn.dynamic_rnn(BasicLSTMCell(H), neigh_vecs, sequence_length = len) followed by the gather of each
 *       sequence's last valid output (aggregators.py:408-433), for n sequences of k steps in ONE launch:
 *         len_g = max(1, sum_{t<k} used[row(g, t)]),  row(g, t) = row_ids ? row_ids[g*k + t] : row0 + g*k + t
 *           (the count of non-zero rows; the recurrence still consumes the FIRST len_g rows, as dynamic_rnn does);
 *         gates_t = P[g*k + t, 0:4H] + h_{t-1} @ Wh   (h_{-1} = c_{-1} = 0), column blocks i, j, f, o;
 *         c_t = c_{t-1} * sigmoid(f + 1) + sigmoid(i) * tanh(j);  h_t = tanh(c_t) * sigmoid(o)   (forget_bias 1.0);
 *         out[g, 0:H] = h_{len_g - 1}.
 *       P is the input projection x_{g,t} @ kernel[0:in] + bias (fp32, row stride ldp >= 4H); Wh = kernel[in:in+H] is
 *       fp32 [H, 4H] row-major.  keep_h / keep_c (fp32 [n, k, H], may be NULL) receive h_t / c_t for t < len_g (rows
 *       t >= len_g are not written); lengths (int32 [n], may be NULL) receives len_g - the backward pass's inputs.
 *       Exact fp32 arithmetic (FFMA, expf / tanhf).  GS_ERR_UNSUPPORTED unless H % 32 == 0 and H <= 256.
 * --------------------------------------------------------------------------------------------- */
int32_t gs_row_used(const void* x, int32_t dtype, int64_t n_rows, int32_t F, int64_t pitch, uint8_t* used, void* stream);
int32_t gs_lstm_seq(const float* P, int64_t ldp, const float* Wh, int32_t H, const uint8_t* used, const int32_t* row_ids,
                    int64_t row0, int64_t n, int32_t k, float* out, int64_t ldo, float* keep_h, float* keep_c,
                    int32_t* lengths, void* stream);

/* ---------------------------------------------------------------------------------------------
 * One pipelined step from HOST buffers in a single call (no per-kernel host work), on three streams:
 *   h2d_stream     : wait ev_done (this slot's previous step no longer reads ids_dev), copy ids host->device,
 *                    record ev_ids
 *   compute_stream : wait ev_ids and ev_drained (this slot's previous result has left the device), launch the
 *                    captured CUDA graph(s) of the step, record ev_done
 *   copy_stream    : wait ev_done, copy the result device->host, record ev_drained
 * so the id upload of step i+1 and the result download of step i-1 both overlap the kernels of step i.
 * All handles are the caller's CUDA objects (cudaGraphExec_t, cudaStream_t, cudaEvent_t as void*); events must
 * have been recorded at least once; host buffers should be pinned.
 * --------------------------------------------------------------------------------------------- */
int32_t gs_pipeline_step(const void* ids_host, void* ids_dev, int64_t ids_bytes, void* const* graph_execs_host,
                         int32_t n_graphs, const void* out_dev, void* out_host, int64_t out_bytes,
                         void* h2d_stream, void* compute_stream, void* copy_stream, void* ev_ids, void* ev_done,
                         void* ev_drained);

/* *counter_dev += inc, on the stream: advances the samplers' device-side call counter once per step (the counter a
 * CUDA-graph replay reads, see gs_sample_padded) when the step's last kernel is not gs_sage_layer_small. */
int32_t gs_bump_counter(uint64_t* counter_dev, uint64_t inc, void* stream);

/* tf.nn.l2_normalize(x, 1)   reference graphsage/models.py:368-370, supervised_models.py:85 */
int32_t gs_l2_normalize_rows(float* x, int64_t n, int32_t C, int64_t ldx, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* GRAPHSAGE_B200_H_ */
