// The LSTM neighbour aggregator's recurrence (reference graphsage/aggregators.py:405-433, SeqAggregator._call):
//   gs_row_used  - sign(reduce_max(abs(x), axis=-1)) per row (:411), over an fp32 or bf16 matrix;
//   gs_lstm_seq  - dynamic_rnn(BasicLSTMCell(H), sequence_length = max(1, sum(used)))(:412-427) plus the gather of
//                  h_{len-1} (:428-433), the whole recurrence of one hop in one launch.
//
// gs_lstm_seq layout: a thread-block cluster of H/32 CTAs per tile of kS sequences.  CTA c owns hidden units
// [32c, 32c + 32) and all four gate columns of them (i, j, f, o), so the cell update is local to the thread that computed
// the gates.  Its Wh column slice [H, 4 x 32] stays in shared memory for the whole launch and c stays in registers.  Each
// step it writes its 32 units of h_t into the next buffer of every cluster CTA's double-buffered h tile [kS, H] through
// distributed shared memory, then one cluster barrier publishes them.  A tile runs to its longest len; rows that have
// finished keep computing (their results are never stored), which keeps every barrier uniform across the cluster.
#include <cooperative_groups.h>

#include "common.cuh"

namespace cg = cooperative_groups;

namespace gs {

constexpr int kLstmS = 32;                       // sequences per tile
constexpr int kLstmThreads = 256;                // 8 warps: warp w owns sequences [4w, 4w + 4), lane = hidden unit
constexpr int kLstmSeqPerThread = kLstmS / (kLstmThreads / 32);

__global__ void row_used_f32_kernel(const float* __restrict__ x, int64_t n_rows, int32_t F, int64_t pitch,
                                    uint8_t* __restrict__ used) {
  const int lane = threadIdx.x & 31;
  const int64_t warps = (int64_t)gridDim.x * (blockDim.x / 32);
  for (int64_t r = (int64_t)blockIdx.x * (blockDim.x / 32) + threadIdx.x / 32; r < n_rows; r += warps) {
    const float* row = x + r * pitch;
    bool nz = false;
    for (int c = lane; c < F; c += 32) nz |= row[c] != 0.0f;
    nz = __any_sync(0xffffffffu, nz);
    if (lane == 0) used[r] = nz ? 1 : 0;
  }
}

__global__ void row_used_bf16_kernel(const uint16_t* __restrict__ x, int64_t n_rows, int32_t F, int64_t pitch,
                                     uint8_t* __restrict__ used) {
  const int lane = threadIdx.x & 31;
  const int64_t warps = (int64_t)gridDim.x * (blockDim.x / 32);
  for (int64_t r = (int64_t)blockIdx.x * (blockDim.x / 32) + threadIdx.x / 32; r < n_rows; r += warps) {
    const uint16_t* row = x + r * pitch;
    bool nz = false;
    for (int c = lane; c < F; c += 32) nz |= (row[c] & 0x7fffu) != 0;     // +-0 are zero
    nz = __any_sync(0xffffffffu, nz);
    if (lane == 0) used[r] = nz ? 1 : 0;
  }
}

__device__ __forceinline__ float sigmoidf_exact(float x) { return 1.0f / (1.0f + expf(-x)); }

// NC = H / 32 = CTAs per cluster.  Dynamic shared memory: Wh slice [H][128] then h[2][kS][H] then len[kS].
template <int NC>
__global__ void __launch_bounds__(kLstmThreads) lstm_seq_kernel(
    const float* __restrict__ P, int64_t ldp, const float* __restrict__ Wh, const uint8_t* __restrict__ used,
    const int32_t* __restrict__ row_ids, int64_t row0, int64_t n, int32_t k, float* __restrict__ out, int64_t ldo,
    float* __restrict__ keep_h, float* __restrict__ keep_c, int32_t* __restrict__ lengths, int64_t n_tiles) {
  constexpr int H = NC * 32;
  extern __shared__ __align__(16) float smem[];
  float* ws = smem;                                        // ws[kk * 128 + gate * 32 + u] = Wh[kk, gate * H + 32c + u]
  float* hbuf = ws + H * 128;                              // hbuf[b][s][kk]
  int* lens = (int*)(hbuf + 2 * kLstmS * H);
  cg::cluster_group cluster = cg::this_cluster();
  const int rank = (int)cluster.block_rank();
  const int u = threadIdx.x & 31;
  const int s0 = (threadIdx.x >> 5) * kLstmSeqPerThread;
  const int unit = rank * 32 + u;

  for (int i = threadIdx.x; i < H * 128; i += kLstmThreads) {
    const int kk = i >> 7, col = i & 127;
    ws[i] = Wh[(int64_t)kk * 4 * H + (col >> 5) * H + rank * 32 + (col & 31)];
  }
  float* peer_h[NC];
#pragma unroll
  for (int r = 0; r < NC; ++r) peer_h[r] = cluster.map_shared_rank(hbuf, r);

  const int64_t n_clusters = gridDim.x / NC;
  for (int64_t tile = blockIdx.x / NC; tile < n_tiles; tile += n_clusters) {
    const int64_t g0 = tile * kLstmS;
    if (threadIdx.x < kLstmS) {                            // len_g = max(1, sum_t used[row(g, t)])   (:411-414)
      const int64_t g = g0 + threadIdx.x;
      int len = 0;
      if (g < n) {
        for (int t = 0; t < k; ++t) {
          const int64_t q = g * k + t;
          len += used[row_ids ? (int64_t)row_ids[q] : row0 + q] ? 1 : 0;
        }
        if (len < 1) len = 1;
        if (lengths && rank == 0) lengths[g] = len;
      }
      lens[threadIdx.x] = len;                             // 0 for the padding rows of a ragged last tile
    }
    for (int i = threadIdx.x; i < kLstmS * H; i += kLstmThreads) hbuf[i] = 0.0f;   // h_{-1} = 0 (zero_state)
    __syncthreads();
    int T = 0;
    for (int s = 0; s < kLstmS; ++s) T = max(T, lens[s]);
    int mylen[kLstmSeqPerThread];
    float c[kLstmSeqPerThread];
#pragma unroll
    for (int i = 0; i < kLstmSeqPerThread; ++i) {
      mylen[i] = lens[s0 + i];
      c[i] = 0.0f;
    }
    cluster.sync();                                        // every CTA's h_{-1} is zero before anyone writes h_0

    for (int t = 0; t < T; ++t) {
      const float* hcur = hbuf + (t & 1) * kLstmS * H;
      float acc[kLstmSeqPerThread][4];
      float pin[kLstmSeqPerThread][4];
#pragma unroll
      for (int i = 0; i < kLstmSeqPerThread; ++i) {      // input projection x_t @ W_x + b, consumed after the h @ Wh loop
        const int64_t g = g0 + s0 + i;
        const float* prow = P + (g < n ? (g * k + t) : 0) * ldp + unit;
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          pin[i][q] = g < n ? __ldg(prow + q * H) : 0.0f;
          acc[i][q] = 0.0f;
        }
      }
#pragma unroll 2
      for (int kk = 0; kk < H; kk += 4) {
        float4 hv[kLstmSeqPerThread];
#pragma unroll
        for (int i = 0; i < kLstmSeqPerThread; ++i) hv[i] = *(const float4*)(hcur + (s0 + i) * H + kk);
#pragma unroll
        for (int d = 0; d < 4; ++d) {
          float w[4];
#pragma unroll
          for (int q = 0; q < 4; ++q) w[q] = ws[(kk + d) * 128 + q * 32 + u];
#pragma unroll
          for (int i = 0; i < kLstmSeqPerThread; ++i) {
            const float hx = d == 0 ? hv[i].x : d == 1 ? hv[i].y : d == 2 ? hv[i].z : hv[i].w;
#pragma unroll
            for (int q = 0; q < 4; ++q) acc[i][q] = fmaf(hx, w[q], acc[i][q]);
          }
        }
      }
      float* hnext_off = hbuf + ((t + 1) & 1) * kLstmS * H;
      const int64_t off_next = hnext_off - hbuf;
#pragma unroll
      for (int i = 0; i < kLstmSeqPerThread; ++i) {
        // BasicLSTMCell: i, j, f, o = split(gates); c = c * sigmoid(f + forget_bias) + sigmoid(i) * tanh(j);
        // h = tanh(c) * sigmoid(o)   (forget_bias = 1.0)
        const float gi = pin[i][0] + acc[i][0], gj = pin[i][1] + acc[i][1];
        const float gf = pin[i][2] + acc[i][2], go = pin[i][3] + acc[i][3];
        const float cn = c[i] * sigmoidf_exact(gf + 1.0f) + sigmoidf_exact(gi) * tanhf(gj);
        const float hn = tanhf(cn) * sigmoidf_exact(go);
        c[i] = cn;
        const int s = s0 + i;
#pragma unroll
        for (int r = 0; r < NC; ++r) peer_h[r][off_next + s * H + unit] = hn;
        if (t < mylen[i]) {
          const int64_t g = g0 + s;
          if (keep_h) keep_h[(g * k + t) * H + unit] = hn;
          if (keep_c) keep_c[(g * k + t) * H + unit] = cn;
          if (t == mylen[i] - 1) out[g * ldo + unit] = hn;        // neigh_h = h_{len-1}   (:428-433)
        }
      }
      cluster.sync();                                      // h_t is complete in every CTA; h_{t-1} is no longer read
    }
  }
}

template <int NC>
int32_t launch_lstm_seq(const float* P, int64_t ldp, const float* Wh, const uint8_t* used, const int32_t* row_ids,
                        int64_t row0, int64_t n, int32_t k, float* out, int64_t ldo, float* keep_h, float* keep_c,
                        int32_t* lengths, cudaStream_t st) {
  constexpr int H = NC * 32;
  const int smem = (H * 128 + 2 * kLstmS * H) * (int)sizeof(float) + kLstmS * (int)sizeof(int);
  const void* fn = (const void*)lstm_seq_kernel<NC>;
  const int32_t rc = ensure_dyn_smem(fn, smem);
  if (rc != GS_OK) return rc;
  const int64_t n_tiles = (n + kLstmS - 1) / kLstmS;
  cudaLaunchConfig_t cfg = {};
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = NC;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.blockDim = dim3(kLstmThreads, 1, 1);
  cfg.dynamicSmemBytes = (size_t)smem;
  cfg.stream = st;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  // persistent clusters: as many as can be resident (one Wh slice load per cluster), never more than there are tiles
  static int resident[64][9] = {};
  int dev = 0;
  GS_CUDA(cudaGetDevice(&dev));
  if (dev < 0 || dev >= 64) dev = 0;
  if (resident[dev][NC] == 0) {
    int clusters = 0;
    cfg.gridDim = dim3(NC * 148, 1, 1);
    if (cudaOccupancyMaxActiveClusters(&clusters, fn, &cfg) != cudaSuccess || clusters <= 0) {
      (void)cudaGetLastError();
      clusters = sm_count() / NC;
    }
    resident[dev][NC] = clusters;
  }
  int64_t clusters = resident[dev][NC];
  if (clusters > n_tiles) clusters = n_tiles;
  cfg.gridDim = dim3((unsigned)(clusters * NC), 1, 1);
  GS_CUDA(cudaLaunchKernelEx(&cfg, lstm_seq_kernel<NC>, P, ldp, Wh, used, row_ids, row0, n, k, out, ldo, keep_h, keep_c,
                             lengths, n_tiles));
  return launch_check("lstm_seq_kernel");
}

}  // namespace gs

extern "C" {

int32_t gs_row_used(const void* x, int32_t dtype, int64_t n_rows, int32_t F, int64_t pitch, uint8_t* used,
                    void* stream) {
  GS_REQUIRE(n_rows >= 0 && F >= 0 && pitch >= F, "gs_row_used: bad sizes");
  if (n_rows == 0) return GS_OK;
  GS_REQUIRE(x && used, "gs_row_used: NULL pointer");
  GS_REQUIRE(dtype == GS_F32 || dtype == GS_BF16, "gs_row_used: dtype %d", dtype);
  int64_t blocks = (n_rows + 7) / 8;
  const int64_t cap = (int64_t)gs::sm_count() * 8;
  if (blocks > cap) blocks = cap;
  if (dtype == GS_F32)
    gs::row_used_f32_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>((const float*)x, n_rows, F, pitch, used);
  else
    gs::row_used_bf16_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>((const uint16_t*)x, n_rows, F, pitch,
                                                                                  used);
  return gs::launch_check("row_used_kernel");
}

int32_t gs_lstm_seq(const float* P, int64_t ldp, const float* Wh, int32_t H, const uint8_t* used, const int32_t* row_ids,
                    int64_t row0, int64_t n, int32_t k, float* out, int64_t ldo, float* keep_h, float* keep_c,
                    int32_t* lengths, void* stream) {
  if (H <= 0 || H % 32 != 0 || H > 256) {
    gs::set_error("gs_lstm_seq: H = %d (needs a multiple of 32, at most 256)", H);
    return GS_ERR_UNSUPPORTED;
  }
  GS_REQUIRE(n >= 0 && k >= 1, "gs_lstm_seq: bad sizes (n=%lld, k=%d)", (long long)n, k);
  if (n == 0) return GS_OK;
  GS_REQUIRE(P && Wh && used && out, "gs_lstm_seq: NULL pointer");
  GS_REQUIRE(ldp >= 4 * (int64_t)H && ldo >= H, "gs_lstm_seq: ldp < 4H or ldo < H");
  cudaStream_t st = (cudaStream_t)stream;
  switch (H / 32) {
    case 1: return gs::launch_lstm_seq<1>(P, ldp, Wh, used, row_ids, row0, n, k, out, ldo, keep_h, keep_c, lengths, st);
    case 2: return gs::launch_lstm_seq<2>(P, ldp, Wh, used, row_ids, row0, n, k, out, ldo, keep_h, keep_c, lengths, st);
    case 3: return gs::launch_lstm_seq<3>(P, ldp, Wh, used, row_ids, row0, n, k, out, ldo, keep_h, keep_c, lengths, st);
    case 4: return gs::launch_lstm_seq<4>(P, ldp, Wh, used, row_ids, row0, n, k, out, ldo, keep_h, keep_c, lengths, st);
    case 5: return gs::launch_lstm_seq<5>(P, ldp, Wh, used, row_ids, row0, n, k, out, ldo, keep_h, keep_c, lengths, st);
    case 6: return gs::launch_lstm_seq<6>(P, ldp, Wh, used, row_ids, row0, n, k, out, ldo, keep_h, keep_c, lengths, st);
    case 7: return gs::launch_lstm_seq<7>(P, ldp, Wh, used, row_ids, row0, n, k, out, ldo, keep_h, keep_c, lengths, st);
    default: return gs::launch_lstm_seq<8>(P, ldp, Wh, used, row_ids, row0, n, k, out, ldo, keep_h, keep_c, lengths, st);
  }
}

}  // extern "C"
