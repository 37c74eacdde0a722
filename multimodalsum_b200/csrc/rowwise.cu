// HBM-bound kernels of the MultimodalSum step: vectorised (128-bit) loads, warp-shuffle reductions, one warp per
// 1024-wide row.  Everything here is memory-bound; the roofline is achieved GB/s vs the measured HBM peak.
//   cast / embedding-gather+LayerNorm(+dropout) / residual+dropout+LayerNorm fwd+bwd / column sums (bias grads) /
//   gate fusion fwd+bwd / label-smoothed cross-entropy fwd+bwd / input preparation (shift_tokens_right, masks,
//   leave-one-out bookkeeping) / table-encoder front end.
#include "common.cuh"
#include "../../include/mmsum_b200.h"

namespace mmsum {

static constexpr int D = 1024;          // d_model (fixed by the reference's table / image heads, src/table_encoder.py:8-12)
static constexpr int VPL = D / 32;      // values per lane = 32
static constexpr float kEps = 1e-5f;

// step_dev (optional): device-resident step counter folded into the stream id inside the kernel, so that a recorded CUDA graph
// of the training step draws fresh masks at every replay (the stream id passed by value would be baked into the graph)
struct DropCfg { unsigned long long seed; uint32_t stream; uint32_t thr16; float scale; const uint32_t* step_dev; };
__host__ inline DropCfg make_drop(float p, unsigned long long seed, uint32_t stream, const uint32_t* step_dev = nullptr) {
  DropCfg d; d.seed = seed; d.stream = stream; d.step_dev = step_dev;
  if (p <= 0.f) { d.thr16 = 65536; d.scale = 1.f; }
  else { uint32_t t = (uint32_t)((1.0 - (double)p) * 65536.0 + 0.5); if (t < 1) t = 1; d.thr16 = t; d.scale = 65536.f / (float)t; }
  return d;
}
__device__ __forceinline__ DropCfg resolve_drop(DropCfg d) {
  if (d.step_dev != nullptr && d.thr16 < 65536) d.stream += d.step_dev[0] * 4096u;
  return d;
}
// dropout multiplier for elements (idx, idx+1) of a tensor; idx even
__device__ __forceinline__ float2 drop_pair(const DropCfg& d, unsigned long long idx) {
  if (d.thr16 >= 65536) return make_float2(1.f, 1.f);
  const uint32_t r = dropout_rand(d.seed, d.stream, idx >> 1);
  return make_float2(((r & 0xFFFF) < d.thr16) ? d.scale : 0.f, ((r >> 16) < d.thr16) ? d.scale : 0.f);
}

// lane owns columns: for j in 0..3: [j*256 + lane*8, +8)
__device__ __forceinline__ void load_row_bf16(const bf16* row, int lane, float (&v)[VPL]) {
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const uint4 u = *reinterpret_cast<const uint4*>(row + j * 256 + lane * 8);
    const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
    for (int e = 0; e < 4; ++e) { const float2 f = unpack_bf16(w[e]); v[j * 8 + 2 * e] = f.x; v[j * 8 + 2 * e + 1] = f.y; }
  }
}
__device__ __forceinline__ void store_row_bf16(bf16* row, int lane, const float (&v)[VPL]) {
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    uint4 u;
    u.x = pack_bf16(v[j * 8 + 0], v[j * 8 + 1]); u.y = pack_bf16(v[j * 8 + 2], v[j * 8 + 3]);
    u.z = pack_bf16(v[j * 8 + 4], v[j * 8 + 5]); u.w = pack_bf16(v[j * 8 + 6], v[j * 8 + 7]);
    *reinterpret_cast<uint4*>(row + j * 256 + lane * 8) = u;
  }
}
__device__ __forceinline__ void load_row_f32(const float* row, int lane, float (&v)[VPL]) {
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const float4 a = *reinterpret_cast<const float4*>(row + j * 256 + lane * 8);
    const float4 b = *reinterpret_cast<const float4*>(row + j * 256 + lane * 8 + 4);
    v[j * 8 + 0] = a.x; v[j * 8 + 1] = a.y; v[j * 8 + 2] = a.z; v[j * 8 + 3] = a.w;
    v[j * 8 + 4] = b.x; v[j * 8 + 5] = b.y; v[j * 8 + 6] = b.z; v[j * 8 + 7] = b.w;
  }
}
__device__ __forceinline__ int col_of(int lane, int i) { return (i >> 3) * 256 + lane * 8 + (i & 7); }
// per-column fp32 vector (gamma, beta) in the same lane layout, coalesced 128-bit loads
__device__ __forceinline__ void load_cols_f32(const float* __restrict__ v, int lane, float (&o)[VPL]) { load_row_f32(v, lane, o); }

__device__ __forceinline__ void ln_stats(const float (&z)[VPL], float& mean, float& rstd) {
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < VPL; ++i) s += z[i];
  mean = warp_sum(s) * (1.f / D);
  float q = 0.f;
#pragma unroll
  for (int i = 0; i < VPL; ++i) { const float d = z[i] - mean; q += d * d; }
  rstd = rsqrtf(warp_sum(q) * (1.f / D) + kEps);
}

// ------------------------------------------------------------------ cast
__global__ void cast_f32_bf16_kernel(const float* __restrict__ src, bf16* __restrict__ dst, long long n) {
  const long long stride = (long long)gridDim.x * blockDim.x * 8;
  for (long long i = ((long long)blockIdx.x * blockDim.x + threadIdx.x) * 8; i < n; i += stride) {
    if (i + 8 <= n) {
      const float4 a = *reinterpret_cast<const float4*>(src + i);
      const float4 b = *reinterpret_cast<const float4*>(src + i + 4);
      uint4 u; u.x = pack_bf16(a.x, a.y); u.y = pack_bf16(a.z, a.w); u.z = pack_bf16(b.x, b.y); u.w = pack_bf16(b.z, b.w);
      *reinterpret_cast<uint4*>(dst + i) = u;
    } else {
      for (long long k = i; k < n; ++k) dst[k] = __float2bfloat16_rn(src[k]);
    }
  }
}

// ------------------------------------------------------------------ embedding gather + LN (+dropout)
// out[row] = dropout(LN(E[ids[row]] + P[row % S + 2] + rating_diff[row / S] * r))     (BartEncoder.forward :368-372,
// BartDecoder.forward :588-597, LearnedPositionalEmbedding :961-969).  Tables are read in fp32 (exact gather).
__global__ void __launch_bounds__(256) embed_ln_fwd_kernel(const int* __restrict__ ids, const float* __restrict__ E,
                                                           const float* __restrict__ P, const float* __restrict__ rating_diff,
                                                           const float* __restrict__ remb, const float* __restrict__ gamma,
                                                           const float* __restrict__ beta, bf16* __restrict__ out,
                                                           float* __restrict__ mean_o, float* __restrict__ rstd_o,
                                                           int rows, int S, DropCfg dc_in, const int* __restrict__ pos_dev) {
  const DropCfg dc = resolve_drop(dc_in);
  const int lane = threadIdx.x & 31;
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= rows) return;
  float z[VPL], p[VPL];
  load_row_f32(E + (long long)ids[row] * D, lane, z);
  // decode steps: every row sits at the same position, read from device memory (the launch is replayed from a CUDA graph)
  const int pos = (pos_dev != nullptr) ? pos_dev[0] : (row % S);
  load_row_f32(P + (long long)(pos + 2) * D, lane, p);
#pragma unroll
  for (int i = 0; i < VPL; ++i) z[i] += p[i];
  if (rating_diff != nullptr) {
    const float rd = rating_diff[row / S];
    load_row_f32(remb, lane, p);
#pragma unroll
    for (int i = 0; i < VPL; ++i) z[i] += rd * p[i];
  }
  float mean, rstd;
  ln_stats(z, mean, rstd);
  if (lane == 0) { mean_o[row] = mean; rstd_o[row] = rstd; }
#pragma unroll
  for (int i = 0; i < VPL; i += 2) {
    const int c = col_of(lane, i);
    const float2 m = drop_pair(dc, (unsigned long long)row * D + c);
    z[i] = ((z[i] - mean) * rstd * gamma[c] + beta[c]) * m.x;
    z[i + 1] = ((z[i + 1] - mean) * rstd * gamma[c + 1] + beta[c + 1]) * m.y;
  }
  store_row_bf16(out + (long long)row * D, lane, z);
}

// backward of the above: dz (fp32, [rows, D]) for the position / rating reductions, scatter-add into dE (pad id
// skipped: nn.Embedding(padding_idx=1)), dgamma/dbeta.
// kOrdered: no dE scatter (embed_group_kernel + embed_scatter_tile/span_kernel add the dz rows per token id instead) and the
// block's dgamma / dbeta sums go to its own row of `partial` [gridDim.x][2 * D] (ordered_colsum_kernel adds them up).
// dE == NULL: no scatter; dgamma == NULL (then dbeta == NULL too): no gamma / beta flush.  dz is always written.
template <bool kOrdered>
__global__ void __launch_bounds__(256) embed_ln_bwd_kernel(const bf16* __restrict__ dout, const bf16* __restrict__ dout2,
                                                           const int* __restrict__ ids,
                                                           const float* __restrict__ E, const float* __restrict__ P,
                                                           const float* __restrict__ rating_diff, const float* __restrict__ remb,
                                                           const float* __restrict__ gamma, const float* __restrict__ mean_i,
                                                           const float* __restrict__ rstd_i, float* __restrict__ dE,
                                                           float* __restrict__ dz_out, float* __restrict__ dgamma,
                                                           float* __restrict__ dbeta, int rows, int S, int pad_id, DropCfg dc_in,
                                                           float* __restrict__ partial) {
  const DropCfg dc = resolve_drop(dc_in);
  __shared__ float sg[8][D / 4];  // staged reduction of dgamma / dbeta across the block's warps (two passes of D/4... see below)
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
  float ag[VPL], ab[VPL];
#pragma unroll
  for (int i = 0; i < VPL; ++i) { ag[i] = 0.f; ab[i] = 0.f; }
  for (int row = blockIdx.x * nw + warp; row < rows; row += gridDim.x * nw) {
    float z[VPL], p[VPL], dy[VPL];
    const int id = ids[row];
    load_row_f32(E + (long long)id * D, lane, z);
    load_row_f32(P + (long long)((row % S) + 2) * D, lane, p);
#pragma unroll
    for (int i = 0; i < VPL; ++i) z[i] += p[i];
    if (rating_diff != nullptr) {
      const float rd = rating_diff[row / S];
      load_row_f32(remb, lane, p);
#pragma unroll
      for (int i = 0; i < VPL; ++i) z[i] += rd * p[i];
    }
    load_row_bf16(dout + (long long)row * D, lane, dy);
    if (dout2 != nullptr) {
      load_row_bf16(dout2 + (long long)row * D, lane, p);
#pragma unroll
      for (int i = 0; i < VPL; ++i) dy[i] += p[i];
    }
    const float mean = mean_i[row], rstd = rstd_i[row];
    float s1 = 0.f, s2 = 0.f;
#pragma unroll
    for (int i = 0; i < VPL; i += 2) {
      const int c = col_of(lane, i);
      const float2 m = drop_pair(dc, (unsigned long long)row * D + c);
      dy[i] *= m.x; dy[i + 1] *= m.y;
    }
#pragma unroll
    for (int i = 0; i < VPL; ++i) {
      const int c = col_of(lane, i);
      const float xh = (z[i] - mean) * rstd;
      ag[i] += dy[i] * xh; ab[i] += dy[i];
      const float dxh = dy[i] * gamma[c];
      s1 += dxh; s2 += dxh * xh;
      z[i] = xh; dy[i] = dxh;
    }
    s1 = warp_sum(s1) * (1.f / D); s2 = warp_sum(s2) * (1.f / D);
    float* dzr = dz_out + (long long)row * D;
    float* der = dE + (long long)id * D;
#pragma unroll
    for (int i = 0; i < VPL; ++i) {
      const int c = col_of(lane, i);
      const float dz = rstd * (dy[i] - s1 - z[i] * s2);
      dzr[c] = dz;
      if (!kOrdered && dE != nullptr && id != pad_id) atomicAdd(der + c, dz);
    }
  }
  if (dgamma == nullptr) return;   // uniform over the block
  // block reduce dgamma/dbeta then one atomic per column per block
  for (int pass = 0; pass < 2; ++pass) {
    float* acc = pass == 0 ? ag : ab;
    float* dst = pass == 0 ? dgamma : dbeta;
    for (int quarter = 0; quarter < 4; ++quarter) {
      __syncthreads();
#pragma unroll
      for (int i = 0; i < 8; ++i) sg[warp][lane * 8 + i] = acc[quarter * 8 + i];
      __syncthreads();
      for (int c = threadIdx.x; c < 256; c += blockDim.x) {
        float s = 0.f;
        for (int w = 0; w < nw; ++w) s += sg[w][c];
        if (kOrdered) partial[(long long)blockIdx.x * 2 * D + pass * D + quarter * 256 + c] = s;
        else          atomicAdd(dst + quarter * 256 + c, s);
      }
    }
  }
}

// dP[t+2] += sum_seq dz[seq*S+t],  dremb += sum_rows rating_diff[seq] * dz[row]   (dP or dremb may be NULL: not written)
// (every dP element has exactly one writer, so its single atomic is already order-free; the S blocks of a column all add into
//  dremb, so kOrdered stores the position's dremb sum to partial[t][c] instead, summed over t by ordered_colsum_kernel)
template <bool kOrdered>
__global__ void __launch_bounds__(256) embed_pos_bwd_kernel(const float* __restrict__ dz, const float* __restrict__ rating_diff,
                                                            float* __restrict__ dP, float* __restrict__ dremb, int n_seq, int S,
                                                            float* __restrict__ partial) {
  // grid: (D/256, S); thread = one column, loops over sequences
  const int c = blockIdx.x * 256 + threadIdx.x;
  const int t = blockIdx.y;
  const bool remb_on = rating_diff != nullptr && dremb != nullptr;
  float s = 0.f, r = 0.f;
  for (int q = 0; q < n_seq; ++q) {
    const float v = dz[((long long)q * S + t) * D + c];
    s += v;
    if (remb_on) r += rating_diff[q] * v;
  }
  if (dP != nullptr) atomicAdd(dP + (long long)(t + 2) * D + c, s);
  if (remb_on) {
    if (kOrdered) partial[(long long)t * D + c] = r;
    else          atomicAdd(dremb + c, r);
  }
}

// ---- ordered (bitwise-reproducible) reductions
// out0[c] += sum_p part[p * width + c] for c < split, out1[c - split] += ... otherwise; the parts are summed in a fixed tree:
// row group g of the block sums parts g, g + 8, g + 16, ... in order, then the 8 group sums are added in order g = 0..7.
__global__ void __launch_bounds__(256) ordered_colsum_kernel(const float* __restrict__ part, int nparts, int width, int split,
                                                             float* __restrict__ out0, float* __restrict__ out1) {
  __shared__ float sm[8][32];
  const int cl = threadIdx.x & 31, grp = threadIdx.x >> 5;
  const int c = blockIdx.x * 32 + cl;
  float s = 0.f;
  if (c < width)
    for (int p = grp; p < nparts; p += 8) s += part[(long long)p * width + c];
  sm[grp][cl] = s;
  __syncthreads();
  if (grp == 0 && c < width) {
    float t = 0.f;
#pragma unroll
    for (int g = 0; g < 8; ++g) t += sm[g][cl];
    if (c < split) out0[c] += t;
    else           out1[c - split] += t;
  }
}

// inclusive block scan over 1024 threads (op: sum or max), scratch `ws` >= 32 ints
template <bool kMax>
__device__ __forceinline__ int block_scan_1024(int v, int* ws) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int u = __shfl_up_sync(0xffffffffu, v, o);
    if (lane >= o) v = kMax ? max(v, u) : v + u;
  }
  if (lane == 31) ws[warp] = v;
  __syncthreads();
  if (warp == 0) {
    int w = ws[lane];
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int u = __shfl_up_sync(0xffffffffu, w, o);
      if (lane >= o) w = kMax ? max(w, u) : w + u;
    }
    ws[lane] = w;
  }
  __syncthreads();
  if (warp > 0) { const int u = ws[warp - 1]; v = kMax ? max(v, u) : v + u; }
  __syncthreads();
  return v;
}

// Stable grouping of the rows by token id (one block of 1024 threads): a counting sort.  cursor [V + 1] ints: histogram, then
// exclusive offsets, and on return the END of each id's group; cursor[V] = number of non-pad rows.  order [rows]: the non-pad
// row indices sorted by (id, row); sid [rows]: the id at each sorted position.  The rows are placed 1024 at a time in row order;
// inside a tile, a bitonic sort of (id << 10 | lane) ranks rows of the same id by row.
__global__ void __launch_bounds__(1024) embed_group_kernel(const int* __restrict__ ids, int rows, int V, int pad_id,
                                                           int* __restrict__ cursor, int* __restrict__ order, int* __restrict__ sid) {
  __shared__ unsigned keys[1024];
  __shared__ int ws[32];
  const int tid = threadIdx.x;
  for (int i = tid; i < V; i += 1024) cursor[i] = 0;
  __syncthreads();
  for (int r = tid; r < rows; r += 1024) {
    const int id = ids[r];
    if (id != pad_id && id >= 0 && id < V) atomicAdd(&cursor[id], 1);    // integer counts: order-free
  }
  __syncthreads();
  const int per = (V + 1023) / 1024;
  const int b0 = min(V, tid * per), b1 = min(V, b0 + per);
  int cnt = 0;
  for (int i = b0; i < b1; ++i) cnt += cursor[i];
  const int incl = block_scan_1024<false>(cnt, ws);
  int run = incl - cnt;
  for (int i = b0; i < b1; ++i) { const int c = cursor[i]; cursor[i] = run; run += c; }
  if (tid == 1023) cursor[V] = incl;
  __syncthreads();
  for (int base = 0; base < rows; base += 1024) {
    const int r = base + tid;
    const int id = r < rows ? ids[r] : -1;
    const bool valid = r < rows && id != pad_id && id >= 0 && id < V;
    keys[tid] = valid ? (((unsigned)id << 10) | (unsigned)tid) : 0xFFFFFFFFu;
    __syncthreads();
    for (int k = 2; k <= 1024; k <<= 1)
      for (int j = k >> 1; j > 0; j >>= 1) {
        const int p = tid ^ j;
        if (p > tid) {
          const unsigned a = keys[tid], b = keys[p];
          if ((a > b) == ((tid & k) == 0)) { keys[tid] = b; keys[p] = a; }
        }
        __syncthreads();
      }
    const unsigned key = keys[tid];
    const unsigned kid = key >> 10;
    const bool first = tid == 0 || (keys[tid - 1] >> 10) != kid;
    const bool last = tid == 1023 || (keys[tid + 1] >> 10) != kid;
    const int start = block_scan_1024<true>(first ? tid : 0, ws);
    const int rank = tid - start;
    const bool v = key != 0xFFFFFFFFu;
    if (v) { order[cursor[kid] + rank] = base + (int)(key & 1023u); sid[cursor[kid] + rank] = (int)kid; }
    __syncthreads();
    if (v && last) cursor[kid] += rank + 1;
    __syncthreads();
  }
}

// dE[id] += sum of the dz rows of that id, in a fixed order, with one read-modify-write per element.  The sorted positions are
// cut into tiles of kScatterTile; embed_scatter_tile_kernel sums each (id, tile) segment in row order.  A group inside one tile
// is added to dE there; a group that spans tiles leaves its first segment in tail[tile] and every later one in head[tile], and
// embed_scatter_span_kernel adds tail + head + head + ... in tile order.  So no group is summed by one long serial chain.
static constexpr int kScatterTile = 64;
__global__ void __launch_bounds__(256) embed_scatter_tile_kernel(const float* __restrict__ dz, const int* __restrict__ sid,
                                                                 const int* __restrict__ order, const int* __restrict__ cursor,
                                                                 int V, float* __restrict__ dE, float* __restrict__ head,
                                                                 float* __restrict__ tail) {
  __shared__ int s_row[kScatterTile], s_id[kScatterTile + 2];     // s_id[0]: id before the tile, s_id[n + 1]: id after it
  const int total = cursor[V];
  const int t = blockIdx.x, p0 = t * kScatterTile;
  if (p0 >= total) return;
  const int n = min(kScatterTile, total - p0);
  if (threadIdx.x < n) { s_row[threadIdx.x] = order[p0 + threadIdx.x]; s_id[threadIdx.x + 1] = sid[p0 + threadIdx.x]; }
  if (threadIdx.x == 0) { s_id[0] = p0 > 0 ? sid[p0 - 1] : -1; s_id[n + 1] = p0 + n < total ? sid[p0 + n] : -1; }
  __syncthreads();
  const int c = blockIdx.y * 256 + threadIdx.x;
  float acc = 0.f;
  int seg = 0;
  for (int i = 0; i < n; ++i) {
    acc += dz[(long long)s_row[i] * D + c];
    if (i == n - 1 || s_id[i + 2] != s_id[i + 1]) {              // the segment ends at i
      const int id = s_id[i + 1];
      if (seg == 0 && s_id[0] == id)                  head[(long long)t * D + c] = acc;   // continues a group
      else if (i == n - 1 && s_id[n + 1] == id)       tail[(long long)t * D + c] = acc;   // starts a group that continues
      else                                            dE[(long long)id * D + c] += acc;   // the whole group
      acc = 0.f;
      seg = i + 1;
    }
  }
}

__global__ void __launch_bounds__(256) embed_scatter_span_kernel(const int* __restrict__ sid, const int* __restrict__ cursor, int V,
                                                                 const float* __restrict__ head, const float* __restrict__ tail,
                                                                 float* __restrict__ dE) {
  const int total = cursor[V];
  const int c = blockIdx.y * 256 + threadIdx.x;
  for (int p = blockIdx.x; p < total; p += gridDim.x) {
    const int id = sid[p];
    if (p > 0 && sid[p - 1] == id) continue;
    const int ts = p / kScatterTile, te = (cursor[id] - 1) / kScatterTile;      // cursor[id]: end of the group
    if (ts == te) continue;
    float acc = tail[(long long)ts * D + c];
    for (int t = ts + 1; t <= te; ++t) acc += head[(long long)t * D + c];
    dE[(long long)id * D + c] += acc;
  }
}

// ------------------------------------------------------------------ residual + dropout + LayerNorm
// out = LN(res + dropout(y))   (EncoderLayer.forward :288-308, DecoderLayer.forward :442-489, post-LN)
// Persistent: the grid covers the SMs a fixed number of times and every warp walks rows with the NEXT row's 8 loads already
// in flight while it normalises the current one (one warp per row and one row per warp ran at 0.55 of the HBM peak: five
// and a fraction waves of short blocks, each exposing its own load latency).
__global__ void __launch_bounds__(256, 2) add_ln_fwd_kernel(const bf16* __restrict__ res, const bf16* __restrict__ y,
                                                            const float* __restrict__ gamma, const float* __restrict__ beta,
                                                            bf16* __restrict__ out, float* __restrict__ mean_o,
                                                            float* __restrict__ rstd_o, int rows, DropCfg dc_in) {
  pdl_launch_dependents();
  pdl_wait();
  const DropCfg dc = resolve_drop(dc_in);
  const int lane = threadIdx.x & 31;
  const int stride = gridDim.x * (blockDim.x >> 5);
  int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= rows) return;
  uint4 ny[4], nr[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    ny[j] = *reinterpret_cast<const uint4*>(y + (long long)row * D + j * 256 + lane * 8);
    nr[j] = *reinterpret_cast<const uint4*>(res + (long long)row * D + j * 256 + lane * 8);
  }
  for (; row < rows; row += stride) {
    uint4 cy[4], cr[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) { cy[j] = ny[j]; cr[j] = nr[j]; }
    const int nxt = row + stride;
    if (nxt < rows) {
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        ny[j] = *reinterpret_cast<const uint4*>(y + (long long)nxt * D + j * 256 + lane * 8);
        nr[j] = *reinterpret_cast<const uint4*>(res + (long long)nxt * D + j * 256 + lane * 8);
      }
    }
    float z[VPL];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const uint32_t wy[4] = {cy[j].x, cy[j].y, cy[j].z, cy[j].w}, wr[4] = {cr[j].x, cr[j].y, cr[j].z, cr[j].w};
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const int i = j * 8 + 2 * e;
        const float2 fy = unpack_bf16(wy[e]), fr = unpack_bf16(wr[e]);
        const float2 m = drop_pair(dc, (unsigned long long)row * D + col_of(lane, i));
        z[i] = fr.x + fy.x * m.x; z[i + 1] = fr.y + fy.y * m.y;
      }
    }
    float mean, rstd;
    ln_stats(z, mean, rstd);
    if (lane == 0) { mean_o[row] = mean; rstd_o[row] = rstd; }
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float4 g0 = __ldg(reinterpret_cast<const float4*>(gamma + j * 256 + lane * 8));
      const float4 g1 = __ldg(reinterpret_cast<const float4*>(gamma + j * 256 + lane * 8 + 4));
      const float4 b0 = __ldg(reinterpret_cast<const float4*>(beta + j * 256 + lane * 8));
      const float4 b1 = __ldg(reinterpret_cast<const float4*>(beta + j * 256 + lane * 8 + 4));
      const float gg[8] = {g0.x, g0.y, g0.z, g0.w, g1.x, g1.y, g1.z, g1.w}, bb[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
      for (int k = 0; k < 8; ++k) z[j * 8 + k] = (z[j * 8 + k] - mean) * rstd * gg[k] + bb[k];
    }
    store_row_bf16(out + (long long)row * D, lane, z);
  }
}

// backward: dout = d1 (+ d2); z recomputed from res, y.  dres = dz (bf16), dy = dz * dropmask (bf16; same buffer
// allowed when dropout is off), dgamma/dbeta accumulated with atomics (fp32).
// (Measured and dropped in round 2: also accumulating the column sums of dy here — the bias gradient of the Linear that
//  produced y — to save the separate colsum launch: a third 16 KB smem accumulator per warp and the extra spills at the
//  168-register cap made this kernel 27 % slower, 55 -> 70 us, more than the side-stream colsum ever cost.)
// dgamma / dbeta partial sums live in shared memory ([warp][value i][lane]: conflict-free), not in 64 registers, so
// three 128-thread blocks fit per SM; one atomic per column per block at the end (kOrdered: the block's column sums go to its row of
// `partial` [gridDim.x][2 * D] instead, summed by ordered_colsum_kernel).
// !kGrads (frozen LayerNorm: dgamma = dbeta = NULL): no accumulators and no flush, the same dres / dy bits.
template <bool kOrdered, bool kGrads = true>
__global__ void __launch_bounds__(128, 3) add_ln_bwd_kernel(const bf16* __restrict__ d1, const bf16* __restrict__ d2,
                                                            const bf16* __restrict__ res, const bf16* __restrict__ y,
                                                            const float* __restrict__ gamma, const float* __restrict__ mean_i,
                                                            const float* __restrict__ rstd_i, bf16* __restrict__ dres,
                                                            bf16* __restrict__ dy_out, float* __restrict__ dgamma,
                                                            float* __restrict__ dbeta, int rows, DropCfg dc_in,
                                                            float* __restrict__ partial) {
  pdl_launch_dependents();
  pdl_wait();
  const DropCfg dc = resolve_drop(dc_in);
  extern __shared__ float sacc[];                      // [4 warps][2][VPL][32]
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
  float* sg = sacc + warp * (2 * VPL * 32);
  float* sb = sg + VPL * 32;
  if (kGrads) {
#pragma unroll
    for (int i = 0; i < VPL; ++i) { sg[i * 32 + lane] = 0.f; sb[i * 32 + lane] = 0.f; }
  }
  for (int row = blockIdx.x * nw + warp; row < rows; row += gridDim.x * nw) {
    // all 12-16 global loads of the row are issued before the first use (the kernel is latency-bound otherwise)
    uint4 ry[4], rr[4], r1[4], r2[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const long long o = (long long)row * D + j * 256 + lane * 8;
      ry[j] = *reinterpret_cast<const uint4*>(y + o);
      rr[j] = *reinterpret_cast<const uint4*>(res + o);
      r1[j] = *reinterpret_cast<const uint4*>(d1 + o);
      r2[j] = (d2 != nullptr) ? *reinterpret_cast<const uint4*>(d2 + o) : make_uint4(0, 0, 0, 0);
    }
    const float mean = mean_i[row], rstd = rstd_i[row];
    float z[VPL], t[VPL];
    uint32_t keep = 0;   // bit i: element i survived dropout
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const uint32_t wy[4] = {ry[j].x, ry[j].y, ry[j].z, ry[j].w}, wr[4] = {rr[j].x, rr[j].y, rr[j].z, rr[j].w};
      const uint32_t w1[4] = {r1[j].x, r1[j].y, r1[j].z, r1[j].w}, w2[4] = {r2[j].x, r2[j].y, r2[j].z, r2[j].w};
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const int i = j * 8 + 2 * e;
        const float2 fy = unpack_bf16(wy[e]), fr = unpack_bf16(wr[e]), f1 = unpack_bf16(w1[e]), f2 = unpack_bf16(w2[e]);
        const float2 m = drop_pair(dc, (unsigned long long)row * D + col_of(lane, i));
        keep |= (m.x != 0.f ? 1u : 0u) << i;
        keep |= (m.y != 0.f ? 1u : 0u) << (i + 1);
        z[i] = (fy.x * m.x + fr.x - mean) * rstd;              // z := xhat
        z[i + 1] = (fy.y * m.y + fr.y - mean) * rstd;
        t[i] = f1.x + f2.x;                                     // t := upstream gradient
        t[i + 1] = f1.y + f2.y;
      }
    }
    float s1 = 0.f, s2 = 0.f;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float4 g0 = *reinterpret_cast<const float4*>(gamma + j * 256 + lane * 8);
      const float4 g1 = *reinterpret_cast<const float4*>(gamma + j * 256 + lane * 8 + 4);
      const float gg[8] = {g0.x, g0.y, g0.z, g0.w, g1.x, g1.y, g1.z, g1.w};
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        const int i = j * 8 + k;
        if (kGrads) {
          sg[i * 32 + lane] += t[i] * z[i];
          sb[i * 32 + lane] += t[i];
        }
        t[i] *= gg[k];                                                          // t := d xhat
        s1 += t[i]; s2 += t[i] * z[i];
      }
    }
    s1 = warp_sum(s1) * (1.f / D); s2 = warp_sum(s2) * (1.f / D);
#pragma unroll
    for (int i = 0; i < VPL; ++i) t[i] = rstd * (t[i] - s1 - z[i] * s2);        // t := dz
    store_row_bf16(dres + (long long)row * D, lane, t);
    if (dy_out != dres) {
#pragma unroll
      for (int i = 0; i < VPL; ++i) t[i] = ((keep >> i) & 1u) ? t[i] * dc.scale : 0.f;
      store_row_bf16(dy_out + (long long)row * D, lane, t);
    }
  }
  if (!kGrads) return;
  __syncthreads();
  // column c = (i>>3)*256 + lane*8 + (i&7)  <->  (i, lane)
  for (int c = threadIdx.x; c < D; c += blockDim.x) {
    const int j = c >> 8, l = (c & 255) >> 3, k = c & 7;
    const int idx = (j * 8 + k) * 32 + l;
    float a = 0.f, bsum = 0.f;
    for (int w = 0; w < nw; ++w) { a += sacc[w * (2 * VPL * 32) + idx]; bsum += sacc[w * (2 * VPL * 32) + VPL * 32 + idx]; }
    if (kOrdered) {
      partial[(long long)blockIdx.x * 2 * D + c] = a;
      partial[(long long)blockIdx.x * 2 * D + D + c] = bsum;
    } else {
      atomicAdd(dgamma + c, a);
      atomicAdd(dbeta + c, bsum);
    }
  }
}

// ------------------------------------------------------------------ column sums (bias gradients)
// out[n] += sum_r x[r, n]   x bf16 [rows, ld]; N multiple of 8 (kOrdered: row chunk y stores its sums to partial[y][n])
template <bool kOrdered>
__global__ void __launch_bounds__(256) colsum_kernel(const bf16* __restrict__ x, long long ld, int rows, int N,
                                                     float* __restrict__ out, int rows_per_block, float* __restrict__ partial) {
  pdl_launch_dependents();
  pdl_wait();
  __shared__ float sm[8][256];
  const int cg = threadIdx.x & 31;        // column group of 8
  const int rl = threadIdx.x >> 5;        // row lane 0..7
  const int c0 = blockIdx.x * 256 + cg * 8;
  const int r_begin = blockIdx.y * rows_per_block;
  const int r_end = min(rows, r_begin + rows_per_block);
  float acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  if (c0 < N) {
    // four independent 16-byte loads in flight per thread: with one, the kernel ran at ~2.4 TB/s (latency-bound)
    int r = r_begin + rl;
    for (; r + 24 < r_end; r += 32) {
      uint4 u[4];
#pragma unroll
      for (int k = 0; k < 4; ++k) u[k] = *reinterpret_cast<const uint4*>(x + (long long)(r + 8 * k) * ld + c0);
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const uint32_t w[4] = {u[k].x, u[k].y, u[k].z, u[k].w};
#pragma unroll
        for (int e = 0; e < 4; ++e) { const float2 f = unpack_bf16(w[e]); acc[2 * e] += f.x; acc[2 * e + 1] += f.y; }
      }
    }
    for (; r < r_end; r += 8) {
      const uint4 u = *reinterpret_cast<const uint4*>(x + (long long)r * ld + c0);
      const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
      for (int e = 0; e < 4; ++e) { const float2 f = unpack_bf16(w[e]); acc[2 * e] += f.x; acc[2 * e + 1] += f.y; }
    }
  }
#pragma unroll
  for (int i = 0; i < 8; ++i) sm[rl][cg * 8 + i] = acc[i];
  __syncthreads();
  const int c = blockIdx.x * 256 + threadIdx.x;
  if (c < N) {
    float s = 0.f;
#pragma unroll
    for (int w = 0; w < 8; ++w) s += sm[w][threadIdx.x];
    if (kOrdered) partial[(long long)blockIdx.y * N + c] = s;
    else          atomicAdd(out + c, s);
  }
}

// ------------------------------------------------------------------ gate fusion (SelfAttention.forward :732-744)
// y = text + alpha*table + beta*img, alpha = relu(tanh(u_a)) * pres_tab[b], beta = relu(tanh(u_b)) * pres_img[b]
__global__ void __launch_bounds__(256) gate_fwd_kernel(const bf16* __restrict__ o3, const bf16* __restrict__ u,
                                                       const uint8_t* __restrict__ pres, bf16* __restrict__ y,
                                                       bf16* __restrict__ ab, long long n, int rows_per_biz) {
  pdl_launch_dependents();
  pdl_wait();
  const long long stride = (long long)gridDim.x * blockDim.x * 8;
  for (long long i = ((long long)blockIdx.x * blockDim.x + threadIdx.x) * 8; i < n; i += stride) {
    const long long row = i / D;
    const int biz = (int)(row / rows_per_biz);
    const float pt = pres[biz * 2] ? 1.f : 0.f, pi = pres[biz * 2 + 1] ? 1.f : 0.f;
    const uint4 t4 = *reinterpret_cast<const uint4*>(o3 + i);
    const uint4 b4 = *reinterpret_cast<const uint4*>(o3 + n + i);
    const uint4 i4 = *reinterpret_cast<const uint4*>(o3 + 2 * n + i);
    const uint4 ua = *reinterpret_cast<const uint4*>(u + i);
    const uint4 ub = *reinterpret_cast<const uint4*>(u + n + i);
    const uint32_t tw[4] = {t4.x, t4.y, t4.z, t4.w}, bw[4] = {b4.x, b4.y, b4.z, b4.w}, iw[4] = {i4.x, i4.y, i4.z, i4.w};
    const uint32_t uaw[4] = {ua.x, ua.y, ua.z, ua.w}, ubw[4] = {ub.x, ub.y, ub.z, ub.w};
    uint32_t yo[4], ao[4], bo[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const float2 tx = unpack_bf16(tw[e]), tb = unpack_bf16(bw[e]), im = unpack_bf16(iw[e]);
      const float2 a = unpack_bf16(uaw[e]), b = unpack_bf16(ubw[e]);
      const float a0 = bf16_round(fmaxf(tanhf(a.x), 0.f) * pt), a1 = bf16_round(fmaxf(tanhf(a.y), 0.f) * pt);
      const float b0 = bf16_round(fmaxf(tanhf(b.x), 0.f) * pi), b1 = bf16_round(fmaxf(tanhf(b.y), 0.f) * pi);
      yo[e] = pack_bf16(tx.x + a0 * tb.x + b0 * im.x, tx.y + a1 * tb.y + b1 * im.y);
      ao[e] = pack_bf16(a0, a1); bo[e] = pack_bf16(b0, b1);
    }
    *reinterpret_cast<uint4*>(y + i) = make_uint4(yo[0], yo[1], yo[2], yo[3]);
    *reinterpret_cast<uint4*>(ab + i) = make_uint4(ao[0], ao[1], ao[2], ao[3]);
    *reinterpret_cast<uint4*>(ab + n + i) = make_uint4(bo[0], bo[1], bo[2], bo[3]);
  }
}
// du_a = dy*table*(alpha>0)*(1-alpha^2), du_b likewise with img / beta
__global__ void __launch_bounds__(256) gate_bwd_u_kernel(const bf16* __restrict__ dy, const bf16* __restrict__ o3,
                                                         const bf16* __restrict__ ab, bf16* __restrict__ du, long long n) {
  pdl_launch_dependents();
  pdl_wait();
  const long long stride = (long long)gridDim.x * blockDim.x * 8;
  for (long long i = ((long long)blockIdx.x * blockDim.x + threadIdx.x) * 8; i < n; i += stride) {
    const uint4 d4 = *reinterpret_cast<const uint4*>(dy + i);
    const uint4 b4 = *reinterpret_cast<const uint4*>(o3 + n + i);
    const uint4 i4 = *reinterpret_cast<const uint4*>(o3 + 2 * n + i);
    const uint4 a4 = *reinterpret_cast<const uint4*>(ab + i);
    const uint4 e4 = *reinterpret_cast<const uint4*>(ab + n + i);
    const uint32_t dw[4] = {d4.x, d4.y, d4.z, d4.w}, bw[4] = {b4.x, b4.y, b4.z, b4.w}, iw[4] = {i4.x, i4.y, i4.z, i4.w};
    const uint32_t aw[4] = {a4.x, a4.y, a4.z, a4.w}, ew[4] = {e4.x, e4.y, e4.z, e4.w};
    uint32_t oa[4], ob[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const float2 d = unpack_bf16(dw[e]), tb = unpack_bf16(bw[e]), im = unpack_bf16(iw[e]);
      const float2 al = unpack_bf16(aw[e]), be = unpack_bf16(ew[e]);
      oa[e] = pack_bf16(al.x > 0.f ? d.x * tb.x * (1.f - al.x * al.x) : 0.f, al.y > 0.f ? d.y * tb.y * (1.f - al.y * al.y) : 0.f);
      ob[e] = pack_bf16(be.x > 0.f ? d.x * im.x * (1.f - be.x * be.x) : 0.f, be.y > 0.f ? d.y * im.y * (1.f - be.y * be.y) : 0.f);
    }
    *reinterpret_cast<uint4*>(du + i) = make_uint4(oa[0], oa[1], oa[2], oa[3]);
    *reinterpret_cast<uint4*>(du + n + i) = make_uint4(ob[0], ob[1], ob[2], ob[3]);
  }
}
// dO3[text] = dy + dca[:, :D] + dcb[:, :D];  dO3[table] = dy*alpha + dca[:, D:];  dO3[img] = dy*beta + dcb[:, D:]
__global__ void __launch_bounds__(256) gate_bwd_o_kernel(const bf16* __restrict__ dy, const bf16* __restrict__ ab,
                                                         const bf16* __restrict__ dca, const bf16* __restrict__ dcb,
                                                         bf16* __restrict__ do3, long long n) {
  pdl_launch_dependents();
  pdl_wait();
  const long long stride = (long long)gridDim.x * blockDim.x * 8;
  for (long long i = ((long long)blockIdx.x * blockDim.x + threadIdx.x) * 8; i < n; i += stride) {
    const long long row = i / D; const int c = (int)(i - row * D);
    const uint4 d4 = *reinterpret_cast<const uint4*>(dy + i);
    const uint4 a4 = *reinterpret_cast<const uint4*>(ab + i);
    const uint4 e4 = *reinterpret_cast<const uint4*>(ab + n + i);
    const uint4 at4 = *reinterpret_cast<const uint4*>(dca + row * 2 * D + c);
    const uint4 ab4 = *reinterpret_cast<const uint4*>(dca + row * 2 * D + D + c);
    const uint4 bt4 = *reinterpret_cast<const uint4*>(dcb + row * 2 * D + c);
    const uint4 bi4 = *reinterpret_cast<const uint4*>(dcb + row * 2 * D + D + c);
    const uint32_t dw[4] = {d4.x, d4.y, d4.z, d4.w}, aw[4] = {a4.x, a4.y, a4.z, a4.w}, ew[4] = {e4.x, e4.y, e4.z, e4.w};
    const uint32_t atw[4] = {at4.x, at4.y, at4.z, at4.w}, abw[4] = {ab4.x, ab4.y, ab4.z, ab4.w};
    const uint32_t btw[4] = {bt4.x, bt4.y, bt4.z, bt4.w}, biw[4] = {bi4.x, bi4.y, bi4.z, bi4.w};
    uint32_t ot[4], ob[4], oi[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const float2 d = unpack_bf16(dw[e]), al = unpack_bf16(aw[e]), be = unpack_bf16(ew[e]);
      const float2 at = unpack_bf16(atw[e]), abv = unpack_bf16(abw[e]), bt = unpack_bf16(btw[e]), bi = unpack_bf16(biw[e]);
      ot[e] = pack_bf16(d.x + at.x + bt.x, d.y + at.y + bt.y);
      ob[e] = pack_bf16(d.x * al.x + abv.x, d.y * al.y + abv.y);
      oi[e] = pack_bf16(d.x * be.x + bi.x, d.y * be.y + bi.y);
    }
    *reinterpret_cast<uint4*>(do3 + i) = make_uint4(ot[0], ot[1], ot[2], ot[3]);
    *reinterpret_cast<uint4*>(do3 + n + i) = make_uint4(ob[0], ob[1], ob[2], ob[3]);
    *reinterpret_cast<uint4*>(do3 + 2 * n + i) = make_uint4(oi[0], oi[1], oi[2], oi[3]);
  }
}

// ------------------------------------------------------------------ label-smoothed cross entropy
// (LabelSmoothingLoss, src/utils.py:32-38; eps < 0 selects nn.CrossEntropyLoss, src/text_pretrain.py:97).
// One block per row: pass 1 online (max, sum exp, sum z, z[y]); pass 2 rewrites the row in place with
// d loss / d logits * gscale (bf16).  Pad targets are NOT ignored (reference quirk Q2).
// lse_rows: the loss pass (write_grad = 0) stores the row's log-sum-exp there; the gradient pass (write_grad = 1) reads it
// instead of repeating pass 1 (one read of the logits instead of two: 5.4 -> 3.7 GB per step at 18432 x 50265).
__global__ void __launch_bounds__(256) ce_fwd_bwd_kernel(bf16* __restrict__ logits, long long ld, int V,
                                                         const int* __restrict__ target, float eps, float gscale,
                                                         const float* __restrict__ gscale_dev,
                                                         float* __restrict__ loss_rows, float* __restrict__ lse_rows,
                                                         int write_grad) {
  __shared__ float red[4][8];
  bf16* row = logits + (long long)blockIdx.x * ld;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int nvec = V >> 3;
  const int y = target[blockIdx.x];
  float lse;
  if (write_grad && lse_rows != nullptr) {
    lse = lse_rows[blockIdx.x];
  } else {
  const float zy = __bfloat162float(row[y]);   // read before the barrier: pass 2 overwrites the row in place
  float m = -INFINITY, s = 0.f, sz = 0.f;
  for (int i = tid; i < nvec; i += 256) {
    const uint4 u = *reinterpret_cast<const uint4*>(row + i * 8);
    const uint32_t w[4] = {u.x, u.y, u.z, u.w};
    float v[8];
#pragma unroll
    for (int e = 0; e < 4; ++e) { const float2 f = unpack_bf16(w[e]); v[2 * e] = f.x; v[2 * e + 1] = f.y; }
    float bm = v[0];
#pragma unroll
    for (int e = 1; e < 8; ++e) bm = fmaxf(bm, v[e]);
    const float mn = fmaxf(m, bm);
    float add = 0.f;
#pragma unroll
    for (int e = 0; e < 8; ++e) { add += __expf(v[e] - mn); sz += v[e]; }
    s = s * __expf(m - mn) + add;
    m = mn;
  }
  for (int i = nvec * 8 + tid; i < V; i += 256) {
    const float v = __bfloat162float(row[i]);
    const float mn = fmaxf(m, v);
    s = s * __expf(m - mn) + __expf(v - mn);
    m = mn; sz += v;
  }
  // block reduce (m, s) and sz
  float wm = warp_max(m);
  s = (m == -INFINITY) ? 0.f : s * __expf(m - wm);   // lanes / warps without data (V < 8*256) hold m = -inf
  s = warp_sum(s); sz = warp_sum(sz);
  if (lane == 0) { red[0][warp] = wm; red[1][warp] = s; red[2][warp] = sz; }
  __syncthreads();
  float M = red[0][0];
#pragma unroll
  for (int w = 1; w < 8; ++w) M = fmaxf(M, red[0][w]);
  float S = 0.f, SZ = 0.f;
#pragma unroll
  for (int w = 0; w < 8; ++w) { S += (red[0][w] == -INFINITY) ? 0.f : red[1][w] * __expf(red[0][w] - M); SZ += red[2][w]; }
  lse = M + logf(S);
  if (tid == 0) {
    if (lse_rows != nullptr) lse_rows[blockIdx.x] = lse;
    const float logp_y = zy - lse;
    float loss;
    if (eps < 0.f) loss = -logp_y;
    else {
      const float sum_logp = SZ - (float)V * lse;
      loss = -(1.f - eps) * logp_y - eps / (float)(V - 1) * (sum_logp - logp_y);
    }
    loss_rows[blockIdx.x] = loss;
  }
  }
  if (!write_grad) return;
  if (gscale_dev != nullptr) gscale *= gscale_dev[0];
  const float off = eps < 0.f ? 0.f : eps / (float)(V - 1);
  const float on = eps < 0.f ? 1.f : 1.f - eps;
  for (int i = tid; i < nvec; i += 256) {
    const uint4 u = *reinterpret_cast<const uint4*>(row + i * 8);
    const uint32_t w[4] = {u.x, u.y, u.z, u.w};
    float v[8];
#pragma unroll
    for (int e = 0; e < 4; ++e) { const float2 f = unpack_bf16(w[e]); v[2 * e] = f.x; v[2 * e + 1] = f.y; }
#pragma unroll
    for (int e = 0; e < 8; ++e) v[e] = (__expf(v[e] - lse) - ((i * 8 + e == y) ? on : off)) * gscale;
    uint4 o; o.x = pack_bf16(v[0], v[1]); o.y = pack_bf16(v[2], v[3]); o.z = pack_bf16(v[4], v[5]); o.w = pack_bf16(v[6], v[7]);
    *reinterpret_cast<uint4*>(row + i * 8) = o;
  }
  for (int i = nvec * 8 + tid; i < V; i += 256) {
    const float v = __bfloat162float(row[i]);
    row[i] = __float2bfloat16_rn((__expf(v - lse) - ((i == y) ? on : off)) * gscale);
  }
}
// out[0] = scale * sum(x)   (single block, deterministic order)
__global__ void __launch_bounds__(1024) sum_rows_kernel(const float* __restrict__ x, int n, float scale, float* __restrict__ out) {
  __shared__ float red[32];
  float s = 0.f;
  for (int i = threadIdx.x; i < n; i += 1024) s += x[i];
  s = warp_sum(s);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x < 32) {
    float v = red[threadIdx.x];
    v = warp_sum(v);
    if (threadIdx.x == 0) out[0] = v * scale;
  }
}

// ------------------------------------------------------------------ step input preparation
// One block per business.  Integer work that must be bit-exact with the reference:
//   dec_ids  = shift_tokens_right(reviews[:, i])   (modeling_multimodalsum.py:225-246, incl. the batch-level
//              BOS/EOS decision taken from element [0,0] of the pass, i.e. reviews[0, i, 0])
//   rating_diff[b,i] = r_i - mean_{j != i} r_j      (multimodal_train.py:154-156)
//   key / entity validity of the text, table and image memory, 1/#valid entities per (target, modality),
//   modality presence per business for the gates (:732-736).
__global__ void __launch_bounds__(128) prep_step_kernel(const int64_t* __restrict__ reviews, const int64_t* __restrict__ reviews_mask,
                                                        const float* __restrict__ rating, const uint8_t* __restrict__ table_valid,
                                                        const uint8_t* __restrict__ img_mask, MmsumPrepArgs a) {
  const int b = blockIdx.x;
  const int R = a.R, S = a.S;
  const int SE = a.S_enc > 0 ? a.S_enc : S;      // encoder frame: the first SE tokens of a review (the rest is pad by contract)
  const int n_ent = R + (a.F > 0 ? 1 : 0) + a.n_img;
  __shared__ int s_bad;
  if (threadIdx.x == 0) s_bad = 0;
  __syncthreads();
  for (int i = threadIdx.x; i < R * S; i += blockDim.x) {
    const int r = i / S, t = i - r * S;
    const long long gi = ((long long)b * R + r) * S + t;
    const long long tok = (long long)reviews[gi];
    a.labels[gi] = (int)tok;
    if (t >= SE && reviews_mask[gi] != 0) s_bad = 1;   // a valid token beyond the encoder frame: the caller's length hint was wrong
    if (t < SE) {
      const long long ge = ((long long)b * R + r) * SE + t;
      a.enc_ids[ge] = (int)tok;
      const uint8_t kv = reviews_mask[gi] != 0 ? 1 : 0;
      a.enc_valid[ge] = kv;
      a.mem_valid[ge] = kv;   // text region of the memory comes first
    }
  }
  __shared__ int s_cnt;
  __syncthreads();
  // per review: index of the last non-pad token, then the shifted row
  for (int r = 0; r < R; ++r) {
    const int64_t* src = reviews + ((long long)b * R + r) * S;
    if (threadIdx.x == 0) s_cnt = 0;
    __syncthreads();
    int local = 0;
    for (int t = threadIdx.x; t < S; t += blockDim.x) local += (src[t] != a.pad_id) ? 1 : 0;
    atomicAdd(&s_cnt, local);
    __syncthreads();
    const int idx_eos = s_cnt - 1;
    const long long first = (long long)reviews[(long long)r * S];  // element [0, 0] of pass r (batch row 0)
    const int start = (first != a.bos_id) ? a.bos_id : a.eos_id;
    for (int t = threadIdx.x; t < S; t += blockDim.x) {
      int v;
      if (t == 0) v = start;
      else { const int tp = t - 1; v = (tp == idx_eos) ? a.pad_id : (int)src[tp]; }
      const long long gi = ((long long)b * R + r) * S + t;
      a.dec_ids[gi] = v;
      a.dec_valid[gi] = (v != a.pad_id) ? 1 : 0;
    }
    __syncthreads();
  }
  // memory validity: table rows then image keys
  const long long T_text = (long long)a.B * R * SE;
  for (int f = threadIdx.x; f < a.F; f += blockDim.x)
    a.mem_valid[T_text + (long long)b * a.F + f] = table_valid[(long long)b * a.F + f];
  const long long T_tab = (long long)a.B * a.F;
  for (int i = threadIdx.x; i < a.n_img * a.img_keys; i += blockDim.x)
    a.mem_valid[T_text + T_tab + (long long)b * a.n_img * a.img_keys + i] = img_mask[(long long)b * a.n_img + i / a.img_keys] ? 1 : 0;
  __syncthreads();
  if (threadIdx.x == 0) {
    // entity validity
    int text_cnt = 0;
    for (int r = 0; r < R; ++r) {
      int any = 0;
      for (int t = 0; t < S; ++t) any |= (reviews_mask[((long long)b * R + r) * S + t] != 0);
      a.ent_valid[(long long)b * n_ent + r] = (uint8_t)any;
      text_cnt += any;
    }
    int tab_any = 0;
    if (a.F > 0) {
      for (int f = 0; f < a.F; ++f) tab_any |= table_valid[(long long)b * a.F + f];
      a.ent_valid[(long long)b * n_ent + R] = (uint8_t)tab_any;
    }
    int img_cnt = 0;
    for (int e = 0; e < a.n_img; ++e) {
      const int v = img_mask[(long long)b * a.n_img + e] ? 1 : 0;
      a.ent_valid[(long long)b * n_ent + R + (a.F > 0 ? 1 : 0) + e] = (uint8_t)v;
      img_cnt += v;
    }
    if (a.pres != nullptr) { a.pres[b * 2] = (uint8_t)tab_any; a.pres[b * 2 + 1] = (uint8_t)(img_cnt > 0); }
    float rsum = 0.f;
    for (int r = 0; r < R; ++r) rsum += rating[(long long)b * R + r];
    for (int r = 0; r < R; ++r) {
      const long long q = (long long)b * R + r;
      const float ri = rating[q];
      // (a violated frame contract must not pass silently: the NaN reaches the decoder embedding and the loss)
      a.rating_diff[q] = s_bad ? __int_as_float(0x7fc00000) : ri - (rsum - ri) / (float)(R - 1);
      const int self_valid = a.ent_valid[(long long)b * n_ent + r];
      const int nt = text_cnt - self_valid;
      a.inv_n[q * a.n_mod + 0] = nt > 0 ? 1.f / (float)nt : 0.f;
      if (a.n_mod > 1) {
        a.inv_n[q * a.n_mod + 1] = tab_any ? 1.f : 0.f;
        a.inv_n[q * a.n_mod + 2] = img_cnt > 0 ? 1.f / (float)img_cnt : 0.f;
      }
    }
  }
}

// ------------------------------------------------------------------ table encoder front end
// Builds X[b, f, 0:D] = field-name embedding, X[b, f, D:2D] = field-value embedding (bf16) and valid[b, f]
// (YelpTableEncoder.forward src/table_encoder.py:27-82, AmazonTableEncoder.forward :108-166).  The frozen-embedding
// gathers read the fp32 table; the tiny bit-code Linear layers (rating / hours / price) are evaluated inline.
__device__ __forceinline__ void masked_sum4(const float* __restrict__ E, const int64_t* __restrict__ tok, int L, int c,
                                            bool mask_pad, float (&acc)[4], int& any) {
  for (int j = 0; j < L; ++j) {
    const long long id = (long long)tok[j];
    if (id != 1) any = 1;
    if (mask_pad && id == 1) continue;
    const float4 v = *reinterpret_cast<const float4*>(E + id * D + c);
    acc[0] += v.x; acc[1] += v.y; acc[2] += v.z; acc[3] += v.w;
  }
}
__device__ __forceinline__ void bits_linear4(const float* __restrict__ W, const int64_t* __restrict__ bits, int nb, int c, float (&acc)[4]) {
  for (int j = 0; j < nb; ++j) {
    const float x = (float)bits[j];
#pragma unroll
    for (int e = 0; e < 4; ++e) acc[e] += x * W[(long long)(c + e) * nb + j];
  }
}
__device__ __forceinline__ void store4(bf16* dst, const float (&v)[4]) {
  uint2 u; u.x = pack_bf16(v[0], v[1]); u.y = pack_bf16(v[2], v[3]);
  *reinterpret_cast<uint2*>(dst) = u;
}

__global__ void __launch_bounds__(256) table_yelp_kernel(MmsumTableArgs a) {
  const int f = blockIdx.x % 47, b = blockIdx.x / 47;
  const int c = threadIdx.x * 4;
  const float* E = a.E;
  float nm[4] = {0.f, 0.f, 0.f, 0.f}, val[4] = {0.f, 0.f, 0.f, 0.f};
  int any = 0, dummy = 0;
  masked_sum4(E, a.field + f * 6, 6, c, true, nm, dummy);
  uint8_t valid = 1;
  if (f == 0) {                       // name [B,24]
    masked_sum4(E, a.v0 + (long long)b * 24, 24, c, true, val, any);
  } else if (f == 1) {                // category [B,6,12]: masked sum over 12, masked mean over 6
    float cnt = 0.f;
    for (int k = 0; k < 6; ++k) {
      float t4[4] = {0.f, 0.f, 0.f, 0.f}; int anyk = 0;
      masked_sum4(E, a.v1 + ((long long)b * 6 + k) * 12, 12, c, true, t4, anyk);
      if (anyk) { cnt += 1.f; for (int e = 0; e < 4; ++e) val[e] += t4[e]; }
    }
    for (int e = 0; e < 4; ++e) val[e] /= (cnt + 1e-6f);
    valid = a.v1[(long long)b * 72] != 1;
  } else if (f < 7) {                 // str_categorical [B,5,3]
    const int64_t* tk = a.v2 + ((long long)b * 5 + (f - 2)) * 3;
    masked_sum4(E, tk, 3, c, true, val, any);
    valid = tk[0] != 1;
  } else if (f < 39) {                // str_boolean [B,32,1]
    const int64_t* tk = a.v3 + (long long)b * 32 + (f - 7);
    masked_sum4(E, tk, 1, c, true, val, any);
    valid = tk[0] != 1;
  } else if (f == 39) {               // rating bits [B,4] -> Linear(4, D)
    bits_linear4(a.W0, a.v4 + (long long)b * 4, 4, c, val);
  } else {                            // hours [B,7,4] -> Linear(4, D)
    const int64_t* hb = a.v5 + ((long long)b * 7 + (f - 40)) * 4;
    bits_linear4(a.W1, hb, 4, c, val);
    valid = (hb[0] + hb[1] + hb[2] + hb[3]) != 0;
  }
  bf16* x = reinterpret_cast<bf16*>(a.X) + ((long long)b * 47 + f) * 2 * D;
  store4(x + c, nm);
  store4(x + D + c, val);
  if (threadIdx.x == 0) a.valid[(long long)b * 47 + f] = valid;
}

__global__ void __launch_bounds__(256) table_amazon_kernel(MmsumTableArgs a) {
  const int f = blockIdx.x % 133, b = blockIdx.x / 133;
  const int c = threadIdx.x * 4;
  const float* E = a.E;
  float nm[4], val[4] = {0.f, 0.f, 0.f, 0.f};
  {  // field names: rows 0..4 their own token, rows 5..132 the 6th (description) token, no pad masking (:108-110)
    const long long id = a.field[f < 5 ? f : 5];
    const float4 v = *reinterpret_cast<const float4*>(E + id * D + c);
    nm[0] = v.x; nm[1] = v.y; nm[2] = v.z; nm[3] = v.w;
  }
  int any = 0;
  uint8_t valid = 1;
  if (f == 0) {                       // price bits [B,11]
    const int64_t* pb = a.v0 + (long long)b * 11;
    bits_linear4(a.W0, pb, 11, c, val);
    long long s = 0; for (int j = 0; j < 11; ++j) s += pb[j];
    valid = s != 0;
  } else if (f == 1) {                // rating bits [B,4]
    bits_linear4(a.W1, a.v1 + (long long)b * 4, 4, c, val);
  } else if (f == 2) {                // brand [B,12]
    masked_sum4(E, a.v2 + (long long)b * 12, 12, c, true, val, any);
    valid = a.v2[(long long)b * 12] != 1;
  } else if (f == 3) {                // name [B,32]
    masked_sum4(E, a.v3 + (long long)b * 32, 32, c, true, val, any);
    valid = a.v3[(long long)b * 32] != 1;
  } else if (f == 4) {                // category [B,3,8,12]: sum over 12, masked mean over 8, masked mean over 3
    float cnt1 = 0.f;
    for (int i = 0; i < 3; ++i) {
      float mid[4] = {0.f, 0.f, 0.f, 0.f}; float cnt2 = 0.f;
      for (int k = 0; k < 8; ++k) {
        float t4[4] = {0.f, 0.f, 0.f, 0.f}; int anyk = 0;
        masked_sum4(E, a.v4 + (((long long)b * 3 + i) * 8 + k) * 12, 12, c, true, t4, anyk);
        if (anyk) { cnt2 += 1.f; for (int e = 0; e < 4; ++e) mid[e] += t4[e]; }
      }
      if (cnt2 > 0.f) { cnt1 += 1.f; for (int e = 0; e < 4; ++e) val[e] += mid[e] / (cnt2 + 1e-6f); }
    }
    for (int e = 0; e < 4; ++e) val[e] /= (cnt1 + 1e-6f);
  } else {                            // description tokens [B,128], one field each, no pad masking of the embedding
    const long long id = a.v5[(long long)b * 128 + (f - 5)];
    const float4 v = *reinterpret_cast<const float4*>(E + id * D + c);
    val[0] = v.x; val[1] = v.y; val[2] = v.z; val[3] = v.w;
    valid = id != 1;
  }
  bf16* x = reinterpret_cast<bf16*>(a.X) + ((long long)b * 133 + f) * 2 * D;
  store4(x + c, nm);
  store4(x + D + c, val);
  if (threadIdx.x == 0) a.valid[(long long)b * 133 + f] = valid;
}

// gradient of the bit-code Linear layers: dW[c, j] += sum_{b, rows} bits[b,row,j] * dX[b, f0+row, D + c]
__global__ void __launch_bounds__(256) table_bits_bwd_kernel(const bf16* __restrict__ dX, const int64_t* __restrict__ bits,
                                                             float* __restrict__ dW, int B, int F, int f0, int nrows, int nb) {
  const int c = blockIdx.x * 256 + threadIdx.x;
  for (int j = 0; j < nb; ++j) {
    float s = 0.f;
    for (int b = 0; b < B; ++b)
      for (int r = 0; r < nrows; ++r) {
        const long long bit = bits[((long long)b * nrows + r) * nb + j];
        if (bit != 0) s += (float)bit * __bfloat162float(dX[((long long)b * F + f0 + r) * 2 * D + D + c]);
      }
    atomicAdd(dW + (long long)c * nb + j, s);
  }
}

static inline int nblocks(long long n, int per_block, int cap) {
  long long b = (n + per_block - 1) / per_block;
  if (b > cap) b = cap;
  if (b < 1) b = 1;
  return (int)b;
}

}  // namespace mmsum

using namespace mmsum;
#define STREAM(s) reinterpret_cast<cudaStream_t>(s)

extern "C" int mmsum_cast_f32_bf16(const float* src, void* dst, int64_t n, void* stream) {
  if (!src || !dst || n < 0) return MMSUM_ERR_INVALID;
  if (n == 0) return 0;
  if ((reinterpret_cast<uintptr_t>(src) & 15) || (reinterpret_cast<uintptr_t>(dst) & 15)) return MMSUM_ERR_INVALID;
  cast_f32_bf16_kernel<<<nblocks(n, 2048, 148 * 16), 256, 0, STREAM(stream)>>>(src, reinterpret_cast<bf16*>(dst), n);
  MMSUM_CHECK_LAUNCH();
  return 0;
}

extern "C" int mmsum_embed_ln_fwd(const int32_t* ids, const float* E, const float* P, const float* rating_diff,
                                  const float* remb, const float* gamma, const float* beta, void* out, float* mean,
                                  float* rstd, int32_t rows, int32_t S, int32_t d_model, float p_drop, uint64_t seed,
                                  uint32_t stream_id, const uint32_t* step_dev, void* stream) {
  if (d_model != D || rows <= 0 || S <= 0 || !ids || !E || !P || !out) return MMSUM_ERR_INVALID;
  embed_ln_fwd_kernel<<<(rows + 7) / 8, 256, 0, STREAM(stream)>>>(ids, E, P, rating_diff, remb, gamma, beta,
                                                                   reinterpret_cast<bf16*>(out), mean, rstd, rows, S,
                                                                   make_drop(p_drop, seed, stream_id, step_dev), nullptr);
  MMSUM_CHECK_LAUNCH();
  return 0;
}

extern "C" int mmsum_embed_ln_decode(const int32_t* ids, const float* E, const float* P, const float* rating_diff,
                                     const float* remb, const float* gamma, const float* beta, void* out, float* mean,
                                     float* rstd, int32_t rows, int32_t d_model, const int32_t* pos_dev, void* stream) {
  if (d_model != D || rows <= 0 || !ids || !E || !P || !out || !pos_dev) return MMSUM_ERR_INVALID;
  embed_ln_fwd_kernel<<<(rows + 7) / 8, 256, 0, STREAM(stream)>>>(ids, E, P, rating_diff, remb, gamma, beta,
                                                                   reinterpret_cast<bf16*>(out), mean, rstd, rows, 1,
                                                                   make_drop(0.f, 0, 0), pos_dev);
  MMSUM_CHECK_LAUNCH();
  return 0;
}

extern "C" int mmsum_embed_ln_bwd(const void* dout, const void* dout2, const int32_t* ids, const float* E, const float* P,
                                  const float* rating_diff, const float* remb, const float* gamma, const float* mean,
                                  const float* rstd, float* dE, float* dP, float* dremb, float* dgamma, float* dbeta,
                                  float* dz_scratch, int32_t rows, int32_t S, int32_t d_model, int32_t pad_id,
                                  float p_drop, uint64_t seed, uint32_t stream_id, const uint32_t* step_dev, void* stream) {
  if (d_model != D || rows <= 0 || S <= 0 || rows % S || !dz_scratch) return MMSUM_ERR_INVALID;
  if ((dgamma == nullptr) != (dbeta == nullptr) || (rating_diff != nullptr && !remb)) return MMSUM_ERR_INVALID;
  const bool want_remb = rating_diff != nullptr && dremb != nullptr;
  if (!dE && !dgamma && !dP && !want_remb) return 0;
  embed_ln_bwd_kernel<false><<<nblocks(rows, 8 * 4, 148 * 4), 256, 0, STREAM(stream)>>>(
      reinterpret_cast<const bf16*>(dout), reinterpret_cast<const bf16*>(dout2), ids, E, P, rating_diff, remb, gamma, mean,
      rstd, dE, dz_scratch, dgamma, dbeta,
      rows, S, pad_id, make_drop(p_drop, seed, stream_id, step_dev), nullptr);
  MMSUM_CHECK_LAUNCH();
  if (dP || want_remb) {
    embed_pos_bwd_kernel<false><<<dim3(D / 256, S), 256, 0, STREAM(stream)>>>(dz_scratch, rating_diff, dP, dremb, rows / S, S, nullptr);
    MMSUM_CHECK_LAUNCH();
  }
  return 0;
}

static int ordered_colsum(const float* part, int nparts, int width, int split, float* out0, float* out1, cudaStream_t stream) {
  ordered_colsum_kernel<<<(width + 31) / 32, 256, 0, stream>>>(part, nparts, width, split, out0, out1);
  MMSUM_CHECK_LAUNCH();
  return 0;
}

// the ordered embedding backward; each of dE, dP, dremb and the pair dgamma / dbeta may be NULL (not computed), not all of them
static int embed_ln_bwd_ordered(const void* dout, const void* dout2, const int32_t* ids, const float* E, const float* P,
                                const float* rating_diff, const float* remb, const float* gamma, const float* mean,
                                const float* rstd, float* dE, float* dP, float* dremb, float* dgamma, float* dbeta,
                                float* dz_scratch, int32_t rows, int32_t S, int32_t d_model, int32_t pad_id,
                                float p_drop, uint64_t seed, uint32_t stream_id, const uint32_t* step_dev, int32_t V,
                                float* workspace, int64_t workspace_elems, void* stream) {
  if (d_model != D || rows <= 0 || S <= 0 || rows % S || !dz_scratch) return MMSUM_ERR_INVALID;
  if (!dout || !ids || !E || !P || !gamma || !mean || !rstd) return MMSUM_ERR_INVALID;
  if ((dgamma == nullptr) != (dbeta == nullptr)) return MMSUM_ERR_INVALID;
  if (rating_diff != nullptr && !remb) return MMSUM_ERR_INVALID;
  const bool want_remb = rating_diff != nullptr && dremb != nullptr;
  if (!dE && !dgamma && !dP && !want_remb) return MMSUM_ERR_INVALID;
  if (V <= 0 || V >= (1 << 22) || !workspace) return MMSUM_ERR_INVALID;
  const int nblk = nblocks(rows, 8 * 4, 148 * 4);
  const int ntiles = (rows + kScatterTile - 1) / kScatterTile;
  if (workspace_elems < (int64_t)nblk * 2 * D + (int64_t)S * D + 2LL * ntiles * D + V + 1 + 2LL * rows) return MMSUM_ERR_INVALID;
  cudaStream_t st = STREAM(stream);
  float* part_ln = workspace;
  float* part_remb = part_ln + (long long)nblk * 2 * D;
  float* head = part_remb + (long long)S * D;
  float* tail = head + (long long)ntiles * D;
  int* cursor = reinterpret_cast<int*>(tail + (long long)ntiles * D);
  int* order = cursor + V + 1;
  int* sid = order + rows;
  embed_ln_bwd_kernel<true><<<nblk, 256, 0, st>>>(
      reinterpret_cast<const bf16*>(dout), reinterpret_cast<const bf16*>(dout2), ids, E, P, rating_diff, remb, gamma, mean,
      rstd, dE, dz_scratch, dgamma, dbeta, rows, S, pad_id, make_drop(p_drop, seed, stream_id, step_dev), part_ln);
  MMSUM_CHECK_LAUNCH();
  if (dgamma != nullptr)
    if (int rc = ordered_colsum(part_ln, nblk, 2 * D, D, dgamma, dbeta, st)) return rc;
  if (dE != nullptr) {
    embed_group_kernel<<<1, 1024, 0, st>>>(ids, rows, V, pad_id, cursor, order, sid);
    MMSUM_CHECK_LAUNCH();
    embed_scatter_tile_kernel<<<dim3(ntiles, D / 256), 256, 0, st>>>(dz_scratch, sid, order, cursor, V, dE, head, tail);
    MMSUM_CHECK_LAUNCH();
    embed_scatter_span_kernel<<<dim3(nblocks(rows, 16, 148 * 4), D / 256), 256, 0, st>>>(sid, cursor, V, head, tail, dE);
    MMSUM_CHECK_LAUNCH();
  }
  if (dP != nullptr || want_remb) {
    embed_pos_bwd_kernel<true><<<dim3(D / 256, S), 256, 0, st>>>(dz_scratch, rating_diff, dP, dremb, rows / S, S, part_remb);
    MMSUM_CHECK_LAUNCH();
  }
  if (want_remb)
    if (int rc = ordered_colsum(part_remb, S, D, D, dremb, nullptr, st)) return rc;
  return 0;
}

extern "C" int mmsum_embed_ln_bwd_ordered(const void* dout, const void* dout2, const int32_t* ids, const float* E, const float* P,
                                          const float* rating_diff, const float* remb, const float* gamma, const float* mean,
                                          const float* rstd, float* dE, float* dP, float* dremb, float* dgamma, float* dbeta,
                                          float* dz_scratch, int32_t rows, int32_t S, int32_t d_model, int32_t pad_id,
                                          float p_drop, uint64_t seed, uint32_t stream_id, const uint32_t* step_dev, int32_t V,
                                          float* workspace, int64_t workspace_elems, void* stream) {
  if (!dE || !dP || !dgamma || !dbeta || (rating_diff != nullptr && !dremb)) return MMSUM_ERR_INVALID;
  return embed_ln_bwd_ordered(dout, dout2, ids, E, P, rating_diff, remb, gamma, mean, rstd, dE, dP, dremb, dgamma, dbeta, dz_scratch,
                              rows, S, d_model, pad_id, p_drop, seed, stream_id, step_dev, V, workspace, workspace_elems, stream);
}

extern "C" int mmsum_embed_ln_bwd_ordered_subset(const void* dout, const void* dout2, const int32_t* ids, const float* E,
                                                 const float* P, const float* rating_diff, const float* remb, const float* gamma,
                                                 const float* mean, const float* rstd, float* dE, float* dP, float* dremb,
                                                 float* dgamma, float* dbeta, float* dz_scratch, int32_t rows, int32_t S,
                                                 int32_t d_model, int32_t pad_id, float p_drop, uint64_t seed, uint32_t stream_id,
                                                 const uint32_t* step_dev, int32_t V, float* workspace, int64_t workspace_elems,
                                                 void* stream) {
  return embed_ln_bwd_ordered(dout, dout2, ids, E, P, rating_diff, remb, gamma, mean, rstd, dE, dP, dremb, dgamma, dbeta, dz_scratch,
                              rows, S, d_model, pad_id, p_drop, seed, stream_id, step_dev, V, workspace, workspace_elems, stream);
}

extern "C" int mmsum_add_ln_fwd(const void* res, const void* y, const float* gamma, const float* beta, void* out,
                                float* mean, float* rstd, int32_t rows, int32_t d_model, float p_drop, uint64_t seed,
                                uint32_t stream_id, const uint32_t* step_dev, void* stream) {
  if (d_model != D || rows <= 0 || !res || !y || !out) return MMSUM_ERR_INVALID;
  MMSUM_LAUNCH_PDL(add_ln_fwd_kernel, nblocks(rows, 8, 148 * 2), 256, 0, STREAM(stream), reinterpret_cast<const bf16*>(res),
                                                                 reinterpret_cast<const bf16*>(y), gamma, beta,
                                                                 reinterpret_cast<bf16*>(out), mean, rstd, rows,
                                                                 make_drop(p_drop, seed, stream_id, step_dev));
  MMSUM_CHECK_LAUNCH();
  return 0;
}

// dgamma = dbeta = NULL: the variant without the gamma / beta reduction (one kernel, nothing to order)
static int add_ln_bwd_frozen(const void* d1, const void* d2, const void* res, const void* y, const float* gamma, const float* mean,
                             const float* rstd, void* dres, void* dy, int32_t rows, float p_drop, uint64_t seed, uint32_t stream_id,
                             const uint32_t* step_dev, void* stream) {
  MMSUM_LAUNCH_PDL((add_ln_bwd_kernel<false, false>), nblocks(rows, 4 * 4, 148 * 3), 128, 0, STREAM(stream),
      reinterpret_cast<const bf16*>(d1), reinterpret_cast<const bf16*>(d2), reinterpret_cast<const bf16*>(res),
      reinterpret_cast<const bf16*>(y), gamma, mean, rstd, reinterpret_cast<bf16*>(dres), reinterpret_cast<bf16*>(dy),
      nullptr, nullptr, rows, make_drop(p_drop, seed, stream_id, step_dev), nullptr);
  MMSUM_CHECK_LAUNCH();
  return 0;
}

extern "C" int mmsum_add_ln_bwd(const void* d1, const void* d2, const void* res, const void* y, const float* gamma,
                                const float* mean, const float* rstd, void* dres, void* dy, float* dgamma, float* dbeta,
                                int32_t rows, int32_t d_model, float p_drop, uint64_t seed, uint32_t stream_id, const uint32_t* step_dev,
                                void* stream) {
  if (d_model != D || rows <= 0 || !d1 || !res || !y || !dres || !dy) return MMSUM_ERR_INVALID;
  if (p_drop > 0.f && dres == dy) return MMSUM_ERR_INVALID;
  if ((dgamma == nullptr) != (dbeta == nullptr)) return MMSUM_ERR_INVALID;
  if (dgamma == nullptr)
    return add_ln_bwd_frozen(d1, d2, res, y, gamma, mean, rstd, dres, dy, rows, p_drop, seed, stream_id, step_dev, stream);
  static std::atomic<unsigned long long> attr{0};
  if (int rc = ensure_dyn_smem(add_ln_bwd_kernel<false>, 4 * 2 * VPL * 32 * 4, attr)) return rc;
  MMSUM_LAUNCH_PDL(add_ln_bwd_kernel<false>, nblocks(rows, 4 * 4, 148 * 3), 128, 4 * 2 * VPL * 32 * 4, STREAM(stream), 
      reinterpret_cast<const bf16*>(d1), reinterpret_cast<const bf16*>(d2), reinterpret_cast<const bf16*>(res),
      reinterpret_cast<const bf16*>(y), gamma, mean, rstd, reinterpret_cast<bf16*>(dres), reinterpret_cast<bf16*>(dy),
      dgamma, dbeta, rows, make_drop(p_drop, seed, stream_id, step_dev), nullptr);
  MMSUM_CHECK_LAUNCH();
  return 0;
}

extern "C" int mmsum_add_ln_bwd_ordered(const void* d1, const void* d2, const void* res, const void* y, const float* gamma,
                                        const float* mean, const float* rstd, void* dres, void* dy, float* dgamma, float* dbeta,
                                        int32_t rows, int32_t d_model, float p_drop, uint64_t seed, uint32_t stream_id,
                                        const uint32_t* step_dev, float* workspace, int64_t workspace_elems, void* stream) {
  if (d_model != D || rows <= 0 || !d1 || !res || !y || !dres || !dy) return MMSUM_ERR_INVALID;
  if (p_drop > 0.f && dres == dy) return MMSUM_ERR_INVALID;
  if ((dgamma == nullptr) != (dbeta == nullptr)) return MMSUM_ERR_INVALID;
  if (dgamma == nullptr)      // no reduction left to order: the workspace is not read
    return add_ln_bwd_frozen(d1, d2, res, y, gamma, mean, rstd, dres, dy, rows, p_drop, seed, stream_id, step_dev, stream);
  const int nblk = nblocks(rows, 4 * 4, 148 * 3);
  if (!workspace || workspace_elems < (int64_t)nblk * 2 * D) return MMSUM_ERR_INVALID;
  static std::atomic<unsigned long long> attr{0};
  if (int rc = ensure_dyn_smem(add_ln_bwd_kernel<true>, 4 * 2 * VPL * 32 * 4, attr)) return rc;
  MMSUM_LAUNCH_PDL(add_ln_bwd_kernel<true>, nblk, 128, 4 * 2 * VPL * 32 * 4, STREAM(stream),
      reinterpret_cast<const bf16*>(d1), reinterpret_cast<const bf16*>(d2), reinterpret_cast<const bf16*>(res),
      reinterpret_cast<const bf16*>(y), gamma, mean, rstd, reinterpret_cast<bf16*>(dres), reinterpret_cast<bf16*>(dy),
      dgamma, dbeta, rows, make_drop(p_drop, seed, stream_id, step_dev), workspace);
  MMSUM_CHECK_LAUNCH();
  return ordered_colsum(workspace, nblk, 2 * D, D, dgamma, dbeta, STREAM(stream));
}

extern "C" int mmsum_colsum(const void* x, int64_t ld, int32_t rows, int32_t N, float* out, void* stream) {
  if (!x || !out || rows <= 0 || N <= 0 || (N % 8) || (ld % 8)) return MMSUM_ERR_INVALID;
  const int gx = (N + 255) / 256;
  int gy = (148 * 4) / gx; if (gy < 1) gy = 1; if (gy > (rows + 63) / 64) gy = (rows + 63) / 64;
  const int rpb = (rows + gy - 1) / gy;
  MMSUM_LAUNCH_PDL(colsum_kernel<false>, dim3(gx, gy), 256, 0, STREAM(stream), reinterpret_cast<const bf16*>(x), ld, rows, N, out, rpb,
                   nullptr);
  MMSUM_CHECK_LAUNCH();
  return 0;
}

extern "C" int mmsum_colsum_ordered(const void* x, int64_t ld, int32_t rows, int32_t N, float* out, float* workspace,
                                    int64_t workspace_elems, void* stream) {
  if (!x || !out || rows <= 0 || N <= 0 || (N % 8) || (ld % 8)) return MMSUM_ERR_INVALID;
  const int gx = (N + 255) / 256;
  int gy = (148 * 4) / gx; if (gy < 1) gy = 1; if (gy > (rows + 63) / 64) gy = (rows + 63) / 64;
  const int rpb = (rows + gy - 1) / gy;
  if (!workspace || workspace_elems < (int64_t)gy * N) return MMSUM_ERR_INVALID;
  MMSUM_LAUNCH_PDL(colsum_kernel<true>, dim3(gx, gy), 256, 0, STREAM(stream), reinterpret_cast<const bf16*>(x), ld, rows, N, out, rpb,
                   workspace);
  MMSUM_CHECK_LAUNCH();
  return ordered_colsum(workspace, gy, N, N, out, nullptr, STREAM(stream));
}

extern "C" int mmsum_gate_fwd(const void* o3, const void* u, const uint8_t* pres, void* y, void* ab, int32_t rows,
                              int32_t rows_per_biz, int32_t d_model, void* stream) {
  if (d_model != D || rows <= 0 || rows_per_biz <= 0) return MMSUM_ERR_INVALID;
  const long long n = (long long)rows * D;
  MMSUM_LAUNCH_PDL(gate_fwd_kernel, nblocks(n, 2048, 148 * 8), 256, 0, STREAM(stream), 
      reinterpret_cast<const bf16*>(o3), reinterpret_cast<const bf16*>(u), pres, reinterpret_cast<bf16*>(y),
      reinterpret_cast<bf16*>(ab), n, rows_per_biz);
  MMSUM_CHECK_LAUNCH();
  return 0;
}
extern "C" int mmsum_gate_bwd_u(const void* dy, const void* o3, const void* ab, void* du, int32_t rows, int32_t d_model, void* stream) {
  if (d_model != D || rows <= 0) return MMSUM_ERR_INVALID;
  const long long n = (long long)rows * D;
  MMSUM_LAUNCH_PDL(gate_bwd_u_kernel, nblocks(n, 2048, 148 * 8), 256, 0, STREAM(stream), 
      reinterpret_cast<const bf16*>(dy), reinterpret_cast<const bf16*>(o3), reinterpret_cast<const bf16*>(ab),
      reinterpret_cast<bf16*>(du), n);
  MMSUM_CHECK_LAUNCH();
  return 0;
}
extern "C" int mmsum_gate_bwd_o(const void* dy, const void* ab, const void* dca, const void* dcb, void* do3, int32_t rows,
                                int32_t d_model, void* stream) {
  if (d_model != D || rows <= 0) return MMSUM_ERR_INVALID;
  const long long n = (long long)rows * D;
  MMSUM_LAUNCH_PDL(gate_bwd_o_kernel, nblocks(n, 2048, 148 * 8), 256, 0, STREAM(stream), 
      reinterpret_cast<const bf16*>(dy), reinterpret_cast<const bf16*>(ab), reinterpret_cast<const bf16*>(dca),
      reinterpret_cast<const bf16*>(dcb), reinterpret_cast<bf16*>(do3), n);
  MMSUM_CHECK_LAUNCH();
  return 0;
}

extern "C" int mmsum_ce_fwd_bwd(void* logits, int64_t ld, int32_t rows, int32_t V, const int32_t* target, float eps,
                                float gscale, const float* gscale_dev, float* loss_rows, float* loss_out, float loss_scale,
                                float* lse_rows, int32_t write_grad, void* stream) {
  if (!logits || !target || !loss_rows || rows <= 0 || V <= 8 || (ld % 8) || ld < V) return MMSUM_ERR_INVALID;
  ce_fwd_bwd_kernel<<<rows, 256, 0, STREAM(stream)>>>(reinterpret_cast<bf16*>(logits), ld, V, target, eps, gscale, gscale_dev, loss_rows,
                                                      lse_rows, write_grad);
  MMSUM_CHECK_LAUNCH();
  if (loss_out != nullptr) {
    sum_rows_kernel<<<1, 1024, 0, STREAM(stream)>>>(loss_rows, rows, loss_scale, loss_out);
    MMSUM_CHECK_LAUNCH();
  }
  return 0;
}

extern "C" int mmsum_prep_step(const int64_t* reviews, const int64_t* reviews_mask, const float* rating,
                               const uint8_t* table_valid, const uint8_t* img_mask, const MmsumPrepArgs* a, void* stream) {
  if (!a || !reviews || !reviews_mask || !rating || a->B <= 0 || a->R < 2 || a->S <= 0) return MMSUM_ERR_INVALID;
  if (a->n_mod != 1 && a->n_mod != 3) return MMSUM_ERR_INVALID;
  if (a->S_enc < 0 || a->S_enc > a->S) return MMSUM_ERR_INVALID;
  if (a->n_mod == 3 && (!table_valid || !img_mask || a->F <= 0 || a->n_img <= 0)) return MMSUM_ERR_INVALID;
  prep_step_kernel<<<a->B, 128, 0, STREAM(stream)>>>(reviews, reviews_mask, rating, table_valid, img_mask, *a);
  MMSUM_CHECK_LAUNCH();
  return 0;
}

extern "C" int mmsum_table_fwd(const MmsumTableArgs* a, void* stream) {
  if (!a || !a->E || !a->field || !a->X || !a->valid || a->B <= 0) return MMSUM_ERR_INVALID;
  if (a->dataset == 0) table_yelp_kernel<<<a->B * 47, 256, 0, STREAM(stream)>>>(*a);
  else if (a->dataset == 1) table_amazon_kernel<<<a->B * 133, 256, 0, STREAM(stream)>>>(*a);
  else return MMSUM_ERR_INVALID;
  MMSUM_CHECK_LAUNCH();
  return 0;
}

extern "C" int mmsum_table_bits_bwd(const void* dX, const int64_t* bits, float* dW, int32_t B, int32_t F, int32_t f0,
                                    int32_t nrows, int32_t nb, void* stream) {
  if (!dX || !bits || !dW || B <= 0 || nrows <= 0 || nb <= 0) return MMSUM_ERR_INVALID;
  table_bits_bwd_kernel<<<D / 256, 256, 0, STREAM(stream)>>>(reinterpret_cast<const bf16*>(dX), bits, dW, B, F, f0, nrows, nb);
  MMSUM_CHECK_LAUNCH();
  return 0;
}
