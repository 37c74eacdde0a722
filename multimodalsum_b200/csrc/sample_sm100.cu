// Device-side sampling of one token per row (generate(do_sample=True), no beam search).
//
// Replaces, per row, the chain the reference runs on [N, V] tensors in _generate_no_beam_search (vendored transformers 3.0.2
// generation_utils.py): postprocess_next_token_scores (enforce_repetition_penalty_, the EOS ban below min_length,
// calc_banned_ngram_tokens), `scores / temperature`, top_k_top_p_filtering(min_tokens_to_keep=1), softmax and
// torch.multinomial, then `tokens_to_add = next_token * unfinished + pad * (1 - unfinished)` and the unfinished update.
// No adjust_logits_during_generation: the reference calls it on the beam path only.
//
// One CTA per row.  The row's fp32 logits are staged once into shared memory (50265 x 4 B = 201 KB, so one CTA per SM) with
// 128-bit loads; every later pass reads shared memory only:
//   1. repetition penalty (each distinct id of the prefix once), EOS ban, n-gram ban (the rule of beam_topk_kernel), / T;
//   2. top-k: radix select (4 x 8-bit digits) of the k-th largest order-preserving uint32 key; keys below it become -inf,
//      so ties at the k-th value survive;
//   3. top-p: a radix select over the same keys weighted by the softmax mass, to find the token whose cumulative mass crosses
//      top_p.  Tokens are ranked by descending score, equal scores by ascending token id (our rule: torch.sort leaves the
//      order of equal values unspecified).  A token is kept iff the mass ranked strictly before it is <= top_p * Z;
//   4. draw: inverse CDF over the kept tokens in vocabulary order, from block prefix sums of exp(s - max).
// The softmax masses are 2^40-scaled integers (exp(s - max) <= 1, so a row sums to < 2^56): every histogram, prefix sum and
// comparison is exact and independent of the order in which threads add, so a draw does not depend on scheduling.
// Randomness: Philox4x32-10 (curand_kernel.h), key = the 64-bit seed, counter = (cur_len, row); one draw is a pure function
// of (seed, row, step), whatever the grid, the number of rows or graph replay.
#include <curand_philox4x32_x.h>   // the counter-based generator of the curand_kernel.h device API, without its global tables

#include "common.cuh"
#include "../../include/mmsum_b200.h"

namespace mmsum {

static constexpr int kSampleThreads = 512;
static constexpr int kSampleWarps = kSampleThreads / 32;
static constexpr int kSampleMaxL = 160;
static constexpr int kSampleMaxSmem = 227 * 1024;
static constexpr int kSampleStaticSmem = 4096;          // histogram, history and scan scratch below (static shared memory)
static constexpr float kMassScale = 1099511627776.0f;  // 2^40

// Order-preserving uint32 image of a score.  -0.0 is folded onto +0.0 first: torch compares them as equal, so they must share
// one key for the top-k / top-p tie rules to match.
__device__ __forceinline__ uint32_t score_key(float v) {
  const uint32_t u = (v == 0.f) ? 0u : __float_as_uint(v);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}

struct SampleSmem {
  unsigned long long hist[256];
  unsigned long long warp_part[kSampleWarps];
  int ids[kSampleMaxL];
  int sel_bin;
  unsigned long long sel_above;
  float red[kSampleWarps];
};

// Warp 0 walks the 256 bins from the highest digit down and finds the first bin at which the running sum reaches `need`.
// Writes the bin and the sum of the bins above it; sel_bin = -1 when the whole histogram stays below `need`.
__device__ void select_bin(SampleSmem& sm, unsigned long long need) {
  if (threadIdx.x < 32) {
    const int lane = threadIdx.x;
    unsigned long long v[8], local = 0;
#pragma unroll
    for (int j = 0; j < 8; ++j) { v[j] = sm.hist[255 - 8 * lane - j]; local += v[j]; }
    unsigned long long incl = local;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const unsigned long long y = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += y;
    }
    const unsigned hit = __ballot_sync(0xffffffffu, incl >= need);
    if (hit == 0) {
      if (lane == 0) sm.sel_bin = -1;
    } else if (lane == __ffs(hit) - 1) {
      unsigned long long acc = incl - local;
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        if (acc + v[j] >= need) { sm.sel_bin = 255 - 8 * lane - j; sm.sel_above = acc; break; }
        acc += v[j];
      }
    }
  }
  __syncthreads();
}

// Exclusive block prefix sum of one value per thread (thread order); returns the thread's offset and the total.
__device__ __forceinline__ unsigned long long block_exclusive_scan(SampleSmem& sm, unsigned long long x,
                                                                    unsigned long long& total) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  unsigned long long incl = x;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const unsigned long long y = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += y;
  }
  if (lane == 31) sm.warp_part[warp] = incl;
  __syncthreads();
  unsigned long long before = 0;
  total = 0;
#pragma unroll
  for (int w = 0; w < kSampleWarps; ++w) {
    if (w < warp) before += sm.warp_part[w];
    total += sm.warp_part[w];
  }
  __syncthreads();
  return before + incl - x;
}

__device__ __forceinline__ unsigned long long mass_of(float s, float M) {
  return s == -INFINITY ? 0ull : __float2ull_rz(expf(s - M) * kMassScale);
}

__global__ void __launch_bounds__(kSampleThreads, 1)
sample_token_kernel(const float* __restrict__ logits, long long ld, int V, long long* __restrict__ ids, int L,
                    const long long* __restrict__ cur_dev, const unsigned long long* __restrict__ seed_dev, int min_length,
                    int ngram, int eos, int pad, float temperature, int top_k, float top_p, float penalty,
                    unsigned char* __restrict__ unfinished, int* __restrict__ next_tok32) {
  extern __shared__ __align__(16) float s[];
  __shared__ SampleSmem sm;
  const int row = blockIdx.x, tid = threadIdx.x;
  const int cur = (int)cur_dev[0];
  if (cur < 1 || cur >= L) return;      // no prefix or no slot left to write: nothing to sample (uniform over the block)
  const float* z = logits + (long long)row * ld;
  long long* hist = ids + (long long)row * L;

  // ---- stage the row (128-bit loads; the host checks alignment) and the prefix
  const int nvec = V >> 2;
  for (int i = tid; i < nvec; i += kSampleThreads)
    reinterpret_cast<float4*>(s)[i] = __ldg(reinterpret_cast<const float4*>(z) + i);
  for (int i = nvec * 4 + tid; i < V; i += kSampleThreads) s[i] = z[i];
  for (int t = tid; t < cur; t += kSampleThreads) sm.ids[t] = (int)hist[t];
  __syncthreads();

  // ---- 1. enforce_repetition_penalty_: every distinct id of positions 0 .. cur-1 once (the first occurrence does it)
  if (penalty != 1.f) {
    for (int t = tid; t < cur; t += kSampleThreads) {
      const int tok = sm.ids[t];
      bool first = tok >= 0 && tok < V;
      for (int j = 0; j < t && first; ++j) first = sm.ids[j] != tok;
      if (first) { const float v = s[tok]; s[tok] = v < 0.f ? v * penalty : v / penalty; }
    }
    __syncthreads();
  }
  // ---- 2. EOS below min_length, 3. n-gram ban (as beam_topk_kernel)
  if (tid == 0 && cur < min_length) s[eos] = -INFINITY;
  if (ngram > 0 && cur >= ngram) {
    for (int i = tid; i <= cur - ngram; i += kSampleThreads) {
      bool hit = true;
      for (int j = 0; j < ngram - 1; ++j) hit = hit && (sm.ids[i + j] == sm.ids[cur - ngram + 1 + j]);
      const int tok = sm.ids[i + ngram - 1];
      if (hit && tok >= 0 && tok < V) s[tok] = -INFINITY;
    }
  }
  __syncthreads();
  // ---- 5. temperature
  if (temperature != 1.f)
    for (int i = tid; i < V; i += kSampleThreads) s[i] = s[i] / temperature;

  // ---- 6a. top-k: the k-th largest key by radix select; smaller keys are removed
  if (top_k > 0 && top_k < V) {
    uint32_t prefix = 0, mask = 0;
    unsigned long long need = (unsigned long long)top_k;
    for (int shift = 24; shift >= 0; shift -= 8) {
      if (tid < 256) sm.hist[tid] = 0;
      __syncthreads();
      // warp-aggregated: logits share few exponent bytes, so per-lane atomics would serialise on a handful of bins
      for (int base = 0; base < V; base += kSampleThreads) {
        const int i = base + tid;
        const uint32_t key = i < V ? score_key(s[i]) : 0u;
        const uint32_t bin = (i < V && (key & mask) == prefix) ? ((key >> shift) & 255) : 256u;
        const unsigned peers = __match_any_sync(0xffffffffu, bin);
        if (bin < 256 && (tid & 31) == __ffs(peers) - 1) atomicAdd(&sm.hist[bin], (unsigned long long)__popc(peers));
      }
      __syncthreads();
      select_bin(sm, need);           // always found: the range holds >= need keys
      prefix |= (uint32_t)sm.sel_bin << shift;
      mask |= 255u << shift;
      need -= sm.sel_above;
      __syncthreads();
    }
    for (int i = tid; i < V; i += kSampleThreads)
      if (score_key(s[i]) < prefix) s[i] = -INFINITY;
  }
  __syncthreads();

  // ---- row maximum of what is left (the reference for the softmax masses)
  float m = -INFINITY;
  for (int i = tid; i < V; i += kSampleThreads) m = fmaxf(m, s[i]);
  m = warp_max(m);
  if ((tid & 31) == 0) sm.red[tid >> 5] = m;
  __syncthreads();
  float M = sm.red[0];
#pragma unroll
  for (int w = 1; w < kSampleWarps; ++w) M = fmaxf(M, sm.red[w]);

  // chunked layout for the ordered passes: thread t owns tokens [t*C, t*C + C); C odd keeps the shared loads conflict-free
  int C = (V + kSampleThreads - 1) / kSampleThreads;
  C |= 1;
  const int c0 = min(tid * C, V), c1 = min(c0 + C, V);

  // ---- 6b. top-p over the remaining tokens
  if (top_p < 1.f && M != -INFINITY) {
    unsigned long long local = 0, Z;
    for (int i = c0; i < c1; ++i) local += mass_of(s[i], M);
    block_exclusive_scan(sm, local, Z);
    const unsigned long long T = (unsigned long long)((double)top_p * (double)Z);
    // the crossing token: the first one (descending key) at which the mass up to and including it exceeds T
    uint32_t prefix = 0, mask = 0;
    unsigned long long above = 0;
    bool keep_all = false;
    for (int shift = 24; shift >= 0; shift -= 8) {
      if (tid < 256) sm.hist[tid] = 0;
      __syncthreads();
      for (int i = tid; i < V; i += kSampleThreads) {
        const float v = s[i];
        const uint32_t key = score_key(v);
        if ((key & mask) == prefix && v != -INFINITY) atomicAdd(&sm.hist[(key >> shift) & 255], mass_of(v, M));
      }
      __syncthreads();
      select_bin(sm, T - above + 1);
      if (sm.sel_bin < 0) { keep_all = true; break; }     // T >= Z: top_p rounds to 1
      prefix |= (uint32_t)sm.sel_bin << shift;
      mask |= 255u << shift;
      above += sm.sel_above;
      __syncthreads();
    }
    if (!keep_all) {
      // tokens of the crossing key, in id order, are kept while the mass before them stays <= T
      const float ks = __uint_as_float((prefix & 0x80000000u) ? (prefix & 0x7fffffffu) : ~prefix);
      const unsigned long long mk = mass_of(ks, M);
      const unsigned long long keep_eq = (T - above) / mk + 1;
      unsigned long long eq_local = 0, eq_total;
      for (int i = c0; i < c1; ++i) eq_local += score_key(s[i]) == prefix;
      unsigned long long rank = block_exclusive_scan(sm, eq_local, eq_total);
      for (int i = c0; i < c1; ++i) {
        const uint32_t key = score_key(s[i]);
        if (key == prefix) { if (rank >= keep_eq) s[i] = -INFINITY; ++rank; }
        else if (key < prefix) s[i] = -INFINITY;
      }
      __syncthreads();
    }
  }

  // ---- 7. draw: r uniform in [0, Z), the first kept token whose inclusive prefix mass exceeds r
  unsigned long long local = 0, Z;
  for (int i = c0; i < c1; ++i) local += mass_of(s[i], M);
  const unsigned long long before = block_exclusive_scan(sm, local, Z);
  const unsigned long long seed = seed_dev[0];
  const uint4 rnd = curand_Philox4x32_10(make_uint4((uint32_t)cur, 0u, (uint32_t)row, 0u),
                                         make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)));
  const unsigned long long r = __umul64hi(((unsigned long long)rnd.y << 32) | rnd.x, Z);
  if (Z == 0) {                         // every token is banned: nothing to draw from; close the row
    if (tid == 0) sm.sel_bin = eos;
  } else if (r >= before && r < before + local) {
    unsigned long long acc = before;
    for (int i = c0; i < c1; ++i) {
      acc += mass_of(s[i], M);
      if (acc > r) { sm.sel_bin = i; break; }
    }
  }
  __syncthreads();

  // ---- loop bookkeeping: tokens_to_add, the history, the decoder's next input, unfinished
  if (tid == 0) {
    const bool live = unfinished[row] != 0;
    const int tok = live ? sm.sel_bin : pad;
    if (cur < L) hist[cur] = tok;
    if (next_tok32 != nullptr) next_tok32[row] = tok;
    if (tok == eos) unfinished[row] = 0;
  }
}

}  // namespace mmsum

using namespace mmsum;

extern "C" int mmsum_sample_token(const float* logits, int64_t ld, int32_t rows, int32_t V, int64_t* ids, int32_t L,
                                  const int64_t* cur_dev, const uint64_t* seed_dev, int32_t min_length, int32_t ngram,
                                  int32_t eos, int32_t pad, float temperature, int32_t top_k, float top_p, float penalty,
                                  uint8_t* unfinished, int32_t* next_tok32, void* stream_v) {
  if (!logits || !ids || !cur_dev || !seed_dev || !unfinished) return MMSUM_ERR_INVALID;
  if (rows <= 0 || V < 32 || L < 2 || L > kSampleMaxL) return MMSUM_ERR_INVALID;
  if ((size_t)V * sizeof(float) + kSampleStaticSmem > (size_t)kSampleMaxSmem) return MMSUM_ERR_INVALID;
  if ((ld % 4) || ld < V || (reinterpret_cast<uintptr_t>(logits) & 15)) return MMSUM_ERR_INVALID;
  if (ngram < 0 || ngram > 8 || min_length < 0 || eos < 0 || eos >= V || pad < 0 || pad >= V) return MMSUM_ERR_INVALID;
  if (!(temperature > 0.f) || top_k < 0 || !(top_p >= 0.f && top_p <= 1.f) || !(penalty >= 1.f)) return MMSUM_ERR_INVALID;
  const int smem = V * (int)sizeof(float);
  static std::atomic<unsigned long long> attr_set{0};
  if (int rc = ensure_dyn_smem(sample_token_kernel, kSampleMaxSmem - kSampleStaticSmem, attr_set)) return rc;
  sample_token_kernel<<<rows, kSampleThreads, smem, reinterpret_cast<cudaStream_t>(stream_v)>>>(
      logits, ld, V, reinterpret_cast<long long*>(ids), L, reinterpret_cast<const long long*>(cur_dev),
      reinterpret_cast<const unsigned long long*>(seed_dev), min_length, ngram, eos, pad, temperature, top_k, top_p, penalty,
      unfinished, next_tok32);
  MMSUM_CHECK_LAUNCH();
  return 0;
}
