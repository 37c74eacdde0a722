// Decode-step attention for beam-search generation (BASELINE config 5; reference: the cached branch of
// SelfAttention.get_head_output, src/transformer/modeling_multimodalsum.py:774-815, 889-920, driven by
// _generate_beam_search :2857-3010).
//
// One decode step feeds ONE query row per hypothesis, so the step is bound by streaming the cached keys / values out of
// HBM (10 GB of cross-attention K|V per token at 64 businesses), not by the tensor pipe.  The training kernels' 128-row
// tcgen05 query tiles waste 97 % of their work here; these kernels are built for the decode shape instead:
//
//   attn_decode_cross_kernel  one CTA per (business, head).  The `beams` query rows of a business attend to the SAME
//       un-expanded per-business memory (the reference expands the memory per beam and re-gathers it every token,
//       :2598-2627, :3004-3010), so K_e / V_e of every entity are read ONCE per business and head: TMA (128B swizzle) ->
//       per-warp smem stage -> ldmatrix -> mma.sync m16n8k16 (bf16, fp32 accumulate; the beams are the M rows, padded to 16)
//       -> per-entity softmax in registers -> P V -> mean over the valid entities of the modality.  Eight warps pull
//       entities from a shared counter; a warp owns ONE 26 KB stage that holds the entity's K, then (loaded during the
//       softmax) its V — eight independent load -> compute chains per SM keep HBM busy where four double-staged warps
//       moving in lock-step did not (203 -> see profiles/r02_decode_* per layer at the config-5 shape).
//   attn_decode_self_kernel   one warp per (hypothesis, head): appends the new position's K|V to the cache and attends to
//       positions 0..t through a per-hypothesis slot table (`hist[n][j]` = cache row that holds position j of hypothesis n),
//       so re-ranking the beams permutes a 128 KB table instead of copying 12 layers of K|V caches (_reorder_cache,
//       :3103-3115).
#include "common.cuh"
#include "../../include/mmsum_b200.h"

#include <cudaTypedefs.h>

namespace mmsum {

int make_tmap(CUtensorMap* out, const void* ptr, int dtype, uint64_t inner, uint64_t outer, uint64_t ld_bytes,
              uint32_t box_inner, uint32_t box_outer);

static constexpr int DHD = 64;
static constexpr int kDecMaxKeys = 208;                 // keys per entity, multiple of 16
static constexpr int kDecStage = kDecMaxKeys * 128;     // 26 KB: one entity's K (or V) head slice, 128 B per key row
static constexpr int kDecWarps = 8;
static constexpr int kDecMaxEnt = 32;
static constexpr int kDecMaxBeams = 8;
static constexpr float kDecLog2e = 1.4426950408889634f;

struct DecItem { int kv_row0; short nkeys, mod; };
struct DecMaps { CUtensorMap kv[3]; };

struct DecSmem {
  uint8_t kv[kDecWarps][kDecStage];      // per warp: the current entity's K, later overwritten by its V
  float oacc[3][kDecMaxBeams][DHD];
  uint64_t bar[kDecWarps];
  DecItem items[kDecMaxEnt];
  int n_items;
  int next_item;
  int turn;                              // ordered accumulation: index of the entity whose output is added next
};

__device__ __forceinline__ void ldsm_x4(uint32_t saddr, uint32_t (&r)[4]) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(saddr));
}
__device__ __forceinline__ void ldsm_x4_t(uint32_t saddr, uint32_t (&r)[4]) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(saddr));
}
// D[16x8] += A[16x16] B[16x8], bf16 operands, fp32 accumulate
__device__ __forceinline__ void mma_16816(float (&d)[4], uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, uint32_t b0, uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3]) : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
}
// byte offset of 16-byte chunk `chunk` of key row `row` inside a 128B-swizzled stage
__device__ __forceinline__ uint32_t sw128(int row, int chunk) { return (uint32_t)(row * 128 + ((chunk ^ (row & 7)) << 4)); }

__global__ void __launch_bounds__(kDecWarps * 32, 1)
attn_decode_cross_kernel(const __grid_constant__ DecMaps maps, const MmsumAttnArgs p) {
  extern __shared__ uint8_t smem_raw[];
  DecSmem& sm = *reinterpret_cast<DecSmem*>(smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u));
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int h = blockIdx.x % p.H, biz = blockIdx.x / p.H;
  const int R = p.R;                                  // beams per business (query rows of this CTA)
  const int g = lane >> 2, t = lane & 3;              // mma fragment coordinates: row group, thread in group

  // ---- valid entities of this business (lane = candidate entity), as in the training kernels
  if (warp == 0) {
    int m = 0, e = lane, found = 0;
    for (m = 0; m < p.n_mod; ++m) {
      if (e < p.mods[m].E) { found = 1; break; }
      e -= p.mods[m].E;
    }
    bool ok = false;
    DecItem it; it.kv_row0 = 0; it.nkeys = 0; it.mod = 0;
    if (found) {
      const MmsumAttnMod& md = p.mods[m];
      ok = (p.ent_valid == nullptr) || p.ent_valid[(long long)biz * p.E_total + md.ent_base + e] != 0;
      it.kv_row0 = (int)(md.kv_row_base + ((long long)biz * md.E + e) * (md.ent_stride > 0 ? md.ent_stride : md.Sk));
      it.nkeys = (short)md.Sk; it.mod = (short)m;
    }
    const uint32_t bal = __ballot_sync(0xffffffffu, ok);
    if (ok) sm.items[__popc(bal & ((1u << lane) - 1u))] = it;
    if (lane == 0) { sm.n_items = __popc(bal); sm.next_item = 0; sm.turn = 0; }
  }
  for (int i = threadIdx.x; i < 3 * kDecMaxBeams * DHD; i += blockDim.x) (&sm.oacc[0][0][0])[i] = 0.f;
  if (threadIdx.x == 32) {
    for (int w = 0; w < kDecWarps; ++w) mbar_init(&sm.bar[w], 1);
    fence_barrier_init();
  }
  __syncthreads();
  const int n_items = sm.n_items;

  // ---- the query rows as mma A fragments (rows >= R are zero), loaded once
  uint32_t qa[4][2];
  {
    const bf16* Q = reinterpret_cast<const bf16*>(p.Q);
#pragma unroll
    for (int ks = 0; ks < 4; ++ks) {
      qa[ks][0] = 0; qa[ks][1] = 0;
      if (g < R) {
        const bf16* q = Q + (long long)(biz * R + g) * p.ldq + p.q_col + h * DHD + ks * 16 + 2 * t;
        qa[ks][0] = *reinterpret_cast<const uint32_t*>(q);
        qa[ks][1] = *reinterpret_cast<const uint32_t*>(q + 8);
      }
    }
  }
  const float sc = p.scale * kDecLog2e;
  const uint32_t k_base = smem_u32(sm.kv[warp]), v_base = k_base;
  auto load_tile = [&](const DecItem& it, int col) {
    const int n16 = (it.nkeys + 15) & ~15;
    mbar_expect_tx(&sm.bar[warp], n16 * 128);
    tma_load_2d(sm.kv[warp], &maps.kv[it.mod], &sm.bar[warp], col + h * DHD, it.kv_row0);
  };
  float oc[8][4];
#pragma unroll
  for (int nd = 0; nd < 8; ++nd) { oc[nd][0] = 0.f; oc[nd][1] = 0.f; oc[nd][2] = 0.f; oc[nd][3] = 0.f; }
  // Entity outputs are added to the CTA accumulator in ENTITY ORDER (bit-reproducible results): the warp that finished entity i
  // waits until entity i-1 has been added, then adds its own output with plain read-modify-writes (it holds the turn) and passes
  // the turn on.  Entities are pulled in increasing order, so they also finish roughly in order and the wait is short; the sum
  // order does not depend on which warp got which entity or on timing.
  auto add_in_order = [&](int i, int m) {
    if (lane == 0) { while (*reinterpret_cast<volatile int*>(&sm.turn) != i) { } }
    __syncwarp();
    __threadfence_block();
    if (g < R) {
#pragma unroll
      for (int nd = 0; nd < 8; ++nd) {
        sm.oacc[m][g][nd * 8 + 2 * t] += oc[nd][0];
        sm.oacc[m][g][nd * 8 + 2 * t + 1] += oc[nd][1];
      }
    }
#pragma unroll
    for (int nd = 0; nd < 8; ++nd) { oc[nd][0] = 0.f; oc[nd][1] = 0.f; oc[nd][2] = 0.f; oc[nd][3] = 0.f; }
    __threadfence_block();
    __syncwarp();
    if (lane == 0) *reinterpret_cast<volatile int*>(&sm.turn) = i + 1;
  };

  uint32_t phase = 0;
  for (;;) {
    int i = 0;
    if (lane == 0) i = atomicAdd(&sm.next_item, 1);
    i = __shfl_sync(0xffffffffu, i, 0);
    if (i >= n_items) break;
    const DecItem it = sm.items[i];
    if (lane == 0) load_tile(it, p.k_col);
    const int nkeys = it.nkeys;
    const int nblk = (nkeys + 15) >> 4;
    // validity words of the entity's keys (bit j of word c: key 32c + j may be attended)
    uint32_t words[7];
#pragma unroll
    for (int c = 0; c < 7; ++c) {
      const int j = c * 32 + lane;
      bool ok = j < nkeys;
      if (ok && p.key_valid != nullptr) ok = p.key_valid[(long long)it.kv_row0 + j] != 0;
      words[c] = __ballot_sync(0xffffffffu, ok);
    }
    const float inv_n = p.inv_n ? p.inv_n[(long long)(biz * R) * p.n_mod + it.mod] : 1.f;

    // ---- S = Q K^T: 16 (beams, padded) x 16 keys per block; only the first 8 rows are kept
    float s[kDecMaxKeys / 16][2][2];
    mbar_wait(&sm.bar[warp], phase);
    phase ^= 1;
#pragma unroll
    for (int kb = 0; kb < kDecMaxKeys / 16; ++kb) {
      if (kb < nblk) {
        float d0[4] = {0.f, 0.f, 0.f, 0.f}, d1[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
        for (int ks = 0; ks < 4; ++ks) {
          // four 8x8 matrices: (keys 0-7, dims lo), (keys 0-7, dims hi), (keys 8-15, dims lo), (keys 8-15, dims hi)
          const int mi = lane >> 3, r = lane & 7;
          const int key = kb * 16 + (mi >> 1) * 8 + r;
          uint32_t b[4];
          ldsm_x4(k_base + sw128(key, 2 * ks + (mi & 1)), b);
          mma_16816(d0, qa[ks][0], 0u, qa[ks][1], 0u, b[0], b[1]);
          mma_16816(d1, qa[ks][0], 0u, qa[ks][1], 0u, b[2], b[3]);
        }
        s[kb][0][0] = d0[0]; s[kb][0][1] = d0[1]; s[kb][1][0] = d1[0]; s[kb][1][1] = d1[1];
      }
    }
    // every lane has consumed the keys: the entity's values stream into the same stage while the softmax runs
    __syncwarp();
    if (lane == 0) load_tile(it, p.v_col);

    // ---- softmax over the entity's keys (row = beam g; the 4 lanes of a group share a row)
    float mx = -INFINITY;
    int n_valid = 0;
#pragma unroll
    for (int c = 0; c < 7; ++c) n_valid += __popc(words[c]);
    const bool all_valid = (n_valid == nkeys);        // warp-uniform: only the 16-key tail block can hold masked keys
#pragma unroll
    for (int kb = 0; kb < kDecMaxKeys / 16; ++kb) {
      if (kb < nblk) {
        if (!all_valid || kb == nblk - 1) {
#pragma unroll
          for (int nt = 0; nt < 2; ++nt)
#pragma unroll
            for (int j = 0; j < 2; ++j) {
              const int key = kb * 16 + nt * 8 + 2 * t + j;
              const bool ok = (words[key >> 5] >> (key & 31)) & 1u;
              s[kb][nt][j] = ok ? s[kb][nt][j] : -INFINITY;
            }
        }
        mx = fmaxf(mx, fmaxf(fmaxf(s[kb][0][0], s[kb][0][1]), fmaxf(s[kb][1][0], s[kb][1][1])));
      }
    }
    mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 1));
    mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 2));
    const float msc = (mx == -INFINITY) ? 0.f : mx * sc;
    float l = 0.f;
#pragma unroll
    for (int kb = 0; kb < kDecMaxKeys / 16; ++kb) {
      if (kb < nblk) {
#pragma unroll
        for (int nt = 0; nt < 2; ++nt)
#pragma unroll
          for (int j = 0; j < 2; ++j) {
            const float e = fast_ex2(fmaf(s[kb][nt][j], sc, -msc));     // exp2(-inf) = 0 for masked keys
            s[kb][nt][j] = e;
            l += e;
          }
      }
    }
    l += __shfl_xor_sync(0xffffffffu, l, 1);
    l += __shfl_xor_sync(0xffffffffu, l, 2);
    const float wgt = (l > 0.f) ? __fdividef(inv_n, l) : 0.f;

    // ---- O += (wgt P) V: P as A fragments straight from the score registers (rows 8..15 are zero)
    mbar_wait(&sm.bar[warp], phase);
    phase ^= 1;
#pragma unroll
    for (int kb = 0; kb < kDecMaxKeys / 16; ++kb) {
      if (kb < nblk) {
        const uint32_t a0 = pack_bf16(s[kb][0][0] * wgt, s[kb][0][1] * wgt);
        const uint32_t a2 = pack_bf16(s[kb][1][0] * wgt, s[kb][1][1] * wgt);
#pragma unroll
        for (int ndp = 0; ndp < 4; ++ndp) {
          // transposed 8x8 loads: (keys 0-7, dims 16ndp..+7), (keys 8-15, same dims), (keys 0-7, dims +8), (keys 8-15, dims +8)
          const int mi = lane >> 3, r = lane & 7;
          const int key = kb * 16 + (mi & 1) * 8 + r;
          uint32_t b[4];
          ldsm_x4_t(v_base + sw128(key, 2 * ndp + (mi >> 1)), b);
          mma_16816(oc[2 * ndp], a0, 0u, a2, 0u, b[0], b[1]);
          mma_16816(oc[2 * ndp + 1], a0, 0u, a2, 0u, b[2], b[3]);
        }
      }
    }
    __syncwarp();          // the stage may be overwritten by the next entity's keys
    add_in_order(i, it.mod);
  }
  __syncthreads();
  // ---- modality outputs: [n_mod][hypothesis][head slice] (a modality without a valid entity yields zeros)
  bf16* Og = reinterpret_cast<bf16*>(p.O);
  for (int idx = threadIdx.x; idx < p.n_mod * R * (DHD / 2); idx += blockDim.x) {
    const int m = idx / (R * (DHD / 2));
    const int rem = idx - m * (R * (DHD / 2));
    const int b = rem / (DHD / 2), d2 = rem - b * (DHD / 2);
    bf16* dst = Og + p.mods[m].o_off + (long long)(biz * R + b) * p.ldo + h * DHD + 2 * d2;
    *reinterpret_cast<uint32_t*>(dst) = pack_bf16(sm.oacc[m][b][2 * d2], sm.oacc[m][b][2 * d2 + 1]);
  }
}

// ----------------------------------------------------------------------------------------------
// causal self-attention of the newest position against the per-layer K|V cache
// ----------------------------------------------------------------------------------------------
static constexpr int kSelfMaxPos = 128;
__global__ void __launch_bounds__(128)
attn_decode_self_kernel(const bf16* __restrict__ qkv, long long ldqkv, bf16* __restrict__ cache, int* __restrict__ hist,
                        const int* __restrict__ pos_dev, bf16* __restrict__ out, long long ldo, int n_hyp, int H, float scale) {
  __shared__ float s_q[4][DHD];
  __shared__ float s_p[4][kSelfMaxPos];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int hpb = blockDim.x >> 5;
  const int n = blockIdx.x / (H / hpb), h = (blockIdx.x % (H / hpb)) * hpb + warp;
  const int D = H * DHD;
  const int tpos = pos_dev[0];
  const bf16* qrow = qkv + (long long)n * ldqkv + h * DHD;
  const bf16* knew = qrow + D;
  const bf16* vnew = qrow + 2 * D;
  // append this position's K|V to the hypothesis' own cache row and record the slot
  bf16* crow = cache + ((long long)n * kSelfMaxPos + tpos) * (2 * D) + h * DHD;
  const uint32_t kw = *reinterpret_cast<const uint32_t*>(knew + 2 * lane);
  const uint32_t vw = *reinterpret_cast<const uint32_t*>(vnew + 2 * lane);
  *reinterpret_cast<uint32_t*>(crow + 2 * lane) = kw;
  *reinterpret_cast<uint32_t*>(crow + D + 2 * lane) = vw;
  if (h == 0 && lane == 0) hist[(long long)n * kSelfMaxPos + tpos] = n;
  {
    const float2 q2 = unpack_bf16(*reinterpret_cast<const uint32_t*>(qrow + 2 * lane));
    s_q[warp][2 * lane] = q2.x; s_q[warp][2 * lane + 1] = q2.y;
  }
  __syncwarp();
  // scores: lane <-> key position (4 per lane); positions < t come from the cache row of the slot that holds them
  const float sc = scale * kDecLog2e;
  float sv[4];
  float mx = -INFINITY;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int j = lane + 32 * i;
    sv[i] = -INFINITY;
    if (j <= tpos) {
      const bf16* kr = (j == tpos) ? knew : cache + ((long long)hist[(long long)n * kSelfMaxPos + j] * kSelfMaxPos + j) * (2 * D) + h * DHD;
      float acc = 0.f;
#pragma unroll
      for (int c = 0; c < 8; ++c) {
        const uint4 u = *reinterpret_cast<const uint4*>(kr + c * 8);
        const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const float2 f = unpack_bf16(w[e]);
          acc = fmaf(f.x, s_q[warp][c * 8 + 2 * e], acc);
          acc = fmaf(f.y, s_q[warp][c * 8 + 2 * e + 1], acc);
        }
      }
      sv[i] = acc;
      mx = fmaxf(mx, acc);
    }
  }
  mx = warp_max(mx);
  float l = 0.f;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const float e = fast_ex2((sv[i] - mx) * sc);
    s_p[warp][lane + 32 * i] = e;
    l += e;
  }
  l = warp_sum(l);
  __syncwarp();
  // context: lane <-> two head dims
  float o0 = 0.f, o1 = 0.f;
  for (int j0 = 0; j0 <= tpos; j0 += 8) {
    uint32_t vv[8];
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      const int j = j0 + u;
      vv[u] = 0u;
      if (j <= tpos) {
        const bf16* vr = (j == tpos) ? vnew : cache + ((long long)hist[(long long)n * kSelfMaxPos + j] * kSelfMaxPos + j) * (2 * D) + D + h * DHD;
        vv[u] = *reinterpret_cast<const uint32_t*>(vr + 2 * lane);
      }
    }
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      const int j = j0 + u;
      if (j <= tpos) {
        const float2 f = unpack_bf16(vv[u]);
        const float pj = s_p[warp][j];
        o0 = fmaf(pj, f.x, o0); o1 = fmaf(pj, f.y, o1);
      }
    }
  }
  const float inv = 1.f / l;
  *reinterpret_cast<uint32_t*>(out + (long long)n * ldo + h * DHD + 2 * lane) = pack_bf16(o0 * inv, o1 * inv);
}

}  // namespace mmsum

using namespace mmsum;

extern "C" int mmsum_attn_decode_cross(const MmsumAttnArgs* a, void* stream_v) {
  if (!a || !a->Q || !a->KV || !a->O) return MMSUM_ERR_INVALID;
  if (a->n_qseq <= 0 || a->H <= 0 || a->R <= 0 || a->R > kDecMaxBeams || (a->n_qseq % a->R) || a->n_mod < 1 || a->n_mod > 3) return MMSUM_ERR_INVALID;
  if ((a->ldq % 2) || (a->ldkv % 8) || (a->ldo % 2) || (a->q_col % 2) || (a->k_col % 8) || (a->v_col % 8)) return MMSUM_ERR_INVALID;
  int ents = 0;
  for (int m = 0; m < a->n_mod; ++m) {
    const MmsumAttnMod& md = a->mods[m];
    if (md.E <= 0 || md.Sk <= 0 || md.Sk > kDecMaxKeys || md.loo) return MMSUM_ERR_INVALID;
    if (md.ent_stride != 0 && md.ent_stride < md.Sk) return MMSUM_ERR_INVALID;
    if (md.o_off % 2) return MMSUM_ERR_INVALID;
    ents += md.E;
  }
  if (ents > kDecMaxEnt || ents > a->E_total) return MMSUM_ERR_INVALID;
  const int n_biz = a->n_qseq / a->R;
  DecMaps mp;
  for (int m = 0; m < 3; ++m) {
    const MmsumAttnMod& md = a->mods[m < a->n_mod ? m : 0];
    const uint64_t rows = (uint64_t)md.kv_row_base + (uint64_t)n_biz * md.E * (md.ent_stride > 0 ? md.ent_stride : md.Sk);
    // box rows rounded up to the 16-key mma block: the rows past Sk are the next entity's (or zero fill), never stale smem
    if (int rc = make_tmap(&mp.kv[m], a->KV, 0, (uint64_t)a->ldkv, rows, (uint64_t)a->ldkv * 2, 64, (uint32_t)((md.Sk + 15) & ~15))) return rc;
  }
  const int smem = (int)sizeof(DecSmem) + 1024;
  static std::atomic<unsigned long long> attr{0};
  if (int rc = ensure_dyn_smem(attn_decode_cross_kernel, smem, attr)) return rc;
  attn_decode_cross_kernel<<<n_biz * a->H, kDecWarps * 32, smem, reinterpret_cast<cudaStream_t>(stream_v)>>>(mp, *a);
  MMSUM_CHECK_LAUNCH();
  return 0;
}

extern "C" int mmsum_attn_decode_self(const void* qkv, int64_t ldqkv, void* cache, int32_t* hist, const int32_t* pos_dev,
                                      void* out, int64_t ldo, int32_t n_hyp, int32_t H, float scale, void* stream_v) {
  if (!qkv || !cache || !hist || !pos_dev || !out || n_hyp <= 0 || H <= 0 || (H % 4) || (ldqkv % 8) || (ldo % 2)) return MMSUM_ERR_INVALID;
  attn_decode_self_kernel<<<n_hyp * (H / 4), 128, 0, reinterpret_cast<cudaStream_t>(stream_v)>>>(
      reinterpret_cast<const bf16*>(qkv), ldqkv, reinterpret_cast<bf16*>(cache), hist, pos_dev, reinterpret_cast<bf16*>(out), ldo,
      n_hyp, H, scale);
  MMSUM_CHECK_LAUNCH();
  return 0;
}
