// tcgen05 / TMEM / TMA multi-entity attention for sm_100a — forward, dQ backward, dK/dV backward.
//
// One family of kernels covers
//   * encoder self-attention        (modeling_multimodalsum.py:746-749, 783-853; key-pad mask)
//   * decoder causal self-attention (same call path + causal triu mask)
//   * the multi-entity, multi-modal cross-attention (:722-745, :768-869): per modality an independent softmax PER
//     ENTITY (review / table / image) and the mean over the entities that have a valid key; the leave-one-out target of
//     multimodal_train.py:150-163 is "entity i is excluded for target i".
// Self-attention is the special case "one modality, one entity, memory = own sequence".
//
// Masking semantics: pad keys of a valid entity get probability exactly 0 (the reference fills -2^16 / -inf, both
// underflow to 0 in fp32 next to any valid key); entities without a valid key are skipped (the reference zeroes them and
// removes them from the divisor); a modality without any valid entity yields 0.
//
// Shapes are the model's: 128 query positions per sequence (one UMMA M=128 tile), head_dim 64, <= 208 keys per entity,
// so a whole entity's score tile lives in TMEM (128 lanes x <=208 fp32 columns) and no online-softmax rescaling is needed.
//
// forward, one CTA per (sequence, head), 192 threads, two CTAs per SM:
//   warp 0    TMA producer: Q once, then K_e / V_e per entity into one smem stage each (128B swizzle)
//   warp 1    MMA issuer:   S_e = Q K_e^T -> TMEM;  O_e = P_e V_e -> TMEM (A operand P_e read from TMEM)
//   warps 2-5 softmax:      thread = query row; tcgen05.ld S, exp2, bf16 P back over the scores in TMEM;
//                           reads O_e back and accumulates (1/n)(1/l_e) O_e in registers; writes the modality outputs
#include <cstdlib>
#include <type_traits>
#include "common.cuh"
#include "../../include/mmsum_b200.h"

namespace mmsum {

static constexpr int SQ = 128;
static constexpr int HD = 64;
static constexpr int kMaxKeys = 208;            // per entity, multiple of 16
static constexpr int kMaxEnt = 24;
static constexpr float kLog2e = 1.4426950408889634f;
static constexpr int kKVStageBytes = kMaxKeys * 128;   // 26624 = 26 * 1024
static constexpr int kPBytes = 4 * SQ * 128;           // four 64-key atoms of [128 rows x 128 B]
static constexpr uint32_t kColS0 = 0;
struct EntItem {
  int kv_row0;     // first KV row of the entity
  int nkeys;       // keys of the entity (Sk of its modality)
  int n16;         // nkeys rounded up to 16
  short mod, ent;  // modality, global entity index
};

// 2 control warps (TMA producer, MMA issuer) + 16 softmax warps: 4 per TMEM lane quarter, each owning every 4th
// 32-column chunk of the score tile and 16 of the 64 output columns.  One warp per scheduler cannot hide the ALU /
// MUFU / TMEM latencies of the softmax (measured IPC 0.26); four can.
static constexpr int kSoftWarps = 16;
static constexpr int kSoftThreads = kSoftWarps * 32;
static constexpr int kAttnThreads = 64 + kSoftThreads;

__device__ __forceinline__ void soft_bar() { asm volatile("bar.sync 1, %0;" ::"n"(kSoftThreads) : "memory"); }

// validity word of chunk c (keys 32c .. 32c+31) of an entity, computed by one warp
__device__ __forceinline__ uint32_t chunk_word(const MmsumAttnArgs& p, const EntItem& it, int c, int lane) {
  const int j = c * 32 + lane;
  bool ok = j < it.nkeys;
  if (ok && p.key_valid != nullptr) ok = p.key_valid[(long long)it.kv_row0 + j] != 0;
  return __ballot_sync(0xffffffffu, ok);
}
// All (entity, chunk) validity words of the CTA, computed up front by warps 1..17 (one global-load latency for the whole
// CTA instead of one per entity on the critical path).  Each entity's score tile is then trimmed to its last valid key
// (n16): pad keys at the tail of a review cost neither MMA columns nor softmax work.
__device__ __forceinline__ void mask_bar() { asm volatile("bar.sync 2, %0;" ::"n"(kSoftThreads + 32) : "memory"); }
__device__ __forceinline__ void build_masks(const MmsumAttnArgs& p, EntItem* items, int n_items, uint32_t (*kmask)[8],
                                            int w, int lane) {   // w = warp - 1 in [0, 17)
  for (int idx = w; idx < n_items * 7; idx += kSoftWarps + 1) {
    const int i = idx / 7, c = idx - i * 7;
    const uint32_t wd = chunk_word(p, items[i], c, lane);
    if (lane == 0) kmask[i][c] = wd;
  }
  mask_bar();
  const int i = w * 32 + lane;
  if (i < n_items) {
    int last = 0;
#pragma unroll
    for (int c = 0; c < 7; ++c) { const uint32_t wd = kmask[i][c]; if (wd) last = c * 32 + 32 - __clz(wd); }
    const int n16 = (last + 15) & ~15;
    items[i].n16 = n16 < 16 ? 16 : n16;
  }
  mask_bar();
}
__device__ __forceinline__ uint32_t causal_word(uint32_t wd, int row, int c) {
  const int lim = row - c * 32;   // keys 32c + j <= row
  return wd & ((lim >= 31) ? 0xffffffffu : (lim < 0 ? 0u : ((2u << lim) - 1u)));
}

struct AttnMaps {
  CUtensorMap q;       // Q rows, box {64, 128}
  CUtensorMap kv[3];   // per modality: KV rows, box {64, Sk}
  CUtensorMap d_o;     // bwd: upstream gradient rows (all modalities stacked), box {64, 128}
};

#ifdef MMSUM_ATTN_TRACE
// debug-only timeline of CTA 0 (build with MMSUM_TRACE=1): g_trace[role][event index] = clock64
__device__ long long g_trace[8][512];
#define TRACE(role, idx) do { if (blockIdx.x == 0 && (idx) < 512) g_trace[role][idx] = clock64(); } while (0)
#else
#define TRACE(role, idx) do { } while (0)
#endif

// The MMA issuer is ONE thread: every ALU instruction between two tcgen05.mma issues is exposed latency (measured: the
// P V issue loop with per-step descriptor construction took ~1300 clk for 13 x 32-clk MMAs).  Descriptors are therefore
// built once per operand and advanced with a single 64-bit add of a compile-time constant.
__device__ __forceinline__ uint64_t desc_adv(uint64_t d, uint32_t bytes) { return d + (uint64_t)(bytes >> 4); }

__device__ __forceinline__ float ex2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// Enumerate the valid entities of one query sequence (executed by one full warp: lane = candidate entity).
__device__ int build_ent_items(const MmsumAttnArgs& p, int qseq, EntItem* items, int lane) {
  const int biz = qseq / p.R;
  const int tgt = qseq - biz * p.R;
  int m = 0, e = lane, found = 0;
  for (m = 0; m < p.n_mod; ++m) {
    if (e < p.mods[m].E) { found = 1; break; }
    e -= p.mods[m].E;
  }
  bool ok = false;
  EntItem it;
  it.kv_row0 = 0; it.nkeys = 0; it.n16 = 0; it.mod = 0; it.ent = 0;
  if (found) {
    const MmsumAttnMod& md = p.mods[m];
    const int ge = md.ent_base + e;
    ok = !(md.loo && e == tgt);
    if (ok && p.ent_valid != nullptr) ok = p.ent_valid[(long long)biz * p.E_total + ge] != 0;
    it.kv_row0 = (int)(md.kv_row_base + ((long long)biz * md.E + e) * (md.ent_stride > 0 ? md.ent_stride : md.Sk));
    it.nkeys = md.Sk;
    it.n16 = (md.Sk + 15) & ~15;
    it.mod = (short)m; it.ent = (short)ge;
  }
  const uint32_t bal = __ballot_sync(0xffffffffu, ok);
  if (ok) items[__popc(bal & ((1u << lane) - 1u))] = it;
  return __popc(bal);
}

// ----------------------------------------------------------------------------------------------
// forward — two INDEPENDENT CTAs per SM
//   A CTA is a single chain (4 softmax warps, thread = query row; 256 TMEM columns; one Q / K / V stage, 69 KB smem) and
//   TWO such CTAs are resident per SM, each with its own MMA warp, score buffer and output accumulator; they interfere only
//   through the shared pipes, and one CTA's set-up / tear-down overlaps the other's items.  Two softmax groups coupled in one
//   CTA would share one in-order MMA warp and ONE output accumulator: P V of item i+1 waits for the read-out of O_i, so the
//   groups ran almost serially (measured ~4.1 k clk per item against ~4.7 k for a single group).
//   TMEM columns: scores [0, 208); P (bf16) over the scores' lower half [0, 104); O at [192, 256) — it overlaps score columns
//   only of 208-wide (image) entities, and only after their exp pass has consumed them.
// ----------------------------------------------------------------------------------------------
static constexpr int kF3Threads = 64 + 4 * 32;
static constexpr uint32_t kF3ColO = 192;
struct Fwd3Smem {
  uint8_t q[SQ * 128];
  uint8_t k[kKVStageBytes];
  uint8_t v[kKVStageBytes];
  uint32_t kmask[kMaxEnt][8];
  EntItem items[kMaxEnt];
  uint64_t q_full, q_empty, k_full, k_empty, v_full, v_empty, s_full, p_full, o_full, o_free;
  uint32_t tmem_slot;
  int n_items;
};
__device__ __forceinline__ void f3_mask_bar() { asm volatile("bar.sync 2, 160;" ::: "memory"); }   // warps 1..5
__device__ __forceinline__ void f3_build_masks(const MmsumAttnArgs& p, EntItem* items, int n_items, uint32_t (*kmask)[8],
                                               int w, int lane) {   // w = warp - 1 in [0, 5)
  for (int idx = w; idx < n_items * 7; idx += 5) {
    const int i = idx / 7, c = idx - i * 7;
    const uint32_t wd = chunk_word(p, items[i], c, lane);
    if (lane == 0) kmask[i][c] = wd;
  }
  f3_mask_bar();
  const int i = w * 32 + lane;
  if (i < n_items) {
    int last = 0;
#pragma unroll
    for (int c = 0; c < 7; ++c) { const uint32_t wd = kmask[i][c]; if (wd) last = c * 32 + 32 - __clz(wd); }
    const int n16 = (last + 15) & ~15;
    items[i].n16 = n16 < 16 ? 16 : n16;
  }
  f3_mask_bar();
}

__global__ void __launch_bounds__(kF3Threads, 2)
attn_fwd_tc3_kernel(const __grid_constant__ AttnMaps maps, const MmsumAttnArgs p, const int head_mode) {
  extern __shared__ uint8_t smem_raw[];
  pdl_launch_dependents();
  pdl_wait();
  Fwd3Smem& sm = *reinterpret_cast<Fwd3Smem*>(smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u));
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // head_mode = heads per CTA (self-attention: the CTA's items are `head_mode` consecutive heads of one sequence); 0 = the
  // items are the entities of one (sequence, head)
  const int parts = head_mode ? p.H / head_mode : 1;
  const int part = head_mode ? (int)(blockIdx.x % parts) : 0;
  const int sidx = head_mode ? (int)(blockIdx.x / parts) : (int)blockIdx.x;
  const int tgt = sidx % p.R;
  const int h = head_mode ? 0 : (int)((sidx / p.R) % p.H);
  const int biz = head_mode ? (int)(sidx / p.R) : (int)(sidx / (p.R * p.H));
  const int qseq = biz * p.R + tgt;
  const int QS = p.q_rows > 0 ? p.q_rows : SQ;      // query rows of a sequence (frame stride); rows >= QS of the tile are dropped
  const int qrow0 = qseq * QS;
  auto item_head = [&](int i) { return head_mode ? part * head_mode + i : h; };

  if (warp == 0) {
    int n = build_ent_items(p, qseq, sm.items, lane);
    if (head_mode) {                       // replicate the single entity once per head
      __syncwarp();
      if (n > 0) {
        const EntItem it0 = sm.items[0];
        __syncwarp();
        if (lane < head_mode) sm.items[lane] = it0;
        n = head_mode;
      }
    }
    if (lane == 0) sm.n_items = n;
  }
  if (threadIdx.x == 32) {
    mbar_init(&sm.q_full, 1); mbar_init(&sm.q_empty, 1);
    mbar_init(&sm.k_full, 1); mbar_init(&sm.k_empty, 1);
    mbar_init(&sm.v_full, 1); mbar_init(&sm.v_empty, 1);
    mbar_init(&sm.s_full, 1); mbar_init(&sm.p_full, 128); mbar_init(&sm.o_full, 1); mbar_init(&sm.o_free, 128);
    fence_barrier_init();
    tma_prefetch_desc(&maps.q);
  }
  // V rows beyond an entity's key count are multiplied by P = 0: they must hold finite values, never stale NaN bits
  for (int i = threadIdx.x; i < kKVStageBytes / 16; i += blockDim.x)
    reinterpret_cast<uint4*>(sm.v)[i] = make_uint4(0, 0, 0, 0);
  if (warp == 1) { tmem_alloc(&sm.tmem_slot, 256); tmem_relinquish(); }
  fence_proxy_async_smem();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = sm.tmem_slot;
  const int n_items = sm.n_items;

  if (warp == 0) {
    if (lane == 0) {
      if (!head_mode) {
        mbar_expect_tx(&sm.q_full, SQ * 128);
        tma_load_2d(sm.q, &maps.q, &sm.q_full, p.q_col + h * HD, qrow0);
      }
      for (int i = 0; i < n_items; ++i) {
        if (head_mode) {
          mbar_wait(&sm.q_empty, (i & 1) ^ 1);
          mbar_expect_tx(&sm.q_full, SQ * 128);
          tma_load_2d(sm.q, &maps.q, &sm.q_full, p.q_col + item_head(i) * HD, qrow0);
        }
        mbar_wait(&sm.k_empty, (i & 1) ^ 1);
        const EntItem it = sm.items[i];
        mbar_expect_tx(&sm.k_full, it.nkeys * 128);
        tma_load_2d(sm.k, &maps.kv[it.mod], &sm.k_full, p.k_col + item_head(i) * HD, it.kv_row0);
      }
    } else if (lane == 1) {
      for (int i = 0; i < n_items; ++i) {
        mbar_wait(&sm.v_empty, (i & 1) ^ 1);
        const EntItem it = sm.items[i];
        mbar_expect_tx(&sm.v_full, it.nkeys * 128);
        tma_load_2d(sm.v, &maps.kv[it.mod], &sm.v_full, p.v_col + item_head(i) * HD, it.kv_row0);
      }
    }
  } else if (warp == 1) {
    f3_build_masks(p, sm.items, n_items, sm.kmask, 0, lane);
    if (n_items > 0) {   // whole warp runs the issue loop; elect.sync picks the issuing lane per instruction
      const uint64_t qdesc = umma_smem_desc_sw128(smem_u32(sm.q), 16, 1024);
      const uint64_t kdesc = umma_smem_desc_sw128(smem_u32(sm.k), 16, 1024);
      const uint64_t vdesc = umma_smem_desc_sw128(smem_u32(sm.v), 8192, 1024);
      if (!head_mode) mbar_wait(&sm.q_full, 0);
      auto issue_s = [&](int i) {
        const EntItem it = sm.items[i];
        if (head_mode) mbar_wait(&sm.q_full, i & 1);
        mbar_wait(&sm.k_full, i & 1);
        // the output accumulator overlaps the score columns of entities wider than 192 keys: wait for its read-out
        if (i > 0 && it.n16 > (int)kF3ColO) mbar_wait(&sm.o_free, (i - 1) & 1);
        tc_fence_after();
        const uint32_t idesc = umma_idesc_bf16(128, it.n16, 0, 0);
#pragma unroll
        for (int kk = 0; kk < 4; ++kk)
          umma_bf16_w(tmem, desc_adv(qdesc, kk * 32), desc_adv(kdesc, kk * 32), idesc, kk > 0);
        umma_commit_w(&sm.s_full);
        umma_commit_w(&sm.k_empty);
        if (head_mode) umma_commit_w(&sm.q_empty);
      };
      issue_s(0);
      const uint32_t idesc_o = umma_idesc_bf16(128, HD, 0, 1);
      for (int i = 0; i < n_items; ++i) {
        const EntItem it = sm.items[i];
        mbar_wait(&sm.v_full, i & 1);
        mbar_wait(&sm.p_full, i & 1);                        // P (bf16) now sits where the scores were
        if (i > 0) mbar_wait(&sm.o_free, (i - 1) & 1);       // the previous entity's O has been read out
        tc_fence_after();
        const int nk = it.n16 >> 4;
#pragma unroll
        for (int kk = 0; kk < kMaxKeys / 16; ++kk)
          if (kk < nk) umma_bf16_ts_w(tmem + kF3ColO, tmem + kk * 8, desc_adv(vdesc, kk * 2048), idesc_o, kk > 0);
        umma_commit_w(&sm.v_empty);
        umma_commit_w(&sm.o_full);
        if (i + 1 < n_items) issue_s(i + 1);                 // overwrites the score buffer: ordered after P V above
      }
    }
  } else {
    // ===================== softmax warps: thread = one query row =====================
    const int q4 = warp & 3;
    const int row = q4 * 32 + lane;
    const uint32_t lane_off = (uint32_t)(q4 * 32) << 16;
    const float sc = p.scale * kLog2e;
    float acc[HD];
#pragma unroll
    for (int i = 0; i < HD; ++i) acc[i] = 0.f;
    bf16* Og = reinterpret_cast<bf16*>(p.O);
    auto store_out = [&](int m, int head) {        // acc -> bf16 output row, then reset
      bf16* dst = Og + p.mods[m].o_off + (long long)(qrow0 + row) * p.ldo + head * HD;
      if (row < QS) {
#pragma unroll
        for (int j = 0; j < HD / 8; ++j) {
          uint4 u;
          u.x = pack_bf16(acc[j * 8 + 0], acc[j * 8 + 1]); u.y = pack_bf16(acc[j * 8 + 2], acc[j * 8 + 3]);
          u.z = pack_bf16(acc[j * 8 + 4], acc[j * 8 + 5]); u.w = pack_bf16(acc[j * 8 + 6], acc[j * 8 + 7]);
          *reinterpret_cast<uint4*>(dst + j * 8) = u;
        }
      }
#pragma unroll
      for (int i = 0; i < HD; ++i) acc[i] = 0.f;
    };
    int cur_mod = 0;
    f3_build_masks(p, sm.items, n_items, sm.kmask, warp - 1, lane);
    const uint32_t scol = tmem + lane_off;
    for (int i = 0; i < n_items; ++i) {
      const EntItem it = sm.items[i];
      const int head = item_head(i);
      const float inv_n = p.inv_n ? p.inv_n[(long long)qseq * p.n_mod + it.mod] : 1.f;
      if (!head_mode) { while (cur_mod < it.mod) { store_out(cur_mod, h); ++cur_mod; } }
      mbar_wait(&sm.s_full, i & 1);
      tc_fence_after();
      // ---- row max ----
      // 32-column chunks; an odd 16-column tail is handled on its own (no exp2 / TMEM traffic for columns that do not exist)
      const int nfull = it.n16 >> 5;
      const bool tail = (it.n16 & 16) != 0;
      // One pass: every 32-column chunk is read from tensor memory ONCE.  P = exp2(s*sc - ref) where ref is an integer reference
      // in the scaled log2 domain that starts at ceil(max of the first chunk) and is raised only when a later chunk exceeds it
      // by more than kSlack — then the bf16 P columns already written and the row sum are rescaled by the exact power of two
      // 2^(ref_old - ref_new).  The softmax is invariant to the reference (P keeps its relative precision in bf16, the sum is
      // fp32, the normalisation divides it out), so this equals the max-first form up to rounding; with real logits the raise
      // never triggers after the first chunk (it needs a score 22 nats above everything seen before) and costs one vote.
      constexpr float kSlack = 32.f;
      float ref = -INFINITY;
      f32x2 l2[2] = {splat2(0.f), splat2(0.f)};
      const f32x2 sc2 = splat2(sc);
      auto one_part = [&](auto ntag, int c) {
        constexpr int NC = decltype(ntag)::value;
        uint32_t wd = sm.kmask[i][c];
        if (p.causal) wd = causal_word(wd, row, c);
        constexpr uint32_t kAll = NC == 32 ? 0xffffffffu : 0xffffu;
        wd &= kAll;
        uint32_t r[NC], pk[NC / 2];
        if constexpr (NC == 32) tmem_ld_32x32(scol + c * 32, r); else tmem_ld_32x16(scol + c * 32, r);
        tmem_ld_wait();
        const bool full = __all_sync(0xffffffffu, wd == kAll);
        float mx4[4] = {-INFINITY, -INFINITY, -INFINITY, -INFINITY};
        if (full) {
#pragma unroll
          for (int j = 0; j < NC; ++j) mx4[j & 3] = fmaxf(mx4[j & 3], __uint_as_float(r[j]));
        } else {
#pragma unroll
          for (int j = 0; j < NC; ++j) mx4[j & 3] = ((wd >> j) & 1u) ? fmaxf(mx4[j & 3], __uint_as_float(r[j])) : mx4[j & 3];
        }
        const float cms = fmaxf(fmaxf(mx4[0], mx4[1]), fmaxf(mx4[2], mx4[3])) * sc;     // -inf when the row has no valid column here
        const bool raise = cms > ref + kSlack;                                           // (ref = -inf: any finite value raises)
        if (__any_sync(0xffffffffu, raise)) {
          const float nref = raise ? ceilf(cms) : ref;
          if (c > 0) {       // rescale what this row has produced so far; rows that do not raise use the factor 1
            const float f = raise ? ex2(ref - nref) : 1.f;                               // exact power of two (0 when ref = -inf)
            const f32x2 f2 = splat2(f);
            for (int cc = 0; cc < c; ++cc) {
              uint32_t q[16];
              tmem_ld_32x16(scol + cc * 16, q);
              tmem_ld_wait();
#pragma unroll
              for (int j = 0; j < 16; ++j) {
                const float2 v = unpack_bf16(q[j]);
                q[j] = pack_bf16(v.x * f, v.y * f);
              }
              tmem_st_32x16(scol + cc * 16, q);
            }
            l2[0] = mul2(l2[0], f2);
            l2[1] = mul2(l2[1], f2);
          }
          ref = nref;
        }
        const f32x2 nref2 = splat2(-ref);
        auto body = [&](auto tag) {
          constexpr bool kFull = decltype(tag)::value;
#pragma unroll
          for (int j = 0; j < NC; j += 2) {
            float a0, a1;
            unpack2(fma2(pack2(__uint_as_float(r[j]), __uint_as_float(r[j + 1])), sc2, nref2), a0, a1);
            float e0 = ex2(a0), e1 = ex2(a1);
            if constexpr (!kFull) { e0 = ((wd >> j) & 1u) ? e0 : 0.f; e1 = ((wd >> (j + 1)) & 1u) ? e1 : 0.f; }
            l2[(j >> 1) & 1] = add2(l2[(j >> 1) & 1], pack2(e0, e1));
            pk[j >> 1] = pack_bf16(e0, e1);
          }
        };
        if (full) body(std::true_type{}); else body(std::false_type{});
        // columns [16c, 16c + NC/2) lie inside score chunks this thread has consumed
        if constexpr (NC == 32) tmem_st_32x16(scol + c * 16, pk); else tmem_st_32x8(scol + c * 16, pk);
      };
#pragma unroll 1
      for (int c = 0; c < nfull; ++c) one_part(std::integral_constant<int, 32>{}, c);
      if (tail) one_part(std::integral_constant<int, 16>{}, nfull);
      const float msc = (ref == -INFINITY) ? 0.f : ref;
      tmem_st_wait();
      tc_fence_before();
      mbar_arrive(&sm.p_full);
      float l4[4];
      unpack2(l2[0], l4[0], l4[1]);
      unpack2(l2[1], l4[2], l4[3]);
      const float l = (l4[0] + l4[1]) + (l4[2] + l4[3]);
      p.LSE[(((long long)qseq * p.H + head) * p.E_total + it.ent) * SQ + row] = (l > 0.f) ? (msc + __log2f(l)) : INFINITY;
      const float wgt = (l > 0.f) ? __fdividef(inv_n, l) : 0.f;
      // ---- this entity's O = P V: fold into the register accumulators ----
      mbar_wait(&sm.o_full, i & 1);
      tc_fence_after();
#pragma unroll
      for (int hh = 0; hh < 2; ++hh) {
        uint32_t r[32];
        tmem_ld_32x32(tmem + lane_off + kF3ColO + hh * 32, r);
        tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < 32; ++j) acc[hh * 32 + j] = fmaf(wgt, __uint_as_float(r[j]), acc[hh * 32 + j]);
      }
      tc_fence_before();
      mbar_arrive(&sm.o_free);
      if (head_mode) store_out(0, head);
    }
    if (head_mode) {
      if (n_items == 0) for (int hh = 0; hh < head_mode; ++hh) store_out(0, item_head(hh));   // null entity: zero rows
    } else {
      while (cur_mod < p.n_mod) { store_out(cur_mod, h); ++cur_mod; }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) { __syncwarp(); tc_fence_after(); tmem_dealloc(tmem, 256); }
}

// ----------------------------------------------------------------------------------------------
// backward, part 1 — one CTA per (sequence, head): dQ and DELTA
//   per entity:  S = Q K^T and dP' = dA V^T into TMEM;  P = exp2(sc*S - LSE) (kept in registers as bf16),
//   delta' = rowsum(P o dP');  dS = scale*inv_n * P o (dP' - delta') -> bf16 smem;  dQ += dS K  (TMEM, all entities)
// ----------------------------------------------------------------------------------------------
static constexpr uint32_t kColDP = 224, kColDQ = 448;

struct BwdQSmem {
  uint8_t q[SQ * 128];
  uint8_t da[SQ * 128];
  uint8_t k[2][kKVStageBytes];
  uint8_t v[2][kKVStageBytes];
  uint8_t ds[kPBytes];
  float red_delta[2][4][SQ];
  uint32_t kmask[kMaxEnt][8];
  EntItem items[kMaxEnt];
  uint64_t q_full, da_full, da_free, qd_full[2], qd_empty[2], k_full[2], k_empty[2], v_full[2], v_empty[2], sdp_full, s_empty, dp_empty, ds_full, ds_free;
  uint32_t tmem_slot;
  int n_items;
};

__global__ void __launch_bounds__(kAttnThreads, 1)
attn_bwd_dq_tc_kernel(const __grid_constant__ AttnMaps maps, const MmsumAttnArgs p, const int head_mode) {
  extern __shared__ uint8_t smem_raw[];
  pdl_launch_dependents();
  pdl_wait();   // launched with programmatic stream serialization: nothing global is touched before this point
  // align inside the shared window with pointer arithmetic on the __shared__ array so the compiler keeps the
  // shared address space (LDS/STS instead of generic LD/ST)
  BwdQSmem& sm = *reinterpret_cast<BwdQSmem*>(smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u));
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // head mode (self-attention, <= 128 keys): the CTA owns a whole sequence and its items are the H heads, so the per-CTA
  // set-up and the load / MMA / softmax latencies are amortised over the heads; each item then has its own Q / dA tiles
  // (2-deep ring: stage 1 lives in the unused upper half of the dS region) and its own dQ, read out of TMEM one item later.
  const int tgt = blockIdx.x % p.R;
  const int h = head_mode ? 0 : (int)((blockIdx.x / p.R) % p.H);
  const int biz = head_mode ? (int)(blockIdx.x / p.R) : (int)(blockIdx.x / (p.R * p.H));
  const int qseq = biz * p.R + tgt;
  const int QS = p.q_rows > 0 ? p.q_rows : SQ;      // query rows of a sequence (frame stride); rows >= QS of the tile are dropped
  const int qrow0 = qseq * QS;
  auto item_head = [&](int i) { return head_mode ? i : h; };
  uint8_t* const q_stage1 = sm.ds + 2 * SQ * 128;
  uint8_t* const da_stage1 = sm.ds + 3 * SQ * 128;

  if (warp == 0) {
    int n = build_ent_items(p, qseq, sm.items, lane);
    if (head_mode) {                       // replicate the single entity once per head
      __syncwarp();
      if (n > 0) {
        const EntItem it0 = sm.items[0];
        __syncwarp();
        if (lane < p.H) sm.items[lane] = it0;
        n = p.H;
      }
    }
    if (lane == 0) sm.n_items = n;
  }
  if (threadIdx.x == 32) {
    mbar_init(&sm.q_full, 1); mbar_init(&sm.da_full, 1); mbar_init(&sm.da_free, 1);
    for (int s = 0; s < 2; ++s) { mbar_init(&sm.qd_full[s], 1); mbar_init(&sm.qd_empty[s], 1); }
    for (int s = 0; s < 2; ++s) {
      mbar_init(&sm.k_full[s], 1); mbar_init(&sm.k_empty[s], 1);
      mbar_init(&sm.v_full[s], 1); mbar_init(&sm.v_empty[s], 1);
    }
    mbar_init(&sm.sdp_full, 1); mbar_init(&sm.s_empty, kSoftThreads); mbar_init(&sm.dp_empty, kSoftThreads);
    mbar_init(&sm.ds_full, kSoftThreads); mbar_init(&sm.ds_free, 1);
    fence_barrier_init();
  }
  for (int i = threadIdx.x; i < 4 * kKVStageBytes / 16; i += blockDim.x)   // K and V stages: finite contents only
    reinterpret_cast<uint4*>(sm.k[0])[i] = make_uint4(0, 0, 0, 0);
  if (warp == 1) { tmem_alloc(&sm.tmem_slot, 512); tmem_relinquish(); }
  fence_proxy_async_smem();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = sm.tmem_slot;
  const int n_items = sm.n_items;

  if (warp == 0) {
    if (lane == 0) {
      if (!head_mode) {
        mbar_expect_tx(&sm.q_full, SQ * 128);
        tma_load_2d(sm.q, &maps.q, &sm.q_full, p.q_col + h * HD, qrow0);
      }
      int cur_mod = -1, n_da = 0;
      for (int i = 0; i < n_items; ++i) {
        const int st = i & 1;
        const EntItem it = sm.items[i];
        if (head_mode) {                   // this head's Q and dA tiles
          mbar_wait(&sm.qd_empty[st], ((i >> 1) & 1) ^ 1);
          mbar_expect_tx(&sm.qd_full[st], 2 * SQ * 128);
          tma_load_2d(st ? q_stage1 : sm.q, &maps.q, &sm.qd_full[st], p.q_col + i * HD, qrow0);
          tma_load_2d(st ? da_stage1 : sm.da, &maps.d_o, &sm.qd_full[st], i * HD, (int)(p.mods[it.mod].o_off / p.ldo) + qrow0);
        } else if (it.mod != cur_mod) {
          mbar_wait(&sm.da_free, (n_da & 1) ^ 1);      // previous modality's dP MMAs have retired
          mbar_expect_tx(&sm.da_full, SQ * 128);
          tma_load_2d(sm.da, &maps.d_o, &sm.da_full, h * HD, (int)(p.mods[it.mod].o_off / p.ldo) + qrow0);
          cur_mod = it.mod; ++n_da;
        }
        // V is only read by dP' = dA V^T (released early); K also feeds dQ += dS K (released late): two rings
        mbar_wait(&sm.v_empty[st], ((i >> 1) & 1) ^ 1);
        mbar_expect_tx(&sm.v_full[st], it.nkeys * 128);
        tma_load_2d(sm.v[st], &maps.kv[it.mod], &sm.v_full[st], p.v_col + item_head(i) * HD, it.kv_row0);
      }
    } else if (lane == 1) {
      for (int i = 0; i < n_items; ++i) {
        const int st = i & 1;
        const EntItem it = sm.items[i];
        mbar_wait(&sm.k_empty[st], ((i >> 1) & 1) ^ 1);
        mbar_expect_tx(&sm.k_full[st], it.nkeys * 128);
        tma_load_2d(sm.k[st], &maps.kv[it.mod], &sm.k_full[st], p.k_col + item_head(i) * HD, it.kv_row0);
      }
    }
  } else if (warp == 1) {
    build_masks(p, sm.items, n_items, sm.kmask, 0, lane);
    if (n_items > 0) {   // whole warp runs the issue loop; elect.sync picks the issuing lane per instruction
      const uint64_t qdesc0 = umma_smem_desc_sw128(smem_u32(sm.q), 16, 1024), dadesc0 = umma_smem_desc_sw128(smem_u32(sm.da), 16, 1024);
      const uint64_t qdesc1 = umma_smem_desc_sw128(smem_u32(q_stage1), 16, 1024), dadesc1 = umma_smem_desc_sw128(smem_u32(da_stage1), 16, 1024);
      const uint64_t dsdesc = umma_smem_desc_sw128(smem_u32(sm.ds), 16, 1024);
      const uint64_t kdesc_k[2] = {umma_smem_desc_sw128(smem_u32(sm.k[0]), 16, 1024), umma_smem_desc_sw128(smem_u32(sm.k[1]), 16, 1024)};
      const uint64_t kdesc_mn[2] = {umma_smem_desc_sw128(smem_u32(sm.k[0]), 8192, 1024), umma_smem_desc_sw128(smem_u32(sm.k[1]), 8192, 1024)};
      const uint64_t vdesc_k[2] = {umma_smem_desc_sw128(smem_u32(sm.v[0]), 16, 1024), umma_smem_desc_sw128(smem_u32(sm.v[1]), 16, 1024)};
      if (!head_mode) mbar_wait(&sm.q_full, 0);
      int cur_mod = -1, n_da = 0;
      auto issue_sdp = [&](int i) {
        const int st = i & 1;
        const EntItem it = sm.items[i];
        const uint64_t qdesc = (head_mode && st) ? qdesc1 : qdesc0, dadesc = (head_mode && st) ? dadesc1 : dadesc0;
        if (head_mode) {
          mbar_wait(&sm.qd_full[st], (i >> 1) & 1);
        } else if (it.mod != cur_mod) { mbar_wait(&sm.da_full, n_da & 1); cur_mod = it.mod; ++n_da; }
        mbar_wait(&sm.k_full[st], (i >> 1) & 1);
        // the S columns are handed back after pass 1 of the previous entity, the dP' columns once pass 2 has
        // re-read them: both products of entity i+1 overlap the softmax work of entity i
        mbar_wait(&sm.s_empty, (i & 1) ^ 1);
        tc_fence_after();
        const uint32_t idesc = umma_idesc_bf16(128, it.n16, 0, 0);
        const uint64_t kd = st ? kdesc_k[1] : kdesc_k[0], vd = st ? vdesc_k[1] : vdesc_k[0];
#pragma unroll
        for (int kk = 0; kk < 4; ++kk)
          umma_bf16_w(tmem + kColS0, desc_adv(qdesc, kk * 32), desc_adv(kd, kk * 32), idesc, kk > 0);
        mbar_wait(&sm.v_full[st], (i >> 1) & 1);
        mbar_wait(&sm.dp_empty, (i & 1) ^ 1);
        tc_fence_after();
#pragma unroll
        for (int kk = 0; kk < 4; ++kk)
          umma_bf16_w(tmem + kColDP, desc_adv(dadesc, kk * 32), desc_adv(vd, kk * 32), idesc, kk > 0);
        umma_commit_w(&sm.sdp_full);
        umma_commit_w(&sm.v_empty[st]);
        // last item of its modality: the dA tile may be replaced once these MMAs retire
        if (head_mode) umma_commit_w(&sm.qd_empty[st]);
        else if (i + 1 >= n_items || sm.items[i + 1].mod != it.mod) umma_commit_w(&sm.da_free);
      };
      issue_sdp(0);
      const uint32_t idesc_q = umma_idesc_bf16(128, HD, 0, 1);
      for (int i = 0; i < n_items; ++i) {
        if (i + 1 < n_items) issue_sdp(i + 1);
        const int st = i & 1;
        const EntItem it = sm.items[i];
        if (lane == 0) TRACE(1, 3 * i);
        mbar_wait(&sm.ds_full, i & 1);
        if (lane == 0) TRACE(1, 3 * i + 1);
        tc_fence_after();
        const uint64_t kd = st ? kdesc_mn[1] : kdesc_mn[0];
        const int nk = it.n16 >> 4;
#pragma unroll
        for (int kk = 0; kk < kMaxKeys / 16; ++kk)
          if (kk < nk)
            umma_bf16_w(tmem + kColDQ, desc_adv(dsdesc, (kk >> 2) * (SQ * 128) + (kk & 3) * 32), desc_adv(kd, kk * 2048), idesc_q,
                      ((i > 0 && !head_mode) || kk > 0) ? 1u : 0u);
        if (lane == 0) TRACE(1, 3 * i + 2);
        umma_commit_w(&sm.k_empty[st]);
        umma_commit_w(&sm.ds_free);
      }
    }
  } else {
    // thread = (query row, column group cg): score chunks cg and cg+4, dQ columns [16cg, 16cg+16)
    const int q4 = warp & 3;
    const int cg = (warp - 2) >> 2;
    const int row = q4 * 32 + lane;
    const uint32_t lane_off = (uint32_t)(q4 * 32) << 16;
    const float sc = p.scale * kLog2e;
    build_masks(p, sm.items, n_items, sm.kmask, warp - 1, lane);
    // dQ columns [16cg, 16cg+16) of this row out of TMEM (caller has waited for the dQ MMAs) -> global, for one head
    auto store_dq = [&](int head) {
      bf16* dQg = reinterpret_cast<bf16*>(p.dQ) + (long long)(qrow0 + row) * p.lddq + p.dq_col + head * HD + cg * 16;
      uint32_t r[16];
      tmem_ld_32x16(tmem + lane_off + kColDQ + cg * 16, r);
      tmem_ld_wait();
      if (row >= QS) return;
#pragma unroll
      for (int j = 0; j < 2; ++j) {
        uint4 u;
        u.x = pack_bf16(__uint_as_float(r[j * 8 + 0]), __uint_as_float(r[j * 8 + 1]));
        u.y = pack_bf16(__uint_as_float(r[j * 8 + 2]), __uint_as_float(r[j * 8 + 3]));
        u.z = pack_bf16(__uint_as_float(r[j * 8 + 4]), __uint_as_float(r[j * 8 + 5]));
        u.w = pack_bf16(__uint_as_float(r[j * 8 + 6]), __uint_as_float(r[j * 8 + 7]));
        *reinterpret_cast<uint4*>(dQg + j * 8) = u;
      }
    };
    // LSE / 1/n of an item are fetched one item ahead: as plain loads at the top of the item their global latency (~500 clk)
    // would sit in front of pass 1 of every item
    auto lse_index = [&](int i) { return (((long long)qseq * p.H + item_head(i)) * p.E_total + sm.items[i].ent) * SQ + row; };
    float lse_nx = 0.f, invn_nx = 1.f;
    if (n_items > 0) {
      lse_nx = p.LSE[lse_index(0)];
      if (p.inv_n) invn_nx = p.inv_n[(long long)qseq * p.n_mod + sm.items[0].mod];
    }
    for (int i = 0; i < n_items; ++i) {
      const EntItem it = sm.items[i];
      const int par = i & 1;
      const int nchunk = (it.n16 + 31) >> 5;
      const bool has[2] = {cg < nchunk, cg + 4 < nchunk};
      uint32_t wd[2];
      wd[0] = has[0] ? sm.kmask[i][cg] : 0u;
      wd[1] = has[1] ? sm.kmask[i][cg + 4] : 0u;
      if (p.causal) { wd[0] = causal_word(wd[0], row, cg); wd[1] = causal_word(wd[1], row, cg + 4); }
      const long long li = lse_index(i);
      const float lse = lse_nx;
      const float inv_n = invn_nx;
      if (i + 1 < n_items) {
        lse_nx = p.LSE[lse_index(i + 1)];
        if (p.inv_n) invn_nx = p.inv_n[(long long)qseq * p.n_mod + sm.items[i + 1].mod];
      }
      if (threadIdx.x == 64) TRACE(3, 5 * i);
      mbar_wait(&sm.sdp_full, i & 1);
      if (threadIdx.x == 64) TRACE(3, 5 * i + 1);
      tc_fence_after();
      // pass 1: P = exp2(sc*S - LSE) (stashed as packed bf16), partial delta' = sum P o dP'
      // pass 2: dS = scale*inv_n * P o (dP' - delta') -> bf16 A-operand tile
      // The S columns go back to the MMA warp after pass 1, the dP' columns as soon as pass 2 has them in registers
      // (entities of <= 4 chunks keep dP' in registers across the delta exchange and release both after pass 1), so
      // the next entity's Q K^T / dA V^T overlap this entity's softmax work.
      const float wgt = p.scale * inv_n;
      float dl4[4] = {0.f, 0.f, 0.f, 0.f};
      // half = 16 score columns: bits [16*half, +16) of the chunk's mask word, packed P words [8*half, +8)
      auto pass1 = [&](const uint32_t w16, const uint32_t (&rs)[16], const uint32_t (&rd)[16], uint32_t (&pk)[8]) {
        // two copies of the loop (warp-uniform choice): predicated-off mask code would still take issue slots
        auto body = [&](auto tag) {
          constexpr bool kFull = decltype(tag)::value;
#pragma unroll
          for (int j = 0; j < 16; j += 2) {
            // scalar FFMA: at this kernel's 96-register cap the pack / unpack moves of packed fp32 pairs cost more than the
            // halved FFMA count saves
            float p0 = ex2(fmaf(__uint_as_float(rs[j]), sc, -lse));
            float p1 = ex2(fmaf(__uint_as_float(rs[j + 1]), sc, -lse));
            float d0 = __uint_as_float(rd[j]), d1 = __uint_as_float(rd[j + 1]);
            // masked columns: the score tile's columns beyond n16 were never written by this entity's MMAs (stale tensor
            // memory, possibly NaN patterns), so both factors are SELECTED to zero — 0 * stale is not 0
            if constexpr (!kFull) {
              const bool b0 = (w16 >> j) & 1u, b1 = (w16 >> (j + 1)) & 1u;
              p0 = b0 ? p0 : 0.f; p1 = b1 ? p1 : 0.f;
              d0 = b0 ? d0 : 0.f; d1 = b1 ? d1 : 0.f;
            }
            dl4[(j >> 1) & 3] = fmaf(p0, d0, dl4[(j >> 1) & 3]);
            dl4[(j >> 1) & 3] = fmaf(p1, d1, dl4[(j >> 1) & 3]);
            pk[j >> 1] = pack_bf16(p0, p1);
          }
        };
        if (__all_sync(0xffffffffu, w16 == 0xffffu)) body(std::true_type{}); else body(std::false_type{});
      };
      auto exchange_delta = [&]() {
        sm.red_delta[par][cg][row] = (dl4[0] + dl4[1]) + (dl4[2] + dl4[3]);
        if (threadIdx.x == 64) TRACE(3, 5 * i + 2);
        soft_bar();
        if (threadIdx.x == 64) TRACE(3, 5 * i + 3);
        const float delta = (sm.red_delta[par][0][row] + sm.red_delta[par][1][row]) +
                            (sm.red_delta[par][2][row] + sm.red_delta[par][3][row]);
        if (cg == 0) p.DELTA[li] = delta;
        return delta * wgt;            // dS = P * (wgt*dP' - wgt*delta')
      };
      auto pass2 = [&](const int c, const int half, const float dw, const uint32_t (&rd)[16], const uint32_t (&pk)[8]) {
        uint8_t* atom = sm.ds + row * 128 + (c >> 1) * (SQ * 128);
#pragma unroll
        for (int g8 = 0; g8 < 2; ++g8) {
          uint32_t o[4];
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const float2 pr = unpack_bf16(pk[g8 * 4 + e]);
            const int j = g8 * 8 + 2 * e;
            o[e] = pack_bf16(pr.x * fmaf(__uint_as_float(rd[j]), wgt, -dw), pr.y * fmaf(__uint_as_float(rd[j + 1]), wgt, -dw));
          }
          const int chunk = (c & 1) * 4 + half * 2 + g8;
          *reinterpret_cast<uint4*>(atom + ((chunk ^ (row & 7)) << 4)) = make_uint4(o[0], o[1], o[2], o[3]);
        }
      };
      // 16-column halves beyond the entity's n16 (the tail of the last chunk when n16 % 32 == 16): the dQ product never reads
      // them, so they are neither loaded nor computed nor stored
      const bool live[2][2] = {{cg * 32 < it.n16, cg * 32 + 16 < it.n16}, {(cg + 4) * 32 < it.n16, (cg + 4) * 32 + 16 < it.n16}};
      if (nchunk <= 4) {
        uint32_t pk[2][8] = {}, rda[16] = {}, rdb[16] = {};
        if (live[0][0]) {
          uint32_t rs[16];
          tmem_ld_32x16(tmem + lane_off + kColS0 + cg * 32, rs);
          tmem_ld_32x16(tmem + lane_off + kColDP + cg * 32, rda);
          tmem_ld_wait();
          pass1(wd[0] & 0xffffu, rs, rda, pk[0]);
        }
        if (live[0][1]) {
          uint32_t rs[16];
          tmem_ld_32x16(tmem + lane_off + kColS0 + cg * 32 + 16, rs);
          tmem_ld_32x16(tmem + lane_off + kColDP + cg * 32 + 16, rdb);
          tmem_ld_wait();
          pass1(wd[0] >> 16, rs, rdb, pk[1]);
        }
        tc_fence_before();
        mbar_arrive(&sm.s_empty);
        mbar_arrive(&sm.dp_empty);
        const float dw = exchange_delta();
        if (i > 0) {                                       // dQ MMA of the previous entity has consumed the dS tile
          mbar_wait(&sm.ds_free, (i - 1) & 1);
          if (head_mode) { tc_fence_after(); store_dq(i - 1); tc_fence_before(); }   // ... and the previous head's dQ is final
        }
        if (live[0][0]) pass2(cg, 0, dw, rda, pk[0]);
        if (live[0][1]) pass2(cg, 1, dw, rdb, pk[1]);
      } else {
        uint32_t pk[4][8] = {};
#pragma unroll
        for (int t = 0; t < 2; ++t) {
          if (has[t]) {
#pragma unroll
            for (int half = 0; half < 2; ++half) {
              if (live[t][half]) {
                uint32_t rs[16], rd[16];
                tmem_ld_32x16(tmem + lane_off + kColS0 + (cg + 4 * t) * 32 + half * 16, rs);
                tmem_ld_32x16(tmem + lane_off + kColDP + (cg + 4 * t) * 32 + half * 16, rd);
                tmem_ld_wait();
                pass1((wd[t] >> (16 * half)) & 0xffffu, rs, rd, pk[t * 2 + half]);
              }
            }
          }
        }
        tc_fence_before();
        mbar_arrive(&sm.s_empty);
        const float dw = exchange_delta();
        if (i > 0) {
          mbar_wait(&sm.ds_free, (i - 1) & 1);
          if (head_mode) { tc_fence_after(); store_dq(i - 1); tc_fence_before(); }
        }
        {
          uint32_t r0[16] = {}, r1[16] = {};
          if (live[0][0]) tmem_ld_32x16(tmem + lane_off + kColDP + cg * 32, r0);
          if (live[0][1]) tmem_ld_32x16(tmem + lane_off + kColDP + cg * 32 + 16, r1);
          tmem_ld_wait();
          if (!has[1]) { tc_fence_before(); mbar_arrive(&sm.dp_empty); }
          if (live[0][0]) pass2(cg, 0, dw, r0, pk[0]);
          if (live[0][1]) pass2(cg, 1, dw, r1, pk[1]);
        }
        if (has[1]) {
          uint32_t r0[16] = {}, r1[16] = {};
          if (live[1][0]) tmem_ld_32x16(tmem + lane_off + kColDP + (cg + 4) * 32, r0);
          if (live[1][1]) tmem_ld_32x16(tmem + lane_off + kColDP + (cg + 4) * 32 + 16, r1);
          tmem_ld_wait();
          tc_fence_before();
          mbar_arrive(&sm.dp_empty);
          if (live[1][0]) pass2(cg + 4, 0, dw, r0, pk[2]);
          if (live[1][1]) pass2(cg + 4, 1, dw, r1, pk[3]);
        }
      }
      if (threadIdx.x == 64) TRACE(3, 5 * i + 4);
      fence_proxy_async_smem();
      mbar_arrive(&sm.ds_full);
    }
    // dQ: read the accumulator once every entity has been folded in (head mode: the last head's)
    if (n_items > 0) {
      mbar_wait(&sm.ds_free, (n_items - 1) & 1);
      tc_fence_after();
      store_dq(head_mode ? n_items - 1 : h);
    } else {
      for (int hh = head_mode ? 0 : h; hh < (head_mode ? p.H : h + 1); ++hh) {
        bf16* dQg = reinterpret_cast<bf16*>(p.dQ) + (long long)(qrow0 + row) * p.lddq + p.dq_col + hh * HD + cg * 16;
        if (row < QS) {
          *reinterpret_cast<uint4*>(dQg) = make_uint4(0, 0, 0, 0);
          *reinterpret_cast<uint4*>(dQg + 8) = make_uint4(0, 0, 0, 0);
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) { __syncwarp(); tc_fence_after(); tmem_dealloc(tmem, 512); }
}

// ----------------------------------------------------------------------------------------------
// backward, part 2 — one CTA per (business, head, entity tile of <=128 keys): dK, dV summed over the consumer targets
//   per target:  S^T = K Q^T and dP'^T = V dA^T into TMEM (keys on the lanes);
//   Pn^T = inv_n * exp2(sc*S^T - LSE[q]);  dS^T = scale * Pn^T o (dP'^T - delta'[q]);  both -> bf16 over their own TMEM columns;
//   dV += Pn^T dA,  dK += dS^T Q  (TMEM accumulators over all targets)
// ----------------------------------------------------------------------------------------------
// Two CTAs share an SM (256 TMEM columns, ~100 KB smem, 320 threads each): one CTA's softmax phase overlaps the other's
// MMA / staging phases, which a single lock-stepped CTA cannot do.  A step is one (consumer target, 64-query half).
static constexpr int QH = 64;                       // queries per step
static constexpr int kKvSoftWarps = 8;
static constexpr int kKvSoftThreads = kKvSoftWarps * 32;
static constexpr int kKvThreads = 64 + kKvSoftThreads;
__device__ __forceinline__ void kv_soft_bar() { asm volatile("bar.sync 1, %0;" ::"n"(kKvSoftThreads) : "memory"); }

// Key tiling of a modality for the dK/dV kernel.  Entities whose key count is not a multiple of 128 (196-key images) are
// tiled as ONE contiguous key range per business (tiles may straddle two entities; every row carries its own entity), so
// 10 x 196 keys cost 16 tiles instead of 20 half-empty ones.  Needs contiguous entities, no leave-one-out, Sk >= 128.
__host__ __device__ inline bool mod_packed(const MmsumAttnMod& md) {
  return md.E > 1 && !md.loo && (md.ent_stride == 0 || md.ent_stride == md.Sk) && md.Sk >= SQ && (md.Sk % SQ) != 0;
}
__host__ __device__ inline int mod_tiles(const MmsumAttnMod& md) {
  return mod_packed(md) ? (md.E * md.Sk + SQ - 1) / SQ : md.E * ((md.Sk + SQ - 1) / SQ);
}
// key tiles of the dK/dV pass: none for a modality whose dK/dV is not wanted (its dKV rows are left as they are)
__host__ __device__ inline int dkv_tiles(const MmsumAttnMod& md) { return md.no_dkv ? 0 : mod_tiles(md); }

static constexpr int kKvStages = 4;                 // Q / dA ring depth (P^T / dS^T stay in TMEM, so smem has room for four)
struct BwdKVSmem {
  uint8_t k[SQ * 128];
  uint8_t v[SQ * 128];
  uint8_t q[kKvStages][QH * 128];      // Q / dA rows of the step's 64 queries (ring)
  uint8_t da[kKvStages][QH * 128];
  float lse[2][2][QH];         // raw LSE / DELTA rows of the current and the next step (cp.async staged), for the (up to)
  float dlt[2][2][QH];         // two entities a packed tile straddles
  float lg_invn[32];           // log2(1/n) of every target for this modality
  uint64_t kv_full, kv_free, qd_full[kKvStages], qd_empty[kKvStages], sdp_full, pds_full, pds_free;
  uint32_t tmem_slot;
};
static constexpr uint32_t kColST = 0, kColDPT = 64, kColDK = 128, kColDV = 192;

__global__ void __launch_bounds__(kKvThreads, 2)
attn_bwd_dkv_tc_kernel(const __grid_constant__ CUtensorMap q64, const __grid_constant__ CUtensorMap do64,
                       const __grid_constant__ CUtensorMap kv128, const MmsumAttnArgs p, int tiles_per_bh,
                       const int head_mode) {
  extern __shared__ uint8_t smem_raw[];
  pdl_launch_dependents();
  pdl_wait();   // launched with programmatic stream serialization: nothing global is touched before this point
  // align inside the shared window with pointer arithmetic on the __shared__ array so the compiler keeps the
  // shared address space (LDS/STS instead of generic LD/ST)
  BwdKVSmem& sm = *reinterpret_cast<BwdKVSmem*>(smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u));
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int QS = p.q_rows > 0 ? p.q_rows : SQ;      // query rows of a sequence (frame stride); queries >= QS are masked
  int rem = blockIdx.x % tiles_per_bh;
  const int bh = blockIdx.x / tiles_per_bh;
  // head mode (self-attention): the CTA owns one (sequence, key tile) and walks a group of heads, so the set-up is paid once
  // and every mbarrier simply keeps counting steps across heads (g = head index * n_steps + step)
  // head_mode = heads per CTA (1 = one head per CTA)
  const int hgroups = p.H / head_mode;
  const int biz = bh / hgroups;
  const int h_begin = (bh % hgroups) * head_mode, h_end = h_begin + head_mode;
  int m = 0;
  for (m = 0; m < p.n_mod; ++m) {
    const int cnt = dkv_tiles(p.mods[m]);
    if (rem < cnt) break;
    rem -= cnt;
  }
  const MmsumAttnMod& md = p.mods[m];
  const bool packed = mod_packed(md);
  int e, key0, nkeys, kvrow0;
  if (packed) {            // tile `rem` of the business' contiguous key range; rows belong to entity e or e + 1
    const int gk0 = rem * SQ;
    e = gk0 / md.Sk;
    key0 = gk0 - e * md.Sk;
    nkeys = min(SQ, md.E * md.Sk - gk0);
    kvrow0 = (int)(md.kv_row_base + (long long)biz * md.E * md.Sk) + gk0;
  } else {
    const int nt = (md.Sk + SQ - 1) / SQ;
    e = rem / nt;
    key0 = (rem % nt) * SQ;
    nkeys = min(SQ, md.Sk - key0);
    kvrow0 = (int)(md.kv_row_base + ((long long)biz * md.E + e) * (md.ent_stride > 0 ? md.ent_stride : md.Sk)) + key0;
  }
  const int e_hi = min(e + 1, md.E - 1);                       // second entity of a packed tile (== e when there is none)
  auto ent_valid_at = [&](int ee) { return (p.ent_valid == nullptr) || (p.ent_valid[(long long)biz * p.E_total + md.ent_base + ee] != 0); };
  const bool ok_lo = ent_valid_at(e), ok_hi = packed && (key0 + SQ > md.Sk) && (e + 1 < md.E) && ent_valid_at(e + 1);
  const bool ent_ok = ok_lo || ok_hi;
  bf16* dKV = reinterpret_cast<bf16*>(p.dKV);

  // consumer targets of this entity (leave-one-out excludes target e); two 64-query steps per target
  int n_tgt = 0;
  for (int tg = 0; tg < p.R; ++tg) n_tgt += (md.loo && tg == e) ? 0 : 1;
  const int n_steps = 2 * n_tgt;
  if (!ent_ok || n_steps == 0) {
    // null entity: its gradient is exactly zero (the buffer is never memset)
    if (warp >= 2) {
      const int row = (warp & 3) * 32 + lane;
      const int cg = (warp - 2) >> 2;
      if (row < nkeys) {
        for (int h = h_begin; h < h_end; ++h) {
          bf16* dk = dKV + (long long)(kvrow0 + row) * p.lddkv + p.dk_col + h * HD + cg * 32;
          bf16* dv = dKV + (long long)(kvrow0 + row) * p.lddkv + p.dv_col + h * HD + cg * 32;
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            *reinterpret_cast<uint4*>(dk + j * 8) = make_uint4(0, 0, 0, 0);
            *reinterpret_cast<uint4*>(dv + j * 8) = make_uint4(0, 0, 0, 0);
          }
        }
      }
    }
    return;
  }

  if (threadIdx.x == 0) {
    mbar_init(&sm.kv_full, 1); mbar_init(&sm.kv_free, 1);
    for (int s = 0; s < kKvStages; ++s) { mbar_init(&sm.qd_full[s], 1); mbar_init(&sm.qd_empty[s], 1); }
    mbar_init(&sm.sdp_full, 1);
    mbar_init(&sm.pds_full, kKvSoftThreads); mbar_init(&sm.pds_free, 1);
    fence_barrier_init();
  }
  if (warp == 1) { tmem_alloc(&sm.tmem_slot, 256); tmem_relinquish(); }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = sm.tmem_slot;
  auto step_target = [&](int s) {   // step -> target index of its 64-query half
    int tg = s >> 1;
    if (md.loo && tg >= e) ++tg;
    return tg;
  };

  if (warp == 0) {
    if (lane == 0) {
      for (int h = h_begin; h < h_end; ++h) {
        const int g0 = (h - h_begin) * n_steps;
        // the K / V tiles are read by the S^T / dP^T products only: the previous head's last pair has retired
        if (h > h_begin) mbar_wait(&sm.kv_free, (h - h_begin - 1) & 1);
        mbar_expect_tx(&sm.kv_full, 2 * SQ * 128);
        tma_load_2d(sm.k, &kv128, &sm.kv_full, p.k_col + h * HD, kvrow0);
        tma_load_2d(sm.v, &kv128, &sm.kv_full, p.v_col + h * HD, kvrow0);
        for (int s = 0; s < n_steps; ++s) {
          const int g = g0 + s, st = g % kKvStages;
          const int qrow0 = (biz * p.R + step_target(s)) * QS + (s & 1) * QH;
          mbar_wait(&sm.qd_empty[st], ((g / kKvStages) & 1) ^ 1);
          mbar_expect_tx(&sm.qd_full[st], 2 * QH * 128);
          tma_load_2d(sm.q[st], &q64, &sm.qd_full[st], p.q_col + h * HD, qrow0);
          tma_load_2d(sm.da[st], &do64, &sm.qd_full[st], h * HD, (int)(md.o_off / p.ldo) + qrow0);
        }
      }
    }
  } else if (warp == 1) {
    {   // whole warp runs the issue loop; elect.sync picks the issuing lane per instruction
      const uint64_t kdesc = umma_smem_desc_sw128(smem_u32(sm.k), 16, 1024), vdesc = umma_smem_desc_sw128(smem_u32(sm.v), 16, 1024);
      // stage descriptors: the stages are QH*128 bytes apart, so stage st = stage 0 advanced by st * QH*128 bytes
      const uint64_t qdesc_k0 = umma_smem_desc_sw128(smem_u32(sm.q[0]), 16, 1024), qdesc_mn0 = umma_smem_desc_sw128(smem_u32(sm.q[0]), 8192, 1024);
      const uint64_t dadesc_k0 = umma_smem_desc_sw128(smem_u32(sm.da[0]), 16, 1024), dadesc_mn0 = umma_smem_desc_sw128(smem_u32(sm.da[0]), 8192, 1024);
      const uint32_t idesc_s = umma_idesc_bf16(128, QH, 0, 0);
      const uint32_t idesc_o = umma_idesc_bf16(128, HD, 0, 1);
      const int g_total = (h_end - h_begin) * n_steps;
      auto issue_sdp = [&](int s) {        // s = global step; the first step of a head waits for that head's K / V
        const int st = s % kKvStages;
        if (s % n_steps == 0) mbar_wait(&sm.kv_full, (s / n_steps) & 1);
        mbar_wait(&sm.qd_full[st], (s / kKvStages) & 1);
        if (lane == 0) TRACE(5, 4 * s);
        if (lane == 0) TRACE(5, 4 * s + 1);
        tc_fence_after();
        const uint64_t qd = desc_adv(qdesc_k0, st * (QH * 128)), dd = desc_adv(dadesc_k0, st * (QH * 128));
#pragma unroll
        for (int kk = 0; kk < 4; ++kk)
          umma_bf16_w(tmem + kColST, desc_adv(kdesc, kk * 32), desc_adv(qd, kk * 32), idesc_s, kk > 0);
#pragma unroll
        for (int kk = 0; kk < 4; ++kk)
          umma_bf16_w(tmem + kColDPT, desc_adv(vdesc, kk * 32), desc_adv(dd, kk * 32), idesc_s, kk > 0);
        umma_commit_w(&sm.sdp_full);
        if (s % n_steps == n_steps - 1) umma_commit_w(&sm.kv_free);   // last reader of this head's K / V tiles
      };
      // P^T / dS^T overwrite the score columns they were computed from and feed the dV / dK products straight out of tensor
      // memory, so the next step's S^T / dP^T products can only follow this step's dV / dK (issue order = execution order):
      // one serial chain per CTA, the co-resident CTA fills the gaps.
      for (int s = 0; s < g_total; ++s) {
        issue_sdp(s);
        const int st = s % kKvStages;
        const uint32_t first = (s % n_steps == 0) ? 0u : 1u;     // first step of a head starts fresh dK / dV accumulators
        mbar_wait(&sm.pds_full, s & 1);
        if (lane == 0) TRACE(5, 4 * s + 2);
        tc_fence_after();
        const uint64_t qd = desc_adv(qdesc_mn0, st * (QH * 128)), dd = desc_adv(dadesc_mn0, st * (QH * 128));
        // k-step kk = 16 queries = 8 packed columns; queries 32cg + [0, 32) sit at columns 32cg + [0, 16) of their score tile
#pragma unroll
        for (int kk = 0; kk < QH / 16; ++kk)   // contraction over the step's 64 queries
          umma_bf16_ts_w(tmem + kColDV, tmem + kColST + (kk >> 1) * 32 + (kk & 1) * 8, desc_adv(dd, kk * 2048), idesc_o, (kk > 0) ? 1u : first);
#pragma unroll
        for (int kk = 0; kk < QH / 16; ++kk)
          umma_bf16_ts_w(tmem + kColDK, tmem + kColDPT + (kk >> 1) * 32 + (kk & 1) * 8, desc_adv(qd, kk * 2048), idesc_o, (kk > 0) ? 1u : first);
        if (lane == 0) TRACE(5, 4 * s + 3);
        umma_commit_w(&sm.qd_empty[st]);
        umma_commit_w(&sm.pds_free);
      }
    }
  } else {
    // thread = (key row, column group cg): 32 of the step's 64 queries, dK / dV columns [32cg, 32cg+32)
    const int q4 = warp & 3;
    const int sw = warp - 2;
    const int cg = sw >> 2;
    const int row = q4 * 32 + lane;            // key within the tile
    const uint32_t lane_off = (uint32_t)(q4 * 32) << 16;
    const float sc = p.scale * kLog2e;
    const int slot = (packed && key0 + row >= md.Sk) ? 1 : 0;  // which of the tile's two entities owns this key row
    const bool kvalid = (row < nkeys) && (slot ? ok_hi : ok_lo) && (p.key_valid == nullptr || p.key_valid[(long long)kvrow0 + row] != 0);
    auto lse_index = [&](int h, int s, int ent) {
      return (((long long)(biz * p.R + step_target(s)) * p.H + h) * p.E_total + md.ent_base + ent) * SQ + (s & 1) * QH + (sw * 32 + lane);
    };
    // LSE / DELTA rows of a step are staged with cp.async one step ahead (no register dependency, so the global
    // latency never sits on the softmax critical path); P absorbs 1/n through  exp2(sc*s - (LSE - log2(1/n)))
    auto stage_rows = [&](int h, int s, int st) {
      const long long i = lse_index(h, s, e);
      cp_async_4(smem_u32(&sm.lse[st][0][sw * 32 + lane]), p.LSE + i);
      cp_async_4(smem_u32(&sm.dlt[st][0][sw * 32 + lane]), p.DELTA + i);
      if (packed) {
        const long long i2 = lse_index(h, s, e_hi);
        cp_async_4(smem_u32(&sm.lse[st][1][sw * 32 + lane]), p.LSE + i2);
        cp_async_4(smem_u32(&sm.dlt[st][1][sw * 32 + lane]), p.DELTA + i2);
      }
    };
    if (sw < 2) stage_rows(h_begin, 0, 0);
    if (threadIdx.x - 64 < (unsigned)p.R && threadIdx.x - 64 < 32u) {
      const int tg = threadIdx.x - 64;
      sm.lg_invn[tg] = p.inv_n ? __log2f(p.inv_n[(long long)(biz * p.R + tg) * p.n_mod + m]) : 0.f;
    }
    for (int h = h_begin; h < h_end; ++h) {
    const int g0 = (h - h_begin) * n_steps;
    for (int s = 0; s < n_steps; ++s) {
      const int g = g0 + s, st = g & 1;
      if (sw < 2) cp_async_wait_all();   // rows of this step (issued one step ago) have landed
      if (threadIdx.x == 64) TRACE(6, 6 * s);
      kv_soft_bar();   // stage st is visible; everybody is done with stage st^1 (read during step s-1)
      if (threadIdx.x == 64) TRACE(6, 6 * s + 1);
      if (sw < 2) {
        if (s + 1 < n_steps) stage_rows(h, s + 1, st ^ 1);
        else if (h + 1 < h_end) stage_rows(h + 1, 0, st ^ 1);
      }
      const float lg = sm.lg_invn[step_target(s)];
      uint32_t wd = kvalid ? 0xffffffffu : 0u;
      if (p.causal) {  // key (key0 + row) <= query ((s&1)*64 + cg*32 + j)  <=>  j >= key0 + row - (s&1)*64 - cg*32
        const int lo = key0 + row - (s & 1) * QH - cg * 32;
        wd &= (lo <= 0) ? 0xffffffffu : (lo >= 32 ? 0u : ~((1u << lo) - 1u));
      }
      // queries beyond the sequence's frame (q_rows < 128): their Q / dA rows belong to the next sequence
      const int qleft = QS - (s & 1) * QH - cg * 32;
      const bool qpartial = qleft < 32;
      if (qpartial) wd &= (qleft <= 0) ? 0u : ((1u << qleft) - 1u);
      mbar_wait(&sm.sdp_full, g & 1);
      if (threadIdx.x == 64) TRACE(6, 6 * s + 2);
      tc_fence_after();
      uint32_t rs[32], rd[32];
      tmem_ld_32x32(tmem + lane_off + kColST + cg * 32, rs);
      tmem_ld_32x32(tmem + lane_off + kColDPT + cg * 32, rd);
      tmem_ld_wait();
      if (threadIdx.x == 64) TRACE(6, 6 * s + 3);
      const f32x2 lg2 = splat2(lg), m1 = splat2(-1.f), sc2 = splat2(sc), scale2 = splat2(p.scale), nscale2 = splat2(-p.scale);
      if (threadIdx.x == 64) TRACE(6, 6 * s + 4);
      // three copies of the loop (warp-uniform choice; predicated-off mask code would still take issue slots):
      //   0 = every score valid;  1 = per-element mask (causal);  2 = the thread's key row is valid or not as a whole (pad keys,
      //   null entity of a packed tile): computed like 0, the packed words are selected at the end (1 instead of 2 selects per score)
      auto body = [&](auto tag) {
      constexpr int kMode = decltype(tag)::value;
#pragma unroll
      for (int g8 = 0; g8 < 4; ++g8) {
        uint32_t po[4], dso[4];
        const float4 l0 = *reinterpret_cast<const float4*>(&sm.lse[st][slot][cg * 32 + g8 * 8]);
        const float4 l1 = *reinterpret_cast<const float4*>(&sm.lse[st][slot][cg * 32 + g8 * 8 + 4]);
        const float4 d0 = *reinterpret_cast<const float4*>(&sm.dlt[st][slot][cg * 32 + g8 * 8]);
        const float4 d1 = *reinterpret_cast<const float4*>(&sm.dlt[st][slot][cg * 32 + g8 * 8 + 4]);
        // packed fp32 pairs (FFMA2 / FMUL2): the softmax warps are issue-bound, so two lanes per instruction count
        const f32x2 nl[4] = {fma2(pack2(l0.x, l0.y), m1, lg2), fma2(pack2(l0.z, l0.w), m1, lg2),
                             fma2(pack2(l1.x, l1.y), m1, lg2), fma2(pack2(l1.z, l1.w), m1, lg2)};      // log2(1/n) - LSE
        const f32x2 nd[4] = {mul2(pack2(d0.x, d0.y), nscale2), mul2(pack2(d0.z, d0.w), nscale2),
                             mul2(pack2(d1.x, d1.y), nscale2), mul2(pack2(d1.z, d1.w), nscale2)};      // -scale * delta'
#pragma unroll
        for (int e2 = 0; e2 < 4; ++e2) {
          const int j = g8 * 8 + 2 * e2;
          float a0, a1;
          unpack2(fma2(pack2(__uint_as_float(rs[j]), __uint_as_float(rs[j + 1])), sc2, nl[e2]), a0, a1);
          float p0 = ex2(a0), p1 = ex2(a1);
          if constexpr (kMode == 1) { p0 = ((wd >> j) & 1u) ? p0 : 0.f; p1 = ((wd >> (j + 1)) & 1u) ? p1 : 0.f; }
          po[e2] = pack_bf16(p0, p1);
          float s0, s1;
          unpack2(mul2(pack2(p0, p1), fma2(pack2(__uint_as_float(rd[j]), __uint_as_float(rd[j + 1])), scale2, nd[e2])), s0, s1);
          // invalid key rows (null entity of a packed tile, pad keys): the forward never wrote their LSE / DELTA rows, which may
          // hold NaN patterns — select, 0 * stale is not 0
          if constexpr (kMode == 1) { s0 = ((wd >> j) & 1u) ? s0 : 0.f; s1 = ((wd >> (j + 1)) & 1u) ? s1 : 0.f; }
          dso[e2] = pack_bf16(s0, s1);
          if constexpr (kMode == 2) { po[e2] = wd ? po[e2] : 0u; dso[e2] = wd ? dso[e2] : 0u; }
        }
        // packed bf16 pairs back over the thread's own score columns (4 words = 8 queries): A operands of dV += Pn^T dA and
        // dK += dS^T Q, read by the tensor core straight from tensor memory
        tmem_st_32x4(tmem + lane_off + kColST + cg * 32 + g8 * 4, po);
        tmem_st_32x4(tmem + lane_off + kColDPT + cg * 32 + g8 * 4, dso);
      }
      };
      if (__all_sync(0xffffffffu, wd == 0xffffffffu)) body(std::integral_constant<int, 0>{});
      else if (p.causal || qpartial) body(std::integral_constant<int, 1>{});
      else body(std::integral_constant<int, 2>{});
      if (threadIdx.x == 64) TRACE(6, 6 * s + 5);
      tmem_st_wait();
      tc_fence_before();
      mbar_arrive(&sm.pds_full);
    }
    mbar_wait(&sm.pds_free, (g0 + n_steps - 1) & 1);
    tc_fence_after();
    {
      // every lane issues the (.sync.aligned) TMEM loads; only lanes that own a key store
      const int srow = row < nkeys ? row : 0;
      bf16* dk = dKV + (long long)(kvrow0 + srow) * p.lddkv + p.dk_col + h * HD + cg * 32;
      bf16* dv = dKV + (long long)(kvrow0 + srow) * p.lddkv + p.dv_col + h * HD + cg * 32;
      uint32_t rk[32], rv[32];
      tmem_ld_32x32(tmem + lane_off + kColDK + cg * 32, rk);
      tmem_ld_32x32(tmem + lane_off + kColDV + cg * 32, rv);
      tmem_ld_wait();
      if (row < nkeys) {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          uint4 u, w2;
          u.x = pack_bf16(__uint_as_float(rk[j * 8 + 0]), __uint_as_float(rk[j * 8 + 1]));
          u.y = pack_bf16(__uint_as_float(rk[j * 8 + 2]), __uint_as_float(rk[j * 8 + 3]));
          u.z = pack_bf16(__uint_as_float(rk[j * 8 + 4]), __uint_as_float(rk[j * 8 + 5]));
          u.w = pack_bf16(__uint_as_float(rk[j * 8 + 6]), __uint_as_float(rk[j * 8 + 7]));
          w2.x = pack_bf16(__uint_as_float(rv[j * 8 + 0]), __uint_as_float(rv[j * 8 + 1]));
          w2.y = pack_bf16(__uint_as_float(rv[j * 8 + 2]), __uint_as_float(rv[j * 8 + 3]));
          w2.z = pack_bf16(__uint_as_float(rv[j * 8 + 4]), __uint_as_float(rv[j * 8 + 5]));
          w2.w = pack_bf16(__uint_as_float(rv[j * 8 + 6]), __uint_as_float(rv[j * 8 + 7]));
          *reinterpret_cast<uint4*>(dk + j * 8) = u;
          *reinterpret_cast<uint4*>(dv + j * 8) = w2;
        }
      }
      tc_fence_before();   // the next head's first dV / dK products overwrite these accumulators
    }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) { __syncwarp(); tc_fence_after(); tmem_dealloc(tmem, 256); }
}

static int validate_tc(const MmsumAttnArgs* a, bool bwd) {
  if (!a || !a->Q || !a->KV || !a->O || !a->LSE) return MMSUM_ERR_INVALID;
  if (a->n_qseq <= 0 || a->H <= 0 || a->R <= 0 || a->n_mod < 1 || a->n_mod > 3) return MMSUM_ERR_INVALID;
  if ((a->n_qseq % a->R) || a->R > 32) return MMSUM_ERR_INVALID;
  if ((a->ldq % 8) || (a->ldkv % 8) || (a->ldo % 8) || (a->q_col % 8) || (a->k_col % 8) || (a->v_col % 8)) return MMSUM_ERR_INVALID;
  int ents = 0;
  for (int m = 0; m < a->n_mod; ++m) {
    if (a->mods[m].E <= 0 || a->mods[m].Sk <= 0 || a->mods[m].Sk > kMaxKeys) return MMSUM_ERR_INVALID;
    if (a->mods[m].ent_stride != 0 && a->mods[m].ent_stride < a->mods[m].Sk) return MMSUM_ERR_INVALID;
    ents += a->mods[m].E;
    if (a->mods[m].o_off % a->ldo) return MMSUM_ERR_INVALID;
  }
  if (ents > kMaxEnt || ents > a->E_total || ents > 32) return MMSUM_ERR_INVALID;
  if (a->causal && (a->n_mod != 1 || a->mods[0].Sk != SQ)) return MMSUM_ERR_INVALID;
  if (a->q_rows != 0 && (a->q_rows < 16 || a->q_rows > SQ || (a->q_rows % 16) || a->causal)) return MMSUM_ERR_INVALID;
  if (bwd) {
    if (!a->DELTA || !a->dQ || !a->dKV) return MMSUM_ERR_INVALID;
    if ((a->lddq % 8) || (a->lddkv % 8) || (a->dq_col % 8) || (a->dk_col % 8) || (a->dv_col % 8)) return MMSUM_ERR_INVALID;
    for (int m = 0; m < a->n_mod; ++m)
      if (a->mods[m].no_dkv != 0 && a->mods[m].no_dkv != 1) return MMSUM_ERR_INVALID;
  }
  return 0;
}

static int build_maps(const MmsumAttnArgs* a, AttnMaps* mp, bool bwd) {
  const int n_biz = a->n_qseq / a->R;
  const uint64_t qrows = (uint64_t)a->n_qseq * (a->q_rows > 0 ? a->q_rows : SQ);   // rows past the last frame: TMA zero fill
  int rc = make_tmap(&mp->q, a->Q, 0, (uint64_t)a->ldq, qrows, (uint64_t)a->ldq * 2, 64, SQ);
  if (rc) return rc;
  for (int m = 0; m < 3; ++m) {
    const MmsumAttnMod& md = a->mods[m < a->n_mod ? m : 0];
    const uint64_t rows = (uint64_t)md.kv_row_base + (uint64_t)n_biz * md.E * (md.ent_stride > 0 ? md.ent_stride : md.Sk);
    rc = make_tmap(&mp->kv[m], a->KV, 0, (uint64_t)a->ldkv, rows, (uint64_t)a->ldkv * 2, 64, (uint32_t)md.Sk);
    if (rc) return rc;
  }
  if (bwd) {
    uint64_t orows = 0;
    for (int m = 0; m < a->n_mod; ++m) {
      const uint64_t r = (uint64_t)(a->mods[m].o_off / a->ldo) + qrows;
      if (r > orows) orows = r;
    }
    rc = make_tmap(&mp->d_o, a->O, 0, (uint64_t)a->ldo, orows, (uint64_t)a->ldo * 2, 64, SQ);
    if (rc) return rc;
  } else {
    mp->d_o = mp->q;
  }
  return 0;
}

}  // namespace mmsum

using namespace mmsum;

// Debugging aids ------------------------------------------------------------------------------

// Fills every SM's shared memory and tensor memory with NaN bit patterns: a kernel that consumes stale on-chip state shows up as
// non-finite / run-to-run different output when launched after this one (tools/gpu_attn_determinism.py).
__global__ void __launch_bounds__(128, 1) debug_poison_kernel(int smem_words) {
  extern __shared__ uint8_t smem_raw[];
  __shared__ uint32_t slot;
  uint32_t* w = reinterpret_cast<uint32_t*>(smem_raw);
  for (int i = threadIdx.x; i < smem_words; i += blockDim.x) w[i] = 0xffffffffu;
  const int warp = threadIdx.x >> 5;
  if (warp == 0) { tmem_alloc(&slot, 512); tmem_relinquish(); }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = slot + ((uint32_t)(warp * 32) << 16);
  uint32_t r[16];
#pragma unroll
  for (int j = 0; j < 16; ++j) r[j] = 0xffffffffu;
  for (int c = 0; c < 512; c += 16) tmem_st_32x16(tmem + c, r);
  tmem_st_wait();
  tc_fence_before();
  __syncthreads();
  if (warp == 0) { tc_fence_after(); tmem_dealloc(slot, 512); }
}
extern "C" int mmsum_debug_poison(void* stream_v) {
  const int bytes = 200 * 1024;
  static std::atomic<unsigned long long> attr{0};
  if (int rc = ensure_dyn_smem(debug_poison_kernel, bytes, attr)) return rc;
  debug_poison_kernel<<<kNumSMs, 128, bytes, reinterpret_cast<cudaStream_t>(stream_v)>>>(bytes / 4);
  MMSUM_CHECK_LAUNCH();
  return 0;
}

extern "C" int mmsum_attn_fwd(const MmsumAttnArgs* a, void* stream_v) {
  if (int rc = validate_tc(a, false)) return rc;
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_v);
  AttnMaps mp;
  if (int rc = build_maps(a, &mp, false)) return rc;
  const int smem = (int)sizeof(Fwd3Smem) + 1024;
  static std::atomic<unsigned long long> attr{0};
  if (int rc = ensure_dyn_smem(attn_fwd_tc3_kernel, smem, attr)) return rc;
  // self-attention shape (one modality, one entity per sequence, no leave-one-out): heads become the CTA's items, so the
  // per-CTA set-up and the load / MMA / softmax latencies are amortised over the heads instead of paid once per head.  Two
  // CTAs per sequence (half of the heads each) so that both CTA slots of every SM are used.
  const int head_mode = (a->n_mod == 1 && a->mods[0].E == 1 && !a->mods[0].loo && a->H <= kMaxEnt && a->n_qseq >= 64) ? 1 : 0;
  const int hpc = head_mode ? ((a->H % 2 == 0 && a->n_qseq <= 2 * kNumSMs) ? a->H / 2 : a->H) : 0;
  MMSUM_LAUNCH_PDL(attn_fwd_tc3_kernel, head_mode ? a->n_qseq * (a->H / hpc) : a->n_qseq * a->H, kF3Threads, smem, stream, mp, *a, hpc);
  MMSUM_CHECK_LAUNCH();
  return 0;
}

extern "C" int mmsum_attn_bwd(const MmsumAttnArgs* a, void* stream_v) {
  if (int rc = validate_tc(a, true)) return rc;
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_v);
  AttnMaps mp;
  if (int rc = build_maps(a, &mp, true)) return rc;
  const int n_biz = a->n_qseq / a->R;
  uint64_t kvrows = 0;
  int tiles = 0;
  for (int m = 0; m < a->n_mod; ++m) {
    const uint64_t r = (uint64_t)a->mods[m].kv_row_base + (uint64_t)n_biz * a->mods[m].E * (a->mods[m].ent_stride > 0 ? a->mods[m].ent_stride : a->mods[m].Sk);
    if (r > kvrows) kvrows = r;
    tiles += dkv_tiles(a->mods[m]);
  }
  CUtensorMap kv128, q64, do64;
  if (int rc = make_tmap(&kv128, a->KV, 0, (uint64_t)a->ldkv, kvrows, (uint64_t)a->ldkv * 2, 64, SQ)) return rc;
  {   // 64-query boxes of Q and of the upstream gradient for the dK/dV kernel's steps
    const uint64_t qrows = (uint64_t)a->n_qseq * (a->q_rows > 0 ? a->q_rows : SQ);
    uint64_t orows = 0;
    for (int m = 0; m < a->n_mod; ++m) {
      const uint64_t r = (uint64_t)(a->mods[m].o_off / a->ldo) + qrows;
      if (r > orows) orows = r;
    }
    if (int rc = make_tmap(&q64, a->Q, 0, (uint64_t)a->ldq, qrows, (uint64_t)a->ldq * 2, 64, QH)) return rc;
    if (int rc = make_tmap(&do64, a->O, 0, (uint64_t)a->ldo, orows, (uint64_t)a->ldo * 2, 64, QH)) return rc;
  }
  const int smem_q = (int)sizeof(BwdQSmem) + 1024, smem_kv = (int)sizeof(BwdKVSmem) + 1024;
  static std::atomic<unsigned long long> attr_q{0}, attr_kv{0};
  if (int rc = ensure_dyn_smem(attn_bwd_dq_tc_kernel, smem_q, attr_q)) return rc;
  if (int rc = ensure_dyn_smem(attn_bwd_dkv_tc_kernel, smem_kv, attr_kv)) return rc;
  // profiling knob (tools/gpu_bench_attn.py): MMSUM_ATTN_BWD_PART=1 launches only dQ/DELTA, =2 only dK/dV
  static const int part = [] { const char* e = getenv("MMSUM_ATTN_BWD_PART"); return e ? atoi(e) : 0; }();
  if (part != 2) {
    // self-attention shape: heads become the CTA's items (needs <= 128 keys: the Q / dA ring borrows the dS upper half)
    const int head_mode = (a->n_mod == 1 && a->mods[0].E == 1 && !a->mods[0].loo && a->mods[0].Sk <= SQ && a->H <= kMaxEnt &&
                           a->n_qseq >= 64) ? 1 : 0;
    MMSUM_LAUNCH_PDL(attn_bwd_dq_tc_kernel, head_mode ? a->n_qseq : a->n_qseq * a->H, kAttnThreads, smem_q, stream, mp, *a, head_mode);
    MMSUM_CHECK_LAUNCH();
  }
  if (part != 1 && tiles > 0) {
    // self-attention shape: 4 heads per CTA (amortises the set-up, still ~2 waves of 2 CTAs/SM at 144 sequences)
    const int heads_per_cta = (a->n_mod == 1 && a->mods[0].E == 1 && !a->mods[0].loo && n_biz >= 64 && a->H % 4 == 0) ? 4 : 1;
    MMSUM_LAUNCH_PDL(attn_bwd_dkv_tc_kernel, n_biz * (a->H / heads_per_cta) * tiles, kKvThreads, smem_kv, stream, q64, do64, kv128, *a,
                     tiles, heads_per_cta);
    MMSUM_CHECK_LAUNCH();
  }
  return 0;
}

#ifdef MMSUM_ATTN_TRACE
extern "C" int mmsum_debug_read_trace(long long* host_out) {
  return (int)cudaMemcpyFromSymbol(host_out, mmsum::g_trace, sizeof(long long) * 8 * 512);
}
#endif
