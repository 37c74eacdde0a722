// tcgen05 / TMEM / TMA GEMM for sm_100a.
//
//   D[M,N] (+)= epilogue( alpha * sum_k A(m,k) * B(n,k) )        bf16 x bf16 -> fp32 accumulate in TMEM
//
// This one kernel serves every dense contraction of the MultimodalSum training step
// (reference: nn.Linear / F.linear call sites in src/transformer/modeling_multimodalsum.py
// :272-273,428-429,695-704,2281 and their autograd backward):
//   fprop   y = x W^T        A = x  [M,K]  K-major      B = W  [N,K]  K-major
//   dgrad   dx = dy W        A = dy [M,N'] K-major      B = W  [N',K'] read as MN-major (no transposed copy)
//   wgrad   dW = dy^T x      A = dy [T,N'] MN-major     B = x  [T,K'] MN-major, split-K + TMA reduce-add (fp32)
//
// Structure (one CTA per SM, persistent over output tiles, 192 threads):
//   warp 0     TMA producer   global -> 128B-swizzled smem ring (kStages deep), mbarrier expect_tx
//   warp 1     MMA issuer     one elected thread issues tcgen05.mma (M=128, N=BN, K=16) into TMEM; tcgen05.commit
//                             releases smem stages and publishes finished accumulators
//   warps 2-9  epilogue       tcgen05.ld TMEM -> registers, alpha/bias/GELU/ReLU/d-activation, bf16 or fp32,
//                             swizzled smem staging, TMA store (or TMA reduce-add for split-K / grad accumulation)
// TMEM holds two accumulator stages (2 x BN fp32 columns) so the epilogue of tile i overlaps the MMAs of tile i+1.
// Ragged M/N/K edges rely on TMA: out-of-bounds loads are zero-filled, out-of-bounds stores are clipped.
//
// CL = 2 (large problems): the persistent CTAs run as thread-block clusters of two — a CTA PAIR on the two SMs of a TPC — and
// one tcgen05.mma.cta_group::2 (M = 256, N = 256, issued by the leader CTA only) computes two adjacent m-tiles of the same
// n-tile.  Each CTA stages its own 128 A rows and HALF of the B tile (128 of the 256 n rows); the tensor cores read the other
// half out of the peer's shared memory, so per k-block a CTA moves 32 KB instead of 48 KB through L2 -> smem and the smem
// operand reads per MMA drop by a third (6 stages fit instead of 4).  Both CTAs' TMA loads complete on the LEADER's full
// barrier; tcgen05.commit.cta_group::2 (multicast) frees the stage in both CTAs and publishes the accumulator halves, which
// each CTA's epilogue warps read from their own tensor memory; accumulator stages are handed back on the leader's barrier.
#include "common.cuh"
#include "../../include/mmsum_b200.h"

#include <cudaTypedefs.h>
#include <mutex>
#include <unordered_map>
#include <string.h>

namespace mmsum {

static constexpr int BM = 128;
static constexpr int BK = 64;       // 64 bf16 = 128 B = one swizzle row
static constexpr int UMMA_K = 16;
static constexpr int kEpiWarps = 8;   // two warps per TMEM lane quarter, each owning alternate 64-column groups
static constexpr int kGemmThreads = 64 + kEpiWarps * 32;
static constexpr int kEpiBufBytes = 32 * 128;  // 32 rows x 128 B per staging buffer

template <int BN, int CL>
struct GemmSmem {
  static constexpr int kABytes = BM * BK * 2;
  static constexpr int kBBytes = (BN / CL) * BK * 2;           // CTA pair: this CTA's half of the B tile
  static constexpr int kStageBytes = kABytes + kBBytes;
  static constexpr int kStages = (CL == 2) ? 6 : ((BN == 256) ? 4 : 6);
  static constexpr int kEpiBytes = kEpiWarps * kEpiBufBytes;     // one staging buffer per epilogue warp
  static constexpr int kBarOffset = kStages * kStageBytes + kEpiBytes;
  static constexpr int kTotal = kBarOffset + 256 + 1024;  // + barriers + alignment slack
};

struct GemmKernelArgs {
  int M, N, K;
  int m_tiles, n_tiles, splits, k_per_split;
  int raster_m_fast;
  float alpha;
  const float* bias;
  int act;        // 0 none, 1 gelu(erf), 2 relu
  int aux_mode;   // 0 none, 1 store pre-activation to aux, 2 multiply by act'(aux)
  bf16* aux;
  long long ld_aux;
  int out_f32;
  int accumulate;
  int k_split;    // > 0: A columns [k_split, K) come from the second A tensor map (concat along K)
  int ws_rows;    // EPI 3: rows of one split's region of the partial workspace (split sp stores at row sp * ws_rows + m)
};

// work unit t -> (m unit, n tile, k split); an m unit is one m-tile (CL = 1) or a pair of adjacent m-tiles (CL = 2)
__device__ __forceinline__ void decode_tile(const GemmKernelArgs& g, int m_units, int t, int& mu, int& nt, int& sp) {
  const int mn = m_units * g.n_tiles;
  sp = t / mn;
  const int r = t - sp * mn;
  if (g.raster_m_fast) { mu = r % m_units; nt = r / m_units; }
  else                 { nt = r % g.n_tiles; mu = r / g.n_tiles; }
}

// EPI: 0 plain epilogue (alpha, bias, ReLU), 1 = GELU/ReLU with the pre-activation saved to aux, 2 = multiply by act'(aux),
//      3 = fp32 split-K partials stored (not reduce-added) to each split's own region of a workspace (ordered split-K)
template <int BN, bool A_MN, bool B_MN, int EPI, int CL>
__global__ void __launch_bounds__(kGemmThreads, 1)
gemm_tcgen05_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmA2,
                    const __grid_constant__ CUtensorMap tmB, const __grid_constant__ CUtensorMap tmD,
                    const __grid_constant__ CUtensorMap tmAux,
                    const GemmKernelArgs g) {
  using L = GemmSmem<BN, CL>;
  extern __shared__ uint8_t smem_raw[];
  // align inside the shared window with pointer arithmetic on the __shared__ array (keeps LDS/STS addressing)
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + L::kBarOffset);
  uint64_t* empty_bar = full_bar + L::kStages;
  uint64_t* tfull_bar = empty_bar + L::kStages;
  uint64_t* tempty_bar = tfull_bar + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty_bar + 2);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int crank = (CL == 2) ? (int)cluster_ctarank() : 0;      // position inside the CTA pair
  const int m_units = (CL == 2) ? (g.m_tiles + 1) / 2 : g.m_tiles;
  const int total_tiles = m_units * g.n_tiles * g.splits;        // work units of a cluster (CL = 2) / a CTA
  const int unit0 = blockIdx.x / CL, unit_stride = gridDim.x / CL;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmA); tma_prefetch_desc(&tmB); tma_prefetch_desc(&tmD);
  }
  if (warp == 1) {
    if (lane == 0) {
      for (int s = 0; s < L::kStages; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
      // CTA pair: one arrival per epilogue warp of BOTH CTAs on the leader's barrier; otherwise one per epilogue thread
      for (int s = 0; s < 2; ++s) { mbar_init(&tfull_bar[s], 1); mbar_init(&tempty_bar[s], CL == 2 ? 2 * kEpiWarps : kEpiWarps * 32); }
      fence_barrier_init();
    }
    __syncwarp();
    if (CL == 2) { tmem_alloc2(tmem_slot, 512); tmem_relinquish2(); }
    else         { tmem_alloc(tmem_slot, 512); tmem_relinquish(); }
  }
  tc_fence_before();
  __syncthreads();
  if (CL == 2) cluster_sync_all();     // the peer's barriers are initialised before anything of ours can signal them
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  pdl_launch_dependents();
  pdl_wait();            // everything above overlapped the previous kernel's tail; global memory is touched only below

  if (warp == 0) {
    // ===================== TMA producer (whole warp runs the loop; lane 0 issues) =====================
    int stage = 0; uint32_t phase = 0;
    for (int t = unit0; t < total_tiles; t += unit_stride) {
      int mu, nt, sp; decode_tile(g, m_units, t, mu, nt, sp);
      const int mt = (CL == 2) ? 2 * mu + crank : mu;
      const int m0 = mt * BM, n0 = nt * BN;
      const int k_begin = sp * g.k_per_split;
      const int k_end = min(g.K, k_begin + g.k_per_split);
      for (int k0 = k_begin; k0 < k_end; k0 += BK) {
        mbar_wait(&empty_bar[stage], phase ^ 1);
        uint8_t* sA = smem + stage * L::kStageBytes;
        uint8_t* sB = sA + L::kABytes;
        if (CL == 2) {
          // both CTAs' loads complete on the LEADER's barrier, which expects the bytes of both stages
          const uint32_t lbar = mapa_u32(smem_u32(&full_bar[stage]), 0);
          if (crank == 0) mbar_expect_tx_w(&full_bar[stage], 2 * L::kStageBytes);
          if (A_MN) {
#pragma unroll
            for (int j = 0; j < BM / 64; ++j) tma_load_2d_2sm_w(sA + j * 8192, &tmA, lbar, m0 + 64 * j, k0);
          } else if (g.k_split > 0 && k0 >= g.k_split) {
            tma_load_2d_2sm_w(sA, &tmA2, lbar, k0 - g.k_split, m0);
          } else {
            tma_load_2d_2sm_w(sA, &tmA, lbar, k0, m0);
          }
          // this CTA's half of the B tile (n rows [crank * BN/2, +BN/2)); the pair's MMA reads the other half from the peer
          if (B_MN) {
#pragma unroll
            for (int j = 0; j < BN / 128; ++j) tma_load_2d_2sm_w(sB + j * 8192, &tmB, lbar, n0 + crank * (BN / 2) + 64 * j, k0);
          } else {
            tma_load_2d_2sm_w(sB, &tmB, lbar, k0, n0 + crank * (BN / 2));
          }
          if (++stage == L::kStages) { stage = 0; phase ^= 1; }
          continue;
        }
        mbar_expect_tx_w(&full_bar[stage], L::kStageBytes);
        if (A_MN) {
#pragma unroll
          for (int j = 0; j < BM / 64; ++j) tma_load_2d_w(sA + j * 8192, &tmA, &full_bar[stage], m0 + 64 * j, k0);
        } else if (g.k_split > 0 && k0 >= g.k_split) {
          tma_load_2d_w(sA, &tmA2, &full_bar[stage], k0 - g.k_split, m0);
        } else {
          tma_load_2d_w(sA, &tmA, &full_bar[stage], k0, m0);
        }
        if (B_MN) {
#pragma unroll
          for (int j = 0; j < BN / 64; ++j) tma_load_2d_w(sB + j * 8192, &tmB, &full_bar[stage], n0 + 64 * j, k0);
        } else {
          tma_load_2d_w(sB, &tmB, &full_bar[stage], k0, n0);
        }
        if (++stage == L::kStages) { stage = 0; phase ^= 1; }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer (whole warp runs the loop; lane 0 issues; CTA pair: the leader CTA only) =====================
    constexpr uint32_t idesc = umma_idesc_bf16(BM * CL, BN, A_MN ? 1 : 0, B_MN ? 1 : 0);
    const uint32_t smem_base = smem_u32(smem);
    int stage = 0; uint32_t phase = 0;
    int as = 0; uint32_t aphase = 0;
    for (int t = unit0; t < total_tiles && crank == 0; t += unit_stride) {
      int mu, nt, sp; decode_tile(g, m_units, t, mu, nt, sp);
      const int k_begin = sp * g.k_per_split;
      const int k_end = min(g.K, k_begin + g.k_per_split);
      mbar_wait(&tempty_bar[as], aphase ^ 1);
      tc_fence_after();
      const uint32_t d_tmem = tmem_base + as * BN;
      uint32_t accum = 0;
      for (int k0 = k_begin; k0 < k_end; k0 += BK) {
        mbar_wait(&full_bar[stage], phase);
        tc_fence_after();
        const uint32_t aaddr = smem_base + stage * L::kStageBytes;
        const uint32_t baddr = aaddr + L::kABytes;
        // K-major: 8-row groups are 1024 B apart (SBO); a K step of 16 elements is +32 B inside the swizzle row.
        // MN-major: 64-wide MN blocks are 8192 B apart (LBO), 8-row K groups 1024 B apart (SBO); K step = 16 rows = 2048 B.
        const uint64_t ad0 = A_MN ? umma_smem_desc_sw128(aaddr, 8192, 1024) : umma_smem_desc_sw128(aaddr, 16, 1024);
        const uint64_t bd0 = B_MN ? umma_smem_desc_sw128(baddr, 8192, 1024) : umma_smem_desc_sw128(baddr, 16, 1024);
#pragma unroll
        for (int kk = 0; kk < BK / UMMA_K; ++kk) {
          if (CL == 2) umma_bf16_2sm_w(d_tmem, ad0 + (uint64_t)((A_MN ? kk * 2048 : kk * 32) >> 4),
                                       bd0 + (uint64_t)((B_MN ? kk * 2048 : kk * 32) >> 4), idesc, accum);
          else         umma_bf16_w(d_tmem, ad0 + (uint64_t)((A_MN ? kk * 2048 : kk * 32) >> 4),
                                   bd0 + (uint64_t)((B_MN ? kk * 2048 : kk * 32) >> 4), idesc, accum);
          accum = 1;
        }
        // frees the smem stage once these MMAs retire (CTA pair: in BOTH CTAs, each producer refills its own stage)
        if (CL == 2) umma_commit_2sm_mc_w(&empty_bar[stage], (uint16_t)3); else umma_commit_w(&empty_bar[stage]);
        if (++stage == L::kStages) { stage = 0; phase ^= 1; }
      }
      // accumulator complete (CTA pair: each CTA's epilogue warps wait on their own barrier for their 128 rows)
      if (CL == 2) umma_commit_2sm_mc_w(&tfull_bar[as], (uint16_t)3); else umma_commit_w(&tfull_bar[as]);
      if (++as == 2) { as = 0; aphase ^= 1; }
    }
  } else {
    // ===================== epilogue warps (2..9) =====================
    // warp = (TMEM lane quarter q, column half eh): 64-column groups eh, eh+2, ... of the tile, 32 columns at a time.
    const int q = warp & 3;            // TMEM lane quarter this warp may access
    const int ew = warp - 2;
    const int eh = ew >> 2;
    uint8_t* stg = smem + L::kStages * L::kStageBytes + ew * kEpiBufBytes;
    const bool bias_vec = (g.bias != nullptr) && ((reinterpret_cast<uintptr_t>(g.bias) & 15u) == 0);
    constexpr int kGroupsPerWarp = BN / 128;      // 64-column groups per warp and tile
    int as = 0; uint32_t aphase = 0;
    for (int t = unit0; t < total_tiles; t += unit_stride) {
      int mu, nt, sp; decode_tile(g, m_units, t, mu, nt, sp);
      const int mt = (CL == 2) ? 2 * mu + crank : mu;
      const int m0 = mt * BM, n0 = nt * BN;
      const int row = m0 + q * 32 + lane;
      // activation-gradient operand (EPI 2): this warp's share of the tile is fetched before the accumulator is
      // complete, so the global-load latency hides behind the MMAs of the tile
      uint4 auxr[EPI == 2 ? kGroupsPerWarp : 1][2][4] = {};
      if (EPI == 2) {
#pragma unroll
        for (int gi = 0; gi < kGroupsPerWarp; ++gi)
#pragma unroll
          for (int half = 0; half < 2; ++half)
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              const int n = n0 + (eh + 2 * gi) * 64 + half * 32 + j * 8;
              if (row < g.M && n + 8 <= g.N) auxr[gi][half][j] = *reinterpret_cast<const uint4*>(g.aux + (size_t)row * g.ld_aux + n);
            }
      }
      mbar_wait(&tfull_bar[as], aphase);
      tc_fence_after();
      const uint32_t tbase = tmem_base + ((uint32_t)(q * 32) << 16) + as * BN;
      // accumulator chunk -> alpha, bias
      auto load_chunk = [&](int c, float (&v)[32]) {
        const int ncol0 = n0 + c * 32;
        uint32_t r[32];
        tmem_ld_32x32(tbase + c * 32, r);
        tmem_ld_wait();
#pragma unroll
        for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]) * g.alpha;
        if (g.bias != nullptr && sp == 0) {
          if (bias_vec && ncol0 + 32 <= g.N) {
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              const float4 b4 = __ldg(reinterpret_cast<const float4*>(g.bias + ncol0) + j);
              v[j * 4 + 0] += b4.x; v[j * 4 + 1] += b4.y; v[j * 4 + 2] += b4.z; v[j * 4 + 3] += b4.w;
            }
          } else {
#pragma unroll
            for (int i = 0; i < 32; ++i) { const int n = ncol0 + i; v[i] += (n < g.N) ? __ldg(g.bias + n) : 0.f; }
          }
        }
      };
      auto pack16 = [&](const float (&v)[32], uint32_t (&o)[16]) {
#pragma unroll
        for (int i = 0; i < 16; ++i) o[i] = pack_bf16(v[2 * i], v[2 * i + 1]);
      };
      // 32 rows x 64 bf16 columns from registers into the swizzled staging tile, then one TMA store
      auto store_group = [&](const CUtensorMap* tm, const uint32_t (&lo)[16], const uint32_t (&hi)[16], int x) {
        if (lane == 0) tma_store_wait_read<0>();   // the previous store has finished reading the staging tile
        __syncwarp();
        uint8_t* b = stg + lane * 128;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          *reinterpret_cast<uint4*>(b + ((j ^ (lane & 7)) << 4)) = make_uint4(lo[j * 4], lo[j * 4 + 1], lo[j * 4 + 2], lo[j * 4 + 3]);
          *reinterpret_cast<uint4*>(b + (((4 + j) ^ (lane & 7)) << 4)) = make_uint4(hi[j * 4], hi[j * 4 + 1], hi[j * 4 + 2], hi[j * 4 + 3]);
        }
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) {
          if (x < g.N && m0 + q * 32 < g.M) tma_store_2d(tm, stg, x, m0 + q * 32);
          tma_store_commit();
        }
      };
#pragma unroll
      for (int gi = 0; gi < kGroupsPerWarp; ++gi) {
        const int grp = eh + 2 * gi;
        if (g.out_f32) {
#pragma unroll 1
          for (int half = 0; half < 2; ++half) {
            const int c = 2 * grp + half;
            const int ncol0 = n0 + c * 32;
            float v[32];
            load_chunk(c, v);
            if (g.act == 2) {
#pragma unroll
              for (int i = 0; i < 32; ++i) v[i] = fmaxf(v[i], 0.f);
            }
            if (lane == 0) tma_store_wait_read<0>();
            __syncwarp();
            uint8_t* b = stg + lane * 128;
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              float4 f = make_float4(v[j * 4 + 0], v[j * 4 + 1], v[j * 4 + 2], v[j * 4 + 3]);
              *reinterpret_cast<float4*>(b + ((j ^ (lane & 7)) << 4)) = f;
            }
            fence_proxy_async_smem();
            __syncwarp();
            if (lane == 0) {
              if (ncol0 < g.N && m0 + q * 32 < g.M) {
                if (EPI == 3)          tma_store_2d(&tmD, stg, ncol0, sp * g.ws_rows + m0 + q * 32);
                else if (g.accumulate) tma_reduce_add_2d(&tmD, stg, ncol0, m0 + q * 32);
                else                   tma_store_2d(&tmD, stg, ncol0, m0 + q * 32);
              }
              tma_store_commit();
            }
          }
        } else {
          uint32_t outp[2][16], prep[EPI == 1 ? 2 : 1][16];
#pragma unroll
          for (int half = 0; half < 2; ++half) {
            float v[32];
            load_chunk(2 * grp + half, v);
            if (EPI == 1 && g.aux_mode == 1) pack16(v, prep[EPI == 1 ? half : 0]);     // pre-activation, saved for the backward epilogue
            if (EPI != 2) {
              if (EPI == 1 && g.aux_mode == 3) {
                // GELU and GELU' from one erf / exp evaluation; the DERIVATIVE is saved, so backward is a single multiply
                float dv[32];
#pragma unroll
                for (int i = 0; i < 32; i += 2) gelu_erf_and_grad2(v[i], v[i + 1], dv[i], dv[i + 1]);
                pack16(dv, prep[EPI == 1 ? half : 0]);
              } else if (g.act == 1) {
#pragma unroll
                for (int i = 0; i < 32; i += 2) gelu_erf2(v[i], v[i + 1]);
              } else if (g.act == 2) {
#pragma unroll
                for (int i = 0; i < 32; ++i) v[i] = fmaxf(v[i], 0.f);
              }
            } else {
              // v *= act'(aux): backward through the activation fused into the dgrad epilogue
#pragma unroll
              for (int j = 0; j < 4; ++j) {
                const uint4 ax = auxr[EPI == 2 ? gi : 0][half][j];
                const uint32_t w[4] = {ax.x, ax.y, ax.z, ax.w};
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                  const float2 h = unpack_bf16(w[e]);
                  if (g.aux_mode == 4) { v[j * 8 + 2 * e] *= h.x; v[j * 8 + 2 * e + 1] *= h.y; }      // aux holds act'(pre-activation)
                  else if (g.act == 1) { gelu_erf_grad_mul2(v[j * 8 + 2 * e], v[j * 8 + 2 * e + 1], h.x, h.y); }
                  else            { v[j * 8 + 2 * e] *= (h.x > 0.f) ? 1.f : 0.f; v[j * 8 + 2 * e + 1] *= (h.y > 0.f) ? 1.f : 0.f; }
                }
              }
            }
            pack16(v, outp[half]);
          }
          if (EPI == 1) store_group(&tmAux, prep[0], prep[EPI == 1 ? 1 : 0], n0 + grp * 64);
          store_group(&tmD, outp[0], outp[1], n0 + grp * 64);
        }
      }
      // all TMEM reads of this accumulator stage are done -> hand it back to the MMA warp
      tc_fence_before();
      if (CL == 2) {   // one arrival per warp on the leader's barrier (its MMA warp owns the accumulator stages of both CTAs)
        __syncwarp();
        if (lane == 0) mbar_arrive_cluster(mapa_u32(smem_u32(&tempty_bar[as]), 0));
      } else {
        mbar_arrive(&tempty_bar[as]);
      }
      if (++as == 2) { as = 0; aphase ^= 1; }
    }
    if (lane == 0) tma_store_wait_all<0>();
  }

  tc_fence_before();
  __syncthreads();
  if (CL == 2) cluster_sync_all();     // neither CTA leaves while the peer may still multicast into it / arrive on its barriers
  if (warp == 1) {
    __syncwarp();
    tc_fence_after();
    if (CL == 2) tmem_dealloc2(tmem_base, 512); else tmem_dealloc(tmem_base, 512);
  }
}

// Ordered split-K: D[m, n] = (((D[m, n] + P_0[m, n]) + P_1[m, n]) + ...) over the splits in index order, one read-modify-write
// per element.  P_s = ws + s * split_stride, row pitch ldw.
__global__ void __launch_bounds__(256) splitk_ordered_reduce_kernel(const float* __restrict__ ws, int splits, long long split_stride,
                                                                    int ldw, float* __restrict__ D, long long ldd, int M, int N) {
  const long long n_el = (long long)M * N;
  for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < n_el; i += (long long)gridDim.x * 256) {
    const int m = (int)(i / N), n = (int)(i - (long long)m * N);
    const float* p = ws + (long long)m * ldw + n;
    float acc = D[(long long)m * ldd + n];
    for (int s = 0; s < splits; ++s) acc += p[s * split_stride];
    D[(long long)m * ldd + n] = acc;
  }
}

// ----------------------------------------------------------------------------
// host side: tensor-map cache + launch
// ----------------------------------------------------------------------------
static PFN_cuTensorMapEncodeTiled g_encode = nullptr;
static std::mutex g_mu;

static int get_encode() {
  if (g_encode) return 0;
  void* fn = nullptr;
  cudaDriverEntryPointQueryResult qres;
  cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres);
  if (e != cudaSuccess || fn == nullptr || qres != cudaDriverEntryPointSuccess) return MMSUM_ERR_DRIVER;
  g_encode = reinterpret_cast<PFN_cuTensorMapEncodeTiled>(fn);
  return 0;
}

struct TmKey {
  const void* ptr; uint64_t inner, outer, ld_bytes; uint32_t box_inner, box_outer; int dtype;
  bool operator==(const TmKey& o) const { return memcmp(this, &o, sizeof(TmKey)) == 0; }
};
struct TmKeyHash {
  size_t operator()(const TmKey& k) const {
    const uint64_t* p = reinterpret_cast<const uint64_t*>(&k);
    uint64_t h = 1469598103934665603ULL;
    for (size_t i = 0; i < sizeof(TmKey) / 8; ++i) { h ^= p[i]; h *= 1099511628211ULL; }
    return (size_t)h;
  }
};
static std::unordered_map<TmKey, CUtensorMap, TmKeyHash> g_tm_cache;

// 2D row-major tensor [outer, inner] with row pitch ld_bytes; box = [box_outer, box_inner]; 128B swizzle.
int make_tmap(CUtensorMap* out, const void* ptr, int dtype /*0 bf16, 1 f32*/, uint64_t inner, uint64_t outer,
                     uint64_t ld_bytes, uint32_t box_inner, uint32_t box_outer) {
  TmKey key;
  memset(&key, 0, sizeof(key));
  key.ptr = ptr; key.inner = inner; key.outer = outer; key.ld_bytes = ld_bytes;
  key.box_inner = box_inner; key.box_outer = box_outer; key.dtype = dtype;
  std::lock_guard<std::mutex> lk(g_mu);
  auto it = g_tm_cache.find(key);
  if (it != g_tm_cache.end()) { *out = it->second; return 0; }
  if (int rc = get_encode()) return rc;
  if ((reinterpret_cast<uintptr_t>(ptr) & 15) || (ld_bytes & 15)) return MMSUM_ERR_INVALID;
  cuuint64_t gdim[2] = {inner, outer};
  cuuint64_t gstr[1] = {ld_bytes};
  cuuint32_t box[2] = {box_inner, box_outer};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = g_encode(out, dtype == 0 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2,
                        const_cast<void*>(ptr), gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                        CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return MMSUM_ERR_DRIVER;
  if (g_tm_cache.size() > 65536) g_tm_cache.clear();
  g_tm_cache.emplace(key, *out);
  return 0;
}

static int num_sms() {
  static std::atomic<int> cached[64];       // per device; 0 = not queried yet
  int dev = 0, v = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return kNumSMs;
  const int c = cached[dev & 63].load(std::memory_order_relaxed);
  if (c > 0) return c;
  if (cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || v <= 0) v = kNumSMs;
  cached[dev & 63].store(v, std::memory_order_relaxed);
  return v;
}

template <int BN, bool A_MN, bool B_MN, int EPI, int CL>
static int launch_gemm(const CUtensorMap& ta, const CUtensorMap& ta2, const CUtensorMap& tb, const CUtensorMap& td,
                       const CUtensorMap& taux,
                       const GemmKernelArgs& ka, int grid, cudaStream_t stream) {
  using L = GemmSmem<BN, CL>;
  static std::atomic<unsigned long long> attr_set{0};     // one per template instantiation
  if (int rc = ensure_dyn_smem(gemm_tcgen05_kernel<BN, A_MN, B_MN, EPI, CL>, L::kTotal, attr_set)) return rc;
  cudaError_t le = launch_pdl_cluster(gemm_tcgen05_kernel<BN, A_MN, B_MN, EPI, CL>, dim3(grid), dim3(kGemmThreads), (size_t)L::kTotal,
                                      stream, CL, ta, ta2, tb, td, taux, ka);
  if (le != cudaSuccess) return (int)le;
  MMSUM_CHECK_LAUNCH();
  return 0;
}

}  // namespace mmsum

using namespace mmsum;

static int launch_gemm_case(int bn, int am, int bm, int epi, int cl, const CUtensorMap& ta, const CUtensorMap& ta2,
                            const CUtensorMap& tb, const CUtensorMap& td, const CUtensorMap& taux, const GemmKernelArgs& ka,
                            int grid, cudaStream_t stream);

// ordered = false: mmsum_gemm_bf16.  ordered = true: mmsum_gemm_bf16_ordered (ws / ws_elems) or, with need != NULL, only the
// workspace size query (nothing is launched and no pointer is read).
static int gemm_impl(const MmsumGemmArgs* a, cudaStream_t stream, bool ordered, float* ws, int64_t ws_elems, int64_t* need) {
  if (need != nullptr) *need = 0;
  if (!a || (need == nullptr && (!a->A || !a->B || !a->D))) return MMSUM_ERR_INVALID;
  if (a->M <= 0 || a->N <= 0 || a->K <= 0) return MMSUM_ERR_INVALID;
  if (!a->out_f32 && a->accumulate) return MMSUM_ERR_INVALID;
  if (a->aux_mode != 0 && (!a->aux || (a->N % 8) != 0 || (a->ld_aux % 8) != 0)) return MMSUM_ERR_INVALID;
  int bn = a->block_n;
  if (bn == 0) {
    bn = (a->N > 128) ? 256 : 128;
    // skinny problems (decode steps: M = a few hundred rows): 128-wide tiles double the number of CTAs that stream the
    // weights and halve each CTA's K loop when 256-wide tiles would leave most of the SMs idle
    // (not for the split-K weight gradients: their K loop supplies the work units, and 256-wide CTA-pair tiles are 12 % faster
    //  there — tools/gpu_gemm_sweep.py)
    const bool splitk_ok = a->out_f32 && a->accumulate && a->A2 == nullptr && a->splits <= 0;
    if (bn == 256 && a->aux_mode == 0 && !splitk_ok &&
        (long long)((a->M + BM - 1) / BM) * ((a->N + 255) / 256) * 2 <= num_sms()) bn = 128;
  }
  if (bn != 128 && bn != 256) return MMSUM_ERR_INVALID;
  if (a->aux_mode != 0) {   // fused-activation epilogues exist for row-major A and 256-wide tiles
    if (a->aux_mode < 0 || a->aux_mode > 4 || a->a_mn_major) return MMSUM_ERR_INVALID;
    if (a->aux_mode == 3 && a->act != 1) return MMSUM_ERR_INVALID;      // the saved derivative exists for GELU
    bn = 256;
  }

  GemmKernelArgs ka;
  ka.M = a->M; ka.N = a->N; ka.K = a->K;
  ka.m_tiles = (a->M + BM - 1) / BM;
  ka.n_tiles = (a->N + bn - 1) / bn;
  const int kblocks = (a->K + BK - 1) / BK;
  int splits = a->splits;
  if (splits <= 0) {
    // auto split-K (fp32 accumulating outputs only): pick the split count that minimises
    //   waves * (k-blocks per split * 512 clk + ~4096 clk of unoverlapped prologue / reduce epilogue)
    // on the persistent grid; the constants were fitted to tools/gpu_gemm_sweep.py on the step's wgrad shapes
    splits = 1;
    const int mn = ka.m_tiles * ka.n_tiles;
    if (a->out_f32 && a->accumulate && a->A2 == nullptr) {
      const int nsm = num_sms();
      long long best = -1;
      for (int sp = 1; sp <= 16 && sp * 8 <= kblocks; ++sp) {
        const int kb = (kblocks + sp - 1) / sp;
        const int eff = (kblocks + kb - 1) / kb;          // splits that actually get work
        const long long waves = ((long long)mn * eff + nsm - 1) / nsm;
        const long long cost = waves * ((long long)kb * 512 + 4096);
        if (best < 0 || cost < best) { best = cost; splits = sp; }
      }
    }
  }
  if (splits > 1 && (!(a->out_f32 && a->accumulate) || a->A2 != nullptr)) return MMSUM_ERR_INVALID;
  int kb_per_split = (kblocks + splits - 1) / splits;
  splits = (kblocks + kb_per_split - 1) / kb_per_split;  // no empty split
  ka.splits = splits;
  ka.k_per_split = kb_per_split * BK;
  ka.raster_m_fast = a->raster_m_fast;
  ka.alpha = a->alpha;
  ka.bias = a->bias;
  ka.act = a->act;
  ka.aux_mode = a->aux_mode;
  ka.aux = reinterpret_cast<bf16*>(a->aux);
  ka.ld_aux = a->ld_aux;
  ka.out_f32 = a->out_f32;
  ka.accumulate = a->accumulate;
  ka.ws_rows = 0;
  // ordered split-K: every split stores its partial tile to its own [m_tiles * 128, ldw] region of `ws`, then one pass adds the
  // regions to D in split order (splits == 1 keeps the single TMA reduce-add per element, which is already one writer)
  const bool ws_mode = ordered && ka.splits > 1;
  const int ldw = (a->N + 3) / 4 * 4;                         // 16-byte row pitch for the tensor map
  const long long split_stride = (long long)ka.m_tiles * BM * ldw;
  if (ws_mode) {
    if (ka.act != 0 || ka.aux_mode != 0) return MMSUM_ERR_INVALID;
    if (need != nullptr) { *need = split_stride * ka.splits; return 0; }
    if (!ws || (reinterpret_cast<uintptr_t>(ws) & 15) || ws_elems < split_stride * ka.splits) return MMSUM_ERR_INVALID;
    ka.ws_rows = ka.m_tiles * BM;
  }
  if (need != nullptr) return 0;

  CUtensorMap ta, ta2, tb, td;
  int rc;
  ka.k_split = 0;
  // A: K-major = [M rows, K cols], box {64(k), 128(m)};  MN-major = [K rows, M cols], box {64(m), 64(k)}
  if (a->A2 != nullptr) {
    // A = [A | A2] concatenated along K at k_split (K-major only; split on a k-block boundary)
    if (a->a_mn_major || a->k_split <= 0 || a->k_split >= a->K || (a->k_split % BK) != 0) return MMSUM_ERR_INVALID;
    ka.k_split = a->k_split;
    rc = make_tmap(&ta, a->A, 0, (uint64_t)a->k_split, (uint64_t)a->M, (uint64_t)a->lda * 2, 64, BM);
    if (rc) return rc;
    rc = make_tmap(&ta2, a->A2, 0, (uint64_t)(a->K - a->k_split), (uint64_t)a->M, (uint64_t)a->lda2 * 2, 64, BM);
  } else {
    if (a->a_mn_major) rc = make_tmap(&ta, a->A, 0, (uint64_t)a->M, (uint64_t)a->K, (uint64_t)a->lda * 2, 64, 64);
    else               rc = make_tmap(&ta, a->A, 0, (uint64_t)a->K, (uint64_t)a->M, (uint64_t)a->lda * 2, 64, BM);
    ta2 = ta;
  }
  if (rc) return rc;
  // CTA pairs (cta_group::2) for problems that fill the machine with 256-wide tiles: +11-15 % on the step's large shapes
  // (profiles/r02_gemm_2sm_ab.txt).  MMSUM_GEMM_CLUSTER=0 switches back to single-CTA tiles for the A/B.
  static const bool cluster_off = [] { const char* e = getenv("MMSUM_GEMM_CLUSTER"); return e && e[0] == '0'; }();
  const int nsm = num_sms();
  const long long pairs = (long long)((ka.m_tiles + 1) / 2) * ka.n_tiles * ka.splits;
  const int cl = (!cluster_off && bn == 256 && ka.m_tiles >= 2 && pairs * 2 >= nsm && (nsm % 2) == 0) ? 2 : 1;
  if (a->b_mn_major) rc = make_tmap(&tb, a->B, 0, (uint64_t)a->N, (uint64_t)a->K, (uint64_t)a->ldb * 2, 64, 64);
  else               rc = make_tmap(&tb, a->B, 0, (uint64_t)a->K, (uint64_t)a->N, (uint64_t)a->ldb * 2, 64, (uint32_t)(bn / cl));
  if (rc) return rc;
  if (ws_mode)    rc = make_tmap(&td, ws, 1, (uint64_t)a->N, (uint64_t)(ka.ws_rows * ka.splits), (uint64_t)ldw * 4, 32, 32);
  else if (a->out_f32) rc = make_tmap(&td, a->D, 1, (uint64_t)a->N, (uint64_t)a->M, (uint64_t)a->ldd * 4, 32, 32);
  else            rc = make_tmap(&td, a->D, 0, (uint64_t)a->N, (uint64_t)a->M, (uint64_t)a->ldd * 2, 64, 32);
  if (rc) return rc;
  CUtensorMap taux = td;   // pre-activation copy (aux_mode 1) leaves through its own map, same tiling as D
  if (a->aux_mode == 1 || a->aux_mode == 3) {
    rc = make_tmap(&taux, a->aux, 0, (uint64_t)a->N, (uint64_t)a->M, (uint64_t)a->ld_aux * 2, 64, 32);
    if (rc) return rc;
  }

  if (ka.splits > 1 && (a->act != 0 || a->aux_mode != 0)) return MMSUM_ERR_INVALID;
  if (a->out_f32 && (a->act == 1 || a->aux_mode != 0)) return MMSUM_ERR_INVALID;   // fused activations are bf16-output only
  const int total = ka.m_tiles * ka.n_tiles * ka.splits;
  int grid = total < nsm ? total : nsm;
  if (cl == 2) grid = (int)(pairs * 2 < nsm ? pairs * 2 : nsm);
  const int am = a->a_mn_major ? 1 : 0, bm = a->b_mn_major ? 1 : 0;
  // aux modes 3 / 4 share the kernels of 1 / 2; EPI 3 = ordered split-K partials
  const int epi = ws_mode ? 3 : ((a->aux_mode == 3) ? 1 : (a->aux_mode == 4 ? 2 : a->aux_mode));
  if (ws_mode) {
    if (int rc2 = launch_gemm_case(bn, am, bm, epi, cl, ta, ta2, tb, td, taux, ka, grid, stream)) return rc2;
    const long long n_el = (long long)a->M * a->N;
    const long long rblocks = (n_el + 255) / 256;
    const int rgrid = (int)(rblocks < (long long)nsm * 8 ? rblocks : (long long)nsm * 8);
    splitk_ordered_reduce_kernel<<<rgrid, 256, 0, stream>>>(ws, ka.splits, split_stride, ldw, reinterpret_cast<float*>(a->D),
                                                             a->ldd, a->M, a->N);
    MMSUM_CHECK_LAUNCH();
    return 0;
  }
  return launch_gemm_case(bn, am, bm, epi, cl, ta, ta2, tb, td, taux, ka, grid, stream);
}

static int launch_gemm_case(int bn, int am, int bm, int epi, int cl, const CUtensorMap& ta, const CUtensorMap& ta2,
                            const CUtensorMap& tb, const CUtensorMap& td, const CUtensorMap& taux, const GemmKernelArgs& ka,
                            int grid, cudaStream_t stream) {
#define MMSUM_GEMM_CASE(BN_, AM_, BM_, EPI_, CL_) \
  if (bn == BN_ && am == AM_ && bm == BM_ && epi == EPI_ && cl == CL_) \
    return launch_gemm<BN_, (AM_ != 0), (BM_ != 0), EPI_, CL_>(ta, ta2, tb, td, taux, ka, grid, stream);
  MMSUM_GEMM_CASE(256, 0, 0, 0, 2)
  MMSUM_GEMM_CASE(256, 0, 1, 0, 2)
  MMSUM_GEMM_CASE(256, 1, 1, 0, 2)
  MMSUM_GEMM_CASE(256, 1, 0, 0, 2)
  MMSUM_GEMM_CASE(256, 0, 0, 1, 2)
  MMSUM_GEMM_CASE(256, 0, 1, 1, 2)
  MMSUM_GEMM_CASE(256, 0, 0, 2, 2)
  MMSUM_GEMM_CASE(256, 0, 1, 2, 2)
  MMSUM_GEMM_CASE(256, 0, 0, 0, 1)
  MMSUM_GEMM_CASE(256, 0, 1, 0, 1)
  MMSUM_GEMM_CASE(256, 1, 1, 0, 1)
  MMSUM_GEMM_CASE(256, 1, 0, 0, 1)
  MMSUM_GEMM_CASE(128, 0, 0, 0, 1)
  MMSUM_GEMM_CASE(128, 0, 1, 0, 1)
  MMSUM_GEMM_CASE(128, 1, 1, 0, 1)
  MMSUM_GEMM_CASE(128, 1, 0, 0, 1)
  // fused-activation epilogues: row-major A (the Linear fprop / dgrad operands), 256-wide tiles
  MMSUM_GEMM_CASE(256, 0, 0, 1, 1)
  MMSUM_GEMM_CASE(256, 0, 1, 1, 1)
  MMSUM_GEMM_CASE(256, 0, 0, 2, 1)
  MMSUM_GEMM_CASE(256, 0, 1, 2, 1)
  // ordered split-K partials (fp32 output, plain epilogue)
  MMSUM_GEMM_CASE(256, 0, 0, 3, 2)
  MMSUM_GEMM_CASE(256, 0, 1, 3, 2)
  MMSUM_GEMM_CASE(256, 1, 1, 3, 2)
  MMSUM_GEMM_CASE(256, 1, 0, 3, 2)
  MMSUM_GEMM_CASE(256, 0, 0, 3, 1)
  MMSUM_GEMM_CASE(256, 0, 1, 3, 1)
  MMSUM_GEMM_CASE(256, 1, 1, 3, 1)
  MMSUM_GEMM_CASE(256, 1, 0, 3, 1)
  MMSUM_GEMM_CASE(128, 0, 0, 3, 1)
  MMSUM_GEMM_CASE(128, 0, 1, 3, 1)
  MMSUM_GEMM_CASE(128, 1, 1, 3, 1)
  MMSUM_GEMM_CASE(128, 1, 0, 3, 1)
#undef MMSUM_GEMM_CASE
  return MMSUM_ERR_INVALID;
}

extern "C" int mmsum_gemm_bf16(const MmsumGemmArgs* a, void* stream) {
  return gemm_impl(a, reinterpret_cast<cudaStream_t>(stream), false, nullptr, 0, nullptr);
}

extern "C" int mmsum_gemm_bf16_ordered(const MmsumGemmArgs* a, float* workspace, int64_t workspace_elems, void* stream) {
  return gemm_impl(a, reinterpret_cast<cudaStream_t>(stream), true, workspace, workspace_elems, nullptr);
}

extern "C" int mmsum_gemm_ordered_workspace(const MmsumGemmArgs* a, int64_t* elems) {
  if (!elems) return MMSUM_ERR_INVALID;
  return gemm_impl(a, nullptr, true, nullptr, 0, elems);
}
