// Shared device/host helpers for the mmsum_b200 kernels (sm_100a only).
// PTX wrappers for mbarrier / TMA / tcgen05, bf16 packing, a counter-based RNG
// for dropout, and warp reductions.  No torch types anywhere in csrc/.
#pragma once
#include <cstdlib>
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include <atomic>

#define MMSUM_OK 0
#define MMSUM_ERR_INVALID (-1)
#define MMSUM_ERR_DRIVER (-2)

// host: launch with the programmatic-stream-serialization attribute (the kernel must call pdl_wait() before touching
// global memory)
template <typename... KArgs, typename... Args>
static inline cudaError_t launch_pdl_cluster(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream,
                                             int cluster_x, Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = stream;
  cudaLaunchAttribute attr[2];
  int n = 0;
  static const bool off = (getenv("MMSUM_NO_PDL") != nullptr);   // A/B switch for measurements
  if (!off) {
    attr[n].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[n].val.programmaticStreamSerializationAllowed = 1;
    ++n;
  }
  if (cluster_x > 1) {
    attr[n].id = cudaLaunchAttributeClusterDimension;
    attr[n].val.clusterDim.x = (unsigned)cluster_x; attr[n].val.clusterDim.y = 1; attr[n].val.clusterDim.z = 1;
    ++n;
  }
  cfg.attrs = attr; cfg.numAttrs = n;
  return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}
template <typename... KArgs, typename... Args>
static inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream,
                                     Args&&... args) {
  return launch_pdl_cluster(kernel, grid, block, smem, stream, 1, static_cast<Args&&>(args)...);
}

#define MMSUM_LAUNCH_PDL(kernel, grid, block, smem, stream, ...)                                          \
  do {                                                                                                   \
    cudaError_t _le = launch_pdl(kernel, dim3(grid), dim3(block), (size_t)(smem), stream, __VA_ARGS__);  \
    if (_le != cudaSuccess) return (int)_le;                                                             \
  } while (0)

// One-time opt-in to > 48 KB of dynamic shared memory, tracked PER DEVICE (bit d of `done`) and safe to race: the attribute
// call is idempotent, the flag is only an optimisation.
template <typename K>
static inline int ensure_dyn_smem(K kernel, int bytes, std::atomic<unsigned long long>& done) {
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return MMSUM_ERR_DRIVER;
  const unsigned long long bit = 1ull << (dev & 63);
  if (done.load(std::memory_order_acquire) & bit) return 0;
  cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
  if (e != cudaSuccess) return (int)e;
  done.fetch_or(bit, std::memory_order_release);
  return 0;
}

#define MMSUM_CHECK_LAUNCH()                         \
  do {                                               \
    cudaError_t _e = cudaGetLastError();             \
    if (_e != cudaSuccess) return (int)_e;           \
  } while (0)

namespace mmsum {

typedef __nv_bfloat16 bf16;
typedef __nv_bfloat162 bf162;

static constexpr int kNumSMs = 148;

// ----------------------------------------------------------------------------
// small math / packing helpers
// ----------------------------------------------------------------------------
__device__ __forceinline__ uint32_t pack_bf16(float lo, float hi) {
  bf162 v = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&v);
}
__device__ __forceinline__ float2 unpack_bf16(uint32_t u) {
  bf162 v = *reinterpret_cast<bf162*>(&u);
  return __bfloat1622float2(v);
}
__device__ __forceinline__ float bf16_round(float x) { return __bfloat162float(__float2bfloat16_rn(x)); }

// erf via Abramowitz-Stegun 7.1.26 (|abs err| <= 1.5e-7, far below the bf16 rounding of every consumer): one MUFU.RCP,
// one MUFU.EX2 and a degree-5 Horner chain instead of libdevice erff (~3x the instructions; the GELU epilogues of the
// fc1 GEMMs were ALU-bound on it).  E = exp(-x^2/2) = exp(-z^2) is shared with the Gaussian pdf term of GELU'.  An FMA-only
// polynomial erf measured slower (DESIGN.md §3): the epilogue is issue-bound on the FMA pipe, and the two MUFU operations of
// this form run beside it for free.
__device__ __forceinline__ float fast_ex2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float fast_rcp(float x) {
  float y;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
// Blackwell packed fp32 pairs (FFMA2 / FMUL2): one issue slot for two lanes of the same elementwise chain.
struct f32x2 { uint64_t r; };
__device__ __forceinline__ f32x2 pack2(float a, float b) { f32x2 o; asm("mov.b64 %0, {%1, %2};" : "=l"(o.r) : "f"(a), "f"(b)); return o; }
__device__ __forceinline__ f32x2 splat2(float a) { return pack2(a, a); }
__device__ __forceinline__ void unpack2(f32x2 v, float& a, float& b) { asm("mov.b64 {%0, %1}, %2;" : "=f"(a), "=f"(b) : "l"(v.r)); }
__device__ __forceinline__ f32x2 fma2(f32x2 a, f32x2 b, f32x2 c) { f32x2 o; asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(o.r) : "l"(a.r), "l"(b.r), "l"(c.r)); return o; }
__device__ __forceinline__ f32x2 mul2(f32x2 a, f32x2 b) { f32x2 o; asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(o.r) : "l"(a.r), "l"(b.r)); return o; }
__device__ __forceinline__ f32x2 add2(f32x2 a, f32x2 b) { f32x2 o; asm("add.rn.f32x2 %0, %1, %2;" : "=l"(o.r) : "l"(a.r), "l"(b.r)); return o; }

// erf(x / sqrt(2)) for a pair; E = exp(-x*x/2)
__device__ __forceinline__ f32x2 erf_as2(float x0, float x1, f32x2 x, f32x2& E) {
  const f32x2 z = pack2(fabsf(x0), fabsf(x1));
  f32x2 d = fma2(z, splat2(0.3275911f * 0.70710678118654752f), splat2(1.f));
  float d0, d1; unpack2(d, d0, d1);
  const f32x2 t = pack2(fast_rcp(d0), fast_rcp(d1));
  const f32x2 a = mul2(x, mul2(x, splat2(-0.72134752044448170f)));
  float a0, a1; unpack2(a, a0, a1);
  E = pack2(fast_ex2(a0), fast_ex2(a1));
  f32x2 q = fma2(t, splat2(1.061405429f), splat2(-1.453152027f));
  q = fma2(q, t, splat2(1.421413741f));
  q = fma2(q, t, splat2(-0.284496736f));
  q = fma2(q, t, splat2(0.254829592f));
  q = mul2(q, t);
  const f32x2 e = fma2(mul2(q, splat2(-1.f)), E, splat2(1.f));
  float e0, e1; unpack2(e, e0, e1);
  return pack2(copysignf(e0, x0), copysignf(e1, x1));
}
__device__ __forceinline__ void gelu_erf2(float& x0, float& x1) {
  const f32x2 x = pack2(x0, x1);
  f32x2 E;
  const f32x2 e = erf_as2(x0, x1, x, E);
  const f32x2 hx = mul2(x, splat2(0.5f));
  unpack2(fma2(hx, e, hx), x0, x1);
}
// GELU and its derivative from one erf / exp evaluation: x := GELU(x), d := GELU'(x)  (the derivative is what the fused fc1
// epilogue saves for backward, so the fc2-dgrad epilogue is a single multiply)
__device__ __forceinline__ void gelu_erf_and_grad2(float& x0, float& x1, float& d0, float& d1) {
  const f32x2 x = pack2(x0, x1);
  f32x2 E;
  const f32x2 e = erf_as2(x0, x1, x, E);
  const f32x2 cdf = fma2(e, splat2(0.5f), splat2(0.5f));
  unpack2(fma2(x, mul2(E, splat2(0.3989422804014327f)), cdf), d0, d1);
  unpack2(mul2(x, cdf), x0, x1);
}
// (g0, g1) *= GELU'(x0), GELU'(x1)
__device__ __forceinline__ void gelu_erf_grad_mul2(float& g0, float& g1, float x0, float x1) {
  const f32x2 x = pack2(x0, x1);
  f32x2 E;
  const f32x2 e = erf_as2(x0, x1, x, E);
  const f32x2 cdf = fma2(e, splat2(0.5f), splat2(0.5f));
  const f32x2 d = fma2(x, mul2(E, splat2(0.3989422804014327f)), cdf);
  unpack2(mul2(pack2(g0, g1), d), g0, g1);
}

// Programmatic dependent launch: a kernel launched with launch_pdl() may begin (set-up only) while its predecessor on the
// stream is still draining; pdl_wait() blocks until the predecessor grid has completed and its writes are visible, so it
// must precede every global-memory access.  pdl_launch_dependents() lets the successor's CTAs be scheduled as SMs free up.
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// ----------------------------------------------------------------------------
// Counter-based RNG for dropout: keep-decision is a pure function of
// (seed, stream id, element index), so forward and backward regenerate the same
// mask without storing it.  (PyTorch's Philox stream cannot be matched — parity
// is defined at dropout 0, SURVEY App. D Q9.)
// ----------------------------------------------------------------------------
// 32-bit integer hash (two multiply-xorshift rounds): ~8 ALU instructions per call; the 64-bit murmur finaliser used
// before made the LayerNorm kernels ALU-bound (two 64-bit multiplies per pair of elements).
__device__ __forceinline__ uint32_t hash_u32(uint32_t h) {
  h ^= h >> 16; h *= 0x21f0aaadu;
  h ^= h >> 15; h *= 0x735a2d97u;
  h ^= h >> 15;
  return h;
}
__device__ __forceinline__ uint32_t dropout_rand(uint64_t seed, uint32_t stream, uint64_t idx) {
  const uint32_t key = (uint32_t)seed ^ (uint32_t)(seed >> 32) ^ (stream * 0x9E3779B1u) ^ ((uint32_t)(idx >> 32) * 0x85EBCA77u);
  return hash_u32((uint32_t)idx * 0x9E3779B1u + key);
}
// keep decision for element idx with keep threshold thr = (uint32)(keep_prob * 2^32)
__device__ __forceinline__ bool dropout_keep(uint64_t seed, uint32_t stream, uint64_t idx, uint32_t thr) {
  return dropout_rand(seed, stream, idx) < thr;
}

// ----------------------------------------------------------------------------
// shared-memory address + mbarrier
// ----------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
// Bounded wait: a protocol bug traps (kernel error) instead of hanging the GPU box.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  uint32_t spins = 0;
  while (!mbar_try_wait(bar, parity)) {
    if (++spins > (1u << 26)) {
      printf("mmsum: mbarrier timeout block %d thread %d\n", blockIdx.x, threadIdx.x);
      __trap();
    }
  }
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "elect.sync _|p, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(pred));
  return pred != 0;
}

// ----------------------------------------------------------------------------
// TMA (cp.async.bulk.tensor) 2D
// ----------------------------------------------------------------------------
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* m) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
}
__device__ __forceinline__ void tma_load_2d(void* smem_dst, const CUtensorMap* m, uint64_t* bar, int x, int y) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(x), "r"(y)
      : "memory");
}
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* m, const void* smem_src, int x, int y) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];"
               ::"l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(smem_src)), "r"(x), "r"(y)
               : "memory");
}
__device__ __forceinline__ void tma_reduce_add_2d(const CUtensorMap* m, const void* smem_src, int x, int y) {
  asm volatile("cp.reduce.async.bulk.tensor.2d.global.shared::cta.add.bulk_group [%0, {%2, %3}], [%1];"
               ::"l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(smem_src)), "r"(x), "r"(y)
               : "memory");
}
__device__ __forceinline__ void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void tma_store_wait_read() {
  asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}
template <int N>
__device__ __forceinline__ void tma_store_wait_all() {
  asm volatile("cp.async.bulk.wait_group %0;" ::"n"(N) : "memory");
}

// ----------------------------------------------------------------------------
// tcgen05 / TMEM
// ----------------------------------------------------------------------------
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_dst, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_dst)), "r"(ncols)
               : "memory");
}
__device__ __forceinline__ void tmem_relinquish() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// D[tmem] (+)= A[smem desc] * B[smem desc]; issued by ONE thread.
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// Warp-converged issue: the WHOLE warp runs the issue loop (so descriptors / coordinates stay in uniform registers and
// the loop is not a chain of R2UR conversions inside a divergent lane-0 branch — measured ~160 clk per issue that way),
// and only the lane chosen by elect.sync (inside the same asm block, so ptxas knows it is a single lane) executes it.
__device__ __forceinline__ void umma_bf16_w(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p, e;\n\t"
      "elect.sync _|e, 0xffffffff;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "@e tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma_commit_w(uint64_t* bar) {
  asm volatile(
      "{\n\t.reg .pred e;\n\t"
      "elect.sync _|e, 0xffffffff;\n\t"
      "@e tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n\t}"
      ::"r"(smem_u32(bar))
      : "memory");
}
__device__ __forceinline__ void mbar_expect_tx_w(uint64_t* bar, uint32_t bytes) {
  asm volatile(
      "{\n\t.reg .pred e;\n\t"
      "elect.sync _|e, 0xffffffff;\n\t"
      "@e mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n\t}"
      ::"r"(smem_u32(bar)), "r"(bytes)
      : "memory");
}
__device__ __forceinline__ void tma_load_2d_w(void* smem_dst, const CUtensorMap* m, uint64_t* bar, int x, int y) {
  asm volatile(
      "{\n\t.reg .pred e;\n\t"
      "elect.sync _|e, 0xffffffff;\n\t"
      "@e cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];\n\t}"
      ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(x), "r"(y)
      : "memory");
}
// ---- thread-block clusters (CTA pairs sharing an operand through TMA multicast)
__device__ __forceinline__ uint32_t cluster_ctarank() { uint32_t r; asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r)); return r; }
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// TMA load delivered to the same shared-memory offset of every CTA in `mask`; each destination CTA's mbarrier at the same
// offset receives the complete_tx for the bytes that land in ITS shared memory
__device__ __forceinline__ void tma_load_2d_mc_w(void* smem_dst, const CUtensorMap* m, uint64_t* bar, int x, int y, uint16_t mask) {
  asm volatile(
      "{\n\t.reg .pred e;\n\t"
      "elect.sync _|e, 0xffffffff;\n\t"
      "@e cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster [%0], [%1, {%3, %4}], [%2], %5;\n\t}"
      ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(x), "r"(y), "h"(mask)
      : "memory");
}
// tcgen05.commit that arrives on the mbarrier at the same offset in every CTA of `mask`
__device__ __forceinline__ void umma_commit_mc_w(uint64_t* bar, uint16_t mask) {
  asm volatile(
      "{\n\t.reg .pred e;\n\t"
      "elect.sync _|e, 0xffffffff;\n\t"
      "@e tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;\n\t}"
      ::"r"(smem_u32(bar)), "h"(mask)
      : "memory");
}
// ---- CTA pairs (cta_group::2): one tcgen05.mma spans two SMs; issued by the leader (cluster rank 0) only
__device__ __forceinline__ uint32_t mapa_u32(uint32_t saddr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(saddr), "r"(rank));
  return r;
}
__device__ __forceinline__ void tmem_alloc2(uint32_t* smem_dst, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_dst)), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tmem_relinquish2() { asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_dealloc2(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
// D (M = 256: lanes 0..127 of BOTH CTAs' tensor memory) (+)= A B^T; A rows / B rows of the second half come from the peer's
// shared memory at the same offsets
__device__ __forceinline__ void umma_bf16_2sm_w(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p, e;\n\t"
      "elect.sync _|e, 0xffffffff;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "@e tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// arrives on the mbarrier at the same offset in every CTA of `mask` once all previously issued pair MMAs have retired
__device__ __forceinline__ void umma_commit_2sm_mc_w(uint64_t* bar, uint16_t mask) {
  asm volatile(
      "{\n\t.reg .pred e;\n\t"
      "elect.sync _|e, 0xffffffff;\n\t"
      "@e tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;\n\t}"
      ::"r"(smem_u32(bar)), "h"(mask)
      : "memory");
}
// TMA load into OWN shared memory whose completion bytes are signalled on an mbarrier given as a shared::cluster address
// (the leader CTA's barrier: the pair's MMA waits for both CTAs' operand halves on one barrier)
__device__ __forceinline__ void tma_load_2d_2sm_w(void* smem_dst, const CUtensorMap* m, uint32_t bar_cluster_addr, int x, int y) {
  asm volatile(
      "{\n\t.reg .pred e;\n\t"
      "elect.sync _|e, 0xffffffff;\n\t"
      "@e cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];\n\t}"
      ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(bar_cluster_addr), "r"(x), "r"(y)
      : "memory");
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t bar_cluster_addr) {
  asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(bar_cluster_addr) : "memory");
}
__device__ __forceinline__ uint32_t uniform_u32(uint32_t v) { return __shfl_sync(0xffffffffu, v, 0); }

// mbarrier arrives once all previously issued tcgen05.mma of this thread retire.
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// A operand from tensor memory (lane = row of A, 32-bit column = two consecutive bf16 K elements), B from shared memory
__device__ __forceinline__ void umma_bf16_ts_w(uint32_t tmem_d, uint32_t tmem_a, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p, e;\n\t"
      "elect.sync _|e, 0xffffffff;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "@e tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}"
      ::"r"(tmem_d), "r"(tmem_a), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// 32 lanes x 16 columns of 32-bit cells, registers -> tensor memory
__device__ __forceinline__ void tmem_st_32x16(uint32_t taddr, const uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};"
      ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]),
        "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
      : "memory");
}
__device__ __forceinline__ void tmem_st_32x8(uint32_t taddr, const uint32_t (&r)[8]) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};"
               ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7])
               : "memory");
}
__device__ __forceinline__ void tmem_st_32x4(uint32_t taddr, const uint32_t (&r)[4]) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x4.b32 [%0], {%1, %2, %3, %4};"
               ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3])
               : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// 32 lanes x 32 columns of fp32: thread t of the warp receives lane (base_lane+t), columns [col, col+32)
__device__ __forceinline__ void tmem_ld_32x32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}

// UMMA shared-memory matrix descriptor (SWIZZLE_128B, sm_100 "version 1").
//   bits [0,14)  start address >> 4      bits [16,30) leading byte offset >> 4
//   bits [32,46) stride byte offset >> 4 bits [46,48) version = 1   bits [61,64) layout (2 = SWIZZLE_128B)
__device__ __forceinline__ uint64_t umma_smem_desc_sw128(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr >> 4) & 0x3FFF);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}
// Instruction descriptor for kind::f16, BF16 x BF16 -> FP32.
//   [4,6) c_format=1(F32)  [7,10) a_format=1(BF16)  [10,13) b_format=1(BF16)
//   [15] a_major (0=K,1=MN)  [16] b_major  [17,23) N>>3  [24,29) M>>4
__host__ __device__ constexpr uint32_t umma_idesc_bf16(int M, int N, int a_mn_major, int b_mn_major) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)a_mn_major << 15) | ((uint32_t)b_mn_major << 16) |
         ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

// ----------------------------------------------------------------------------
// cp.async (per-thread global -> shared copies with no register dependency)
// ----------------------------------------------------------------------------
__device__ __forceinline__ void cp_async_4(uint32_t saddr, const void* gptr) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(saddr), "l"(gptr) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }

// 32 lanes x 16 columns of fp32
__device__ __forceinline__ void tmem_ld_32x16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}

// host: cached cuTensorMapEncodeTiled for a 2D row-major tensor [outer, inner] (dtype 0 = bf16, 1 = f32), 128B swizzle
int make_tmap(CUtensorMap* out, const void* ptr, int dtype, uint64_t inner, uint64_t outer, uint64_t ld_bytes,
              uint32_t box_inner, uint32_t box_outer);

}  // namespace mmsum
