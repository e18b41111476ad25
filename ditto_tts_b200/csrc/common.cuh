// Shared device/host helpers for libditto_b200 (sm_100a only).
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include <atomic>
#include <string>

#include "../../include/ditto_b200.h"

#if defined(__CUDA_ARCH__) && !defined(__CUDA_ARCH_FEAT_SM100_ALL) && !defined(__CUDA_ARCH_FEAT_SM103_ALL)
#error "libditto_b200 must be compiled for sm_100a (-gencode arch=compute_100a,code=sm_100a)"
#endif

#ifndef DITTO_F7_TRACE   // developer timeline of the flash768 kernels (F7Tr below), off by default
#define DITTO_F7_TRACE 0
#endif

namespace ditto {

typedef __nv_bfloat16 bf16;

// ---------------------------------------------------------------- host-side error plumbing
void set_error(const std::string& msg);
int cuda_fail(cudaError_t err, const char* what, const char* file, int line);
extern std::atomic<long long> g_launches;
inline void count_launch(int n = 1) { g_launches.fetch_add(n, std::memory_order_relaxed); }

#define DITTO_CUDA(call)                                                         \
  do {                                                                           \
    cudaError_t _e = (call);                                                     \
    if (_e != cudaSuccess) return ::ditto::cuda_fail(_e, #call, __FILE__, __LINE__); \
  } while (0)

#define DITTO_LAUNCH_CHECK()                                                     \
  do {                                                                           \
    ::ditto::count_launch();                                                     \
    cudaError_t _e = cudaPeekAtLastError();                                      \
    if (_e != cudaSuccess) return ::ditto::cuda_fail(_e, "kernel launch", __FILE__, __LINE__); \
  } while (0)

#define DITTO_REQUIRE(cond, code, msg)                                           \
  do {                                                                           \
    if (!(cond)) {                                                               \
      ::ditto::set_error(std::string(msg) + " [" #cond "]");                     \
      return (code);                                                             \
    }                                                                            \
  } while (0)

#define DITTO_TRY(expr)                                                          \
  do {                                                                           \
    int _rc = (expr);                                                            \
    if (_rc != 0) return _rc;                                                    \
  } while (0)

// ---------------------------------------------------------------- per-kernel-class timing (CUDA events, opt-in)
enum ProfClass {
  PC_TC_PROJ_IN = 0, PC_TC_QKV, PC_TC_SELF_SCORES, PC_TC_SELF_PV, PC_TC_CROSS_Q, PC_TC_CROSS_SCORES, PC_TC_CROSS_PV,
  PC_TC_CROSS_OUT, PC_TC_GLU, PC_TC_FC2, PC_TC_PROJ_OUT, PC_TC_TEXT_KV, PC_TC_OTHER,
  PC_SGEMM, PC_LAYERNORM, PC_ADALN, PC_ROPE, PC_SOFTMAX, PC_CFG_UPDATE, PC_ELEMENTWISE, PC_TC_CROSS_FUSED, PC_FLASH_ATTN, PC_FLASH768,
  PC_CROSS_FLASH, PC_COUNT
};
extern bool g_prof_enabled;
struct ProfScope {  // records start/stop events around the launches issued in its lifetime (no-op unless enabled)
  int slot = -1;
  cudaStream_t st;
  ProfScope(int cls, cudaStream_t stream, double flops, double bytes);
  ~ProfScope();
};

inline int64_t ceil_div(int64_t a, int64_t b) { return (a + b - 1) / b; }
inline int64_t round_up(int64_t a, int64_t b) { return ceil_div(a, b) * b; }

// ---------------------------------------------------------------- device helpers
#ifdef __CUDACC__

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

__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
  __nv_bfloat162 p = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&p);
}
__device__ __forceinline__ float2 unpack_bf16x2(uint32_t u) {
  __nv_bfloat162 p = *reinterpret_cast<__nv_bfloat162*>(&u);
  return __bfloat1622float2(p);
}

__device__ __forceinline__ float silu_f(float x) { return x / (1.0f + __expf(-x)); }
// exact-erf GELU, nn.GELU() default (DiT.py:96)
__device__ __forceinline__ float gelu_erf_f(float x) { return 0.5f * x * (1.0f + erff(x * 0.70710678118654752440f)); }
__device__ __forceinline__ float sigmoid_f(float x) { return 1.0f / (1.0f + __expf(-x)); }

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return static_cast<uint32_t>(__cvta_generic_to_shared(p)); }

// ---- warp-uniform control (single-thread-issue roles) ----------------------------------------------
// tcgen05.mma / cp.async.bulk.tensor / tcgen05.commit take their operands from UNIFORM registers.  When the issuing code sits
// inside `if (lane == 0)`, every operand lives in a vector register of a divergent region and the compiler wraps each
// instruction in a "waterfall" (ELECT + five R2UR.BROADCAST + loop): ~21 SASS instructions per MMA, more than a 64- or
// 128-cycle MMA lasts -- the issuer, not the tensor pipe, paced the kernels (ncu: 33 % tensor-active in flash_attn768 with the
// issuing warp never waiting on a barrier).  Instead the WHOLE warp runs the role's loops on provably warp-uniform values
// (warp index through a shuffle, constants, kernel parameters) and one elected lane executes the instruction.
__device__ __forceinline__ int warp_id_uniform() { return __shfl_sync(0xffffffffu, static_cast<int>(threadIdx.x >> 5), 0); }
__device__ __forceinline__ bool elect_one() {   // one lane of the (fully converged) warp
  uint32_t pred;
  asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
  return pred != 0;
}

// ---- mbarrier ------------------------------------------------------------------------------------
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
// Bounded wait (~4 s of SM clock): a protocol bug traps (-> cudaErrorLaunchFailure) instead of hanging the box.  No printf:
// a call in the spin loop makes every wait an ABI call site and spills the 56-register control warps.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  if (mbar_try_wait(bar, parity)) return;
  const long long start = clock64();
  uint32_t spins = 0;
  while (!mbar_try_wait(bar, parity)) {
    if ((++spins & 0x3FFu) == 0 && clock64() - start > 8000000000ll) __trap();
  }
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// ---- TMA -----------------------------------------------------------------------------------------
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* m) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
}
// 4-D tiled load global -> shared, completion on an mbarrier (complete_tx::bytes).
__device__ __forceinline__ void tma_load_4d(const CUtensorMap* m, uint64_t* bar, void* smem, int c0, int c1, int c2,
                                            int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
      ::"r"(smem_u32(smem)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}

// ---- tcgen05 / TMEM --------------------------------------------------------------------------------
__device__ __forceinline__ void tcgen05_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tcgen05_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

template <int kCols>
__device__ __forceinline__ void tmem_alloc(uint32_t* dst_smem) {  // one full warp
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "n"(kCols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
template <int kCols>
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr) {  // same warp that allocated
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "n"(kCols) : "memory");
}

// D[tmem] (+)= A[smem desc] * B[smem desc]; bf16 x bf16 -> fp32, issued by ONE thread.
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                          uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// mbarrier arrive once all previously issued tcgen05.mma of this thread have completed
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}
// ... on the barrier at this offset in every CTA of `mask` (cluster ranks)
__device__ __forceinline__ void umma_commit_mc(uint64_t* bar, uint16_t mask) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(smem_u32(bar)),
               "h"(mask)
               : "memory");
}

// ---- cta_group::2 (one SM pair = CTAs 2k, 2k+1 of a cluster; the even CTA issues) -------------------
constexpr uint32_t kPeerBitMask = 0xFEFFFFFFu;  // shared::cluster address of the same offset in the even CTA of the pair

__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// shared::cluster address of the same shared-memory offset in the CTA of cluster rank `rank`
__device__ __forceinline__ uint32_t mapa_shared(uint32_t addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
  return r;
}
// remote shared-memory store that signals the destination CTA's mbarrier with complete_tx (4 or 8 bytes): data and
// notification travel together through the async proxy, so the sender needs no release fence (a release-scoped arrive
// would first have to drain this thread's outstanding global stores).
__device__ __forceinline__ void st_async_f32(uint32_t remote_addr, float v, uint32_t remote_bar) {
  asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.b32 [%0], %1, [%2];" ::"r"(remote_addr),
               "r"(__float_as_uint(v)), "r"(remote_bar)
               : "memory");
}
__device__ __forceinline__ void st_async_f32x2(uint32_t remote_addr, float a, float b, uint32_t remote_bar) {
  asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.v2.b32 [%0], {%1, %2}, [%3];" ::"r"(remote_addr),
               "r"(__float_as_uint(a)), "r"(__float_as_uint(b)), "r"(remote_bar)
               : "memory");
}
// shared::cta -> peer's shared memory, completion (complete_tx) on the peer's mbarrier
__device__ __forceinline__ void bulk_copy_to_peer(uint32_t remote_dst, uint32_t local_src, uint32_t bytes, uint32_t remote_bar) {
  asm volatile("cp.async.bulk.shared::cluster.shared::cta.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(remote_dst),
               "r"(local_src), "r"(bytes), "r"(remote_bar)
               : "memory");
}
// TMA load into this CTA's shared memory; the bytes are counted on the PAIR LEADER's copy of `bar`
__device__ __forceinline__ void tma_load_4d_2sm(const CUtensorMap* m, uint64_t* bar, void* smem, int c0, int c1, int c2, int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
      ::"r"(smem_u32(smem)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar) & kPeerBitMask), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}
__device__ __forceinline__ void umma_bf16_2sm(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, {%5, %5, %5, %5, %5, %5, %5, %5}, p;\n\t}"
      ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate), "r"(0u)
      : "memory");
}
// arrive (once the issued MMAs retire) on the barrier at this offset in every CTA of `mask` (cluster ranks)
__device__ __forceinline__ void umma_commit_2sm_mc(uint64_t* bar, uint16_t mask) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
               ::"r"(smem_u32(bar)), "h"(mask)
               : "memory");
}
// ... in BOTH CTAs of the pair that forms a two-CTA cluster
__device__ __forceinline__ void umma_commit_2sm(uint64_t* bar) { umma_commit_2sm_mc(bar, static_cast<uint16_t>(3)); }
__device__ __forceinline__ void mbar_arrive_leader(uint64_t* bar) {  // arrive on the leader CTA's copy of `bar`
  asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(smem_u32(bar) & kPeerBitMask) : "memory");
}
// the same with cluster-scope release: what the arriving thread wrote (shared memory, TMEM after tcgen05.wait::st) is
// visible to the leader CTA's thread that observes the phase with mbar_wait_cluster
__device__ __forceinline__ void mbar_arrive_leader_release(uint64_t* bar) {
  asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(smem_u32(bar) & kPeerBitMask) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait_cluster(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ void mbar_wait_cluster(uint64_t* bar, uint32_t parity) {   // bounded like mbar_wait
  if (mbar_try_wait_cluster(bar, parity)) return;
  const long long start = clock64();
  uint32_t spins = 0;
  while (!mbar_try_wait_cluster(bar, parity)) {
    if ((++spins & 0x3FFu) == 0 && clock64() - start > 8000000000ll) __trap();
  }
}

// 32 lanes x 32 consecutive fp32 columns: thread i of the warp gets TMEM lane (lane_base + i).
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
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// UMMA shared-memory matrix descriptor (cute::UMMA::SmemDescriptor, mma_sm100_desc.hpp):
// [0,14) start>>4 | [16,30) LBO>>4 | [32,46) SBO>>4 | [46,48) version=1 | [61,64) layout (2 = SWIZZLE_128B)
__device__ __forceinline__ uint64_t umma_smem_desc(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((smem_addr & 0x3FFFFu) >> 4);
  d |= static_cast<uint64_t>((lbo_bytes >> 4) & 0x3FFFu) << 16;
  d |= static_cast<uint64_t>((sbo_bytes >> 4) & 0x3FFFu) << 32;
  d |= static_cast<uint64_t>(1) << 46;
  d |= static_cast<uint64_t>(2) << 61;
  return d;
}
// UMMA instruction descriptor, kind::f16 (cute::UMMA::InstrDescriptor): D=f32, A=B=bf16.
__host__ __device__ constexpr uint32_t umma_idesc_bf16(int M, int N, bool a_mn_major, bool b_mn_major) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((a_mn_major ? 1u : 0u) << 15) | ((b_mn_major ? 1u : 0u) << 16) |
         (static_cast<uint32_t>(N >> 3) << 17) | (static_cast<uint32_t>(M >> 4) << 24);
}


// ---- epilogue helpers shared by the tcgen05 kernels (gemm_tc.cu, cross_fused.cu) -------------------
__device__ __forceinline__ float quad_max(float v) {
  v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, 1));
  return fmaxf(v, __shfl_xor_sync(0xffffffffu, v, 2));
}
__device__ __forceinline__ float quad_sum(float v) {
  v += __shfl_xor_sync(0xffffffffu, v, 1);
  return v + __shfl_xor_sync(0xffffffffu, v, 2);
}
// LayerNorm row statistics of the fused epilogues, free of the cancellation of E[v^2] - mean^2 (which loses the variance
// once |mean| / spread ~ 1e3).  A partial is (mean, M2 = sum (v - mean)^2) of n values.  A thread accumulates d = v - K and
// d^2 against its own first value K of the row, which keeps both sums at the scale of the row's spread, and turns them into
// a partial; partials of equal counts merge by Chan's pairwise formula.  ln_merge is symmetric in a and b, so every lane of
// a shuffle and both CTAs of an exchange get the same bits.
__device__ __forceinline__ float2 ln_partial(float K, float sd, float sdd, float inv_n) {
  const float m = sd * inv_n;
  return make_float2(K + m, fmaf(-sd, m, sdd));
}
// a, b: partials of n values each
__device__ __forceinline__ float2 ln_merge(float2 a, float2 b, float n) {
  const float d = b.x - a.x;
  return make_float2(0.5f * (a.x + b.x), (a.y + b.y) + d * d * (0.5f * n));
}
// merge of the four partials (n values each) of a lane quad; every lane gets the quad's partial of 4 n values
__device__ __forceinline__ float2 ln_quad_merge(float2 s, float n) {
  s = ln_merge(s, make_float2(__shfl_xor_sync(0xffffffffu, s.x, 1), __shfl_xor_sync(0xffffffffu, s.y, 1)), n);
  return ln_merge(s, make_float2(__shfl_xor_sync(0xffffffffu, s.x, 2), __shfl_xor_sync(0xffffffffu, s.y, 2)), 2.f * n);
}
__device__ __forceinline__ float ex2_approx(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float rcp_approx(float x) {
  float y;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
// tcgen05.ld.16x256b: a warp gets a 16-row x 64-column block of the accumulator in the mma-fragment layout -- thread t
// holds, for every 8-column block kb, columns kb*8 + (t%4)*2 + {0,1} of rows t/4 (r[4kb], r[4kb+1]) and t/4 + 8
// (r[4kb+2], r[4kb+3]).
__device__ __forceinline__ void tmem_ld_16x64(uint32_t taddr, uint32_t (&r)[32]) {  // 16 lanes x 64 fp32 columns
  asm volatile(
      "tcgen05.ld.sync.aligned.16x256b.x8.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_st_16x64(uint32_t taddr, const uint32_t (&r)[32]) {  // inverse of tmem_ld_16x64
  asm volatile(
      "tcgen05.st.sync.aligned.16x256b.x8.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
      "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};"
      ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]),
        "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]), "r"(r[16]), "r"(r[17]), "r"(r[18]), "r"(r[19]),
        "r"(r[20]), "r"(r[21]), "r"(r[22]), "r"(r[23]), "r"(r[24]), "r"(r[25]), "r"(r[26]), "r"(r[27]), "r"(r[28]), "r"(r[29]),
        "r"(r[30]), "r"(r[31])
      : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void prefetch_l2(const void* p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }

// Register re-distribution between the warp roles of the 384-thread tcgen05 kernels (setmaxnreg): warps 0-3 shrink, the two
// epilogue warpgroups grow.
constexpr int REGS_CTRL = 56, REGS_EPI = 224;
static_assert(128 * REGS_CTRL + 256 * REGS_EPI <= 65536, "register re-distribution exceeds the register file");
__device__ __forceinline__ void regs_shrink_ctrl() { asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(REGS_CTRL)); }
__device__ __forceinline__ void regs_grow_epi() { asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(REGS_EPI)); }

// Developer timeline of the two flash768 kernels (build with -DDITTO_F7_TRACE=1 through DITTO_NVCC_EXTRA;
// tools/f7_trace.py): cluster 0 records (tag, item-relative SM clock) pairs of its MMA issuer, TMA producer and first
// softmax warp into the buffer handed to ditto_debug_set_counters.  Compiled out by default.
constexpr int F7_TR_MAX = 512;   // events per (CTA, role)
constexpr int F7_TR_ROLES = 3;   // 0 MMA issuer, 1 softmax warp 0, 2 TMA producer
struct F7Tr {
  unsigned long long* b; int n; long long t0;
  __device__ __forceinline__ void init(unsigned long long* buf, int rank, int role, bool on, long long t_sync) {
    b = (DITTO_F7_TRACE && buf != nullptr && on) ? buf + (rank * F7_TR_ROLES + role) * F7_TR_MAX : nullptr; n = 0; t0 = t_sync;
  }
  __device__ __forceinline__ void ev(int kind, int j) {
    if (DITTO_F7_TRACE && b != nullptr && n < F7_TR_MAX)
      b[n++] = (static_cast<unsigned long long>(kind * 256 + (j & 255)) << 40) | (static_cast<unsigned long long>(clock64() - t0) & 0xFFFFFFFFFFull);
  }
  __device__ __forceinline__ void val(int kind, int j, long long v) {
    if (DITTO_F7_TRACE && b != nullptr && n < F7_TR_MAX)
      b[n++] = (static_cast<unsigned long long>(kind * 256 + (j & 255)) << 40) | (static_cast<unsigned long long>(v) & 0xFFFFFFFFFFull);
  }
};


#endif  // __CUDACC__
}  // namespace ditto
