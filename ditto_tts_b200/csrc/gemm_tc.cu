// bf16 GEMM on the 5th-generation tensor cores of sm_100a:
//   TMA (cp.async.bulk.tensor, 128B swizzle) -> 4-stage shared-memory ring -> tcgen05.mma (one elected thread,
//   UMMA 128x256x16) -> fp32 accumulators in TMEM (2 x 256 columns, double buffered) -> tcgen05.ld -> fused epilogue.
// Persistent: one CTA per SM loops over (batch, m, n) tiles, n fastest so that concurrently running CTAs share the
// A row-block in L2.  Warp roles: 0 = TMA producer, 1 = MMA issuer, 2 = TMEM allocator, 4..11 = epilogue.
//
// Epilogues (fused, so that no elementwise pass re-reads the GEMM output from HBM):
//   STORE     out = alpha*acc (+bias) (+fp32 residual), fp32 or bf16, optional extra bf16 copy
//   GEGLU     columns interleaved [fc1(16) | gate(16)]: hid = GELU_erf(a+ba) * sigmoid(g+bg)          (DiT.py:153-155)
//   QKV_ROPE  column-permuted q/k so that the RoPE partner (j, j+d/2) sits PD columns away in the tile  (DiT.py:52-72)
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <unordered_map>
#include <mutex>
#include <tuple>
#include <type_traits>

#include "kernels.cuh"

namespace ditto {

namespace {

// ditto_debug_set_counters(): the wait-cycle counters of the paired kernel cost registers in the 56-register control
// warps, so they are compiled in only with -DDITTO_DBG_COUNTERS=1 (the entry point stays, the counters read 0 otherwise)
#ifndef DITTO_DBG_COUNTERS
#define DITTO_DBG_COUNTERS 0
#endif
constexpr bool kDbgCounters = DITTO_DBG_COUNTERS != 0;

constexpr int BLOCK_M = 128;
constexpr int BLOCK_N = 256;
constexpr int BLOCK_K = 64;   // 64 bf16 = 128 B = one swizzle span
constexpr int UMMA_K = 16;
constexpr int STAGES = 4;
constexpr int A_STAGE_BYTES = BLOCK_M * BLOCK_K * 2;  // 16 KiB
constexpr int B_STAGE_BYTES = BLOCK_N * BLOCK_K * 2;  // 32 KiB
constexpr int STAGE_BYTES = A_STAGE_BYTES + B_STAGE_BYTES;
constexpr int NUM_THREADS = 384;
constexpr int EPI_WARP0 = 4;
constexpr int NUM_EPI_WARPS = 8;
constexpr int TMEM_COLS = 512;
constexpr int BARRIER_BYTES = 256;
constexpr int EPI_STAGE_BYTES = 32 * 32 * 4;  // per epilogue warp
constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + BARRIER_BYTES + 1024 /*align slack*/;
static_assert(SMEM_BYTES <= 232448, "exceeds the 227 KiB shared memory of an sm_100 CTA");

// kernel variants (template parameter EPI of the kernels); the public TcEpilogue maps onto them in launch_tc_gemm
enum KernelEpi {
  K_STORE_F32 = 0,        // fp32 out = alpha*acc + bias                      (N even)
  K_STORE_F32_RESID = 1,  // fp32 out = alpha*acc + bias + fp32 residual (+ bf16 copy), in place allowed   (N even)
  K_STORE_BF16 = 2,       // bf16 out = alpha*acc + bias                      (N even)
  K_STORE_GENERIC = 3,    // any combination / odd N: fully predicated slow path
  K_GEGLU = 4,
  K_QKV_ROPE = 5
};

struct DevParams {
  int M, N, K;
  int batch_inner, batch_outer;
  int m_tiles, n_tiles, num_tiles, num_kb;
  int a_bi, a_bo, b_bi, b_bo;  // which batch coordinates each operand consumes
  float alpha;
  const float* bias; long long sb_inner, sb_outer;
  void* out; int out_bf16;
  long long ldo, so_inner, so_outer;
  const float* resid;
  long long ldr, sr_inner, sr_outer, resid_row_mod;
  bf16* out2; long long ldo2;
  const float* rope_freq;
  int rope_half, rope_pd, seq_T, hidden;
  const int* rope_pos;  // optional [M] row -> position table (ragged batches); nullptr: position = row % seq_T
  int rope_fast;        // weights packed for the lean pd = 128 epilogue (TcGemmParams::rope_perm16)
  int glu_fast;         // [fc1; gate] rows packed for the lean GEGLU epilogue (TcGemmParams::glu_perm16)
  int out_perm4;        // fp32 + residual result in the 16-byte column order (TcGemmParams::out_perm4)
  const float* row_lsum; int row_lparts; long long sl_inner, sl_outer;  // optional per-row 1/sum scale (fast STORE paths)
  // Deferred LayerNorm (DiT.py:105,143,151 without a LayerNorm pass over HBM).
  //  producer (STORE_F32_RESID): besides the fp32 result and its bf16 copy (out2), every epilogue warp writes the
  //    (sum, sum of squares) of its 128-column slab of each row to stat_out[row][part]  (deterministic: no atomics);
  //  consumer (QKV_ROPE / GEGLU): A is the raw bf16 residual stream, the weights carry gamma (W' = W diag(gamma)), and
  //    LN(h) W^T + b = rstd (h W'^T) - rstd mean c + b',  c_n = sum_k W'_nk,  b' = b + W beta,  applied per row here.
  float2* stat_out; int stat_parts; long long stat_rows_outer; int stat_parts_item;
  const float2* ln_stat; int ln_parts; float ln_inv_h; const float* ln_c;
  // developer diagnostics (ditto_debug_set_counters): clock cycles, summed over CTAs, that the pair kernel's MMA issuer
  // spent [0] waiting for operands, [1] waiting for a free accumulator, [2] in total; the TMA producer [3] waiting for a
  // free ring slot, [4] in total.  nullptr = off.
  unsigned long long* dbg;
};

// ---------------------------------------------------------------------------------------------------
// epilogue math
// ---------------------------------------------------------------------------------------------------
// per-row LayerNorm coefficients from the producer's partial statistics: LN(h)_k = a h_k + nm  (before gamma / beta);
// eps 1e-5, biased variance (nn.LayerNorm).  stat == nullptr: identity (a = 1, nm = 0).
__device__ __forceinline__ void ln_row_coef(const float2* stat, int parts, long long row, bool ok, float inv_h, float& a, float& nm) {
  a = 1.f; nm = 0.f;
  if (stat == nullptr || !ok) return;
  const float2* sp = stat + row * parts;
  float s = 0.f, q = 0.f;
  for (int c = 0; c < parts; ++c) {
    const float2 v = __ldg(sp + c);
    s += v.x; q += v.y;
  }
  const float mean = s * inv_h;
  const float var = fmaxf(fmaf(-mean, mean, q * inv_h), 0.f);
  a = rsqrtf(var + 1e-5f);
  nm = -mean * a;
}

// cos/sin of a = float(pos) * inv_freq (the reference's fp32 angle, DiT.py:56-59) for |a| up to a few thousand radians:
// two-constant Cody-Waite reduction to [-pi, pi] (k * 6.28125 is exact), then the MUFU approximations (abs. error ~5e-7).
__device__ __forceinline__ void sincos_reduced(float a, float& s, float& c) {
  const float k = rintf(a * 0.15915494309189535f);
  float r = fmaf(k, -6.28125f, a);
  r = fmaf(k, -1.9353071795864769e-3f, r);
  s = __sinf(r);
  c = __cosf(r);
}

// GELU_erf(a) * sigmoid(g) with 3 MUFU ops (2x ex2, 1x rcp shared by both factors) and ~12 FP32 ops.
//   Phi(a) = 0.5 (1 + erf(a / sqrt 2)) ~= sigmoid(2 a s(a^2)), s = odd-polynomial fit of atanh(erf)/a on |a| <= 6
//   (|GELU error| <= 1.3e-5, 150x below the bf16 rounding of the result; the fp32 path uses erff).
//   out = a / ((1 + exp(-2 a s)) (1 + exp(-g)));  an overflowing exponential gives 1/inf = 0, never inf * 0.
__device__ __forceinline__ float geglu_fast(float a, float g) {
  const float ac = fminf(fmaxf(a, -6.0f), 6.0f);
  const float a2 = ac * ac;
  float sp = fmaf(a2, 2.377971153e-05f, 7.501817227e-04f);   // coefficients pre-multiplied by -2 log2(e)
  sp = fmaf(a2, sp, -1.060307563e-01f);
  sp = fmaf(a2, sp, -2.301608248e+00f);
  const float e1 = ex2_approx(ac * sp);                       // exp(-2 a s)
  const float e2 = ex2_approx(g * -1.4426950408889634f);      // exp(-g)
  return a * rcp_approx((1.0f + e1) * (1.0f + e2));
}

// ---------------------------------------------------------------------------------------------------
// Epilogue, register-direct: tcgen05.ld.16x256b hands each warp a 16-row x 64-column block of the accumulator in the
// classic mma-fragment layout -- thread t holds, for every 8-column block kb, columns kb*8 + (t%4)*2 + {0,1} of rows
// t/4 and t/4 + 8.  Four neighbouring threads therefore cover 32 contiguous bytes (fp32) of a row, so plain st.global
// writes whole 32-B sectors; no shared-memory staging (the UMMA operand reads own the smem bandwidth), the bias of a
// column pair is loaded once for all rows, and RoPE / GLU partners (a multiple of 8 columns apart) sit in the same thread.
// ---------------------------------------------------------------------------------------------------
// Residual fragment of one 16 x 64 block in the accumulator-fragment layout: v[2*kb + rr] = columns
// (col0 + kb*8 + q2, +1) of row rowA + 8*rr.  Loaded BEFORE the matching TMEM load is waited for (and one block ahead of
// the stores), so that the global-load latency overlaps the MMA / the previous block's stores.  The residual may alias
// the output (in-place h += ...): every element is read and written by the same thread exactly once, so reading a later
// block early is safe.
struct ResFrag { float2 v[16]; };

__device__ __forceinline__ void load_resid_block(const DevParams& p, int lane, long long rowA, int col0, long long res_off,
                                                 ResFrag& f) {
  const int q2 = (lane & 3) * 2;
#pragma unroll
  for (int rr = 0; rr < 2; ++rr) {
    const long long row = rowA + rr * 8;
    const bool row_ok = row < p.M;
    const long long rrow =
        p.resid_row_mod > 0 ? static_cast<long long>(static_cast<unsigned>(row) % static_cast<unsigned>(p.resid_row_mod)) : row;
    const float* rp = p.resid + res_off + rrow * p.ldr + col0 + q2;
#pragma unroll
    for (int kb = 0; kb < 8; ++kb) {
      const int col = col0 + kb * 8 + q2;
      float2 t = make_float2(0.f, 0.f);
      if (row_ok && col + 1 < p.N) t = *reinterpret_cast<const float2*>(rp + kb * 8);
      else if (row_ok && col < p.N) t.x = rp[kb * 8];
      f.v[2 * kb + rr] = t;
    }
  }
}

__device__ __forceinline__ float2 load_bias2(const float* bias, int col, int N) {
  float2 b = make_float2(0.f, 0.f);
  if (bias != nullptr && col < N) {
    if (col + 1 < N) b = __ldg(reinterpret_cast<const float2*>(bias + col));  // read-only path: hoistable above stores
    else b.x = __ldg(bias + col);
  }
  return b;
}

// v = alpha * (a0, a1) + bias + resid for columns (col, col+1) of `row` -> out (+ bf16 copy)
__device__ __forceinline__ void store_pair(const DevParams& p, long long row, int col, float a0, float a1, float2 bias2, float2 res2,
                                           long long out_off) {
  if (col >= p.N) return;
  const bool both = col + 1 < p.N;
  const float v0 = fmaf(p.alpha, a0, bias2.x) + res2.x, v1 = fmaf(p.alpha, a1, bias2.y) + res2.y;
  const long long o = out_off + row * p.ldo + col;
  if (p.out_bf16) {
    bf16* dst = static_cast<bf16*>(p.out) + o;
    if (both) *reinterpret_cast<uint32_t*>(dst) = pack_bf16x2(v0, v1);
    else dst[0] = __float2bfloat16_rn(v0);
  } else {
    float* dst = static_cast<float*>(p.out) + o;
    if (both) *reinterpret_cast<float2*>(dst) = make_float2(v0, v1);
    else dst[0] = v0;
  }
  if (p.out2 != nullptr) {
    bf16* d2 = p.out2 + out_off + row * p.ldo2 + col;
    if (both) *reinterpret_cast<uint32_t*>(d2) = pack_bf16x2(v0, v1);
    else d2[0] = __float2bfloat16_rn(v0);
  }
}

// plain store of a loaded 16 x 64 block whose first column is global column col0
__device__ __forceinline__ void store_block64(const DevParams& p, const uint32_t (&r)[32], int lane, long long rowA, int col0,
                                              const float* bias, long long out_off, const ResFrag& res) {
  const int q2 = (lane & 3) * 2;
  const bool okA = rowA < p.M, okB = rowA + 8 < p.M;
  float2 b2[8];
#pragma unroll
  for (int kb = 0; kb < 8; ++kb) b2[kb] = load_bias2(bias, col0 + kb * 8 + q2, p.N);
#pragma unroll
  for (int kb = 0; kb < 8; ++kb) {
    const int col = col0 + kb * 8 + q2;
    if (okA) store_pair(p, rowA, col, __uint_as_float(r[4 * kb]), __uint_as_float(r[4 * kb + 1]), b2[kb], res.v[2 * kb], out_off);
    if (okB)
      store_pair(p, rowA + 8, col, __uint_as_float(r[4 * kb + 2]), __uint_as_float(r[4 * kb + 3]), b2[kb], res.v[2 * kb + 1], out_off);
  }
}

// ---------------------------------------------------------------------------------------------------
// Fast STORE epilogues (N even; fp32 / fp32+residual / bf16): compile-time output type, 64-bit vector accesses only, two
// row predicates + one column predicate per 8-column group, immediate address offsets.  ~5x fewer instructions than
// the generic path, which made every K <= 3072 GEMM epilogue-bound (ncu: issue-slot and instruction-cache limited).
// Block order per warp: column half cb (64 columns) outer, 16-row half hh inner; the residual of block i+1 is
// requested before block i is stored.
// ---------------------------------------------------------------------------------------------------
// FULL: the warp's whole 32 x 128 slab is inside the matrix -> no predicates at all (the common case; the edge variant
// costs ~3x the instructions, mostly branches around predicated loads and 64-bit compares).
template <bool RESID, bool FULL>
__device__ __forceinline__ void load_resid_fast(const float* rpA, const float* rpB, bool okA, bool okB, int col0t, int N, float2 (&f)[16]) {
  if (!RESID) return;
#pragma unroll
  for (int kb = 0; kb < 8; ++kb) {
    if (FULL) {
      f[2 * kb] = *reinterpret_cast<const float2*>(rpA + kb * 8);
      f[2 * kb + 1] = *reinterpret_cast<const float2*>(rpB + kb * 8);
    } else {
      const bool cok = col0t + kb * 8 < N;
      f[2 * kb] = (okA && cok) ? *reinterpret_cast<const float2*>(rpA + kb * 8) : make_float2(0.f, 0.f);
      f[2 * kb + 1] = (okB && cok) ? *reinterpret_cast<const float2*>(rpB + kb * 8) : make_float2(0.f, 0.f);
    }
  }
}

// outA / outB (and o2A / o2B): this thread's element (row, col0t) of the two rows it owns in the block
// STATS: st = {sum A, sumsq A, sum B, sumsq B} of the stored values of this thread's two rows (deferred LayerNorm)
template <int EPI, bool FULL, typename OutT, bool STATS = false>
__device__ __forceinline__ void store_blk_fast(const uint32_t (&r)[32], const float2 (&b2)[8], const float2 (&f)[16], OutT* outA, OutT* outB,
                                               bf16* o2A, bf16* o2B, bool okA, bool okB, int col0t, int N, float alphaA, float alphaB,
                                               float* st = nullptr) {
  constexpr bool RESID = EPI == K_STORE_F32_RESID;
  constexpr bool OBF = EPI == K_STORE_BF16;
#pragma unroll
  for (int kb = 0; kb < 8; ++kb) {
    float2 vA, vB;
    vA.x = fmaf(alphaA, __uint_as_float(r[4 * kb]), b2[kb].x);
    vA.y = fmaf(alphaA, __uint_as_float(r[4 * kb + 1]), b2[kb].y);
    vB.x = fmaf(alphaB, __uint_as_float(r[4 * kb + 2]), b2[kb].x);
    vB.y = fmaf(alphaB, __uint_as_float(r[4 * kb + 3]), b2[kb].y);
    if (RESID) {
      vA.x += f[2 * kb].x; vA.y += f[2 * kb].y;
      vB.x += f[2 * kb + 1].x; vB.y += f[2 * kb + 1].y;
    }
    const bool cok = FULL || col0t + kb * 8 < N;
    const bool sA = FULL || (okA && cok), sB = FULL || (okB && cok);
    if (STATS && cok) {
      st[0] += vA.x + vA.y; st[1] = fmaf(vA.x, vA.x, fmaf(vA.y, vA.y, st[1]));
      st[2] += vB.x + vB.y; st[3] = fmaf(vB.x, vB.x, fmaf(vB.y, vB.y, st[3]));
    }
    if (OBF) {
      if (sA) *reinterpret_cast<uint32_t*>(outA + kb * 8) = pack_bf16x2(vA.x, vA.y);
      if (sB) *reinterpret_cast<uint32_t*>(outB + kb * 8) = pack_bf16x2(vB.x, vB.y);
    } else {
      if (sA) *reinterpret_cast<float2*>(outA + kb * 8) = vA;
      if (sB) *reinterpret_cast<float2*>(outB + kb * 8) = vB;
      if (RESID && o2A != nullptr) {  // bf16 copy of the updated residual stream (operand of the next GEMM)
        if (sA) *reinterpret_cast<uint32_t*>(o2A + kb * 8) = pack_bf16x2(vA.x, vA.y);
        if (sB) *reinterpret_cast<uint32_t*>(o2B + kb * 8) = pack_bf16x2(vB.x, vB.y);
      }
    }
  }
}

template <int EPI, bool FULL, bool STATS>
__device__ __forceinline__ void epilogue_store_fast_impl(const DevParams& p, int lane, int half_sel, uint32_t t_row, int row0, int n_blk,
                                                         long long out_off, long long res_off, long long bias_off, long long ls_off,
                                                         long long st_off, uint64_t* full_bar, uint32_t full_parity) {
  constexpr bool RESID = EPI == K_STORE_F32_RESID;
  constexpr bool OBF = EPI == K_STORE_BF16;
  typedef typename std::conditional<OBF, bf16, float>::type OutT;
  const int g = lane >> 2, q2 = (lane & 3) * 2;
  const int colt = n_blk * BLOCK_N + half_sel * 128 + q2;  // this thread's first column of the tile
  const int N = p.N, M = p.M;
  // rows of this thread: row0 + hh*16 + rr*8 + g
  const int r00 = row0 + g;
  const bool ok00 = FULL || r00 < M, ok01 = FULL || r00 + 8 < M, ok10 = FULL || r00 + 16 < M, ok11 = FULL || r00 + 24 < M;
  const bool half1 = FULL || row0 + 16 < M;  // warp-uniform: the second 16-row block has rows inside the matrix
  const float *rp00 = nullptr, *rp01 = nullptr, *rp10 = nullptr, *rp11 = nullptr;
  if (RESID) {
    const float* rb = p.resid + res_off + colt;
    if (p.resid_row_mod > 0) {
      const unsigned md = static_cast<unsigned>(p.resid_row_mod);
      rp00 = rb + static_cast<long long>(static_cast<unsigned>(r00) % md) * p.ldr;
      rp01 = rb + static_cast<long long>(static_cast<unsigned>(r00 + 8) % md) * p.ldr;
      rp10 = rb + static_cast<long long>(static_cast<unsigned>(r00 + 16) % md) * p.ldr;
      rp11 = rb + static_cast<long long>(static_cast<unsigned>(r00 + 24) % md) * p.ldr;
    } else {
      rp00 = rb + static_cast<long long>(r00) * p.ldr;
      rp01 = rp00 + 8 * p.ldr;
      rp10 = rp00 + 16 * p.ldr;
      rp11 = rp00 + 24 * p.ldr;
    }
  }
  // per-row accumulator scale: alpha, or alpha / (sum of the row's partial softmax denominators)
  float a00 = p.alpha, a01 = p.alpha, a10 = p.alpha, a11 = p.alpha;
  if (p.row_lsum != nullptr) {
    const float* lp = p.row_lsum + ls_off + static_cast<long long>(r00) * p.row_lparts;
    float s00 = 0.f, s01 = 0.f, s10 = 0.f, s11 = 0.f;
    for (int c = 0; c < p.row_lparts; ++c) {
      if (ok00) s00 += __ldg(lp + c);
      if (ok01) s01 += __ldg(lp + 8 * p.row_lparts + c);
      if (ok10) s10 += __ldg(lp + 16 * p.row_lparts + c);
      if (ok11) s11 += __ldg(lp + 24 * p.row_lparts + c);
    }
    a00 = ok00 ? p.alpha / s00 : 0.f; a01 = ok01 ? p.alpha / s01 : 0.f;
    a10 = ok10 ? p.alpha / s10 : 0.f; a11 = ok11 ? p.alpha / s11 : 0.f;
  }
  float2 f0[16], f1[16];
  load_resid_fast<RESID, FULL>(rp00, rp01, ok00, ok01, colt, N, f0);
  // bias of the first column half, requested before the accumulator wait; the second half is requested while the
  // first is being stored
  const float* bias = p.bias ? p.bias + bias_off : nullptr;
  float2 b2[8];
#pragma unroll
  for (int kb = 0; kb < 8; ++kb)
    b2[kb] = (bias != nullptr && (FULL || colt + kb * 8 < N)) ? __ldg(reinterpret_cast<const float2*>(bias + colt + kb * 8)) : make_float2(0.f, 0.f);
  // output pointers of row r00 (the other rows are 8 / 16 / 24 rows further)
  OutT* o00 = static_cast<OutT*>(p.out) + out_off + static_cast<long long>(r00) * p.ldo + colt;
  const long long o8 = 8 * p.ldo;
  bf16* q00 = (RESID && p.out2 != nullptr) ? p.out2 + out_off + static_cast<long long>(r00) * p.ldo2 + colt : nullptr;
  const long long q8 = 8 * p.ldo2;
  mbar_wait(full_bar, full_parity);
  tcgen05_fence_after();
  if (row0 >= M) return;  // warp-uniform (cluster padding tile or fully out-of-range row group)
  float st0[4] = {0.f, 0.f, 0.f, 0.f}, st1[4] = {0.f, 0.f, 0.f, 0.f};  // STATS: rows (r00, r00+8) and (r00+16, r00+24)
#pragma unroll 1
  for (int cb = 0; cb < 2; ++cb) {
    const int col0t = colt + cb * 64;
    if (!FULL && col0t - q2 >= N) break;  // warp-uniform
    uint32_t r[32];
    // ---- hh = 0
    tmem_ld_16x64(t_row + static_cast<uint32_t>(half_sel * 128 + cb * 64), r);
    if (half1) load_resid_fast<RESID, FULL>(rp10 + cb * 64, rp11 + cb * 64, ok10, ok11, col0t, N, f1);
    tmem_ld_wait();
    store_blk_fast<EPI, FULL, OutT, STATS>(r, b2, f0, o00 + cb * 64, o00 + o8 + cb * 64, q00 ? q00 + cb * 64 : nullptr,
                                           q00 ? q00 + q8 + cb * 64 : nullptr, ok00, ok01, col0t, N, a00, a01, st0);
    // ---- hh = 1
    if (half1) tmem_ld_16x64(t_row + (16u << 16) + static_cast<uint32_t>(half_sel * 128 + cb * 64), r);
    if (cb == 0 && (FULL || col0t - q2 + 64 < N)) load_resid_fast<RESID, FULL>(rp00 + 64, rp01 + 64, ok00, ok01, col0t + 64, N, f0);
    if (half1) {
      tmem_ld_wait();
      store_blk_fast<EPI, FULL, OutT, STATS>(r, b2, f1, o00 + 2 * o8 + cb * 64, o00 + 3 * o8 + cb * 64,
                                             q00 ? q00 + 2 * q8 + cb * 64 : nullptr, q00 ? q00 + 3 * q8 + cb * 64 : nullptr, ok10, ok11,
                                             col0t, N, a10, a11, st1);
    }
    if (cb == 0) {
#pragma unroll
      for (int kb = 0; kb < 8; ++kb)
        b2[kb] = (bias != nullptr && (FULL || colt + 64 + kb * 8 < N)) ? __ldg(reinterpret_cast<const float2*>(bias + colt + 64 + kb * 8))
                                                                       : make_float2(0.f, 0.f);
    }
  }
  if (STATS) {
    // this warp's slab = part (2 n_blk + half_sel) of the row; a slab without any column inside the matrix writes nothing
    // (its part index is >= stat_parts_item and does not exist)
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      st0[i] = quad_sum(st0[i]);
      st1[i] = quad_sum(st1[i]);
    }
    if ((lane & 3) == 0 && (FULL || colt - q2 < N)) {
      float2* sp = p.stat_out + st_off + static_cast<long long>(r00) * p.stat_parts + (n_blk * 2 + half_sel);
      const long long s8 = 8ll * p.stat_parts;
      if (ok00) sp[0] = make_float2(st0[0], st0[1]);
      if (ok01) sp[s8] = make_float2(st0[2], st0[3]);
      if (ok10) sp[2 * s8] = make_float2(st1[0], st1[1]);
      if (ok11) sp[3 * s8] = make_float2(st1[2], st1[3]);
    }
  }
}

// fp32 result + fp32 residual with 16-byte accesses (TcGemmParams::out_perm4): the producer of the B operand stored its
// columns so that accumulator column 8 kb + 2 q + e of every 64-column block is output column 16 (kb / 2) + 4 q + 2 (kb % 2) + e.
// A thread then owns four consecutive floats per 16-column group and a quad 64 contiguous bytes of a row: half the LSU
// wavefronts of the float2 path for the same bytes (the P.V epilogue is bound by exactly those: +37 MB of 4-byte stores
// cost it 18 us).  No bias, no bf16 copy, no statistics; per-row 1 / sum scale supported.
template <bool FULL>
__device__ __forceinline__ void perm4_load(const float* ra, const float* rb, bool okA, bool okB, float4 (&f)[8]) {
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    f[j] = (FULL || okA) ? *reinterpret_cast<const float4*>(ra + j * 16) : make_float4(0.f, 0.f, 0.f, 0.f);
    f[4 + j] = (FULL || okB) ? *reinterpret_cast<const float4*>(rb + j * 16) : make_float4(0.f, 0.f, 0.f, 0.f);
  }
}
template <bool FULL>
__device__ __forceinline__ void perm4_store(const uint32_t (&r)[32], const float4 (&f)[8], float* oa, float* ob, bool okA, bool okB, float aA,
                                            float aB) {
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const int k0 = 2 * j, k1 = 2 * j + 1;
    float4 vA, vB;
    vA.x = fmaf(aA, __uint_as_float(r[4 * k0]), f[j].x);
    vA.y = fmaf(aA, __uint_as_float(r[4 * k0 + 1]), f[j].y);
    vA.z = fmaf(aA, __uint_as_float(r[4 * k1]), f[j].z);
    vA.w = fmaf(aA, __uint_as_float(r[4 * k1 + 1]), f[j].w);
    vB.x = fmaf(aB, __uint_as_float(r[4 * k0 + 2]), f[4 + j].x);
    vB.y = fmaf(aB, __uint_as_float(r[4 * k0 + 3]), f[4 + j].y);
    vB.z = fmaf(aB, __uint_as_float(r[4 * k1 + 2]), f[4 + j].z);
    vB.w = fmaf(aB, __uint_as_float(r[4 * k1 + 3]), f[4 + j].w);
    if (FULL || okA) *reinterpret_cast<float4*>(oa + j * 16) = vA;
    if (FULL || okB) *reinterpret_cast<float4*>(ob + j * 16) = vB;
  }
}
template <bool FULL>
__device__ __forceinline__ void epilogue_store_perm4(const DevParams& p, int lane, int half_sel, uint32_t t_row, int row0, int n_blk,
                                                     long long out_off, long long res_off, long long ls_off, uint64_t* full_bar,
                                                     uint32_t full_parity) {
  const int g = lane >> 2, q = lane & 3;
  const int colt = n_blk * BLOCK_N + half_sel * 128 + q * 4;  // first output column of this thread
  const int M = p.M;
  const int r00 = row0 + g;
  const bool ok00 = FULL || r00 < M, ok01 = FULL || r00 + 8 < M, ok10 = FULL || r00 + 16 < M, ok11 = FULL || r00 + 24 < M;
  const bool half1 = FULL || row0 + 16 < M;  // warp-uniform
  float a00 = p.alpha, a01 = p.alpha, a10 = p.alpha, a11 = p.alpha;
  if (p.row_lsum != nullptr) {
    const float* lp = p.row_lsum + ls_off + static_cast<long long>(r00) * p.row_lparts;
    float s00 = 0.f, s01 = 0.f, s10 = 0.f, s11 = 0.f;
    for (int c = 0; c < p.row_lparts; ++c) {
      if (ok00) s00 += __ldg(lp + c);
      if (ok01) s01 += __ldg(lp + 8 * p.row_lparts + c);
      if (ok10) s10 += __ldg(lp + 16 * p.row_lparts + c);
      if (ok11) s11 += __ldg(lp + 24 * p.row_lparts + c);
    }
    a00 = ok00 ? p.alpha / s00 : 0.f; a01 = ok01 ? p.alpha / s01 : 0.f;
    a10 = ok10 ? p.alpha / s10 : 0.f; a11 = ok11 ? p.alpha / s11 : 0.f;
  }
  const float* rp00 = p.resid + res_off + static_cast<long long>(r00) * p.ldr + colt;
  const long long r8 = 8 * p.ldr;
  float* o00 = static_cast<float*>(p.out) + out_off + static_cast<long long>(r00) * p.ldo + colt;
  const long long o8 = 8 * p.ldo;
  float4 f0[8], f1[8];
  perm4_load<FULL>(rp00, rp00 + r8, ok00, ok01, f0);
  mbar_wait(full_bar, full_parity);
  tcgen05_fence_after();
  if (row0 >= M) return;  // warp-uniform
#pragma unroll 1
  for (int cb = 0; cb < 2; ++cb) {
    uint32_t r[32];
    tmem_ld_16x64(t_row + static_cast<uint32_t>(half_sel * 128 + cb * 64), r);
    if (half1) perm4_load<FULL>(rp00 + 2 * r8 + cb * 64, rp00 + 3 * r8 + cb * 64, ok10, ok11, f1);
    tmem_ld_wait();
    perm4_store<FULL>(r, f0, o00 + cb * 64, o00 + o8 + cb * 64, ok00, ok01, a00, a01);
    if (half1) tmem_ld_16x64(t_row + (16u << 16) + static_cast<uint32_t>(half_sel * 128 + cb * 64), r);
    if (cb == 0) perm4_load<FULL>(rp00 + 64, rp00 + r8 + 64, ok00, ok01, f0);
    if (half1) {
      tmem_ld_wait();
      perm4_store<FULL>(r, f1, o00 + 2 * o8 + cb * 64, o00 + 3 * o8 + cb * 64, ok10, ok11, a10, a11);
    }
  }
}

template <int EPI>
__device__ __forceinline__ void epilogue_store_fast(const DevParams& p, int lane, int half_sel, uint32_t t_row, long long row0,
                                                    int n_blk, long long out_off, long long res_off, long long bias_off,
                                                    long long ls_off, long long st_off, uint64_t* full_bar, uint32_t full_parity) {
  const int r0 = static_cast<int>(row0);  // rows of one GEMM fit in 31 bits (checked at launch)
  const bool full = r0 + 32 <= p.M && n_blk * BLOCK_N + half_sel * 128 + 128 <= p.N;  // warp-uniform
  if (EPI == K_STORE_F32_RESID && p.out_perm4) {  // warp-uniform; N % 128 == 0 checked at launch
    if (n_blk * BLOCK_N + half_sel * 128 >= p.N) {  // this warp's 128 columns lie past the matrix: only the accumulator hand-shake
      mbar_wait(full_bar, full_parity);
      tcgen05_fence_after();
      return;
    }
    if (full) epilogue_store_perm4<true>(p, lane, half_sel, t_row, r0, n_blk, out_off, res_off, ls_off, full_bar, full_parity);
    else epilogue_store_perm4<false>(p, lane, half_sel, t_row, r0, n_blk, out_off, res_off, ls_off, full_bar, full_parity);
    return;
  }
  if (EPI == K_STORE_F32_RESID && p.stat_out != nullptr) {  // warp-uniform
    if (full)
      epilogue_store_fast_impl<EPI, true, EPI == K_STORE_F32_RESID>(p, lane, half_sel, t_row, r0, n_blk, out_off, res_off, bias_off, ls_off,
                                                                    st_off, full_bar, full_parity);
    else
      epilogue_store_fast_impl<EPI, false, EPI == K_STORE_F32_RESID>(p, lane, half_sel, t_row, r0, n_blk, out_off, res_off, bias_off, ls_off,
                                                                     st_off, full_bar, full_parity);
    return;
  }
  if (full)
    epilogue_store_fast_impl<EPI, true, false>(p, lane, half_sel, t_row, r0, n_blk, out_off, res_off, bias_off, ls_off, st_off, full_bar,
                                               full_parity);
  else
    epilogue_store_fast_impl<EPI, false, false>(p, lane, half_sel, t_row, r0, n_blk, out_off, res_off, bias_off, ls_off, st_off, full_bar,
                                                full_parity);
}

// bf16 store of one 16 x 64 block: v = a_row acc + (n_row c + b)  (plain bias store when the row coefficients are (1, 0))
__device__ __forceinline__ void store_blk_bf16_ln(const uint32_t (&r)[32], const float2 (&b2)[8], const float2 (&c2)[8], bf16* outA, bf16* outB,
                                                  bool okA, bool okB, int col0t, int N, float aA, float nA, float aB, float nB) {
#pragma unroll
  for (int kb = 0; kb < 8; ++kb) {
    const bool cok = col0t + kb * 8 < N;
    const float tAx = fmaf(nA, c2[kb].x, b2[kb].x), tAy = fmaf(nA, c2[kb].y, b2[kb].y);
    const float tBx = fmaf(nB, c2[kb].x, b2[kb].x), tBy = fmaf(nB, c2[kb].y, b2[kb].y);
    if (okA && cok)
      *reinterpret_cast<uint32_t*>(outA + kb * 8) =
          pack_bf16x2(fmaf(aA, __uint_as_float(r[4 * kb]), tAx), fmaf(aA, __uint_as_float(r[4 * kb + 1]), tAy));
    if (okB && cok)
      *reinterpret_cast<uint32_t*>(outB + kb * 8) =
          pack_bf16x2(fmaf(aB, __uint_as_float(r[4 * kb + 2]), tBx), fmaf(aB, __uint_as_float(r[4 * kb + 3]), tBy));
  }
}

// ---------------------------------------------------------------------------------------------------
// Lean QKV + RoPE epilogue for the common case (pair distance 128 = head_dim 768, cos/sin computed on the fly, no deferred
// LayerNorm, row % T positions, tile completely inside the matrix).  The generic path below spends ~21 instructions per
// output element, 40 % of them address / predicate / branch work, and with two epilogue warps per scheduler that latency
// chain -- not the tensor pipe -- set the pace of the GEMM (ncu: 46 % tensor-active).  Here: no predicates, packed f32x2
// arithmetic (bias add, Cody-Waite reduction, rotation), ~6 instructions per element.  Arithmetic identical to the generic
// path (same reduction constants, same MUFU approximations).
// ---------------------------------------------------------------------------------------------------
__device__ __forceinline__ void sincos_reduced2(float2 a, float2& s, float2& c) {
  const float2 t = __fmul2_rn(a, make_float2(0.15915494309189535f, 0.15915494309189535f));
  const float2 k = make_float2(rintf(t.x), rintf(t.y));
  float2 r = __ffma2_rn(k, make_float2(-6.28125f, -6.28125f), a);
  r = __ffma2_rn(k, make_float2(-1.9353071795864769e-3f, -1.9353071795864769e-3f), r);
  s = make_float2(__sinf(r.x), __sinf(r.y));
  c = make_float2(__cosf(r.x), __cosf(r.y));
}

// Store-friendly column order (TcGemmParams::rope_perm16): inside every 64-column block of the packed weight the engine
// additionally permutes the rows so that accumulator column kb * 8 + 2 q + e (the fragment a thread holds) is OUTPUT column
// q * 16 + kb * 2 + e of the block: a thread's 16 values of a row are then 16 consecutive bf16 = two 16-byte stores, and a
// quad writes whole 128-byte lines (was: 4-byte stores, 16 bytes per line and instruction -- the top stall of this
// epilogue in ncu).  Biases follow the GEMM column (they are packed with the weight); rotary frequencies and output
// addresses follow the output column.
// 128-bit global store with the cache-streaming (evict-first) policy
__device__ __forceinline__ void st_global_cs_v4(void* ptr, const uint32_t (&w)[4]) {
  asm volatile("st.global.cs.v4.b32 [%0], {%1, %2, %3, %4};" ::"l"(ptr), "r"(w[0]), "r"(w[1]), "r"(w[2]), "r"(w[3]) : "memory");
}
// 256-bit global store (sm_100+): eight packed bf16 pairs = 16 consecutive outputs; the address must be 32-byte aligned
__device__ __forceinline__ void st_global_v8(void* ptr, const uint32_t (&w)[8]) {
  asm volatile("st.global.v8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"l"(ptr), "r"(w[0]), "r"(w[1]), "r"(w[2]), "r"(w[3]),
               "r"(w[4]), "r"(w[5]), "r"(w[6]), "r"(w[7])
               : "memory");
}

template <bool FULL>
__device__ __forceinline__ void rope_epilogue_fast128(const DevParams& p, int lane, int half_sel, uint32_t t_row, long long row0, int n_blk,
                                                      long long out_off, const float* bias, uint64_t* full_bar, uint32_t full_parity) {
  const int g = lane >> 2, q = lane & 3, q2 = q * 2;
  const int b1 = half_sel * 64;                      // tile column of this warp's x1 block; partners 128 columns further
  const int pc1 = n_blk * BLOCK_N + b1;              // permuted GEMM column
  const bool is_v = pc1 >= 2 * p.hidden;             // warp-uniform: v third = identity layout, plain bias store
  int jbase = 0, dbase = pc1, off2 = 128;
  if (!is_v) {
    const int region = pc1 / p.hidden;               // 0 = q, 1 = k
    const int lp = pc1 - region * p.hidden;
    const int grp = lp >> 8, w = lp & 255;           // groups of 2 * 128 permuted columns; w < 128 by construction
    const int e0 = grp * 128;
    const int head = e0 / p.rope_half;
    jbase = e0 - head * p.rope_half + w;
    dbase = region * p.hidden + head * 2 * p.rope_half + jbase;
    off2 = p.rope_half;
  }
  float2 fr[8], bx1[8], bx2[8];
#pragma unroll
  for (int kb = 0; kb < 8; ++kb) {
    bx1[kb] = __ldg(reinterpret_cast<const float2*>(bias + pc1 + q2 + kb * 8));
    bx2[kb] = __ldg(reinterpret_cast<const float2*>(bias + pc1 + 128 + q2 + kb * 8));
    fr[kb] = is_v ? make_float2(0.f, 0.f) : __ldg(reinterpret_cast<const float2*>(p.rope_freq + jbase + q * 16 + kb * 2));
  }
  float fpos[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const long long rr = row0 + g + 8 * i;
    fpos[i] = p.rope_pos != nullptr ? static_cast<float>((FULL || rr < p.M) ? __ldg(p.rope_pos + rr) : 0)
                                    : static_cast<float>(static_cast<unsigned>(rr) % static_cast<unsigned>(p.seq_T));
  }
  mbar_wait(full_bar, full_parity);
  tcgen05_fence_after();
  if (!FULL && row0 >= p.M) return;                  // warp-uniform
  bf16* o1 = static_cast<bf16*>(p.out) + out_off + (row0 + g) * p.ldo + dbase + q * 16;
#pragma unroll 1
  for (int hh = 0; hh < 2; ++hh) {
    if (!FULL && row0 + hh * 16 >= p.M) break;       // warp-uniform
    uint32_t r1[32], r2[32];
    const uint32_t tbase = t_row + (static_cast<uint32_t>(hh * 16) << 16) + b1;
    tmem_ld_16x64(tbase, r1);
    tmem_ld_16x64(tbase + 128, r2);
    bf16* oA = o1 + static_cast<long long>(hh * 16) * p.ldo;
    bf16* oB = oA + 8 * p.ldo;
    const bool okA = FULL || row0 + hh * 16 + g < p.M, okB = FULL || row0 + hh * 16 + g + 8 < p.M;
    const float2 pA = make_float2(fpos[2 * hh], fpos[2 * hh]), pB = make_float2(fpos[2 * hh + 1], fpos[2 * hh + 1]);
    uint32_t w1A[8], w1B[8], w2A[8], w2B[8];         // packed bf16 pairs: output columns q * 16 + 2 kb (+1) of both blocks
    tmem_ld_wait();
    if (is_v) {
#pragma unroll
      for (int kb = 0; kb < 8; ++kb) {
        const float2 a1 = __fadd2_rn(make_float2(__uint_as_float(r1[4 * kb]), __uint_as_float(r1[4 * kb + 1])), bx1[kb]);
        const float2 c1 = __fadd2_rn(make_float2(__uint_as_float(r1[4 * kb + 2]), __uint_as_float(r1[4 * kb + 3])), bx1[kb]);
        const float2 a2 = __fadd2_rn(make_float2(__uint_as_float(r2[4 * kb]), __uint_as_float(r2[4 * kb + 1])), bx2[kb]);
        const float2 c2 = __fadd2_rn(make_float2(__uint_as_float(r2[4 * kb + 2]), __uint_as_float(r2[4 * kb + 3])), bx2[kb]);
        w1A[kb] = pack_bf16x2(a1.x, a1.y);
        w1B[kb] = pack_bf16x2(c1.x, c1.y);
        w2A[kb] = pack_bf16x2(a2.x, a2.y);
        w2B[kb] = pack_bf16x2(c2.x, c2.y);
      }
    } else {
#pragma unroll
      for (int kb = 0; kb < 8; ++kb) {
        float2 sA, cA, sB, cB;   // angle = float(pos) * inv_freq[j] exactly as the reference forms it (DiT.py:56-59)
        sincos_reduced2(__fmul2_rn(pA, fr[kb]), sA, cA);
        sincos_reduced2(__fmul2_rn(pB, fr[kb]), sB, cB);
        const float2 x1A = __fadd2_rn(make_float2(__uint_as_float(r1[4 * kb]), __uint_as_float(r1[4 * kb + 1])), bx1[kb]);
        const float2 x1B = __fadd2_rn(make_float2(__uint_as_float(r1[4 * kb + 2]), __uint_as_float(r1[4 * kb + 3])), bx1[kb]);
        const float2 x2A = __fadd2_rn(make_float2(__uint_as_float(r2[4 * kb]), __uint_as_float(r2[4 * kb + 1])), bx2[kb]);
        const float2 x2B = __fadd2_rn(make_float2(__uint_as_float(r2[4 * kb + 2]), __uint_as_float(r2[4 * kb + 3])), bx2[kb]);
        // x1' = x1 cos - x2 sin ; x2' = x2 cos + x1 sin   (DiT.py:52-54,72)
        const float2 nA = make_float2(-sA.x, -sA.y), nB = make_float2(-sB.x, -sB.y);
        const float2 y1A = __ffma2_rn(x2A, nA, __fmul2_rn(x1A, cA)), y2A = __ffma2_rn(x1A, sA, __fmul2_rn(x2A, cA));
        const float2 y1B = __ffma2_rn(x2B, nB, __fmul2_rn(x1B, cB)), y2B = __ffma2_rn(x1B, sB, __fmul2_rn(x2B, cB));
        w1A[kb] = pack_bf16x2(y1A.x, y1A.y);
        w2A[kb] = pack_bf16x2(y2A.x, y2A.y);
        w1B[kb] = pack_bf16x2(y1B.x, y1B.y);
        w2B[kb] = pack_bf16x2(y2B.x, y2B.y);
      }
    }
    // one 32-byte store per thread and block: a thread fills whole 32-byte sectors, a quad a whole 128-byte line (two
    // 16-byte stores would write half sectors each)
    if (okA) {
      st_global_v8(oA, w1A);
      st_global_v8(oA + off2, w2A);
    }
    if (okB) {
      st_global_v8(oB, w1B);
      st_global_v8(oB + off2, w2B);
    }
  }
}

// ---------------------------------------------------------------------------------------------------
// Lean GEGLU epilogue (TcGemmParams::glu_perm16): no deferred LayerNorm, N % 256 == 0, packed f32x2 arithmetic, and the
// [fc1; gate] rows of the packed weight ordered so that a thread's 8 outputs of a row and 64-column block are consecutive:
// accumulator 8-column block kb = gi * 4 + kk holds, for kk < 2, the fc1 rows (kk >= 2: the gate rows, block kb - 2) of
// outputs  q * 8 + (gi * 2 + kk) * 2 + e  (column kb * 8 + 2 q + e) -> one 16-byte store per row instead of four 4-byte ones.
// ---------------------------------------------------------------------------------------------------
__device__ __forceinline__ float2 geglu_fast2(float2 a, float2 g) {   // geglu_fast on a pair, same operations
  const float2 ac = make_float2(fminf(fmaxf(a.x, -6.0f), 6.0f), fminf(fmaxf(a.y, -6.0f), 6.0f));
  const float2 a2 = __fmul2_rn(ac, ac);
  float2 sp = __ffma2_rn(a2, make_float2(2.377971153e-05f, 2.377971153e-05f), make_float2(7.501817227e-04f, 7.501817227e-04f));
  sp = __ffma2_rn(a2, sp, make_float2(-1.060307563e-01f, -1.060307563e-01f));
  sp = __ffma2_rn(a2, sp, make_float2(-2.301608248e+00f, -2.301608248e+00f));
  const float2 t1 = __fmul2_rn(ac, sp), t2 = __fmul2_rn(g, make_float2(-1.4426950408889634f, -1.4426950408889634f));
  const float2 e1 = make_float2(ex2_approx(t1.x), ex2_approx(t1.y)), e2 = make_float2(ex2_approx(t2.x), ex2_approx(t2.y));
  const float2 one = make_float2(1.0f, 1.0f);
  const float2 den = __fmul2_rn(__fadd2_rn(one, e1), __fadd2_rn(one, e2));
  return __fmul2_rn(a, make_float2(rcp_approx(den.x), rcp_approx(den.y)));
}

template <bool FULL>
__device__ __forceinline__ void geglu_epilogue_fast(const DevParams& p, int lane, int half_sel, uint32_t t_row, long long row0, int n_blk,
                                                    long long out_off, const float* bias, uint64_t* full_bar, uint32_t full_parity) {
  const int g = lane >> 2, q = lane & 3, q2 = q * 2;
  const int colw = n_blk * BLOCK_N + half_sel * 128;   // first GEMM column of this warp's 128
  float2 bb[2][8];
#pragma unroll
  for (int cb = 0; cb < 2; ++cb)
#pragma unroll
    for (int kb = 0; kb < 8; ++kb) bb[cb][kb] = __ldg(reinterpret_cast<const float2*>(bias + colw + cb * 64 + kb * 8 + q2));
  mbar_wait(full_bar, full_parity);
  tcgen05_fence_after();
  if (!FULL && row0 >= p.M) return;                    // warp-uniform
  bf16* outp = static_cast<bf16*>(p.out) + out_off + (row0 + g) * p.ldo + (colw >> 1) + q * 8;
#pragma unroll
  for (int cb = 0; cb < 2; ++cb) {
#pragma unroll 1
    for (int hh = 0; hh < 2; ++hh) {
      if (!FULL && row0 + hh * 16 >= p.M) break;       // warp-uniform
      uint32_t r[32];
      tmem_ld_16x64(t_row + (static_cast<uint32_t>(hh * 16) << 16) + half_sel * 128 + cb * 64, r);
      tmem_ld_wait();
      uint32_t wA[4], wB[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {                    // j = gi * 2 + kk
        const int ka = (j >> 1) * 4 + (j & 1), kg = ka + 2;
        const float2 aA = __fadd2_rn(make_float2(__uint_as_float(r[4 * ka]), __uint_as_float(r[4 * ka + 1])), bb[cb][ka]);
        const float2 gA = __fadd2_rn(make_float2(__uint_as_float(r[4 * kg]), __uint_as_float(r[4 * kg + 1])), bb[cb][kg]);
        const float2 aB = __fadd2_rn(make_float2(__uint_as_float(r[4 * ka + 2]), __uint_as_float(r[4 * ka + 3])), bb[cb][ka]);
        const float2 gB = __fadd2_rn(make_float2(__uint_as_float(r[4 * kg + 2]), __uint_as_float(r[4 * kg + 3])), bb[cb][kg]);
        const float2 oA = geglu_fast2(aA, gA), oB = geglu_fast2(aB, gB);
        wA[j] = pack_bf16x2(oA.x, oA.y);
        wB[j] = pack_bf16x2(oB.x, oB.y);
      }
      bf16* o = outp + static_cast<long long>(hh * 16) * p.ldo + cb * 32;
      // streaming stores: the hidden activations (147 MB at C2, 2.4 GB at C4) are read once by fc2 and must not push the A
      // row blocks, which 24 column tiles re-read, out of L2
      if (FULL || row0 + hh * 16 + g < p.M) st_global_cs_v4(o, wA);
      if (FULL || row0 + hh * 16 + g + 8 < p.M) st_global_cs_v4(o + 8 * p.ldo, wB);
    }
  }
}

// The same for pair distance 32 (head_dim 64 and other d / 2 = 32 (2k + 1)): a 64-column block holds 32 x1 columns (8-column
// blocks kb 0..3) and their 32 partners (kb 4..7).  Store-friendly order inside the block: accumulator column 8 kb + 2 q + e is
// x1 element q * 8 + kb * 2 + e (kb < 4) resp. its partner (kb >= 4), so a thread's 8 x1' and 8 x2' outputs of a row are two
// 16-byte stores; v blocks use the q * 16 + kb * 2 + e order of the pd = 128 path.
template <bool FULL>
__device__ __forceinline__ void rope_epilogue_fast32(const DevParams& p, int lane, int half_sel, uint32_t t_row, long long row0, int n_blk,
                                                     long long out_off, const float* bias, uint64_t* full_bar, uint32_t full_parity) {
  const int g = lane >> 2, q = lane & 3, q2 = q * 2;
  float fpos[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const long long rr = row0 + g + 8 * i;
    fpos[i] = p.rope_pos != nullptr ? static_cast<float>((FULL || rr < p.M) ? __ldg(p.rope_pos + rr) : 0)
                                    : static_cast<float>(static_cast<unsigned>(rr) % static_cast<unsigned>(p.seq_T));
  }
  bool waited = false;
#pragma unroll 1
  for (int u = 0; u < 2; ++u) {
    const int b1 = half_sel * 128 + u * 64;            // tile column of this 64-column block
    const int pc1 = n_blk * BLOCK_N + b1;              // permuted GEMM column
    const bool is_v = pc1 >= 2 * p.hidden;             // warp-uniform
    int jbase = 0, dbase = pc1;
    if (!is_v) {
      const int region = pc1 / p.hidden;
      const int lp = pc1 - region * p.hidden;
      const int grp = lp >> 6;                         // groups of 2 * 32 permuted columns
      const int e0 = grp * 32;
      const int head = e0 / p.rope_half;
      jbase = e0 - head * p.rope_half;
      dbase = region * p.hidden + head * 2 * p.rope_half + jbase;
    }
    float2 fr[4], bx[8];
#pragma unroll
    for (int kb = 0; kb < 8; ++kb) bx[kb] = __ldg(reinterpret_cast<const float2*>(bias + pc1 + q2 + kb * 8));
#pragma unroll
    for (int kb = 0; kb < 4; ++kb)
      fr[kb] = is_v ? make_float2(0.f, 0.f) : __ldg(reinterpret_cast<const float2*>(p.rope_freq + jbase + q * 8 + kb * 2));
    if (!waited) {
      mbar_wait(full_bar, full_parity);
      tcgen05_fence_after();
      waited = true;
    }
    if (!FULL && row0 >= p.M) continue;                // warp-uniform
    bf16* o1 = static_cast<bf16*>(p.out) + out_off + (row0 + g) * p.ldo + dbase;
#pragma unroll 1
    for (int hh = 0; hh < 2; ++hh) {
      if (!FULL && row0 + hh * 16 >= p.M) break;       // warp-uniform
      uint32_t r[32];
      tmem_ld_16x64(t_row + (static_cast<uint32_t>(hh * 16) << 16) + b1, r);
      bf16* oA = o1 + static_cast<long long>(hh * 16) * p.ldo;
      bf16* oB = oA + 8 * p.ldo;
      const bool okA = FULL || row0 + hh * 16 + g < p.M, okB = FULL || row0 + hh * 16 + g + 8 < p.M;
      tmem_ld_wait();
      if (is_v) {
        uint32_t wA[8], wB[8];
#pragma unroll
        for (int kb = 0; kb < 8; ++kb) {
          const float2 a = __fadd2_rn(make_float2(__uint_as_float(r[4 * kb]), __uint_as_float(r[4 * kb + 1])), bx[kb]);
          const float2 c = __fadd2_rn(make_float2(__uint_as_float(r[4 * kb + 2]), __uint_as_float(r[4 * kb + 3])), bx[kb]);
          wA[kb] = pack_bf16x2(a.x, a.y);
          wB[kb] = pack_bf16x2(c.x, c.y);
        }
        if (okA) {
          reinterpret_cast<uint4*>(oA + q * 16)[0] = make_uint4(wA[0], wA[1], wA[2], wA[3]);
          reinterpret_cast<uint4*>(oA + q * 16)[1] = make_uint4(wA[4], wA[5], wA[6], wA[7]);
        }
        if (okB) {
          reinterpret_cast<uint4*>(oB + q * 16)[0] = make_uint4(wB[0], wB[1], wB[2], wB[3]);
          reinterpret_cast<uint4*>(oB + q * 16)[1] = make_uint4(wB[4], wB[5], wB[6], wB[7]);
        }
        continue;
      }
      const float2 pA = make_float2(fpos[2 * hh], fpos[2 * hh]), pB = make_float2(fpos[2 * hh + 1], fpos[2 * hh + 1]);
      uint32_t w1A[4], w2A[4], w1B[4], w2B[4];
#pragma unroll
      for (int kb = 0; kb < 4; ++kb) {
        float2 sA, cA, sB, cB;
        sincos_reduced2(__fmul2_rn(pA, fr[kb]), sA, cA);
        sincos_reduced2(__fmul2_rn(pB, fr[kb]), sB, cB);
        const int k2 = kb + 4;
        const float2 x1A = __fadd2_rn(make_float2(__uint_as_float(r[4 * kb]), __uint_as_float(r[4 * kb + 1])), bx[kb]);
        const float2 x1B = __fadd2_rn(make_float2(__uint_as_float(r[4 * kb + 2]), __uint_as_float(r[4 * kb + 3])), bx[kb]);
        const float2 x2A = __fadd2_rn(make_float2(__uint_as_float(r[4 * k2]), __uint_as_float(r[4 * k2 + 1])), bx[k2]);
        const float2 x2B = __fadd2_rn(make_float2(__uint_as_float(r[4 * k2 + 2]), __uint_as_float(r[4 * k2 + 3])), bx[k2]);
        const float2 nA = make_float2(-sA.x, -sA.y), nB = make_float2(-sB.x, -sB.y);
        const float2 y1A = __ffma2_rn(x2A, nA, __fmul2_rn(x1A, cA)), y2A = __ffma2_rn(x1A, sA, __fmul2_rn(x2A, cA));
        const float2 y1B = __ffma2_rn(x2B, nB, __fmul2_rn(x1B, cB)), y2B = __ffma2_rn(x1B, sB, __fmul2_rn(x2B, cB));
        w1A[kb] = pack_bf16x2(y1A.x, y1A.y);
        w2A[kb] = pack_bf16x2(y2A.x, y2A.y);
        w1B[kb] = pack_bf16x2(y1B.x, y1B.y);
        w2B[kb] = pack_bf16x2(y2B.x, y2B.y);
      }
      if (okA) {
        *reinterpret_cast<uint4*>(oA + q * 8) = make_uint4(w1A[0], w1A[1], w1A[2], w1A[3]);
        *reinterpret_cast<uint4*>(oA + p.rope_half + q * 8) = make_uint4(w2A[0], w2A[1], w2A[2], w2A[3]);
      }
      if (okB) {
        *reinterpret_cast<uint4*>(oB + q * 8) = make_uint4(w1B[0], w1B[1], w1B[2], w1B[3]);
        *reinterpret_cast<uint4*>(oB + p.rope_half + q * 8) = make_uint4(w2B[0], w2B[1], w2B[2], w2B[3]);
      }
    }
  }
  if (!waited) {
    mbar_wait(full_bar, full_parity);
    tcgen05_fence_after();
  }
}

// One accumulator tile: this warp's 32 rows (two 16-lane halves) x its 128 of the 256 tile columns.  Waits for the
// accumulator itself (after the first residual block has been requested).
template <int EPI>
__device__ __forceinline__ void epilogue_tile(const DevParams& p, int lane, int half_sel, uint32_t t_row, long long row0, int n_blk,
                                              long long out_off, long long res_off, long long bias_off, long long ls_off,
                                              long long st_off, uint64_t* full_bar, uint32_t full_parity) {
  if (EPI == K_STORE_F32 || EPI == K_STORE_F32_RESID || EPI == K_STORE_BF16) {
    epilogue_store_fast<EPI>(p, lane, half_sel, t_row, row0, n_blk, out_off, res_off, bias_off, ls_off, st_off, full_bar, full_parity);
    return;
  }
  const int g = lane >> 2, q2 = (lane & 3) * 2;
  const float* bias = p.bias ? p.bias + bias_off : nullptr;

  if (EPI == K_STORE_GENERIC) {
    // block `it` of this warp: rows row0 + (it&1)*16 .. +16, tile columns half_sel*128 + (it>>1)*64 .. +64
    const bool has_res = p.resid != nullptr;
    ResFrag rf[2];
#pragma unroll
    for (int i = 0; i < 16; ++i) rf[0].v[i] = rf[1].v[i] = make_float2(0.f, 0.f);
    const int colbase = n_blk * BLOCK_N + half_sel * 128;
    if (has_res && row0 < p.M && colbase < p.N) load_resid_block(p, lane, row0 + g, colbase, res_off, rf[0]);
    mbar_wait(full_bar, full_parity);
    tcgen05_fence_after();
    if (row0 >= p.M) return;  // warp-uniform: nothing to store for a fully out-of-range row group
#pragma unroll
    for (int it = 0; it < 4; ++it) {
      const int hh = it & 1, cb = it >> 1;
      const int tcol = half_sel * 128 + cb * 64;
      const int col0 = n_blk * BLOCK_N + tcol;
      const bool valid = col0 < p.N && row0 + hh * 16 < p.M;  // warp-uniform
      uint32_t r[32];
      if (valid) tmem_ld_16x64(t_row + (static_cast<uint32_t>(hh * 16) << 16) + tcol, r);
      if (it + 1 < 4 && has_res) {  // request the next block's residual before this block's stores
        const int nh = (it + 1) & 1, ncb = (it + 1) >> 1;
        const int ncol0 = n_blk * BLOCK_N + half_sel * 128 + ncb * 64;
        if (ncol0 < p.N && row0 + nh * 16 < p.M) load_resid_block(p, lane, row0 + nh * 16 + g, ncol0, res_off, rf[(it + 1) & 1]);
      }
      if (valid) {
        tmem_ld_wait();
        store_block64(p, r, lane, row0 + hh * 16 + g, col0, bias, out_off, rf[it & 1]);
      }
    }
  } else if (EPI == K_GEGLU) {
    if (p.glu_fast) {  // weights packed in the store-friendly order: every tile takes the lean epilogue
      if (row0 + 32 <= p.M) geglu_epilogue_fast<true>(p, lane, half_sel, t_row, row0, n_blk, out_off, bias, full_bar, full_parity);
      else geglu_epilogue_fast<false>(p, lane, half_sel, t_row, row0, n_blk, out_off, bias, full_bar, full_parity);
      return;
    }
    // 64 accumulator columns = two interleave groups [a16 | g16]; a_j and g_j (16 columns apart) live in the same thread.
    // Biases of this thread's column pairs for both 64-column halves are requested before the accumulator wait.
    // Deferred LayerNorm (ln_stat != nullptr): a = rstd acc + (nm c + b') per row -- one extra FMA per element; without
    // it the row coefficients are (1, 0) and the expression reduces to acc + b.
    float2 ba[8], bg[8], ca2[8], cg2[8];
    const bool dln = p.ln_stat != nullptr;
#pragma unroll
    for (int j = 0; j < 8; ++j) {  // j = cb*4 + gi*2 + m
      const int cg0 = n_blk * BLOCK_N + half_sel * 128 + (j >> 2) * 64 + ((j >> 1) & 1) * 32;  // first column of the group
      const int ca = cg0 + (j & 1) * 8 + q2;
      const bool ok = cg0 < p.N;
      ba[j] = ok ? __ldg(reinterpret_cast<const float2*>(bias + ca)) : make_float2(0.f, 0.f);
      bg[j] = ok ? __ldg(reinterpret_cast<const float2*>(bias + ca + 16)) : make_float2(0.f, 0.f);
      ca2[j] = (ok && dln) ? __ldg(reinterpret_cast<const float2*>(p.ln_c + ca)) : make_float2(0.f, 0.f);
      cg2[j] = (ok && dln) ? __ldg(reinterpret_cast<const float2*>(p.ln_c + ca + 16)) : make_float2(0.f, 0.f);
    }
    float lnA0, lnN0, lnA1, lnN1, lnA2, lnN2, lnA3, lnN3;  // rows row0 + g + {0, 8, 16, 24}
    ln_row_coef(p.ln_stat, p.ln_parts, row0 + g, row0 + g < p.M, p.ln_inv_h, lnA0, lnN0);
    ln_row_coef(p.ln_stat, p.ln_parts, row0 + g + 8, row0 + g + 8 < p.M, p.ln_inv_h, lnA1, lnN1);
    ln_row_coef(p.ln_stat, p.ln_parts, row0 + g + 16, row0 + g + 16 < p.M, p.ln_inv_h, lnA2, lnN2);
    ln_row_coef(p.ln_stat, p.ln_parts, row0 + g + 24, row0 + g + 24 < p.M, p.ln_inv_h, lnA3, lnN3);
    mbar_wait(full_bar, full_parity);
    tcgen05_fence_after();
    if (row0 >= p.M) return;
    bf16* outp = static_cast<bf16*>(p.out) + out_off;
#pragma unroll
    for (int cb = 0; cb < 2; ++cb) {
      const int tcol = half_sel * 128 + cb * 64;
      const int col0 = n_blk * BLOCK_N + tcol;
      if (col0 >= p.N) break;
#pragma unroll 1
      for (int hh = 0; hh < 2; ++hh) {
        if (row0 + hh * 16 >= p.M) break;
        const long long rowA = row0 + hh * 16 + g;
        uint32_t r[32];
        tmem_ld_16x64(t_row + (static_cast<uint32_t>(hh * 16) << 16) + tcol, r);
        tmem_ld_wait();
        const bool okA = rowA < p.M, okB = rowA + 8 < p.M;
        const float aA = hh ? lnA2 : lnA0, nA = hh ? lnN2 : lnN0, aB = hh ? lnA3 : lnA1, nB = hh ? lnN3 : lnN1;
#pragma unroll
        for (int gi = 0; gi < 2; ++gi) {
          if (col0 + gi * 32 >= p.N) break;           // N % 32 == 0: a group is all-or-nothing
#pragma unroll
          for (int m = 0; m < 2; ++m) {
            const int ka = gi * 4 + m, kg = ka + 2;   // 8-column blocks of the a and the g values
            const float2 b_a = ba[cb * 4 + gi * 2 + m], b_g = bg[cb * 4 + gi * 2 + m];
            const float2 c_a = ca2[cb * 4 + gi * 2 + m], c_g = cg2[cb * 4 + gi * 2 + m];
            const int oc = ((col0 + gi * 32) >> 1) + m * 8 + q2;
            if (okA)
              *reinterpret_cast<uint32_t*>(outp + rowA * p.ldo + oc) =
                  pack_bf16x2(geglu_fast(fmaf(aA, __uint_as_float(r[4 * ka]), fmaf(nA, c_a.x, b_a.x)),
                                         fmaf(aA, __uint_as_float(r[4 * kg]), fmaf(nA, c_g.x, b_g.x))),
                              geglu_fast(fmaf(aA, __uint_as_float(r[4 * ka + 1]), fmaf(nA, c_a.y, b_a.y)),
                                         fmaf(aA, __uint_as_float(r[4 * kg + 1]), fmaf(nA, c_g.y, b_g.y))));
            if (okB)
              *reinterpret_cast<uint32_t*>(outp + (rowA + 8) * p.ldo + oc) =
                  pack_bf16x2(geglu_fast(fmaf(aB, __uint_as_float(r[4 * ka + 2]), fmaf(nB, c_a.x, b_a.x)),
                                         fmaf(aB, __uint_as_float(r[4 * kg + 2]), fmaf(nB, c_g.x, b_g.x))),
                              geglu_fast(fmaf(aB, __uint_as_float(r[4 * ka + 3]), fmaf(nB, c_a.y, b_a.y)),
                                         fmaf(aB, __uint_as_float(r[4 * kg + 3]), fmaf(nB, c_g.y, b_g.y))));
          }
        }
      }
    }
  } else {  // K_QKV_ROPE
    if (p.rope_fast) {  // weights packed in the store-friendly column order: every tile takes the lean epilogue
      const bool full = row0 + 32 <= p.M;
      if (p.rope_pd == 128) {
        if (full) rope_epilogue_fast128<true>(p, lane, half_sel, t_row, row0, n_blk, out_off, bias, full_bar, full_parity);
        else rope_epilogue_fast128<false>(p, lane, half_sel, t_row, row0, n_blk, out_off, bias, full_bar, full_parity);
      } else {
        if (full) rope_epilogue_fast32<true>(p, lane, half_sel, t_row, row0, n_blk, out_off, bias, full_bar, full_parity);
        else rope_epilogue_fast32<false>(p, lane, half_sel, t_row, row0, n_blk, out_off, bias, full_bar, full_parity);
      }
      return;
    }
    // units of (x1 block, partner block PD columns further); PD = 32: both inside one 64-column load.  Everything that
    // is read from global memory (rotary frequencies, biases) is requested BEFORE the accumulator wait: with the L2 busy
    // feeding the operand ring, a dependent load after the wait costs ~1 us and made this epilogue the bottleneck (ncu).
    const int pd = p.rope_pd;
    const int units = pd == 32 ? 2 : 1;
    const bool dln = p.ln_stat != nullptr;           // deferred LayerNorm: x = rstd acc + (nm c + b') before the rotation
    float lnA0, lnN0, lnA1, lnN1, lnA2, lnN2, lnA3, lnN3;  // rows row0 + g + {0, 8, 16, 24}
    ln_row_coef(p.ln_stat, p.ln_parts, row0 + g, row0 + g < p.M, p.ln_inv_h, lnA0, lnN0);
    ln_row_coef(p.ln_stat, p.ln_parts, row0 + g + 8, row0 + g + 8 < p.M, p.ln_inv_h, lnA1, lnN1);
    ln_row_coef(p.ln_stat, p.ln_parts, row0 + g + 16, row0 + g + 16 < p.M, p.ln_inv_h, lnA2, lnN2);
    ln_row_coef(p.ln_stat, p.ln_parts, row0 + g + 24, row0 + g + 24 < p.M, p.ln_inv_h, lnA3, lnN3);
    // sequence positions of the thread's four rows (requested before the accumulator wait, like every other global read)
    unsigned pos4[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const long long rr = row0 + g + 8 * i;
      pos4[i] = p.rope_pos != nullptr ? (rr < p.M ? static_cast<unsigned>(__ldg(p.rope_pos + rr)) : 0u)
                                      : static_cast<unsigned>(rr) % static_cast<unsigned>(p.seq_T);
    }
    bool waited = false;
#pragma unroll 1
    for (int u = 0; u < units; ++u) {
      const int b1 = pd == 128 ? half_sel * 64 : (pd == 64 ? half_sel * 128 : half_sel * 128 + u * 64);  // tile column of x1
      const int pc1 = n_blk * BLOCK_N + b1;
      const bool in_range = pc1 < p.N;                  // warp-uniform
      const bool is_v = pc1 >= 2 * p.hidden;            // v third: identity layout, plain bias store
      const int nkb = pd == 32 ? 4 : 8;                 // 8-column blocks of x1 values in this unit
      int jbase = 0, dbase = 0;
      if (in_range && !is_v) {
        const int region = pc1 / p.hidden;              // 0 = q, 1 = k
        const int lp = pc1 - region * p.hidden;         // permuted column inside the region
        const int grp = lp / (2 * pd), w = lp - grp * 2 * pd;  // w < PD by construction
        const int e0 = grp * pd;                        // first "x1 element" index of this group
        const int head = e0 / p.rope_half;
        jbase = e0 - head * p.rope_half + w;            // rotary frequency index of the block's first column
        dbase = region * p.hidden + head * 2 * p.rope_half + jbase;
      }
      float2 fr[8], bx1[8], bx2[8], cx1[8], cx2[8];
#pragma unroll
      for (int kb = 0; kb < 8; ++kb) {
        fr[kb] = bx1[kb] = bx2[kb] = cx1[kb] = cx2[kb] = make_float2(0.f, 0.f);
        if (!in_range) continue;
        if (is_v) {  // plain blocks at pc1 and (PD != 32) pc1 + PD
          bx1[kb] = __ldg(reinterpret_cast<const float2*>(bias + pc1 + q2 + kb * 8));
          if (dln) cx1[kb] = __ldg(reinterpret_cast<const float2*>(p.ln_c + pc1 + q2 + kb * 8));
          if (pd != 32) {
            bx2[kb] = __ldg(reinterpret_cast<const float2*>(bias + pc1 + pd + q2 + kb * 8));
            if (dln) cx2[kb] = __ldg(reinterpret_cast<const float2*>(p.ln_c + pc1 + pd + q2 + kb * 8));
          }
        } else if (kb < nkb) {
          fr[kb] = __ldg(reinterpret_cast<const float2*>(p.rope_freq + jbase + q2 + kb * 8));
          bx1[kb] = __ldg(reinterpret_cast<const float2*>(bias + pc1 + q2 + kb * 8));
          bx2[kb] = __ldg(reinterpret_cast<const float2*>(bias + pc1 + pd + q2 + kb * 8));
          if (dln) {
            cx1[kb] = __ldg(reinterpret_cast<const float2*>(p.ln_c + pc1 + q2 + kb * 8));
            cx2[kb] = __ldg(reinterpret_cast<const float2*>(p.ln_c + pc1 + pd + q2 + kb * 8));
          }
        }
      }
      if (!waited) {
        mbar_wait(full_bar, full_parity);
        tcgen05_fence_after();
        waited = true;
      }
      if (row0 >= p.M || !in_range) continue;           // warp-uniform
#pragma unroll 1
      for (int hh = 0; hh < 2; ++hh) {
        if (row0 + hh * 16 >= p.M) break;
        const long long rowA = row0 + hh * 16 + g;
        const uint32_t tbase = t_row + (static_cast<uint32_t>(hh * 16) << 16);
        uint32_t r1[32], r2[32];
        tmem_ld_16x64(tbase + b1, r1);
        if (pd != 32) tmem_ld_16x64(tbase + b1 + pd, r2);
        const bool okA = rowA < p.M, okB = rowA + 8 < p.M;
        const float aA = hh ? lnA2 : lnA0, nA = hh ? lnN2 : lnN0, aB = hh ? lnA3 : lnA1, nB = hh ? lnN3 : lnN1;
        if (is_v) {
          tmem_ld_wait();
          bf16* vo = static_cast<bf16*>(p.out) + out_off + rowA * p.ldo + pc1 + q2;
          store_blk_bf16_ln(r1, bx1, cx1, vo, vo + 8 * p.ldo, okA, okB, pc1 + q2, p.N, aA, nA, aB, nB);
          if (pd != 32) store_blk_bf16_ln(r2, bx2, cx2, vo + pd, vo + 8 * p.ldo + pd, okA, okB, pc1 + pd + q2, p.N, aA, nA, aB, nB);
          continue;
        }
        const unsigned posA = hh ? pos4[2] : pos4[0], posB = hh ? pos4[3] : pos4[1];
        const float fposA = static_cast<float>(posA), fposB = static_cast<float>(posB);
        bf16* outp = static_cast<bf16*>(p.out) + out_off + rowA * p.ldo + dbase + q2;
        tmem_ld_wait();
#pragma unroll
        for (int kb = 0; kb < 8; ++kb) {
          if (kb >= nkb) break;
          const int k2 = (kb + 4) & 7;  // partner block inside r1 when PD == 32
#pragma unroll
          for (int rr = 0; rr < 2; ++rr) {
            float2 c2, s2;   // angle = float(pos) * inv_freq[j] exactly as the reference forms it
            const float fp = rr == 0 ? fposA : fposB;
            sincos_reduced(fp * fr[kb].x, s2.x, c2.x);
            sincos_reduced(fp * fr[kb].y, s2.y, c2.y);
            const float ar = rr == 0 ? aA : aB, nr = rr == 0 ? nA : nB;
            const float x1a = fmaf(ar, __uint_as_float(r1[4 * kb + 2 * rr]), fmaf(nr, cx1[kb].x, bx1[kb].x));
            const float x1b = fmaf(ar, __uint_as_float(r1[4 * kb + 2 * rr + 1]), fmaf(nr, cx1[kb].y, bx1[kb].y));
            const float x2a = fmaf(ar, __uint_as_float(pd == 32 ? r1[4 * k2 + 2 * rr] : r2[4 * kb + 2 * rr]), fmaf(nr, cx2[kb].x, bx2[kb].x));
            const float x2b =
                fmaf(ar, __uint_as_float(pd == 32 ? r1[4 * k2 + 2 * rr + 1] : r2[4 * kb + 2 * rr + 1]), fmaf(nr, cx2[kb].y, bx2[kb].y));
            if (rr == 0 ? okA : okB) {
              bf16* dst = outp + rr * 8 * p.ldo + kb * 8;
              // explicit rounding order (product with cos first), the same as the packed arithmetic of the lean path: a row
              // gives bit-identical results whichever of the two epilogues its tile takes
              *reinterpret_cast<uint32_t*>(dst) = pack_bf16x2(__fmaf_rn(x2a, -s2.x, __fmul_rn(x1a, c2.x)), __fmaf_rn(x2b, -s2.y, __fmul_rn(x1b, c2.y)));
              *reinterpret_cast<uint32_t*>(dst + p.rope_half) =
                  pack_bf16x2(__fmaf_rn(x1a, s2.x, __fmul_rn(x2a, c2.x)), __fmaf_rn(x1b, s2.y, __fmul_rn(x2b, c2.y)));
            }
          }
        }
      }
    }
    if (!waited) {  // not reachable (units >= 1), kept so that the accumulator wait is provably on every path
      mbar_wait(full_bar, full_parity);
      tcgen05_fence_after();
    }
  }
}

// ---------------------------------------------------------------------------------------------------
// Cluster multicast (scores kernel): a TMA load written into the shared memory of every CTA in `mask`, and an MMA commit
// that arrives on the barrier at the same offset in every CTA in `mask`.
// ---------------------------------------------------------------------------------------------------
__device__ __forceinline__ void tma_load_4d_mc(const CUtensorMap* m, uint64_t* bar, void* smem, int c0, int c1, int c2, int c3,
                                               uint16_t mask) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.tile.mbarrier::complete_tx::bytes.multicast::cluster [%0], [%1, {%3, %4, %5, %6}], "
      "[%2], %7;" ::"r"(smem_u32(smem)),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "h"(mask)
      : "memory");
}

// Register re-distribution between the warp roles (setmaxnreg, one instruction per warpgroup): warps 0-3 (TMA producer,
// MMA issuer, TMEM allocator, idle) shrink to 56 registers, the two epilogue warpgroups grow from the launch-bound limit
// of 168 to 224 -- the fused epilogues (RoPE, GLU, residual + statistics) keep two accumulator blocks, their constants and
// the prefetched residual live at once and spilled at 168.
template <int EPI, bool B_KN>
__global__ void __launch_bounds__(NUM_THREADS, 1)
    tc_gemm_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_b, const DevParams p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw_addr = smem_u32(smem_raw);
  uint8_t* smem = smem_raw + ((1024u - (raw_addr & 1023u)) & 1023u);  // SWIZZLE_128B needs 1024-B aligned stages
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + STAGES * STAGE_BYTES);
  uint64_t* empty_bar = full_bar + STAGES;
  uint64_t* tmem_full = empty_bar + STAGES;
  uint64_t* tmem_empty = tmem_full + 2;
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(tmem_empty + 2);

  const int warp = warp_id_uniform();   // control warps run on warp-uniform values (see common.cuh: elect_one)
  const int lane = threadIdx.x & 31;
  // tile = (batch item, m_blk, n_blk), n_blk fastest

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmap_a);
    tma_prefetch_desc(&tmap_b);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init(&tmem_full[s], 1);
      mbar_init(&tmem_empty[s], NUM_EPI_WARPS);
    }
    fence_barrier_init();
  }
  if (warp == 2) tmem_alloc<TMEM_COLS>(tmem_ptr);
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem_base = *tmem_ptr;

  if (warp == 0) {
    // =========================== TMA producer (whole warp, one elected lane issues) ===========================
    regs_shrink_ctrl();
    const bool leader = elect_one();
    int stage = 0;
    uint32_t phase = 0;
    for (int tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x) {
      const int n_blk = tile % p.n_tiles;
      const int rest = tile / p.n_tiles;
      const int m_blk = rest % p.m_tiles;
      const int b = rest / p.m_tiles;
      const int bo = b / p.batch_inner, bi = b - bo * p.batch_inner;
      const int abi = p.a_bi ? bi : 0, abo = p.a_bo ? bo : 0;
      const int bbi = p.b_bi ? bi : 0, bbo = p.b_bo ? bo : 0;
      for (int kb = 0; kb < p.num_kb; ++kb) {
        mbar_wait(&empty_bar[stage], phase ^ 1u);
        if (leader) {
          uint8_t* sa = smem + stage * STAGE_BYTES;
          uint8_t* sb = sa + A_STAGE_BYTES;
          mbar_expect_tx(&full_bar[stage], STAGE_BYTES);
          tma_load_4d(&tmap_a, &full_bar[stage], sa, kb * BLOCK_K, m_blk * BLOCK_M, abi, abo);
          if (!B_KN) {
            tma_load_4d(&tmap_b, &full_bar[stage], sb, kb * BLOCK_K, n_blk * BLOCK_N, bbi, bbo);
          } else {
#pragma unroll
            for (int j = 0; j < BLOCK_N / 64; ++j)  // [64 k-rows x 64 n] boxes, N-contiguous (MN-major operand)
              tma_load_4d(&tmap_b, &full_bar[stage], sb + j * (BLOCK_K * 128), n_blk * BLOCK_N + j * 64, kb * BLOCK_K, bbi, bbo);
          }
        }
        __syncwarp();
        if (++stage == STAGES) { stage = 0; phase ^= 1u; }
      }
    }
  } else if (warp == 1) {
    // =========================== MMA issuer (whole warp, one elected lane issues) ===========================
    regs_shrink_ctrl();
    const bool leader = elect_one();
    constexpr uint32_t idesc = umma_idesc_bf16(BLOCK_M, BLOCK_N, false, B_KN);
    // operand descriptors of ring slot 0; a slot / k-step only adds to the 14-bit address field (16-byte units, no carry:
    // shared memory ends below 256 KiB)
    const uint64_t da0 = umma_smem_desc(smem_u32(smem), 16, 1024);
    const uint64_t db0 = B_KN ? umma_smem_desc(smem_u32(smem) + A_STAGE_BYTES, BLOCK_K * 128, 1024)
                              : umma_smem_desc(smem_u32(smem) + A_STAGE_BYTES, 16, 1024);
    int stage = 0;
    uint32_t phase = 0;
    int as = 0;
    uint32_t aphase = 0;
    for (int tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x) {
      mbar_wait(&tmem_empty[as], aphase ^ 1u);  // epilogue has drained this accumulator stage
      tcgen05_fence_after();
      const uint32_t d_tmem = tmem_base + static_cast<uint32_t>(as * BLOCK_N);
      for (int kb = 0; kb < p.num_kb; ++kb) {
        mbar_wait(&full_bar[stage], phase);
        tcgen05_fence_after();
        if (leader) {
          const uint64_t da = da0 + static_cast<uint64_t>((stage * STAGE_BYTES) >> 4), db = db0 + static_cast<uint64_t>((stage * STAGE_BYTES) >> 4);
#pragma unroll
          for (int k = 0; k < BLOCK_K / UMMA_K; ++k)
            umma_bf16(d_tmem, da + ((k * (UMMA_K * 2)) >> 4), db + ((B_KN ? k * (UMMA_K * 128) : k * (UMMA_K * 2)) >> 4), idesc,
                      (kb | k) != 0 ? 1u : 0u);
          umma_commit(&empty_bar[stage]);  // smem slot reusable once these MMAs retire
        }
        __syncwarp();
        if (++stage == STAGES) { stage = 0; phase ^= 1u; }
      }
      if (leader) umma_commit(&tmem_full[as]);  // accumulator complete -> epilogue
      __syncwarp();
      if (++as == 2) { as = 0; aphase ^= 1u; }
    }
  } else if (warp >= EPI_WARP0) {
    // =========================== epilogue: TMEM -> registers -> global ===========================
    regs_grow_epi();
    const int ew = warp - EPI_WARP0;
    const int quarter = warp & 3;  // TMEM lanes [32*quarter, +32) are the ones this warp may touch
    const int half_sel = ew >> 2;  // which 4 of the 8 column chunks
    int as = 0;
    uint32_t aphase = 0;
    for (int tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x) {
      const int n_blk = tile % p.n_tiles;
      const int rest = tile / p.n_tiles;
      const int m_blk = rest % p.m_tiles;
      const int b = rest / p.m_tiles;
      const int bo = b / p.batch_inner, bi = b - bo * p.batch_inner;
      const long long out_off = bo * p.so_outer + bi * p.so_inner;
      const long long res_off = bo * p.sr_outer + bi * p.sr_inner;
      const long long bias_off = bo * p.sb_outer + bi * p.sb_inner;
      const long long row0 = static_cast<long long>(m_blk) * BLOCK_M + quarter * 32;
      const uint32_t t_row = tmem_base + (static_cast<uint32_t>(quarter * 32) << 16) + static_cast<uint32_t>(as * BLOCK_N);
      const long long ls_off = bo * p.sl_outer + bi * p.sl_inner;
      const long long st_off = (bo * p.stat_rows_outer) * p.stat_parts + static_cast<long long>(bi) * p.stat_parts_item;
      epilogue_tile<EPI>(p, lane, half_sel, t_row, row0, n_blk, out_off, res_off, bias_off, ls_off, st_off, &tmem_full[as], aphase);
      tcgen05_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tmem_empty[as]);
      if (++as == 2) { as = 0; aphase ^= 1u; }
    }
  } else {
    regs_shrink_ctrl();  // warps 2 and 3 idle; the whole warpgroup has to execute the setmaxnreg
  }

  __syncwarp();
  tcgen05_fence_before();
  __syncthreads();
  if (warp == 2) {
    tcgen05_fence_after();
    tmem_dealloc<TMEM_COLS>(tmem_base);
  }
}

// =====================================================================================================
// cta_group::2 variant: a cluster of two CTAs (one SM pair) computes a 256 x 256 tile.  Each CTA loads its own 128 rows
// of A and HALF of the B tile (128 of the 256 N-rows); the leader CTA issues tcgen05.mma.cta_group::2 (UMMA 256x256x16)
// which reads both halves, so B is fetched into shared memory once per SM pair: 32 KiB per stage and CTA -> 6 stages.
// Accumulators: each CTA's TMEM holds its own 128 rows.  K-major ("NK") B only, no batching (weight GEMMs).
// =====================================================================================================
constexpr int P_STAGES = 6;
constexpr int P_B_STAGE_BYTES = (BLOCK_N / 2) * BLOCK_K * 2;  // 16 KiB
constexpr int P_STAGE_BYTES = A_STAGE_BYTES + P_B_STAGE_BYTES;  // 32 KiB
constexpr int P_SMEM_BYTES = P_STAGES * P_STAGE_BYTES + BARRIER_BYTES + 1024;
static_assert(P_SMEM_BYTES <= 232448, "exceeds the 227 KiB shared memory of an sm_100 CTA");
static_assert((2 * P_STAGES + 4) * 8 + 4 <= BARRIER_BYTES, "barrier block too small");
template <int EPI>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(NUM_THREADS, 1)
    tc_gemm_pair_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_b, const DevParams p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw_addr = smem_u32(smem_raw);
  uint8_t* smem = smem_raw + ((1024u - (raw_addr & 1023u)) & 1023u);
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + P_STAGES * P_STAGE_BYTES);
  uint64_t* empty_bar = full_bar + P_STAGES;
  uint64_t* tmem_full = empty_bar + P_STAGES;
  uint64_t* tmem_empty = tmem_full + 2;
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(tmem_empty + 2);

  const int warp = warp_id_uniform();
  const int lane = threadIdx.x & 31;
  const uint32_t rank = __shfl_sync(0xffffffffu, cluster_ctarank(), 0);   // provably warp-uniform (see common.cuh: elect_one)
  const int num_pairs = gridDim.x >> 1;
  const int pair_id = blockIdx.x >> 1;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmap_a);
    tma_prefetch_desc(&tmap_b);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < P_STAGES; ++s) {
      mbar_init(&full_bar[s], 1);   // leader's copy is the one in use: 1 arrive (expect_tx) + bytes of both CTAs
      mbar_init(&empty_bar[s], 1);  // one multicast commit per use, delivered to both CTAs
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init(&tmem_full[s], 1);
      mbar_init(&tmem_empty[s], 2 * NUM_EPI_WARPS);  // leader's copy: epilogue warps of both CTAs
    }
    fence_barrier_init();
  }
  if (warp == 2) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_ptr)), "n"(TMEM_COLS) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
  }
  __syncwarp();
  tcgen05_fence_before();
  cluster_sync_all();  // peer barriers initialised and TMEM allocated on both SMs before any remote arrive / MMA
  tcgen05_fence_after();
  const uint32_t tmem_base = *tmem_ptr;

  // tile = (m_pair, n_blk), n fastest; M is covered in 256-row pair tiles
  const int m_pairs = (p.M + 2 * BLOCK_M - 1) / (2 * BLOCK_M);
  const int num_tiles = m_pairs * p.n_tiles;

  if (warp == 0) {
    // TMA producer: whole warp on warp-uniform values, one elected lane issues
    regs_shrink_ctrl();
    const bool leader = elect_one();
    int stage = 0;
    uint32_t phase = 0;
    long long w_slot = 0;
    const long long t_begin = (kDbgCounters && p.dbg) ? clock64() : 0;
    for (int tile = pair_id; tile < num_tiles; tile += num_pairs) {
      const int n_blk = tile % p.n_tiles, m_pair = tile / p.n_tiles;
      const int m0 = m_pair * 2 * BLOCK_M + static_cast<int>(rank) * BLOCK_M;
      const int n0 = n_blk * BLOCK_N + static_cast<int>(rank) * (BLOCK_N / 2);
      for (int kb = 0; kb < p.num_kb; ++kb) {
        if (kDbgCounters && p.dbg) {
          const long long t0 = clock64();
          mbar_wait(&empty_bar[stage], phase ^ 1u);
          w_slot += clock64() - t0;
        } else {
          mbar_wait(&empty_bar[stage], phase ^ 1u);
        }
        if (leader) {
          uint8_t* sa = smem + stage * P_STAGE_BYTES;
          uint8_t* sb = sa + A_STAGE_BYTES;
          if (rank == 0) mbar_expect_tx(&full_bar[stage], 2 * P_STAGE_BYTES);
          tma_load_4d_2sm(&tmap_a, &full_bar[stage], sa, kb * BLOCK_K, m0, 0, 0);
          tma_load_4d_2sm(&tmap_b, &full_bar[stage], sb, kb * BLOCK_K, n0, 0, 0);
        }
        __syncwarp();
        if (++stage == P_STAGES) { stage = 0; phase ^= 1u; }
      }
    }
    if (kDbgCounters && p.dbg && rank == 0 && leader) {
      atomicAdd(p.dbg + EPI * 8 + 3, static_cast<unsigned long long>(w_slot));
      atomicAdd(p.dbg + EPI * 8 + 4, static_cast<unsigned long long>(clock64() - t_begin));
    }
  } else if (warp == 1) {
    regs_shrink_ctrl();
    if (rank == 0) {   // the leader CTA issues for the pair; whole warp on warp-uniform values, one elected lane issues
      const bool leader = elect_one();
      constexpr uint32_t idesc = umma_idesc_bf16(2 * BLOCK_M, BLOCK_N, false, false);
      const uint64_t da0 = umma_smem_desc(smem_u32(smem), 16, 1024);
      const uint64_t db0 = umma_smem_desc(smem_u32(smem) + A_STAGE_BYTES, 16, 1024);
      int stage = 0;
      uint32_t phase = 0;
      int as = 0;
      uint32_t aphase = 0;
      long long w_ops = 0, w_acc = 0;
      const long long t_begin = (kDbgCounters && p.dbg) ? clock64() : 0;
      for (int tile = pair_id; tile < num_tiles; tile += num_pairs) {
        if (kDbgCounters && p.dbg) {
          const long long t0 = clock64();
          mbar_wait(&tmem_empty[as], aphase ^ 1u);
          w_acc += clock64() - t0;
        } else {
          mbar_wait(&tmem_empty[as], aphase ^ 1u);
        }
        tcgen05_fence_after();
        const uint32_t d_tmem = tmem_base + static_cast<uint32_t>(as * BLOCK_N);
        for (int kb = 0; kb < p.num_kb; ++kb) {
          if (kDbgCounters && p.dbg) {
            const long long t0 = clock64();
            mbar_wait(&full_bar[stage], phase);
            w_ops += clock64() - t0;
          } else {
            mbar_wait(&full_bar[stage], phase);
          }
          tcgen05_fence_after();
          if (leader) {
            const uint64_t da = da0 + static_cast<uint64_t>((stage * P_STAGE_BYTES) >> 4), db = db0 + static_cast<uint64_t>((stage * P_STAGE_BYTES) >> 4);
#pragma unroll
            for (int k = 0; k < BLOCK_K / UMMA_K; ++k)
              umma_bf16_2sm(d_tmem, da + ((k * (UMMA_K * 2)) >> 4), db + ((k * (UMMA_K * 2)) >> 4), idesc, (kb | k) != 0 ? 1u : 0u);
            umma_commit_2sm(&empty_bar[stage]);
          }
          __syncwarp();
          if (++stage == P_STAGES) { stage = 0; phase ^= 1u; }
        }
        if (leader) umma_commit_2sm(&tmem_full[as]);
        __syncwarp();
        if (++as == 2) { as = 0; aphase ^= 1u; }
      }
      if (kDbgCounters && p.dbg && leader) {
        atomicAdd(p.dbg + EPI * 8 + 0, static_cast<unsigned long long>(w_ops));
        atomicAdd(p.dbg + EPI * 8 + 1, static_cast<unsigned long long>(w_acc));
        atomicAdd(p.dbg + EPI * 8 + 2, static_cast<unsigned long long>(clock64() - t_begin));
      }
    }
  } else if (warp >= EPI_WARP0) {
    regs_grow_epi();
    const int ew = warp - EPI_WARP0;
    const int quarter = warp & 3;
    const int half_sel = ew >> 2;
    int as = 0;
    uint32_t aphase = 0;
    for (int tile = pair_id; tile < num_tiles; tile += num_pairs) {
      const int n_blk = tile % p.n_tiles, m_pair = tile / p.n_tiles;
      const long long row0 = static_cast<long long>(m_pair) * 2 * BLOCK_M + rank * BLOCK_M + quarter * 32;
      const uint32_t t_row = tmem_base + (static_cast<uint32_t>(quarter * 32) << 16) + static_cast<uint32_t>(as * BLOCK_N);
      epilogue_tile<EPI>(p, lane, half_sel, t_row, row0, n_blk, 0, 0, 0, 0, 0, &tmem_full[as], aphase);
      tcgen05_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive_leader(&tmem_empty[as]);
      if (++as == 2) { as = 0; aphase ^= 1u; }
    }
  } else {
    regs_shrink_ctrl();  // warps 2 and 3 idle; the whole warpgroup has to execute the setmaxnreg
  }

  __syncwarp();
  tcgen05_fence_before();
  cluster_sync_all();  // nobody leaves while the peer may still signal its barriers / read its shared memory
  if (warp == 2) {
    tcgen05_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(TMEM_COLS) : "memory");
  }
}

// =====================================================================================================
// Fused attention scores + softmax (flash-style: the fp32 score tile lives in TMEM only).
//   One cluster of `csize` CTAs per work item (batch item, 128 query rows); CTA `rank` computes the 128 x 256 score tile
//   of key columns [256 rank, +256) with the same TMA ring / tcgen05 main loop as the GEMM above (K = head dim), then
//     pass 1  row maxima of the tile (accumulator fragments -> quad shuffles), written into EVERY peer's shared memory
//             (st.shared::cluster) and announced on the peer's mbarrier (remote arrive, release.cluster);
//     pass 2  p = 2^(s' - max') in log2 domain, bf16 store of P, row sums.
//   csize == 1: a third pass stores the normalised probabilities.  csize > 1: P stays unnormalised (values in (0, 1]) and
//   the partial sums go to lpart[row][rank]; the P.V GEMM applies 1 / sum in its epilogue (DevParams::row_lsum).
//   Persistent over work items with double-buffered TMEM, so the exchange of item i overlaps the MMAs of item i + 1.
// =====================================================================================================
constexpr int SM_MAX_CLUSTER = 16;
constexpr int SM_STAT_BYTES = 2 * SM_MAX_CLUSTER * BLOCK_M * 4;  // [acc stage][peer rank][row] row maxima
constexpr int SM_SMEM_BYTES = STAGES * STAGE_BYTES + BARRIER_BYTES + SM_STAT_BYTES + 1024;
static_assert(SM_SMEM_BYTES <= 232448, "exceeds the 227 KiB shared memory of an sm_100 CTA");

struct SmDev {
  int M, N, K;
  int batch_inner, batch_outer;
  int m_tiles, num_items, num_kb;
  int a_bi, a_bo, b_bi, b_bo;
  float alpha2;                 // alpha * log2(e)
  const float* bias; long long sb_inner, sb_outer;
  bf16* P; long long ldp, sp_inner, sp_outer;
  int npad;
  float* lpart; long long sl_inner, sl_outer;
  int csize;   // key tiles per row = CTAs per cluster
  const int* col_len;   // optional [batch_outer] valid key columns of each outer batch item (masked text); null: N
  // deferred LayerNorm of the query operand (HAS_BIAS variant): s = alpha (rstd acc - rstd mean c[col]) + bias[col];
  // statistics row = outer batch index * M + query row; c has the layout / strides of bias
  const float2* ln_stat; int ln_parts; float ln_inv_h; const float* ln_c;
};

__device__ __forceinline__ uint32_t cluster_nctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_nctarank;" : "=r"(r));
  return r;
}
template <bool HAS_BIAS>
__global__ void __launch_bounds__(NUM_THREADS, 1)
    tc_scores_softmax_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_b, const SmDev p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw_addr = smem_u32(smem_raw);
  uint8_t* smem = smem_raw + ((1024u - (raw_addr & 1023u)) & 1023u);
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + STAGES * STAGE_BYTES);
  uint64_t* empty_bar = full_bar + STAGES;
  uint64_t* tmem_full = empty_bar + STAGES;
  uint64_t* tmem_empty = tmem_full + 2;
  uint64_t* stat_bar = tmem_empty + 2;  // [2]
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(stat_bar + 2);
  float* stat = reinterpret_cast<float*>(smem + STAGES * STAGE_BYTES + BARRIER_BYTES);  // [2][SM_MAX_CLUSTER][BLOCK_M]

  const int warp = warp_id_uniform();
  const int lane = threadIdx.x & 31;
  // CTA `rank` of the cluster computes the work item's query block against key tile `rank`; the Q block is multicast to
  // the whole cluster, the row maxima are exchanged across it
  const int csize = p.csize;
  const int rank = csize > 1 ? static_cast<int>(cluster_ctarank()) : 0;
  const uint16_t cluster_mask = static_cast<uint16_t>((1u << csize) - 1u);
  const int num_clusters = gridDim.x / csize;
  const int cluster_id = blockIdx.x / csize;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmap_a);
    tma_prefetch_desc(&tmap_b);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], static_cast<uint32_t>(csize));   // a slot is free once every CTA's MMAs have read its Q block
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init(&tmem_full[s], 1);
      mbar_init(&tmem_empty[s], NUM_EPI_WARPS);
      mbar_init(&stat_bar[s], 1);  // one local arrive.expect_tx per use; the row maxima arrive as st.async transactions
    }
    fence_barrier_init();
  }
  if (warp == 2) tmem_alloc<TMEM_COLS>(tmem_ptr);
  tcgen05_fence_before();
  __syncthreads();
  if (csize > 1) cluster_sync_all();  // every peer's barriers are initialised before the first remote arrive / multicast
  tcgen05_fence_after();
  const uint32_t tmem_base = *tmem_ptr;

  if (warp == 0) {
    // =========================== TMA producer (whole warp, one elected lane issues) ===========================
    regs_shrink_ctrl();
    const bool leader = elect_one();
    int stage = 0;
    uint32_t phase = 0;
    for (int item = cluster_id; item < p.num_items; item += num_clusters) {
      const int m_blk = item % p.m_tiles;
      const int b = item / p.m_tiles;
      const int bo = b / p.batch_inner, bi = b - bo * p.batch_inner;
      const int abi = p.a_bi ? bi : 0, abo = p.a_bo ? bo : 0;
      const int bbi = p.b_bi ? bi : 0, bbo = p.b_bo ? bo : 0;
      for (int kb = 0; kb < p.num_kb; ++kb) {
        mbar_wait(&empty_bar[stage], phase ^ 1u);
        if (leader) {
          uint8_t* sa = smem + stage * STAGE_BYTES;
          uint8_t* sb = sa + A_STAGE_BYTES;
          mbar_expect_tx(&full_bar[stage], STAGE_BYTES);
          if (csize == 1)
            tma_load_4d(&tmap_a, &full_bar[stage], sa, kb * BLOCK_K, m_blk * BLOCK_M, abi, abo);
          else if (kb % csize == rank)   // the CTAs take turns fetching the Q block for the whole cluster
            tma_load_4d_mc(&tmap_a, &full_bar[stage], sa, kb * BLOCK_K, m_blk * BLOCK_M, abi, abo, cluster_mask);
          tma_load_4d(&tmap_b, &full_bar[stage], sb, kb * BLOCK_K, rank * BLOCK_N, bbi, bbo);
        }
        __syncwarp();
        if (++stage == STAGES) { stage = 0; phase ^= 1u; }
      }
    }
  } else if (warp == 1) {
    // =========================== MMA issuer (whole warp, one elected lane issues) ===========================
    regs_shrink_ctrl();
    const bool leader = elect_one();
    constexpr uint32_t idesc = umma_idesc_bf16(BLOCK_M, BLOCK_N, false, false);
    const uint64_t da0 = umma_smem_desc(smem_u32(smem), 16, 1024);
    const uint64_t db0 = umma_smem_desc(smem_u32(smem) + A_STAGE_BYTES, 16, 1024);
    int stage = 0;
    uint32_t phase = 0;
    int as = 0;
    uint32_t aphase = 0;
    for (int item = cluster_id; item < p.num_items; item += num_clusters) {
      mbar_wait(&tmem_empty[as], aphase ^ 1u);
      tcgen05_fence_after();
      const uint32_t d_tmem = tmem_base + static_cast<uint32_t>(as * BLOCK_N);
      for (int kb = 0; kb < p.num_kb; ++kb) {
        mbar_wait(&full_bar[stage], phase);
        tcgen05_fence_after();
        if (leader) {
          const uint64_t da = da0 + static_cast<uint64_t>((stage * STAGE_BYTES) >> 4), db = db0 + static_cast<uint64_t>((stage * STAGE_BYTES) >> 4);
#pragma unroll
          for (int k = 0; k < BLOCK_K / UMMA_K; ++k)
            umma_bf16(d_tmem, da + ((k * (UMMA_K * 2)) >> 4), db + ((k * (UMMA_K * 2)) >> 4), idesc, (kb | k) != 0 ? 1u : 0u);
          if (csize == 1) umma_commit(&empty_bar[stage]);
          else umma_commit_mc(&empty_bar[stage], cluster_mask);   // every CTA's slot may hold a Q block this CTA multicast
        }
        __syncwarp();
        if (++stage == STAGES) { stage = 0; phase ^= 1u; }
      }
      if (leader) umma_commit(&tmem_full[as]);
      __syncwarp();
      if (++as == 2) { as = 0; aphase ^= 1u; }
    }
  } else if (warp >= EPI_WARP0) {
    // =========================== softmax epilogue ===========================
    regs_grow_epi();
    // warp -> TMEM lanes [32 (warp & 3), +32); its 16-row half hsel = (warp - EPI_WARP0) >> 2; all 256 tile columns
    const int ew = warp - EPI_WARP0;
    const int quarter = warp & 3, hsel = ew >> 2;
    const int g = lane >> 2, q2 = (lane & 3) * 2;
    const int trow = quarter * 32 + hsel * 16;  // first tile row of this warp
    const int col_base = rank * BLOCK_N;        // first key column of this CTA
    const bool writer = (lane & 3) == 0;
    int as = 0;
    uint32_t aphase = 0;
    for (int item = cluster_id; item < p.num_items; item += num_clusters) {
      const int m_blk = item % p.m_tiles;
      const int b = item / p.m_tiles;
      const int bo = b / p.batch_inner, bi = b - bo * p.batch_inner;
      // valid key columns of this item: columns [nv, N) are masked keys and get probability 0 like the padding.  Always >= 1
      // (key 0 is valid), so rank 0 sees a finite row maximum; a CTA whose whole tile is masked contributes -inf to the
      // exchange and a zero partial sum.  Full 64-column blocks below nv keep the lean path.
      const int nv = p.col_len != nullptr ? min(p.N, __ldg(p.col_len + bo)) : p.N;
      // second row: rowA + 8
      const long long rowA = static_cast<long long>(m_blk) * BLOCK_M + trow + g;
      const bool okA = rowA < p.M, okB = rowA + 8 < p.M;
      const float* bias = HAS_BIAS ? p.bias + bo * p.sb_outer + bi * p.sb_inner : nullptr;
      const float* lnc = (HAS_BIAS && p.ln_stat != nullptr) ? p.ln_c + bo * p.sb_outer + bi * p.sb_inner : nullptr;
      const uint32_t t_row = tmem_base + (static_cast<uint32_t>(trow) << 16) + static_cast<uint32_t>(as * BLOCK_N);
      // s' = aX acc + (nX c + bias log2e): (alpha2, 0) without the deferred LayerNorm
      float aA = p.alpha2, nA = 0.f, aB = p.alpha2, nB = 0.f;
      if (HAS_BIAS && lnc != nullptr) {
        const long long srow = static_cast<long long>(bo) * p.M + rowA;
        ln_row_coef(p.ln_stat, p.ln_parts, srow, okA, p.ln_inv_h, aA, nA);
        ln_row_coef(p.ln_stat, p.ln_parts, srow + 8, okB, p.ln_inv_h, aB, nB);
        aA *= p.alpha2; nA *= p.alpha2; aB *= p.alpha2; nB *= p.alpha2;
      }
      mbar_wait(&tmem_full[as], aphase);
      tcgen05_fence_after();

      // ---- pass 1: row maxima of this tile (log2 domain: s' = (alpha acc + bias) log2 e)
      float mA = -INFINITY, mB = -INFINITY;
#pragma unroll 1
      for (int cbk = 0; cbk < 4; ++cbk) {
        const int col0 = col_base + cbk * 64 + q2;
        if (col0 - q2 >= nv) break;  // warp-uniform
        uint32_t r[32];
        tmem_ld_16x64(t_row + cbk * 64, r);
        if (!HAS_BIAS && col0 - q2 + 64 <= nv) {
          // lean block (no bias, all 64 columns valid): s' = alpha2 acc with alpha2 > 0, so the maximum is taken on the raw
          // accumulators and scaled once -- 1 instruction per element instead of ~7 (the generic block below predicates and
          // rescales every element; ncu: 21 instructions per score made this epilogue, not the MMA, the pace of the kernel)
          tmem_ld_wait();
          float rA = -INFINITY, rB = -INFINITY;
#pragma unroll
          for (int kb = 0; kb < 8; ++kb) {
            rA = fmaxf(rA, fmaxf(__uint_as_float(r[4 * kb]), __uint_as_float(r[4 * kb + 1])));
            rB = fmaxf(rB, fmaxf(__uint_as_float(r[4 * kb + 2]), __uint_as_float(r[4 * kb + 3])));
          }
          mA = fmaxf(mA, rA * p.alpha2);
          mB = fmaxf(mB, rB * p.alpha2);
          continue;
        }
        float2 bb[8], cc[8];
#pragma unroll
        for (int kb = 0; kb < 8; ++kb) {
          bb[kb] = cc[kb] = make_float2(0.f, 0.f);
          if (HAS_BIAS) {
            const int c = col0 + kb * 8;
            if (c < nv) bb[kb].x = __ldg(bias + c) * 1.4426950408889634f;
            if (c + 1 < nv) bb[kb].y = __ldg(bias + c + 1) * 1.4426950408889634f;
            if (lnc != nullptr) {
              if (c < nv) cc[kb].x = __ldg(lnc + c);
              if (c + 1 < nv) cc[kb].y = __ldg(lnc + c + 1);
            }
          }
        }
        tmem_ld_wait();
#pragma unroll
        for (int kb = 0; kb < 8; ++kb) {
          const int c = col0 + kb * 8;
          if (c < nv) {
            mA = fmaxf(mA, fmaf(aA, __uint_as_float(r[4 * kb]), fmaf(nA, cc[kb].x, bb[kb].x)));
            mB = fmaxf(mB, fmaf(aB, __uint_as_float(r[4 * kb + 2]), fmaf(nB, cc[kb].x, bb[kb].x)));
          }
          if (c + 1 < nv) {
            mA = fmaxf(mA, fmaf(aA, __uint_as_float(r[4 * kb + 1]), fmaf(nA, cc[kb].y, bb[kb].y)));
            mB = fmaxf(mB, fmaf(aB, __uint_as_float(r[4 * kb + 3]), fmaf(nB, cc[kb].y, bb[kb].y)));
          }
        }
      }
      mA = quad_max(mA);
      mB = quad_max(mB);

      // ---- exchange through distributed shared memory: every writer lane sends its two row maxima to every CTA of the
      //      cluster (own CTA included); each CTA expects csize * 64 lanes * 8 bytes per work item
      if (csize > 1) {
        if (ew == 0 && lane == 0) mbar_expect_tx(&stat_bar[as], static_cast<uint32_t>(csize * NUM_EPI_WARPS * 8 * 8));
        if (writer) {
          const uint32_t slotA = smem_u32(stat + (as * SM_MAX_CLUSTER + rank) * BLOCK_M + trow + g);
          const uint32_t barl = smem_u32(&stat_bar[as]);
          for (int c = 0; c < csize; ++c) {
            const uint32_t ra = mapa_shared(slotA, static_cast<uint32_t>(c));
            const uint32_t rb = mapa_shared(barl, static_cast<uint32_t>(c));
            st_async_f32(ra, mA, rb);
            st_async_f32(ra + 8 * 4, mB, rb);
          }
        }
        mbar_wait(&stat_bar[as], aphase);
        const float* sp = stat + as * SM_MAX_CLUSTER * BLOCK_M + trow + g;
        for (int c = 0; c < csize; ++c) {
          mA = fmaxf(mA, sp[c * BLOCK_M]);
          mB = fmaxf(mB, sp[c * BLOCK_M + 8]);
        }
        __syncwarp();
      }

      // ---- pass 2: exponentials, row sums; csize > 1: store the unnormalised P
      bf16* Pb = p.P + bo * p.sp_outer + bi * p.sp_inner;
      bf16* pA = Pb + rowA * p.ldp;
      bf16* pB = pA + 8 * p.ldp;
      float sumA = 0.f, sumB = 0.f;
      const bool store2 = csize > 1;
#pragma unroll 1
      for (int cbk = 0; cbk < 4; ++cbk) {
        const int col0 = col_base + cbk * 64 + q2;
        if (col0 - q2 >= p.npad) break;  // warp-uniform (npad >= N)
        uint32_t r[32];
        tmem_ld_16x64(t_row + cbk * 64, r);
        if (!HAS_BIAS && store2 && col0 - q2 + 64 <= nv) {
          // lean block: exp2(alpha2 acc - m) in one FMA + MUFU per element, packed row sums, unpredicated column logic
          tmem_ld_wait();
          float2 sA2 = make_float2(0.f, 0.f), sB2 = make_float2(0.f, 0.f);
          bf16* qA = pA + col0;
          bf16* qB = pB + col0;
#pragma unroll
          for (int kb = 0; kb < 8; ++kb) {
            const float2 eA = make_float2(ex2_approx(fmaf(__uint_as_float(r[4 * kb]), p.alpha2, -mA)),
                                          ex2_approx(fmaf(__uint_as_float(r[4 * kb + 1]), p.alpha2, -mA)));
            const float2 eB = make_float2(ex2_approx(fmaf(__uint_as_float(r[4 * kb + 2]), p.alpha2, -mB)),
                                          ex2_approx(fmaf(__uint_as_float(r[4 * kb + 3]), p.alpha2, -mB)));
            sA2 = __fadd2_rn(sA2, eA);
            sB2 = __fadd2_rn(sB2, eB);
            if (okA) *reinterpret_cast<uint32_t*>(qA + kb * 8) = pack_bf16x2(eA.x, eA.y);
            if (okB) *reinterpret_cast<uint32_t*>(qB + kb * 8) = pack_bf16x2(eB.x, eB.y);
          }
          sumA += sA2.x + sA2.y;
          sumB += sB2.x + sB2.y;
          continue;
        }
        float2 bb[8], cc[8];
#pragma unroll
        for (int kb = 0; kb < 8; ++kb) {
          bb[kb] = cc[kb] = make_float2(0.f, 0.f);
          if (HAS_BIAS) {
            const int c = col0 + kb * 8;
            if (c < nv) bb[kb].x = __ldg(bias + c) * 1.4426950408889634f;
            if (c + 1 < nv) bb[kb].y = __ldg(bias + c + 1) * 1.4426950408889634f;
            if (lnc != nullptr) {
              if (c < nv) cc[kb].x = __ldg(lnc + c);
              if (c + 1 < nv) cc[kb].y = __ldg(lnc + c + 1);
            }
          }
        }
        tmem_ld_wait();
#pragma unroll
        for (int kb = 0; kb < 8; ++kb) {
          const int c = col0 + kb * 8;
          const bool v0 = c < nv, v1 = c + 1 < nv;
          const float a0 = v0 ? ex2_approx(fmaf(aA, __uint_as_float(r[4 * kb]), fmaf(nA, cc[kb].x, bb[kb].x)) - mA) : 0.f;
          const float a1 = v1 ? ex2_approx(fmaf(aA, __uint_as_float(r[4 * kb + 1]), fmaf(nA, cc[kb].y, bb[kb].y)) - mA) : 0.f;
          const float b0 = v0 ? ex2_approx(fmaf(aB, __uint_as_float(r[4 * kb + 2]), fmaf(nB, cc[kb].x, bb[kb].x)) - mB) : 0.f;
          const float b1 = v1 ? ex2_approx(fmaf(aB, __uint_as_float(r[4 * kb + 3]), fmaf(nB, cc[kb].y, bb[kb].y)) - mB) : 0.f;
          sumA += a0 + a1;
          sumB += b0 + b1;
          if (store2 && c < p.npad) {  // npad is even: the pair (c, c + 1) is inside the row
            if (okA) *reinterpret_cast<uint32_t*>(pA + c) = pack_bf16x2(a0, a1);
            if (okB) *reinterpret_cast<uint32_t*>(pB + c) = pack_bf16x2(b0, b1);
          }
        }
      }
      sumA = quad_sum(sumA);
      sumB = quad_sum(sumB);
      if (csize > 1) {
        if (writer) {
          float* lp = p.lpart + bo * p.sl_outer + bi * p.sl_inner + rowA * csize + rank;
          if (okA) lp[0] = sumA;
          if (okB) lp[8 * csize] = sumB;
        }
      } else {
        // ---- pass 3 (single tile): normalised probabilities
        const float iA = 1.0f / sumA, iB = 1.0f / sumB;
#pragma unroll 1
        for (int cbk = 0; cbk < 4; ++cbk) {
          const int col0 = col_base + cbk * 64 + q2;
          if (col0 - q2 >= p.npad) break;
          uint32_t r[32];
          tmem_ld_16x64(t_row + cbk * 64, r);
          float2 bb[8], cc[8];
#pragma unroll
          for (int kb = 0; kb < 8; ++kb) {
            bb[kb] = cc[kb] = make_float2(0.f, 0.f);
            if (HAS_BIAS) {
              const int c = col0 + kb * 8;
              if (c < nv) bb[kb].x = __ldg(bias + c) * 1.4426950408889634f;
              if (c + 1 < nv) bb[kb].y = __ldg(bias + c + 1) * 1.4426950408889634f;
              if (lnc != nullptr) {
                if (c < nv) cc[kb].x = __ldg(lnc + c);
                if (c + 1 < nv) cc[kb].y = __ldg(lnc + c + 1);
              }
            }
          }
          tmem_ld_wait();
#pragma unroll
          for (int kb = 0; kb < 8; ++kb) {
            const int c = col0 + kb * 8;
            if (c >= p.npad) continue;
            const bool v0 = c < nv, v1 = c + 1 < nv;
            const float a0 = v0 ? ex2_approx(fmaf(aA, __uint_as_float(r[4 * kb]), fmaf(nA, cc[kb].x, bb[kb].x)) - mA) * iA : 0.f;
            const float a1 = v1 ? ex2_approx(fmaf(aA, __uint_as_float(r[4 * kb + 1]), fmaf(nA, cc[kb].y, bb[kb].y)) - mA) * iA : 0.f;
            const float b0 = v0 ? ex2_approx(fmaf(aB, __uint_as_float(r[4 * kb + 2]), fmaf(nB, cc[kb].x, bb[kb].x)) - mB) * iB : 0.f;
            const float b1 = v1 ? ex2_approx(fmaf(aB, __uint_as_float(r[4 * kb + 3]), fmaf(nB, cc[kb].y, bb[kb].y)) - mB) * iB : 0.f;
            if (okA) *reinterpret_cast<uint32_t*>(pA + c) = pack_bf16x2(a0, a1);
            if (okB) *reinterpret_cast<uint32_t*>(pB + c) = pack_bf16x2(b0, b1);
          }
        }
      }
      tcgen05_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tmem_empty[as]);
      if (++as == 2) { as = 0; aphase ^= 1u; }
    }
  } else {
    regs_shrink_ctrl();  // warps 2 and 3 idle; the whole warpgroup has to execute the setmaxnreg
  }

  __syncwarp();
  tcgen05_fence_before();
  __syncthreads();
  if (csize > 1) cluster_sync_all();  // nobody leaves while a peer may still write into this CTA / signal its barriers
  if (warp == 2) {
    tcgen05_fence_after();
    tmem_dealloc<TMEM_COLS>(tmem_base);
  }
}

// ---------------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn g_encode = nullptr;
unsigned long long* g_dbg = nullptr;
constexpr int kMaxDevices = 64;
DeviceState g_dev_state[kMaxDevices];
std::mutex g_dev_mutex;
std::map<std::tuple<int, const void*, int>, int> g_max_clusters;  // (device, kernel, cluster size) -> max_active_clusters

struct MapKey {
  uint64_t v[9];
  bool operator==(const MapKey& o) const { return memcmp(v, o.v, sizeof(v)) == 0; }
};
struct MapKeyHash {
  size_t operator()(const MapKey& k) const {
    uint64_t h = 0x9E3779B97F4A7C15ull;
    for (uint64_t x : k.v) h = (h ^ x) * 0xBF58476D1CE4E5B9ull + (h >> 29);
    return static_cast<size_t>(h);
  }
};

// 4-D bf16 map: dims (cols, rows, inner, outer), box (box_cols, box_rows, 1, 1), 128B swizzle, zero OOB fill.
int make_map(CUtensorMap* m, const TcOperand& op, int64_t n_inner, int64_t n_outer, int box_cols, int box_rows) {
  DITTO_REQUIRE((reinterpret_cast<uintptr_t>(op.ptr) & 15) == 0, DITTO_E_BADARG, "tc_gemm: operand base must be 16-B aligned");
  DITTO_REQUIRE(op.ld % 8 == 0 && op.s_inner % 8 == 0 && op.s_outer % 8 == 0, DITTO_E_UNSUPPORTED,
                "tc_gemm: operand strides must be multiples of 8 bf16 (16 B)");
  const int64_t row_bytes = op.ld * 2;
  // a dimension of extent 1 still needs a legal (non-zero, 16-B multiple) stride
  const int64_t inner_bytes = (op.s_inner ? op.s_inner : op.rows * op.ld) * 2;
  const int64_t outer_bytes = (op.s_outer ? op.s_outer : std::max<int64_t>(n_inner, 1) * (op.s_inner ? op.s_inner : op.rows * op.ld)) * 2;
  cuuint64_t dims[4] = {static_cast<cuuint64_t>(op.cols), static_cast<cuuint64_t>(op.rows),
                        static_cast<cuuint64_t>(op.s_inner ? n_inner : 1), static_cast<cuuint64_t>(op.s_outer ? n_outer : 1)};
  cuuint64_t strides[3] = {static_cast<cuuint64_t>(row_bytes), static_cast<cuuint64_t>(inner_bytes),
                           static_cast<cuuint64_t>(outer_bytes)};
  cuuint32_t box[4] = {static_cast<cuuint32_t>(box_cols), static_cast<cuuint32_t>(box_rows), 1, 1};
  cuuint32_t estr[4] = {1, 1, 1, 1};
  // A descriptor is a pure function of (base, extents, strides, box): an eager caller that steps a model in a loop asks for
  // the same few dozen maps every step, so they are kept in a small per-thread cache (pointer/shape-keyed, SURVEY 8b)
  // instead of being re-encoded by the driver on every launch.  Graph replay never comes here.
  const MapKey key{{reinterpret_cast<uint64_t>(op.ptr), dims[0], dims[1], dims[2], dims[3], strides[0], strides[1], strides[2],
                    (static_cast<uint64_t>(box_cols) << 32) | static_cast<uint64_t>(box_rows)}};
  thread_local std::unordered_map<MapKey, CUtensorMap, MapKeyHash> cache;
  auto it = cache.find(key);
  if (it != cache.end()) {
    *m = it->second;
    return 0;
  }
  CUresult r = g_encode(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<bf16*>(op.ptr), dims, strides, box, estr,
                        CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled failed with CUresult " + std::to_string(static_cast<int>(r)) + " (cols=" +
              std::to_string(op.cols) + " rows=" + std::to_string(op.rows) + " ld=" + std::to_string(op.ld) + ")");
    return DITTO_E_CUDA;
  }
  if (cache.size() >= 2048) cache.clear();   // bounded: serving with ever-changing shapes / buffers just re-encodes
  cache.emplace(key, *m);
  return 0;
}

template <int EPI>
int set_attr_pair() {
  DITTO_CUDA(cudaFuncSetAttribute(tc_gemm_pair_kernel<EPI>, cudaFuncAttributeMaxDynamicSharedMemorySize, P_SMEM_BYTES));
  return 0;
}

template <int EPI, bool B_KN>
int set_attr() {
  DITTO_CUDA(cudaFuncSetAttribute(tc_gemm_kernel<EPI, B_KN>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES));
  return 0;
}


}  // namespace

void tc_gemm_set_debug_counters(unsigned long long* dev_ptr) { g_dbg = dev_ptr; }
unsigned long long* tc_gemm_debug_counters() { return g_dbg; }
int tc_make_map(CUtensorMap* m, const TcOperand& op, int64_t n_inner, int64_t n_outer, int box_cols, int box_rows) {
  return make_map(m, op, n_inner, n_outer, box_cols, box_rows);
}
int tc_num_sms() {
  DeviceState* ds = device_state();
  return ds ? ds->num_sms : 0;
}

DeviceState* device_state() {
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= kMaxDevices) {
    set_error("libditto_b200: cudaGetDevice failed (or device ordinal >= 64)");
    return nullptr;
  }
  return &g_dev_state[dev];
}

int max_active_clusters(const void* func, int csize, int threads, int smem_bytes) {
  DeviceState* ds = device_state();
  int dev = 0;
  if (ds == nullptr || cudaGetDevice(&dev) != cudaSuccess) return -1;
  std::lock_guard<std::mutex> lock(g_dev_mutex);
  const auto key = std::make_tuple(dev, func, csize);
  auto it = g_max_clusters.find(key);
  if (it == g_max_clusters.end()) {
    int n = 0;
    if (cudaFuncSetAttribute(func, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes) == cudaSuccess &&
        (csize <= 8 || cudaFuncSetAttribute(func, cudaFuncAttributeNonPortableClusterSizeAllowed, 1) == cudaSuccess)) {
      cudaLaunchAttribute attr;
      attr.id = cudaLaunchAttributeClusterDimension;
      attr.val.clusterDim.x = static_cast<unsigned>(csize);
      attr.val.clusterDim.y = 1;
      attr.val.clusterDim.z = 1;
      cudaLaunchConfig_t cfg = {};
      cfg.gridDim = dim3(static_cast<unsigned>(csize * std::max(ds->num_sms, 1)), 1, 1);
      cfg.blockDim = dim3(static_cast<unsigned>(threads), 1, 1);
      cfg.dynamicSmemBytes = static_cast<size_t>(smem_bytes);
      cfg.attrs = &attr;
      cfg.numAttrs = 1;
      if (cudaOccupancyMaxActiveClusters(&n, func, &cfg) != cudaSuccess) n = 0;
    }
    (void)cudaGetLastError();   // a failed set-up or query must not surface at the next launch check
    it = g_max_clusters.emplace(key, n > 0 ? n : -1).first;
  }
  return it->second;
}

int launch_clusters(const void* func, int csize, int threads, int smem_bytes, int64_t work_items, void** args, cudaStream_t st) {
  DeviceState* ds = device_state();
  if (ds == nullptr) return DITTO_E_CUDA;
  const int capacity = csize == 1 ? ds->num_sms : max_active_clusters(func, csize, threads, smem_bytes);
  DITTO_REQUIRE(capacity > 0, DITTO_E_UNSUPPORTED, "tc_gemm: this cluster size cannot be scheduled on the device");
  cudaLaunchAttribute attr;
  attr.id = cudaLaunchAttributeClusterDimension;
  attr.val.clusterDim.x = static_cast<unsigned>(csize);
  attr.val.clusterDim.y = 1;
  attr.val.clusterDim.z = 1;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(static_cast<unsigned>(csize * std::min<int64_t>(capacity, work_items)), 1, 1);
  cfg.blockDim = dim3(static_cast<unsigned>(threads), 1, 1);
  cfg.dynamicSmemBytes = static_cast<size_t>(smem_bytes);
  cfg.stream = st;
  cfg.attrs = &attr;
  cfg.numAttrs = csize > 1 ? 1 : 0;
  DITTO_CUDA(cudaLaunchKernelExC(&cfg, func, args));
  count_launch();
  return 0;
}

// Per device: kernel attributes (dynamic shared memory opt-in, non-portable cluster sizes) and the SM count belong to the
// device that is current when they are set / read, so a process that holds engines on several GPUs initialises each one.
int tc_gemm_init() {
  DeviceState* ds = device_state();
  if (ds == nullptr) return DITTO_E_CUDA;
  if (ds->tc_init) return 0;
  std::lock_guard<std::mutex> lock(g_dev_mutex);
  if (ds->tc_init) return 0;
  if (g_encode == nullptr) {
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult qres;
    DITTO_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres));
    DITTO_REQUIRE(fn != nullptr && qres == cudaDriverEntryPointSuccess, DITTO_E_CUDA, "cuTensorMapEncodeTiled not available");
    g_encode = reinterpret_cast<EncodeTiledFn>(fn);
  }
  int dev = 0;
  DITTO_CUDA(cudaGetDevice(&dev));
  int major = 0, sms = 0;
  DITTO_CUDA(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev));
  DITTO_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  DITTO_REQUIRE(major == 10, DITTO_E_UNSUPPORTED, "libditto_b200 needs an sm_100a device (B200)");
  ds->num_sms = sms;
  DITTO_TRY((set_attr<K_STORE_F32, false>()));
  DITTO_TRY((set_attr<K_STORE_F32, true>()));
  DITTO_TRY((set_attr<K_STORE_F32_RESID, false>()));
  DITTO_TRY((set_attr<K_STORE_F32_RESID, true>()));
  DITTO_TRY((set_attr<K_STORE_BF16, false>()));
  DITTO_TRY((set_attr<K_STORE_BF16, true>()));
  DITTO_TRY((set_attr<K_STORE_GENERIC, false>()));
  DITTO_TRY((set_attr<K_STORE_GENERIC, true>()));
  DITTO_TRY((set_attr<K_GEGLU, false>()));
  DITTO_TRY((set_attr<K_QKV_ROPE, false>()));
  DITTO_TRY((set_attr_pair<K_STORE_F32>()));
  DITTO_TRY((set_attr_pair<K_STORE_F32_RESID>()));
  DITTO_TRY((set_attr_pair<K_STORE_BF16>()));
  DITTO_TRY((set_attr_pair<K_STORE_GENERIC>()));
  DITTO_TRY((set_attr_pair<K_GEGLU>()));
  DITTO_TRY((set_attr_pair<K_QKV_ROPE>()));
  DITTO_CUDA(cudaFuncSetAttribute(tc_scores_softmax_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, SM_SMEM_BYTES));
  DITTO_CUDA(cudaFuncSetAttribute(tc_scores_softmax_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, SM_SMEM_BYTES));
  DITTO_CUDA(cudaFuncSetAttribute(tc_scores_softmax_kernel<false>, cudaFuncAttributeNonPortableClusterSizeAllowed, 1));
  DITTO_CUDA(cudaFuncSetAttribute(tc_scores_softmax_kernel<true>, cudaFuncAttributeNonPortableClusterSizeAllowed, 1));
  ds->tc_init = true;
  return 0;
}

int launch_tc_gemm(const TcGemmParams& q, cudaStream_t st) {
  DITTO_TRY(tc_gemm_init());
  DITTO_REQUIRE(q.M > 0 && q.N > 0 && q.K > 0 && q.batch_inner >= 1 && q.batch_outer >= 1, DITTO_E_BADARG, "tc_gemm: bad sizes");
  DITTO_REQUIRE(q.A.ptr && q.B.ptr && q.out, DITTO_E_BADARG, "tc_gemm: null operand");
  const int elt = q.out_bf16 ? 8 : 4;
  DITTO_REQUIRE(q.ldo % elt == 0 && q.so_inner % elt == 0 && q.so_outer % elt == 0, DITTO_E_UNSUPPORTED,
                "tc_gemm: output strides must keep 16-B alignment");
  if (q.resid) DITTO_REQUIRE(q.ldr % 4 == 0 && q.sr_inner % 4 == 0 && q.sr_outer % 4 == 0, DITTO_E_UNSUPPORTED, "tc_gemm: resid strides");
  if (q.out2) DITTO_REQUIRE(q.ldo2 % 8 == 0 && !q.out_bf16, DITTO_E_UNSUPPORTED, "tc_gemm: out2 needs fp32 primary output");
  if (q.epilogue == TC_EPI_GEGLU)
    DITTO_REQUIRE(q.N % 32 == 0 && q.bias && q.out_bf16 && !q.b_kn, DITTO_E_UNSUPPORTED, "tc_gemm: GEGLU epilogue constraints");
  if (q.epilogue == TC_EPI_QKV_ROPE)
    DITTO_REQUIRE(q.bias && q.out_bf16 && !q.b_kn && q.rope_freq && q.N == 3 * q.hidden &&
                      (q.rope_pd == 32 || q.rope_pd == 64 || q.rope_pd == 128) && q.rope_half % q.rope_pd == 0 &&
                      q.hidden % (2 * q.rope_pd) == 0 && q.seq_T > 0 && q.alpha == 1.f && !q.resid && !q.out2,
                  DITTO_E_UNSUPPORTED, "tc_gemm: QKV_ROPE epilogue constraints");

  CUtensorMap ma, mb;
  TcOperand A = q.A, B = q.B;
  // paired (cta_group::2) kernel for the large un-batched weight GEMMs
  const int g_num_sms = tc_num_sms();
  const bool pair = !q.b_kn && q.batch_inner == 1 && q.batch_outer == 1 && q.M >= 2 * BLOCK_M && (g_num_sms % 2 == 0);
  DITTO_TRY(make_map(&ma, A, q.batch_inner, q.batch_outer, BLOCK_K, BLOCK_M));
  if (pair)
    DITTO_TRY(make_map(&mb, B, 1, 1, BLOCK_K, BLOCK_N / 2));
  else if (!q.b_kn)
    DITTO_TRY(make_map(&mb, B, q.batch_inner, q.batch_outer, BLOCK_K, BLOCK_N));
  else
    DITTO_TRY(make_map(&mb, B, q.batch_inner, q.batch_outer, 64, BLOCK_K));

  DevParams p;
  p.M = q.M; p.N = q.N; p.K = q.K;
  p.batch_inner = q.batch_inner; p.batch_outer = q.batch_outer;
  p.m_tiles = static_cast<int>(ceil_div(q.M, BLOCK_M));
  p.n_tiles = static_cast<int>(ceil_div(q.N, BLOCK_N));
  const int64_t tiles = static_cast<int64_t>(p.m_tiles) * p.n_tiles * q.batch_inner * q.batch_outer;
  DITTO_REQUIRE(tiles < (1ll << 31), DITTO_E_UNSUPPORTED, "tc_gemm: too many tiles");
  p.num_tiles = static_cast<int>(tiles);
  p.num_kb = static_cast<int>(ceil_div(q.K, BLOCK_K));
  p.a_bi = q.A.s_inner ? 1 : 0; p.a_bo = q.A.s_outer ? 1 : 0;
  p.b_bi = q.B.s_inner ? 1 : 0; p.b_bo = q.B.s_outer ? 1 : 0;
  p.alpha = q.alpha; p.bias = q.bias; p.sb_inner = q.sb_inner; p.sb_outer = q.sb_outer;
  p.out = q.out; p.out_bf16 = q.out_bf16 ? 1 : 0;
  p.ldo = q.ldo; p.so_inner = q.so_inner; p.so_outer = q.so_outer;
  p.resid = q.resid; p.ldr = q.ldr; p.sr_inner = q.sr_inner; p.sr_outer = q.sr_outer; p.resid_row_mod = q.resid_row_mod;
  p.out2 = q.out2; p.ldo2 = q.ldo2;
  p.rope_freq = q.rope_freq;
  p.rope_half = q.rope_half; p.rope_pd = q.rope_pd; p.seq_T = q.seq_T; p.hidden = q.hidden; p.rope_pos = q.rope_pos; p.rope_fast = q.rope_perm16 ? 1 : 0; p.glu_fast = q.glu_perm16 ? 1 : 0; p.out_perm4 = q.out_perm4 ? 1 : 0;
  p.row_lsum = q.row_lsum; p.row_lparts = q.row_lparts; p.sl_inner = q.sl_inner; p.sl_outer = q.sl_outer;
  p.stat_out = q.stat_out; p.stat_parts = q.stat_parts; p.stat_rows_outer = q.stat_rows_outer;
  p.stat_parts_item = static_cast<int>(ceil_div(q.N, 128));
  p.ln_stat = q.ln_stat; p.ln_parts = q.ln_parts; p.ln_inv_h = q.ln_width > 0 ? 1.0f / static_cast<float>(q.ln_width) : 0.f;
  p.ln_c = q.ln_c;
  if (q.stat_out != nullptr)
    DITTO_REQUIRE(q.epilogue == TC_EPI_STORE && q.resid && !q.out_bf16 && q.N % 2 == 0 &&
                      q.stat_parts == q.batch_inner * p.stat_parts_item && (q.batch_outer == 1 || q.stat_rows_outer >= q.M),
                  DITTO_E_UNSUPPORTED, "tc_gemm: row statistics need the fp32 + residual STORE epilogue and matching stat_parts");
  if (q.ln_stat != nullptr)
    DITTO_REQUIRE((q.epilogue == TC_EPI_GEGLU || q.epilogue == TC_EPI_QKV_ROPE) && q.ln_c && q.ln_parts > 0 && q.ln_width > 0 &&
                      q.batch_inner == 1 && q.batch_outer == 1,
                  DITTO_E_UNSUPPORTED, "tc_gemm: deferred LayerNorm is implemented in the GEGLU / QKV_ROPE epilogues only");
  p.dbg = g_dbg;

  unsigned grid = static_cast<unsigned>(std::min<int64_t>(tiles, g_num_sms));
  ProfScope prof(q.tag, st, 2.0 * q.M * q.N * q.K * q.batch_inner * q.batch_outer, 0.0);
  if (q.out_perm4)
    DITTO_REQUIRE(q.epilogue == TC_EPI_STORE && !q.out_bf16 && q.resid != nullptr && q.bias == nullptr && q.out2 == nullptr &&
                      q.stat_out == nullptr && q.resid_row_mod == 0 && q.N % 128 == 0 && q.ldo % 4 == 0 && q.ldr % 4 == 0 &&
                      q.so_inner % 4 == 0 && q.so_outer % 4 == 0 && q.sr_inner % 4 == 0 && q.sr_outer % 4 == 0,
                  DITTO_E_BADARG, "tc_gemm: out_perm4 needs an fp32 result with residual, no bias / copy / statistics, N % 128 == 0");
  if (q.glu_perm16)
    DITTO_REQUIRE(q.epilogue == TC_EPI_GEGLU && q.ln_stat == nullptr && q.N % BLOCK_N == 0 && q.out_bf16 && q.ldo % 8 == 0 && q.bias != nullptr,
                  DITTO_E_BADARG, "tc_gemm: glu_perm16 needs the GEGLU epilogue, no deferred LayerNorm, a bias and N % 256 == 0");
  if (q.rope_perm16)
    DITTO_REQUIRE(q.epilogue == TC_EPI_QKV_ROPE && (q.rope_pd == 128 || q.rope_pd == 32) && q.ln_stat == nullptr &&
                      q.N % BLOCK_N == 0 && q.hidden % BLOCK_N == 0 && q.out_bf16 && q.ldo % 16 == 0 &&
                      (reinterpret_cast<uintptr_t>(q.out) & 31) == 0 && (q.batch_inner * q.batch_outer == 1 || (q.so_inner % 16 == 0 && q.so_outer % 16 == 0)),
                  DITTO_E_BADARG, "tc_gemm: rope_perm16 needs pd = 128 or 32, no deferred LayerNorm, N and hidden % 256 == 0, "
                                  "a 32-byte aligned output with a row stride of a multiple of 16 (32-byte stores)");
  // kernel variant: the lean compile-time epilogues cover the hot cases, anything else takes the generic one
  int ke;
  if (q.epilogue == TC_EPI_GEGLU) ke = K_GEGLU;
  else if (q.epilogue == TC_EPI_QKV_ROPE) ke = K_QKV_ROPE;
  else if (q.epilogue != TC_EPI_STORE) {
    set_error("tc_gemm: unknown epilogue");
    return DITTO_E_BADARG;
  } else if (q.N % 2 != 0) ke = K_STORE_GENERIC;
  else if (!q.out_bf16) ke = q.resid ? K_STORE_F32_RESID : (q.out2 ? K_STORE_GENERIC : K_STORE_F32);
  else ke = (q.resid || q.out2) ? K_STORE_GENERIC : K_STORE_BF16;
  if (q.row_lsum != nullptr)
    DITTO_REQUIRE(ke == K_STORE_F32 || ke == K_STORE_F32_RESID || ke == K_STORE_BF16, DITTO_E_UNSUPPORTED,
                  "tc_gemm: row_lsum needs a fast STORE epilogue (even N)");
#define DITTO_LAUNCH_PAIR(E) tc_gemm_pair_kernel<E><<<grid, NUM_THREADS, P_SMEM_BYTES, st>>>(ma, mb, p)
#define DITTO_FUNC_1CTA(E, KN) reinterpret_cast<const void*>(&tc_gemm_kernel<E, KN>)
  if (pair) {
    const int64_t pair_tiles = ceil_div(q.M, 2 * BLOCK_M) * p.n_tiles;
    grid = static_cast<unsigned>(2 * std::min<int64_t>(pair_tiles, g_num_sms / 2));
    switch (ke) {
      case K_STORE_F32: DITTO_LAUNCH_PAIR(K_STORE_F32); break;
      case K_STORE_F32_RESID: DITTO_LAUNCH_PAIR(K_STORE_F32_RESID); break;
      case K_STORE_BF16: DITTO_LAUNCH_PAIR(K_STORE_BF16); break;
      case K_STORE_GENERIC: DITTO_LAUNCH_PAIR(K_STORE_GENERIC); break;
      case K_GEGLU: DITTO_LAUNCH_PAIR(K_GEGLU); break;
      default: DITTO_LAUNCH_PAIR(K_QKV_ROPE); break;
    }
    DITTO_LAUNCH_CHECK();
    return 0;
  }
  const void* func;
  if (q.b_kn) {
    switch (ke) {
      case K_STORE_F32: func = DITTO_FUNC_1CTA(K_STORE_F32, true); break;
      case K_STORE_F32_RESID: func = DITTO_FUNC_1CTA(K_STORE_F32_RESID, true); break;
      case K_STORE_BF16: func = DITTO_FUNC_1CTA(K_STORE_BF16, true); break;
      default: func = DITTO_FUNC_1CTA(K_STORE_GENERIC, true); break;  // GEGLU / ROPE with b_kn were rejected above
    }
  } else {
    switch (ke) {
      case K_STORE_F32: func = DITTO_FUNC_1CTA(K_STORE_F32, false); break;
      case K_STORE_F32_RESID: func = DITTO_FUNC_1CTA(K_STORE_F32_RESID, false); break;
      case K_STORE_BF16: func = DITTO_FUNC_1CTA(K_STORE_BF16, false); break;
      case K_STORE_GENERIC: func = DITTO_FUNC_1CTA(K_STORE_GENERIC, false); break;
      case K_GEGLU: func = DITTO_FUNC_1CTA(K_GEGLU, false); break;
      default: func = DITTO_FUNC_1CTA(K_QKV_ROPE, false); break;
    }
  }
  // no cluster: TMA multicast of the operands across CTAs of adjacent tiles was measured on B200 (profiles/README.md) and
  // lost -- for these epilogue-heavy batched attention GEMMs the lock-step coupling costs more than the saved L2 traffic
  void* args[3] = {&ma, &mb, &p};
  return launch_clusters(func, 1, NUM_THREADS, SMEM_BYTES, tiles, args, st);
}
#undef DITTO_LAUNCH_PAIR
#undef DITTO_FUNC_1CTA


// ---------------------------------------------------------------------------------------------------
// fused scores + softmax launcher
// ---------------------------------------------------------------------------------------------------

int tc_scores_softmax_csize(int N) {
  const int64_t c = ceil_div(N, BLOCK_N);
  return (N > 0 && c <= SM_MAX_CLUSTER) ? static_cast<int>(c) : 0;
}

int launch_tc_scores_softmax(const TcScoresSoftmaxParams& q, cudaStream_t st) {
  DITTO_TRY(tc_gemm_init());
  DITTO_REQUIRE(q.M > 0 && q.N > 0 && q.K > 0 && q.batch_inner >= 1 && q.batch_outer >= 1, DITTO_E_BADARG, "tc_scores_softmax: bad sizes");
  DITTO_REQUIRE(q.Q.ptr && q.Km.ptr && q.P, DITTO_E_BADARG, "tc_scores_softmax: null operand");
  const int csize = tc_scores_softmax_csize(q.N);
  DITTO_REQUIRE(csize > 0, DITTO_E_UNSUPPORTED, "tc_scores_softmax: too many key columns for one cluster");
  DITTO_REQUIRE(q.npad >= q.N && q.npad % 2 == 0 && q.npad <= q.ldp, DITTO_E_BADARG, "tc_scores_softmax: npad");
  DITTO_REQUIRE(q.ldp % 8 == 0 && q.sp_inner % 8 == 0 && q.sp_outer % 8 == 0, DITTO_E_UNSUPPORTED, "tc_scores_softmax: P strides");
  DITTO_REQUIRE(csize == 1 || q.lpart != nullptr, DITTO_E_BADARG, "tc_scores_softmax: lpart required for multi-tile rows");
  CUtensorMap ma, mb;
  DITTO_TRY(make_map(&ma, q.Q, q.batch_inner, q.batch_outer, BLOCK_K, BLOCK_M));
  DITTO_TRY(make_map(&mb, q.Km, q.batch_inner, q.batch_outer, BLOCK_K, BLOCK_N));
  SmDev p;
  p.M = q.M; p.N = q.N; p.K = q.K;
  p.batch_inner = q.batch_inner; p.batch_outer = q.batch_outer;
  p.m_tiles = static_cast<int>(ceil_div(q.M, BLOCK_M));
  const int64_t items = static_cast<int64_t>(p.m_tiles) * q.batch_inner * q.batch_outer;
  DITTO_REQUIRE(items < (1ll << 31), DITTO_E_UNSUPPORTED, "tc_scores_softmax: too many work items");
  p.num_items = static_cast<int>(items);
  p.num_kb = static_cast<int>(ceil_div(q.K, BLOCK_K));
  p.a_bi = q.Q.s_inner ? 1 : 0; p.a_bo = q.Q.s_outer ? 1 : 0;
  p.b_bi = q.Km.s_inner ? 1 : 0; p.b_bo = q.Km.s_outer ? 1 : 0;
  p.alpha2 = q.alpha * 1.4426950408889634f;
  p.bias = q.bias; p.sb_inner = q.sb_inner; p.sb_outer = q.sb_outer;
  p.P = q.P; p.ldp = q.ldp; p.sp_inner = q.sp_inner; p.sp_outer = q.sp_outer;
  p.npad = q.npad;
  p.lpart = q.lpart; p.sl_inner = q.sl_inner; p.sl_outer = q.sl_outer;
  p.csize = csize;
  p.col_len = q.col_len;
  p.ln_stat = q.ln_stat; p.ln_parts = q.ln_parts; p.ln_inv_h = q.ln_width > 0 ? 1.0f / static_cast<float>(q.ln_width) : 0.f;
  p.ln_c = q.ln_c;
  if (q.ln_stat != nullptr)
    DITTO_REQUIRE(q.bias && q.ln_c && q.ln_parts > 0 && q.ln_width > 0, DITTO_E_BADARG, "tc_scores_softmax: deferred LayerNorm arguments");
  // flops: the contraction; bytes: nothing (the fused softmax saves 12 B per score of HBM round trips)
  ProfScope prof(q.tag, st, 2.0 * q.M * q.N * q.K * q.batch_inner * q.batch_outer, 0.0);
  const void* func = q.bias != nullptr ? reinterpret_cast<const void*>(&tc_scores_softmax_kernel<true>)
                                       : reinterpret_cast<const void*>(&tc_scores_softmax_kernel<false>);
  void* args[3] = {&ma, &mb, &p};
  return launch_clusters(func, csize, NUM_THREADS, SM_SMEM_BYTES, items, args, st);
}

}  // namespace ditto
