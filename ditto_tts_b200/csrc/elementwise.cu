// HBM-bound kernels of the DiT denoiser hot path: LayerNorm / AdaLN, RoPE, softmax, gated activation,
// CFG-combine + DDPM update, q_sample, casts and weight packing.  All coalesced + 128-bit vectorised.
#include <vector>

#include "kernels.cuh"

namespace ditto {

// =====================================================================================================
// casts / packing
// =====================================================================================================
__global__ void cast_bf16_kernel(const float* __restrict__ x, bf16* __restrict__ y, int64_t n) {
  int64_t i = (static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x) * 4;
  const int64_t stride = static_cast<int64_t>(gridDim.x) * blockDim.x * 4;
  for (; i + 3 < n; i += stride) {
    float4 v = *reinterpret_cast<const float4*>(x + i);
    uint2 o;
    o.x = pack_bf16x2(v.x, v.y);
    o.y = pack_bf16x2(v.z, v.w);
    *reinterpret_cast<uint2*>(y + i) = o;
  }
  if (i < n) {  // tail (n % 4 != 0): the one thread that lands on it
    for (int64_t j = i; j < n && j < i + 4; ++j) y[j] = __float2bfloat16_rn(x[j]);
  }
}

int launch_cast_bf16(const float* x, bf16* y, int64_t n, cudaStream_t st) {
  if (n <= 0) return 0;
  DITTO_REQUIRE((reinterpret_cast<uintptr_t>(x) & 15) == 0 && (reinterpret_cast<uintptr_t>(y) & 7) == 0,
                DITTO_E_BADARG, "cast_bf16: misaligned pointer");
  int64_t blocks = std::min<int64_t>(ceil_div(n, 4 * 256), 148 * 16);
  ProfScope prof(PC_ELEMENTWISE, st, 0.0, static_cast<double>(n) * 6);
  cast_bf16_kernel<<<static_cast<unsigned>(blocks), 256, 0, st>>>(x, y, n);
  DITTO_LAUNCH_CHECK();
  return 0;
}

// rows [rows, K] fp32 -> bf16 with an output-row permutation: y[r] = x[perm(r)]  (perm built on the host: GLU interleave
// of [fc1 16 | gate 16] row blocks, RoPE pairing of the q and k thirds of in_proj -- see engine.cu)
// With gamma / beta (deferred LayerNorm folded into the weight, see gemm_tc.cu DevParams):
//   y[r][k] = bf16(x[src][k] gamma[k]),  csum[r] = sum_k float(y[r][k]),  bias_out[r] = bias_in[src] + sum_k x[src][k] beta[k]
__global__ void pack_rows_kernel(const float* __restrict__ x, bf16* __restrict__ y, float* __restrict__ bias_out,
                                 const float* __restrict__ bias_in, const int* __restrict__ perm, int rows, int K,
                                 const float* __restrict__ gamma, const float* __restrict__ beta, float* __restrict__ csum) {
  const int r = blockIdx.x;
  const int src = perm ? perm[r] : r;
  const float* xr = x + static_cast<int64_t>(src) * K;
  bf16* yr = y + static_cast<int64_t>(r) * K;
  float cs = 0.f, bs = 0.f;
  for (int c = threadIdx.x; c < K; c += blockDim.x) {
    const float w = xr[c];
    const bf16 q = __float2bfloat16_rn(gamma ? w * gamma[c] : w);
    yr[c] = q;
    cs += __bfloat162float(q);
    if (beta) bs = fmaf(w, beta[c], bs);
  }
  __shared__ float red[2][8];
  cs = warp_sum(cs);
  bs = warp_sum(bs);
  if ((threadIdx.x & 31) == 0) { red[0][threadIdx.x >> 5] = cs; red[1][threadIdx.x >> 5] = bs; }
  __syncthreads();
  if (threadIdx.x == 0) {
    cs = bs = 0.f;
    for (int i = 0; i < static_cast<int>(blockDim.x >> 5); ++i) { cs += red[0][i]; bs += red[1][i]; }
    if (bias_out) bias_out[r] = bias_in[src] + bs;
    if (csum) csum[r] = cs;
  }
}

int launch_pack_rows(const float* x, bf16* y, float* bias_out, const float* bias_in, const int* perm, int rows, int K,
                     cudaStream_t st, const float* gamma, const float* beta, float* csum) {
  pack_rows_kernel<<<rows, 256, 0, st>>>(x, y, bias_out, bias_in, perm, rows, K, gamma, beta, csum);
  DITTO_LAUNCH_CHECK();
  return 0;
}

// out[g * Sp + s] = sum_k x[(g * S + s) * K + k] for s < S, 0 for S <= s < Sp  (row sums of the gamma-scaled folded keys)
__global__ void rowsum_bf16_kernel(const bf16* __restrict__ x, float* __restrict__ out, int64_t total, int S, int Sp, int K) {
  const int lane = threadIdx.x & 31;
  const int64_t o = static_cast<int64_t>(blockIdx.x) * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (o >= total) return;
  const int s_idx = static_cast<int>(o % Sp);
  const int64_t g = o / Sp;
  float acc = 0.f;
  if (s_idx < S) {
    const bf16* row = x + (g * S + s_idx) * K;
    for (int i = lane; i < K; i += 32) acc += __bfloat162float(row[i]);
  }
  acc = warp_sum(acc);
  if (lane == 0) out[o] = acc;
}
int launch_rowsum_bf16(const bf16* x, float* out, int64_t groups, int S, int Sp, int K, cudaStream_t st) {
  const int64_t total = groups * Sp;
  rowsum_bf16_kernel<<<static_cast<unsigned>(ceil_div(total, 8)), 256, 0, st>>>(x, out, total, S, Sp, K);
  DITTO_LAUNCH_CHECK();
  return 0;
}

// =====================================================================================================
// LayerNorm (eps 1e-5, biased variance, two-pass statistics in fp32) -- one warp per row
// =====================================================================================================
constexpr int LN_MAXV = 8;  // float4 per lane kept in registers -> H <= 1024

template <typename OutT>
__device__ __forceinline__ void store4(OutT* p, float a, float b, float c, float d);
template <>
__device__ __forceinline__ void store4<float>(float* p, float a, float b, float c, float d) {
  *reinterpret_cast<float4*>(p) = make_float4(a, b, c, d);
}
template <>
__device__ __forceinline__ void store4<bf16>(bf16* p, float a, float b, float c, float d) {
  uint2 o;
  o.x = pack_bf16x2(a, b);
  o.y = pack_bf16x2(c, d);
  *reinterpret_cast<uint2*>(p) = o;
}

// statistics of a row held in registers: v[i] valid for i < nv (per-lane float4 slots)
__device__ __forceinline__ void row_stats(const float4 (&v)[LN_MAXV], int nv_lane, int H, float& mean, float& rstd) {
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < LN_MAXV; ++i)
    if (i < nv_lane) s += (v[i].x + v[i].y) + (v[i].z + v[i].w);
  mean = warp_sum(s) / static_cast<float>(H);
  float q = 0.f;
#pragma unroll
  for (int i = 0; i < LN_MAXV; ++i)
    if (i < nv_lane) {
      float a = v[i].x - mean, b = v[i].y - mean, c = v[i].z - mean, d = v[i].w - mean;
      q += (a * a + b * b) + (c * c + d * d);
    }
  rstd = rsqrtf(warp_sum(q) / static_cast<float>(H) + 1e-5f);
}

template <typename OutT>
__global__ void __launch_bounds__(256) layernorm_kernel(const float* __restrict__ x, const float* __restrict__ gamma,
                                                        const float* __restrict__ beta, OutT* __restrict__ y,
                                                        int64_t rows, int H) {
  const int lane = threadIdx.x & 31;
  const int nvec = H >> 2;                            // float4 per row
  const int nv_lane = (nvec - lane + 31) >> 5;        // slots of this lane
  const int64_t warps = static_cast<int64_t>(gridDim.x) * (blockDim.x >> 5);
  // grid-stride over rows (grid = a whole number of resident blocks per SM: no partial last wave)
  for (int64_t row = static_cast<int64_t>(blockIdx.x) * (blockDim.x >> 5) + (threadIdx.x >> 5); row < rows; row += warps) {
    const float* xr = x + row * H;
    float4 v[LN_MAXV];
#pragma unroll
    for (int i = 0; i < LN_MAXV; ++i)
      if (i < nv_lane) v[i] = *reinterpret_cast<const float4*>(xr + ((i << 5) + lane) * 4);
    float mean, rstd;
    row_stats(v, nv_lane, H, mean, rstd);
    OutT* yr = y + row * H;
#pragma unroll
    for (int i = 0; i < LN_MAXV; ++i)
      if (i < nv_lane) {
        const int c = ((i << 5) + lane) * 4;
        float4 g = gamma ? __ldg(reinterpret_cast<const float4*>(gamma + c)) : make_float4(1.f, 1.f, 1.f, 1.f);
        float4 b = beta ? __ldg(reinterpret_cast<const float4*>(beta + c)) : make_float4(0.f, 0.f, 0.f, 0.f);
        store4<OutT>(yr + c, (v[i].x - mean) * rstd * g.x + b.x, (v[i].y - mean) * rstd * g.y + b.y,
                     (v[i].z - mean) * rstd * g.z + b.z, (v[i].w - mean) * rstd * g.w + b.w);
      }
  }
}

int launch_layernorm(const float* x, const float* gamma, const float* beta, void* y, bool out_bf16, int64_t rows, int H,
                     cudaStream_t st) {
  DITTO_REQUIRE(H % 4 == 0 && H <= LN_MAXV * 128 && H > 0, DITTO_E_UNSUPPORTED, "layernorm: need H % 4 == 0 and H <= 1024");
  if (rows <= 0) return 0;
  const unsigned blocks = static_cast<unsigned>(std::min<int64_t>(ceil_div(rows, 8), 148 * 8));
  ProfScope prof(PC_LAYERNORM, st, 0.0, static_cast<double>(rows) * H * (out_bf16 ? 6 : 8));
  if (out_bf16)
    layernorm_kernel<bf16><<<blocks, 256, 0, st>>>(x, gamma, beta, static_cast<bf16*>(y), rows, H);
  else
    layernorm_kernel<float><<<blocks, 256, 0, st>>>(x, gamma, beta, static_cast<float*>(y), rows, H);
  DITTO_LAUNCH_CHECK();
  return 0;
}

// =====================================================================================================
// Global AdaLN fused with the first block's LayerNorm (DiT.py:25-40 then DiT.py:105):
//   h = LN_noaffine(x) * (1 + ts + xs) + (tb + xb)      -> fp32 residual stream
//   u = LN(h) * gamma1 + beta1                          -> GEMM operand (bf16 or fp32)
//   xcast = bf16(x)                                     -> operand of proj_in (written once per distinct x row)
// ts|tb = time_table[t[seq]] (per-step constants), xs|xb = text_mod[seq] (per-utterance constants).
// =====================================================================================================
template <typename OutT>
__global__ void __launch_bounds__(256)
    adaln_ln_kernel(const float* __restrict__ x, int64_t n_x, const float* __restrict__ time_table,
                    const float* __restrict__ text_mod, const int64_t* __restrict__ t, int steps,
                    const float* __restrict__ gamma, const float* __restrict__ beta, float* __restrict__ h,
                    OutT* __restrict__ u, bf16* __restrict__ xcast, int64_t n_seq, int T, int H, float2* __restrict__ stat,
                    bool xcast_all, int* __restrict__ row_pos) {
  const int lane = threadIdx.x & 31;
  const int64_t row = static_cast<int64_t>(blockIdx.x) * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= n_seq * T) return;
  const int64_t seq = row / T;
  const int64_t pos = row - seq * T;
  const int64_t xrow = (seq % n_x) * T + pos;
  int64_t tt = t != nullptr ? t[seq] : seq;   // t == nullptr: the table already holds one row per sequence (ditto_adaln)
  tt = tt < 0 ? 0 : (tt >= steps ? steps - 1 : tt);
  const float* tm = time_table + tt * 2 * H;
  const float* xm = text_mod + seq * 2 * H;
  const int nvec = H >> 2;
  const int nv_lane = (nvec - lane + 31) >> 5;
  const float* xr = x + xrow * H;
  float4 v[LN_MAXV];
#pragma unroll
  for (int i = 0; i < LN_MAXV; ++i)
    if (i < nv_lane) v[i] = *reinterpret_cast<const float4*>(xr + ((i << 5) + lane) * 4);
  if (xcast != nullptr && (xcast_all || seq < n_x)) {  // bf16 copy of x: once per distinct x, or per sequence (ragged batches)
    bf16* xc = xcast + (xcast_all ? row : xrow) * H;
#pragma unroll
    for (int i = 0; i < LN_MAXV; ++i)
      if (i < nv_lane) store4<bf16>(xc + ((i << 5) + lane) * 4, v[i].x, v[i].y, v[i].z, v[i].w);
  }
  if (row_pos != nullptr && lane == 0) row_pos[row] = static_cast<int>(pos);  // RoPE position table of a ragged batch
  float mean, rstd;
  row_stats(v, nv_lane, H, mean, rstd);
#pragma unroll
  for (int i = 0; i < LN_MAXV; ++i)
    if (i < nv_lane) {
      const int c = ((i << 5) + lane) * 4;
      const float4 ts = *reinterpret_cast<const float4*>(tm + c);
      const float4 tb = *reinterpret_cast<const float4*>(tm + H + c);
      const float4 xs = *reinterpret_cast<const float4*>(xm + c);
      const float4 xb = *reinterpret_cast<const float4*>(xm + H + c);
      // scale = 1 + time_scale + text_scale ; shift = time_shift + text_shift   (DiT.py:34-35, same order)
      v[i].x = (v[i].x - mean) * rstd * ((1.f + ts.x) + xs.x) + (tb.x + xb.x);
      v[i].y = (v[i].y - mean) * rstd * ((1.f + ts.y) + xs.y) + (tb.y + xb.y);
      v[i].z = (v[i].z - mean) * rstd * ((1.f + ts.z) + xs.z) + (tb.z + xb.z);
      v[i].w = (v[i].w - mean) * rstd * ((1.f + ts.w) + xs.w) + (tb.w + xb.w);
      *reinterpret_cast<float4*>(h + row * H + c) = v[i];
    }
  if (u == nullptr) return;  // GlobalAdaLN alone (ditto_adaln)
  if (stat != nullptr) {
    // deferred LayerNorm: u = bf16(h) and the row's (sum, sum of squares); the consuming GEMM epilogue normalises
    float sm = 0.f, sq = 0.f;
#pragma unroll
    for (int i = 0; i < LN_MAXV; ++i)
      if (i < nv_lane) {
        sm += (v[i].x + v[i].y) + (v[i].z + v[i].w);
        sq += (v[i].x * v[i].x + v[i].y * v[i].y) + (v[i].z * v[i].z + v[i].w * v[i].w);
        store4<OutT>(u + row * H + ((i << 5) + lane) * 4, v[i].x, v[i].y, v[i].z, v[i].w);
      }
    sm = warp_sum(sm);
    sq = warp_sum(sq);
    if (lane == 0) stat[row] = make_float2(sm, sq);
    return;
  }
  row_stats(v, nv_lane, H, mean, rstd);
#pragma unroll
  for (int i = 0; i < LN_MAXV; ++i)
    if (i < nv_lane) {
      const int c = ((i << 5) + lane) * 4;
      const float4 g = *reinterpret_cast<const float4*>(gamma + c);
      const float4 b = *reinterpret_cast<const float4*>(beta + c);
      store4<OutT>(u + row * H + c, (v[i].x - mean) * rstd * g.x + b.x, (v[i].y - mean) * rstd * g.y + b.y,
                   (v[i].z - mean) * rstd * g.z + b.z, (v[i].w - mean) * rstd * g.w + b.w);
    }
}

// The same for the hot case (bf16 operand, fused LN1, no deferred statistics, H = NV * 128): the row's float4 slots are a
// compile-time count, so there are no predicated slots and the per-slot address arithmetic folds into immediates (933 -> ~450 warp
// instructions per row).
template <int NV>
__global__ void __launch_bounds__(256)
    adaln_ln_fast_kernel(const float* __restrict__ x, int64_t n_x, const float* __restrict__ time_table,
                         const float* __restrict__ text_mod, const int64_t* __restrict__ t, int steps,
                         const float* __restrict__ gamma, const float* __restrict__ beta, float* __restrict__ h,
                         bf16* __restrict__ u, bf16* __restrict__ xcast, int64_t n_seq, int T, bool xcast_all, int* __restrict__ row_pos) {
  constexpr int H = NV * 128;
  constexpr float kInvH = 1.0f / static_cast<float>(H);
  const int lane = threadIdx.x & 31;
  const int64_t row = static_cast<int64_t>(blockIdx.x) * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= n_seq * T) return;
  const int64_t seq = row / T;
  const int64_t pos = row - seq * T;
  const int64_t xrow = (seq % n_x) * T + pos;
  int64_t tt = t != nullptr ? t[seq] : seq;
  tt = tt < 0 ? 0 : (tt >= steps ? steps - 1 : tt);
  const float4* xr = reinterpret_cast<const float4*>(x + xrow * H) + lane;
  const float4* tm = reinterpret_cast<const float4*>(time_table + tt * 2 * H) + lane;
  const float4* xm = reinterpret_cast<const float4*>(text_mod + seq * 2 * H) + lane;
  float4 v[NV], sc[NV], sh[NV];
#pragma unroll
  for (int i = 0; i < NV; ++i) v[i] = xr[i * 32];
#pragma unroll
  for (int i = 0; i < NV; ++i) {   // requested before the first reduction: their latency hides behind the statistics of x
    const float4 ts = __ldg(tm + i * 32), tb = __ldg(tm + H / 4 + i * 32);
    const float4 xs = __ldg(xm + i * 32), xb = __ldg(xm + H / 4 + i * 32);
    // scale = 1 + time_scale + text_scale ; shift = time_shift + text_shift   (DiT.py:34-35, same order)
    sc[i] = make_float4((1.f + ts.x) + xs.x, (1.f + ts.y) + xs.y, (1.f + ts.z) + xs.z, (1.f + ts.w) + xs.w);
    sh[i] = make_float4(tb.x + xb.x, tb.y + xb.y, tb.z + xb.z, tb.w + xb.w);
  }
  if (xcast != nullptr && (xcast_all || seq < n_x)) {
    uint2* xc = reinterpret_cast<uint2*>(xcast + (xcast_all ? row : xrow) * H) + lane;
#pragma unroll
    for (int i = 0; i < NV; ++i) xc[i * 32] = make_uint2(pack_bf16x2(v[i].x, v[i].y), pack_bf16x2(v[i].z, v[i].w));
  }
  if (row_pos != nullptr && lane == 0) row_pos[row] = static_cast<int>(pos);
  auto stats = [&](float& mean, float& rstd) {   // two-pass, the same arithmetic as row_stats
    float sm = 0.f;
#pragma unroll
    for (int i = 0; i < NV; ++i) sm += (v[i].x + v[i].y) + (v[i].z + v[i].w);
    mean = warp_sum(sm) * kInvH;
    float q = 0.f;
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      const float a = v[i].x - mean, b = v[i].y - mean, c = v[i].z - mean, d = v[i].w - mean;
      q += (a * a + b * b) + (c * c + d * d);
    }
    rstd = rsqrtf(warp_sum(q) * kInvH + 1e-5f);
  };
  float mean, rstd;
  stats(mean, rstd);
  float4* hr = reinterpret_cast<float4*>(h + row * H) + lane;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    v[i].x = (v[i].x - mean) * rstd * sc[i].x + sh[i].x;
    v[i].y = (v[i].y - mean) * rstd * sc[i].y + sh[i].y;
    v[i].z = (v[i].z - mean) * rstd * sc[i].z + sh[i].z;
    v[i].w = (v[i].w - mean) * rstd * sc[i].w + sh[i].w;
    hr[i * 32] = v[i];
  }
  stats(mean, rstd);
  const float4* gp = reinterpret_cast<const float4*>(gamma) + lane;
  const float4* bp = reinterpret_cast<const float4*>(beta) + lane;
  uint2* ur = reinterpret_cast<uint2*>(u + row * H) + lane;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const float4 g = __ldg(gp + i * 32), b = __ldg(bp + i * 32);
    ur[i * 32] = make_uint2(pack_bf16x2((v[i].x - mean) * rstd * g.x + b.x, (v[i].y - mean) * rstd * g.y + b.y),
                            pack_bf16x2((v[i].z - mean) * rstd * g.z + b.z, (v[i].w - mean) * rstd * g.w + b.w));
  }
}

int launch_adaln_ln(const float* x, int64_t n_x, const float* time_table, const float* text_mod, const int64_t* t,
                    int steps, const float* gamma, const float* beta, float* h, void* u, bool u_bf16, bf16* xcast,
                    int64_t n_seq, int T, int H, cudaStream_t st, float2* stat, bool xcast_all, int* row_pos) {
  DITTO_REQUIRE(H % 4 == 0 && H <= LN_MAXV * 128, DITTO_E_UNSUPPORTED, "adaln: need H % 4 == 0 and H <= 1024");
  const unsigned blocks = static_cast<unsigned>(ceil_div(n_seq * T, 8));
  ProfScope prof(PC_ADALN, st, 0.0, static_cast<double>(n_seq) * T * H * (u_bf16 ? 10 + 2 : 12));
  if (u_bf16 && u != nullptr && stat == nullptr && gamma != nullptr && beta != nullptr && (H == 768 || H == 256 || H == 512 || H == 1024)) {
    bf16* ub = static_cast<bf16*>(u);
    switch (H) {   // compile-time row width: no predicated slots
      case 768: adaln_ln_fast_kernel<6><<<blocks, 256, 0, st>>>(x, n_x, time_table, text_mod, t, steps, gamma, beta, h, ub, xcast, n_seq, T, xcast_all, row_pos); break;
      case 256: adaln_ln_fast_kernel<2><<<blocks, 256, 0, st>>>(x, n_x, time_table, text_mod, t, steps, gamma, beta, h, ub, xcast, n_seq, T, xcast_all, row_pos); break;
      case 512: adaln_ln_fast_kernel<4><<<blocks, 256, 0, st>>>(x, n_x, time_table, text_mod, t, steps, gamma, beta, h, ub, xcast, n_seq, T, xcast_all, row_pos); break;
      default: adaln_ln_fast_kernel<8><<<blocks, 256, 0, st>>>(x, n_x, time_table, text_mod, t, steps, gamma, beta, h, ub, xcast, n_seq, T, xcast_all, row_pos); break;
    }
  } else if (u_bf16)
    adaln_ln_kernel<bf16><<<blocks, 256, 0, st>>>(x, n_x, time_table, text_mod, t, steps, gamma, beta, h,
                                                  static_cast<bf16*>(u), xcast, n_seq, T, H, stat, xcast_all, row_pos);
  else
    adaln_ln_kernel<float><<<blocks, 256, 0, st>>>(x, n_x, time_table, text_mod, t, steps, gamma, beta, h,
                                                   static_cast<float*>(u), xcast, n_seq, T, H, stat, xcast_all, row_pos);
  DITTO_LAUNCH_CHECK();
  return 0;
}

// =====================================================================================================
// RoPE tables and application (DiT.py:46-72): angle[p][j] = float(p) * inv_freq[j] (fp32 product, as einsum)
// =====================================================================================================
__global__ void rope_table_kernel(const float* __restrict__ inv_freq, float* __restrict__ cos_t, float* __restrict__ sin_t,
                                  float* __restrict__ freq_out, int max_T, int half, int head_dim) {
  const int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= static_cast<int64_t>(max_T) * half) return;
  const int p = static_cast<int>(i / half), j = static_cast<int>(i % half);
  const float f = inv_freq ? inv_freq[j] : 1.0f / powf(10000.f, static_cast<float>(2 * j) / static_cast<float>(head_dim));
  const float a = static_cast<float>(p) * f;
  if (p == 0 && freq_out != nullptr) freq_out[j] = f;  // the frequencies the fused QKV epilogue multiplies positions with
  cos_t[i] = cosf(a);  // accurate (non fast-math) range reduction: angles reach ~2.2e3 rad
  sin_t[i] = sinf(a);
}

int launch_rope_table(const float* inv_freq, float* cos_t, float* sin_t, float* freq_out, int max_T, int half, int head_dim,
                      cudaStream_t st) {
  const int64_t n = static_cast<int64_t>(max_T) * half;
  rope_table_kernel<<<static_cast<unsigned>(ceil_div(n, 256)), 256, 0, st>>>(inv_freq, cos_t, sin_t, freq_out, max_T, half, head_dim);
  DITTO_LAUNCH_CHECK();
  return 0;
}

// in place on the q and k thirds of qkv [M, ld] (q at col 0, k at col H); pairs (j, j + d/2) inside each head
template <typename T>
__global__ void rope_kernel(T* __restrict__ qkv, int64_t ld, const float* __restrict__ cos_t,
                            const float* __restrict__ sin_t, int64_t rows, int seq_T, int H, int head_dim) {
  const int half = head_dim >> 1;
  const int pairs_per_row = H >> 1;                 // per q (and per k)
  const int64_t total = rows * pairs_per_row * 2;   // q and k
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < total;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int64_t row = i / (pairs_per_row * 2);
    int r = static_cast<int>(i - row * pairs_per_row * 2);
    const int which = r / pairs_per_row;            // 0 = q, 1 = k
    r -= which * pairs_per_row;
    const int head = r / half, j = r - head * half;
    const int pos = static_cast<int>(row % seq_T);
    const float c = cos_t[static_cast<int64_t>(pos) * half + j], s = sin_t[static_cast<int64_t>(pos) * half + j];
    T* p = qkv + row * ld + which * H + head * head_dim + j;
    const float x1 = static_cast<float>(p[0]), x2 = static_cast<float>(p[half]);
    p[0] = static_cast<T>(x1 * c - x2 * s);       // t*cos + (-x2)*sin
    p[half] = static_cast<T>(x2 * c + x1 * s);    // t*cos + ( x1)*sin
  }
}

int launch_rope(void* qkv, bool is_bf16, int64_t ld, const float* cos_t, const float* sin_t, int64_t rows, int seq_T,
                int H, int head_dim, cudaStream_t st) {
  const int64_t total = rows * H;
  const unsigned blocks = static_cast<unsigned>(std::min<int64_t>(ceil_div(total, 256), 148 * 32));
  ProfScope prof(PC_ROPE, st, 0.0, static_cast<double>(rows) * H * 2 * (is_bf16 ? 4 : 8));
  if (is_bf16)
    rope_kernel<bf16><<<blocks, 256, 0, st>>>(static_cast<bf16*>(qkv), ld, cos_t, sin_t, rows, seq_T, H, head_dim);
  else
    rope_kernel<float><<<blocks, 256, 0, st>>>(static_cast<float*>(qkv), ld, cos_t, sin_t, rows, seq_T, H, head_dim);
  DITTO_LAUNCH_CHECK();
  return 0;
}

// =====================================================================================================
// row softmax over fp32 scores -> P (bf16 or fp32, may alias the input when fp32).  One warp per row.
// =====================================================================================================
template <typename OutT, bool kFast>
__global__ void __launch_bounds__(256) softmax_kernel(const float* __restrict__ s, int64_t lds, OutT* __restrict__ p,
                                                      int64_t ldp, int64_t rows, int cols) {
  const int lane = threadIdx.x & 31;
  const int64_t row = static_cast<int64_t>(blockIdx.x) * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= rows) return;
  const float* sr = s + row * lds;
  OutT* pr = p + row * ldp;
  float m = -INFINITY;
  for (int c = lane; c < cols; c += 32) m = fmaxf(m, sr[c]);
  m = warp_max(m);
  float sum = 0.f;
  for (int c = lane; c < cols; c += 32) sum += kFast ? __expf(sr[c] - m) : expf(sr[c] - m);
  sum = warp_sum(sum);
  const float inv = 1.0f / sum;
  for (int c = lane; c < cols; c += 32) {
    const float e = kFast ? __expf(sr[c] - m) : expf(sr[c] - m);
    pr[c] = static_cast<OutT>(e * inv);
  }
  // zero the padding columns so that a full-width read never sees garbage
  for (int c = cols + lane; c < ldp; c += 32) pr[c] = static_cast<OutT>(0.f);
}

// single-pass variant for rows of at most 32 * kMaxV columns: the row lives in registers (one HBM read, one write)
template <typename OutT, bool kFast, int kMaxV>
__global__ void __launch_bounds__(256) softmax_reg_kernel(const float* __restrict__ s, int64_t lds, OutT* __restrict__ p,
                                                          int64_t ldp, int64_t rows, int cols) {
  const int lane = threadIdx.x & 31;
  const int64_t row = static_cast<int64_t>(blockIdx.x) * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= rows) return;
  const float* sr = s + row * lds;
  OutT* pr = p + row * ldp;
  float v[kMaxV];
  float m = -INFINITY;
#pragma unroll
  for (int i = 0; i < kMaxV; ++i) {
    const int c = i * 32 + lane;
    v[i] = c < cols ? sr[c] : -INFINITY;
    m = fmaxf(m, v[i]);
  }
  m = warp_max(m);
  float sum = 0.f;
#pragma unroll
  for (int i = 0; i < kMaxV; ++i) {
    v[i] = kFast ? __expf(v[i] - m) : expf(v[i] - m);  // exp(-inf) = 0 for the padding slots
    sum += v[i];
  }
  sum = warp_sum(sum);
  const float inv = 1.0f / sum;
#pragma unroll
  for (int i = 0; i < kMaxV; ++i) {
    const int c = i * 32 + lane;
    if (c < ldp) pr[c] = static_cast<OutT>(c < cols ? v[i] * inv : 0.f);  // padding columns are zeroed
  }
}

int launch_softmax(const float* s, int64_t lds, void* p, bool p_bf16, int64_t ldp, int64_t rows, int cols, cudaStream_t st) {
  if (rows <= 0) return 0;
  const unsigned blocks = static_cast<unsigned>(ceil_div(rows, 8));
  ProfScope prof(PC_SOFTMAX, st, 0.0, static_cast<double>(rows) * cols * (p_bf16 ? 6 : 8));
  const bool reg_ok = ldp <= 1024;
  if (p_bf16) {
    bf16* pp = static_cast<bf16*>(p);
    if (reg_ok && ldp <= 128) softmax_reg_kernel<bf16, true, 4><<<blocks, 256, 0, st>>>(s, lds, pp, ldp, rows, cols);
    else if (reg_ok && ldp <= 256) softmax_reg_kernel<bf16, true, 8><<<blocks, 256, 0, st>>>(s, lds, pp, ldp, rows, cols);
    else if (reg_ok && ldp <= 768) softmax_reg_kernel<bf16, true, 24><<<blocks, 256, 0, st>>>(s, lds, pp, ldp, rows, cols);
    else if (reg_ok) softmax_reg_kernel<bf16, true, 32><<<blocks, 256, 0, st>>>(s, lds, pp, ldp, rows, cols);
    else softmax_kernel<bf16, true><<<blocks, 256, 0, st>>>(s, lds, pp, ldp, rows, cols);
  } else {
    float* pp = static_cast<float*>(p);
    if (reg_ok && ldp <= 256) softmax_reg_kernel<float, false, 8><<<blocks, 256, 0, st>>>(s, lds, pp, ldp, rows, cols);
    else if (reg_ok) softmax_reg_kernel<float, false, 32><<<blocks, 256, 0, st>>>(s, lds, pp, ldp, rows, cols);
    else softmax_kernel<float, false><<<blocks, 256, 0, st>>>(s, lds, pp, ldp, rows, cols);
  }
  DITTO_LAUNCH_CHECK();
  return 0;
}

// =====================================================================================================
// fp32-path gated activation: hid = GELU_erf(a) * sigmoid(g)  (DiT.py:153-155)
// =====================================================================================================
__global__ void geglu_f32_kernel(const float* __restrict__ a, const float* __restrict__ g, float* __restrict__ out, int64_t n) {
  for (int64_t i = (static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x) * 4; i < n;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x * 4) {
    const float4 av = *reinterpret_cast<const float4*>(a + i);
    const float4 gv = *reinterpret_cast<const float4*>(g + i);
    float4 o;
    o.x = gelu_erf_f(av.x) * (1.0f / (1.0f + expf(-gv.x)));
    o.y = gelu_erf_f(av.y) * (1.0f / (1.0f + expf(-gv.y)));
    o.z = gelu_erf_f(av.z) * (1.0f / (1.0f + expf(-gv.z)));
    o.w = gelu_erf_f(av.w) * (1.0f / (1.0f + expf(-gv.w)));
    *reinterpret_cast<float4*>(out + i) = o;
  }
}
int launch_geglu_f32(const float* a, const float* g, float* out, int64_t n, cudaStream_t st) {
  DITTO_REQUIRE(n % 4 == 0, DITTO_E_UNSUPPORTED, "geglu: n % 4");
  const unsigned blocks = static_cast<unsigned>(std::min<int64_t>(ceil_div(n, 1024), 148 * 16));
  geglu_f32_kernel<<<blocks, 256, 0, st>>>(a, g, out, n);
  DITTO_LAUNCH_CHECK();
  return 0;
}

__global__ void silu_kernel(float* __restrict__ x, int64_t n) {
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const float v = x[i];
    x[i] = v / (1.0f + expf(-v));
  }
}
int launch_silu(float* x, int64_t n, cudaStream_t st) {
  silu_kernel<<<static_cast<unsigned>(std::min<int64_t>(ceil_div(n, 256), 148 * 8)), 256, 0, st>>>(x, n);
  DITTO_LAUNCH_CHECK();
  return 0;
}

// silu(mean_S(text)) : text [n, S, D] -> out [n, D]   (DiT.py:27 + the SiLU of text_mlp, DiT.py:19)
__global__ void mean_silu_kernel(const float* __restrict__ text, float* __restrict__ out, int S, int D) {
  const int seq = blockIdx.y;
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= D) return;
  const float* p = text + static_cast<int64_t>(seq) * S * D + c;
  float acc = 0.f;
  for (int s = 0; s < S; ++s) acc += p[static_cast<int64_t>(s) * D];
  const float m = acc / static_cast<float>(S);
  out[static_cast<int64_t>(seq) * D + c] = m / (1.0f + expf(-m));
}
int launch_mean_silu(const float* text, float* out, int64_t n, int S, int D, cudaStream_t st) {
  dim3 grid(static_cast<unsigned>(ceil_div(D, 128)), static_cast<unsigned>(n));
  mean_silu_kernel<<<grid, 128, 0, st>>>(text, out, S, D);
  DITTO_LAUNCH_CHECK();
  return 0;
}

// folded cross-attention score bias: sb[seq, head, s] = scale * sum_i K[seq*S + s, head*d + i] * bq[head*d + i]; zero pad
__global__ void fold_bias_kernel(const bf16* __restrict__ kv, int64_t ld, const float* __restrict__ bq, float* __restrict__ sb,
                                 int64_t total, int S, int Sp, int heads, int d, float scale) {
  const int lane = threadIdx.x & 31;
  const int64_t o = static_cast<int64_t>(blockIdx.x) * (blockDim.x >> 5) + (threadIdx.x >> 5);  // (seq, head, s in [0, Sp))
  if (o >= total) return;
  const int s_idx = static_cast<int>(o % Sp);
  const int head = static_cast<int>((o / Sp) % heads);
  const int64_t seq = o / (static_cast<int64_t>(Sp) * heads);
  float acc = 0.f;
  if (s_idx < S) {
    const bf16* row = kv + (seq * S + s_idx) * ld + head * d;
    for (int i = lane; i < d; i += 32) acc += __bfloat162float(row[i]) * bq[head * d + i];
  }
  acc = warp_sum(acc);
  if (lane == 0) sb[o] = s_idx < S ? scale * acc : 0.f;
}
int launch_fold_bias(const bf16* kv, int64_t ld, const float* bq, float* sb, int64_t n, int S, int Sp, int heads, int d, float scale,
                     cudaStream_t st) {
  const int64_t total = n * heads * Sp;
  fold_bias_kernel<<<static_cast<unsigned>(ceil_div(total, 8)), 256, 0, st>>>(kv, ld, bq, sb, total, S, Sp, heads, d, scale);
  DITTO_LAUNCH_CHECK();
  return 0;
}

// one block per sequence.  A sequence whose text rows are all equal has equal rows of V Wo^T, so its cross-attention output
// softmax(scores) (V Wo^T) + bo is the row vfold[0] + bo whatever the scores are.  Bitwise equality of the inputs is what
// makes the rows of the folded projections equal: the GEMMs that build them treat every row alike.
__global__ void const_text_kernel(const float* __restrict__ text, int S, int D, const bf16* __restrict__ vfold, int64_t vf_seq,
                                  bool vf_perm4, const float* __restrict__ bo, uint8_t* __restrict__ flag, float* __restrict__ crow,
                                  int H) {
  const int64_t seq = blockIdx.x;
  if (flag != nullptr) {
    const uint32_t* t = reinterpret_cast<const uint32_t*>(text) + seq * S * D;
    int diff = 0;
    for (int64_t i = D + threadIdx.x; i < static_cast<int64_t>(S) * D; i += blockDim.x) diff |= t[i] != t[i % D];
    diff = __syncthreads_or(diff);
    if (threadIdx.x == 0) flag[seq] = diff ? 0 : 1;
  }
  const bf16* v = vfold + seq * vf_seq;
  for (int c = threadIdx.x; c < H; c += blockDim.x) {
    // perm4 (gemm_resid_ln_weight_row): plain column 64 blk + 16 (kb / 2) + 4 q + 2 (kb % 2) + e sits at 64 blk + 8 kb + 2 q + e
    const int cp = c & 63, kb = 2 * (cp >> 4) + ((cp & 3) >> 1);
    const int src = vf_perm4 ? (c - cp) + 8 * kb + 2 * ((cp & 15) >> 2) + (cp & 1) : c;
    crow[seq * H + c] = __bfloat162float(v[src]) + bo[c];
  }
}
int launch_const_text(const float* text, int64_t n, int S, int D, const bf16* vfold, int64_t vf_seq, bool vf_perm4, const float* bo,
                      uint8_t* flag, float* crow, int H, cudaStream_t st) {
  DITTO_REQUIRE(!vf_perm4 || H % 64 == 0, DITTO_E_BADARG, "const_text: perm4 column order needs H % 64 == 0");
  const_text_kernel<<<static_cast<unsigned>(n), 256, 0, st>>>(text, S, D, vfold, vf_seq, vf_perm4, bo, flag, crow, H);
  DITTO_LAUNCH_CHECK();
  return 0;
}

// V [T, d] slices of qkv (ld) -> Vt [n*heads, d, Tp] (keys contiguous): fallback operand layout for P@V
__global__ void transpose_v_kernel(const bf16* __restrict__ v, int64_t ld, bf16* __restrict__ vt, int T, int Tp, int heads,
                                   int d) {
  __shared__ bf16 tile[32][33];
  const int b = blockIdx.z;  // seq * heads + head
  const int seq = b / heads, head = b % heads;
  const bf16* src = v + (static_cast<int64_t>(seq) * T) * ld + head * d;
  bf16* dst = vt + static_cast<int64_t>(b) * d * Tp;
  const int t0 = blockIdx.x * 32, c0 = blockIdx.y * 32;
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int tt = t0 + i, c = c0 + threadIdx.x;
    tile[i][threadIdx.x] = (tt < T && c < d) ? src[static_cast<int64_t>(tt) * ld + c] : __float2bfloat16(0.f);
  }
  __syncthreads();
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int c = c0 + i, tt = t0 + threadIdx.x;
    if (c < d && tt < Tp) dst[static_cast<int64_t>(c) * Tp + tt] = tile[threadIdx.x][i];
  }
}
int launch_transpose_v(const bf16* v, int64_t ld, bf16* vt, int64_t n_seq, int T, int Tp, int heads, int d, cudaStream_t st) {
  dim3 grid(static_cast<unsigned>(ceil_div(Tp, 32)), static_cast<unsigned>(ceil_div(d, 32)), static_cast<unsigned>(n_seq * heads));
  transpose_v_kernel<<<grid, dim3(32, 8), 0, st>>>(v, ld, vt, T, Tp, heads, d);
  DITTO_LAUNCH_CHECK();
  return 0;
}

// =====================================================================================================
// CFG combine + DDPM ancestral update, one pass (SpeechGenerator.py:137-147 + the guidance extension)
//   coef[t] = { 1/sqrt(alpha_t), (1-alpha_t)/sqrt(1-acp_t), [t>0]*sqrt(beta_t) }
// 20 B/element with guidance + noise (4 reads, 1 write), 128-bit accesses, grid = multiple of 148.
// =====================================================================================================
// one element: eps = eps_u + w (eps_c - eps_u);  x_out = c1 (x - c2 eps) + c3 z   -- explicit roundings so that the variant
// with caller-supplied noise and the one that draws it in the kernel agree bit for bit
__device__ __forceinline__ float cfg_combine(float ec, float eu, float w) { return __fmaf_rn(w, __fsub_rn(ec, eu), eu); }
__device__ __forceinline__ float ddpm_update(float x, float e, float z, float c1, float c2, float c3) {
  return __fmaf_rn(c3, z, __fmul_rn(c1, __fmaf_rn(-c2, e, x)));
}

__global__ void __launch_bounds__(256)
    cfg_ddpm_update_kernel(const float4* __restrict__ eps_c, const float4* __restrict__ eps_u, const float4* __restrict__ x,
                           const float4* __restrict__ z, const int64_t* __restrict__ t, const float* __restrict__ coef,
                           int steps, float w, float4* __restrict__ out, int64_t vec_per_seq, int64_t total_vec) {
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < total_vec;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int64_t seq = i / vec_per_seq;
    int64_t tt = t[seq];
    tt = tt < 0 ? 0 : (tt >= steps ? steps - 1 : tt);
    const float c1 = coef[tt * 3 + 0], c2 = coef[tt * 3 + 1], c3 = coef[tt * 3 + 2];
    float4 e = eps_c[i];
    if (eps_u != nullptr) {
      const float4 u = eps_u[i];
      e = make_float4(cfg_combine(e.x, u.x, w), cfg_combine(e.y, u.y, w), cfg_combine(e.z, u.z, w), cfg_combine(e.w, u.w, w));
    }
    const float4 xv = x[i];
    const float4 zv = z != nullptr ? z[i] : make_float4(0.f, 0.f, 0.f, 0.f);   // + c3 * 0 == the reference's masked noise term
    out[i] = make_float4(ddpm_update(xv.x, e.x, zv.x, c1, c2, c3), ddpm_update(xv.y, e.y, zv.y, c1, c2, c3),
                         ddpm_update(xv.z, e.z, zv.z, c1, c2, c3), ddpm_update(xv.w, e.w, zv.w, c1, c2, c3));
  }
}

int launch_cfg_ddpm_update(const float* eps_c, const float* eps_u, const float* x, const float* z, const int64_t* t,
                           const float* coef, int steps, float w, float* out, int64_t B, int64_t elems_per_seq,
                           cudaStream_t st) {
  DITTO_REQUIRE(elems_per_seq % 4 == 0, DITTO_E_UNSUPPORTED, "cfg_ddpm_update: elems_per_seq % 4");
  const int64_t total_vec = B * elems_per_seq / 4;
  if (total_vec == 0) return 0;
  const int64_t want = ceil_div(total_vec, 256 * 4);  // ~4 vectors per thread
  const unsigned blocks = static_cast<unsigned>(std::min<int64_t>(round_up(want, 148), 148 * 32));
  ProfScope prof(PC_CFG_UPDATE, st, 0.0, static_cast<double>(total_vec) * 16 * (3 + (eps_u ? 1 : 0) + (z ? 1 : 0)));
  cfg_ddpm_update_kernel<<<blocks, 256, 0, st>>>(
      reinterpret_cast<const float4*>(eps_c), reinterpret_cast<const float4*>(eps_u), reinterpret_cast<const float4*>(x),
      reinterpret_cast<const float4*>(z), t, coef, steps, w, reinterpret_cast<float4*>(out), elems_per_seq / 4, total_vec);
  DITTO_LAUNCH_CHECK();
  return 0;
}

// =====================================================================================================
// The same with the step's noise drawn in the kernel: z = randn_like(x) of SpeechGenerator.py:145 without the separate
// generator launch and its 8 B / element of HBM round trip.  Philox4x32-10 (Salmon et al., SC'11: the counter-based generator
// behind curand and torch's CUDA randn) keyed by the 64-bit seed, counter = (vector index, draw counter); four uniforms ->
// two Box-Muller pairs -> the four normals of one float4.  The draw counter lives in device memory so that a captured CUDA
// graph draws fresh noise on every replay; with `advance` the LAST block to finish (ticket counter) adds 1 to it and
// subtracts 1 from every t[i] -- the bookkeeping of `for t_val in reversed(range(steps))` (SpeechGenerator.py:161-162).
// rng: device uint64[4] = {seed, draw counter, ticket (kept 0 between launches), reserved}.
// =====================================================================================================
__device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint2 k) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint32_t hi0 = __umulhi(0xD2511F53u, c.x), lo0 = 0xD2511F53u * c.x;
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, c.z), lo1 = 0xCD9E8D57u * c.z;
    c = make_uint4(hi1 ^ c.y ^ k.x, lo1, hi0 ^ c.w ^ k.y, lo0);
    k.x += 0x9E3779B9u;
    k.y += 0xBB67AE85u;
  }
  return c;
}
// four N(0, 1) samples for vector index v of draw `draw`
__device__ __forceinline__ float4 philox_normal4(unsigned long long seed, unsigned long long draw, unsigned long long v) {
  const uint4 r = philox4x32_10(make_uint4(static_cast<uint32_t>(v), static_cast<uint32_t>(v >> 32), static_cast<uint32_t>(draw),
                                           static_cast<uint32_t>(draw >> 32)),
                                make_uint2(static_cast<uint32_t>(seed), static_cast<uint32_t>(seed >> 32)));
  // u in (0, 1): 24 random bits + half an ulp, so that log(u) is finite and cos / sin see [0, 2 pi)
  const float u0 = fmaf(static_cast<float>(r.x >> 8), 5.9604644775390625e-08f, 2.98023223876953125e-08f);
  const float u1 = fmaf(static_cast<float>(r.z >> 8), 5.9604644775390625e-08f, 2.98023223876953125e-08f);
  const float a0 = static_cast<float>(r.y >> 8) * (6.283185307179586f * 5.9604644775390625e-08f);
  const float a1 = static_cast<float>(r.w >> 8) * (6.283185307179586f * 5.9604644775390625e-08f);
  const float m0 = sqrtf(-1.3862943611198906f * __log2f(u0)), m1 = sqrtf(-1.3862943611198906f * __log2f(u1));  // sqrt(-2 ln u)
  float s0, c0, s1, c1;
  __sincosf(a0, &s0, &c0);
  __sincosf(a1, &s1, &c1);
  return make_float4(m0 * c0, m0 * s0, m1 * c1, m1 * s1);
}

// `advance` of the in-kernel-noise update kernels: called by every block after its last read of rng / t
__device__ __forceinline__ void last_block_advances(unsigned long long* rng, int64_t* t, int64_t n_t, unsigned long long draw) {
  // every thread of every block has read rng / t before its block takes a ticket; the block holding the last ticket owns them
  __shared__ int s_last;
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    const unsigned long long tk = atomicAdd(rng + 2, 1ull);
    s_last = tk == static_cast<unsigned long long>(gridDim.x) - 1ull;
  }
  __syncthreads();
  if (!s_last) return;
  __threadfence();
  for (int64_t i = threadIdx.x; i < n_t; i += blockDim.x) t[i] -= 1;
  if (threadIdx.x == 0) {
    rng[1] = draw + 1ull;
    rng[2] = 0ull;
  }
}

__global__ void __launch_bounds__(256)
    cfg_ddpm_update_rng_kernel(const float4* __restrict__ eps_c, const float4* __restrict__ eps_u, const float4* __restrict__ x,
                               unsigned long long* rng, int64_t* t, int64_t n_t, const float* __restrict__ coef, int steps, float w,
                               float4* __restrict__ out, int64_t vec_per_seq, int64_t total_vec, int64_t vec_offset, int advance) {
  const unsigned long long seed = rng[0], draw = rng[1];
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < total_vec;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int64_t seq = i / vec_per_seq;
    int64_t tt = t[seq];
    tt = tt < 0 ? 0 : (tt >= steps ? steps - 1 : tt);
    const float c1 = coef[tt * 3 + 0], c2 = coef[tt * 3 + 1], c3 = coef[tt * 3 + 2];
    float4 e = eps_c[i];
    if (eps_u != nullptr) {
      const float4 u = eps_u[i];
      e = make_float4(cfg_combine(e.x, u.x, w), cfg_combine(e.y, u.y, w), cfg_combine(e.z, u.z, w), cfg_combine(e.w, u.w, w));
    }
    const float4 xv = x[i];
    const float4 zv = philox_normal4(seed, draw, static_cast<unsigned long long>(vec_offset + i));
    out[i] = make_float4(ddpm_update(xv.x, e.x, zv.x, c1, c2, c3), ddpm_update(xv.y, e.y, zv.y, c1, c2, c3),
                         ddpm_update(xv.z, e.z, zv.z, c1, c2, c3), ddpm_update(xv.w, e.w, zv.w, c1, c2, c3));
  }
  if (advance) last_block_advances(rng, t, n_t, draw);
}

int launch_cfg_ddpm_update_rng(const float* eps_c, const float* eps_u, const float* x, unsigned long long* rng, int64_t* t, int64_t n_t,
                               const float* coef, int steps, float w, float* out, int64_t B, int64_t elems_per_seq,
                               int64_t elem_offset, bool advance, cudaStream_t st) {
  DITTO_REQUIRE(elems_per_seq % 4 == 0 && elem_offset % 4 == 0, DITTO_E_UNSUPPORTED, "cfg_ddpm_update_rng: elems_per_seq % 4");
  const int64_t total_vec = B * elems_per_seq / 4;
  if (total_vec == 0) return advance ? launch_step_advance(rng, t, n_t, st) : 0;
  const int64_t want = ceil_div(total_vec, 256 * 4);
  const unsigned blocks = static_cast<unsigned>(std::min<int64_t>(round_up(want, 148), 148 * 32));
  ProfScope prof(PC_CFG_UPDATE, st, 0.0, static_cast<double>(total_vec) * 16 * (3 + (eps_u ? 1 : 0)));
  cfg_ddpm_update_rng_kernel<<<blocks, 256, 0, st>>>(reinterpret_cast<const float4*>(eps_c), reinterpret_cast<const float4*>(eps_u),
                                                     reinterpret_cast<const float4*>(x), rng, t, n_t, coef, steps, w,
                                                     reinterpret_cast<float4*>(out), elems_per_seq / 4, total_vec, elem_offset / 4,
                                                     advance ? 1 : 0);
  DITTO_LAUNCH_CHECK();
  return 0;
}

// =====================================================================================================
// CFG combine + multistep update (DPM-Solver++(2M), Lu et al. 2022 Alg. 2, and its SDE variant), one pass:
//   x_out = c1 (x - c2 eps) + c3 z + c4 hist        hist <- d1 (x - d2 eps)   (the x0 prediction of this step)
//   coef_ms[t] = {c1, c2, c3, c4, d1, d2}, computed on the host (schedules.dpmpp_2m_coef).
// The first term is ddpm_update with the same roundings, the history term one more fma; a row with c4 == 0 (first-order
// steps) neither reads hist nor adds the term, so x_out is bit-identical to cfg_ddpm_update_kernel with (c1, c2, c3) and
// whatever hist held before the first step (uninitialised, NaN) cannot reach it.  c4 is uniform per sequence (one row per
// t[seq]), so the branch does not diverge inside a sequence's vectors.  x_out may alias x and hist is updated in place:
// every thread reads its elements before it writes them.  +8 B / element over the DDPM kernel (hist read + write).
// =====================================================================================================
__device__ __forceinline__ float x0_pred(float x, float e, float d1, float d2) { return __fmul_rn(d1, __fmaf_rn(-d2, e, x)); }

// one row of the table; the hist read is issued together with the other loads of the element (before the noise is drawn),
// predicated on c4 so that first-order rows never touch it
struct MultistepRow {
  float c1, c2, c3, c4, d1, d2;
};
__device__ __forceinline__ MultistepRow multistep_row(const float* __restrict__ coef, const int64_t* t, int64_t seq, int steps) {
  int64_t tt = t[seq];
  tt = tt < 0 ? 0 : (tt >= steps ? steps - 1 : tt);
  const float* r = coef + tt * 6;
  return MultistepRow{r[0], r[1], r[2], r[3], r[4], r[5]};
}
__device__ __forceinline__ float4 multistep_hist(const float4* __restrict__ hist, int64_t i, float c4) {
  return c4 != 0.f ? hist[i] : make_float4(0.f, 0.f, 0.f, 0.f);
}
__device__ __forceinline__ void multistep_store(const MultistepRow& c, float4 xv, float4 e, float4 zv, float4 h,
                                                float4* __restrict__ out, float4* __restrict__ hist, int64_t i) {
  float4 o = make_float4(ddpm_update(xv.x, e.x, zv.x, c.c1, c.c2, c.c3), ddpm_update(xv.y, e.y, zv.y, c.c1, c.c2, c.c3),
                         ddpm_update(xv.z, e.z, zv.z, c.c1, c.c2, c.c3), ddpm_update(xv.w, e.w, zv.w, c.c1, c.c2, c.c3));
  if (c.c4 != 0.f)
    o = make_float4(__fmaf_rn(c.c4, h.x, o.x), __fmaf_rn(c.c4, h.y, o.y), __fmaf_rn(c.c4, h.z, o.z), __fmaf_rn(c.c4, h.w, o.w));
  hist[i] = make_float4(x0_pred(xv.x, e.x, c.d1, c.d2), x0_pred(xv.y, e.y, c.d1, c.d2), x0_pred(xv.z, e.z, c.d1, c.d2),
                        x0_pred(xv.w, e.w, c.d1, c.d2));
  out[i] = o;
}

__global__ void __launch_bounds__(256)
    cfg_multistep_update_kernel(const float4* __restrict__ eps_c, const float4* __restrict__ eps_u, const float4* __restrict__ x,
                                const float4* __restrict__ z, const int64_t* __restrict__ t, const float* __restrict__ coef,
                                int steps, float w, float4* __restrict__ out, float4* __restrict__ hist, int64_t vec_per_seq,
                                int64_t total_vec) {
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < total_vec;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const MultistepRow c = multistep_row(coef, t, i / vec_per_seq, steps);
    float4 e = eps_c[i];
    if (eps_u != nullptr) {
      const float4 u = eps_u[i];
      e = make_float4(cfg_combine(e.x, u.x, w), cfg_combine(e.y, u.y, w), cfg_combine(e.z, u.z, w), cfg_combine(e.w, u.w, w));
    }
    const float4 xv = x[i];
    const float4 zv = z != nullptr ? z[i] : make_float4(0.f, 0.f, 0.f, 0.f);
    const float4 h = multistep_hist(hist, i, c.c4);
    multistep_store(c, xv, e, zv, h, out, hist, i);
  }
}

int launch_cfg_multistep_update(const float* eps_c, const float* eps_u, const float* x, const float* z, const int64_t* t,
                                const float* coef, int steps, float w, float* out, float* hist, int64_t B, int64_t elems_per_seq,
                                cudaStream_t st) {
  DITTO_REQUIRE(elems_per_seq % 4 == 0, DITTO_E_UNSUPPORTED, "cfg_multistep_update: elems_per_seq % 4");
  const int64_t total_vec = B * elems_per_seq / 4;
  if (total_vec == 0) return 0;
  const int64_t want = ceil_div(total_vec, 256 * 4);
  const unsigned blocks = static_cast<unsigned>(std::min<int64_t>(round_up(want, 148), 148 * 32));
  ProfScope prof(PC_CFG_UPDATE, st, 0.0, static_cast<double>(total_vec) * 16 * (5 + (eps_u ? 1 : 0) + (z ? 1 : 0)));
  cfg_multistep_update_kernel<<<blocks, 256, 0, st>>>(
      reinterpret_cast<const float4*>(eps_c), reinterpret_cast<const float4*>(eps_u), reinterpret_cast<const float4*>(x),
      reinterpret_cast<const float4*>(z), t, coef, steps, w, reinterpret_cast<float4*>(out), reinterpret_cast<float4*>(hist),
      elems_per_seq / 4, total_vec);
  DITTO_LAUNCH_CHECK();
  return 0;
}

// the same with the noise drawn in the kernel: Philox stream, element offsets and `advance` bookkeeping exactly as
// cfg_ddpm_update_rng_kernel (the normals equal ditto_randn's at the same {seed, draw})
__global__ void __launch_bounds__(256)
    cfg_multistep_update_rng_kernel(const float4* __restrict__ eps_c, const float4* __restrict__ eps_u, const float4* __restrict__ x,
                                    unsigned long long* rng, int64_t* t, int64_t n_t, const float* __restrict__ coef, int steps,
                                    float w, float4* __restrict__ out, float4* __restrict__ hist, int64_t vec_per_seq,
                                    int64_t total_vec, int64_t vec_offset, int advance) {
  const unsigned long long seed = rng[0], draw = rng[1];
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < total_vec;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const MultistepRow c = multistep_row(coef, t, i / vec_per_seq, steps);
    float4 e = eps_c[i];
    if (eps_u != nullptr) {
      const float4 u = eps_u[i];
      e = make_float4(cfg_combine(e.x, u.x, w), cfg_combine(e.y, u.y, w), cfg_combine(e.z, u.z, w), cfg_combine(e.w, u.w, w));
    }
    const float4 xv = x[i];
    const float4 h = multistep_hist(hist, i, c.c4);
    const float4 zv = philox_normal4(seed, draw, static_cast<unsigned long long>(vec_offset + i));
    multistep_store(c, xv, e, zv, h, out, hist, i);
  }
  if (advance) last_block_advances(rng, t, n_t, draw);
}

int launch_cfg_multistep_update_rng(const float* eps_c, const float* eps_u, const float* x, unsigned long long* rng, int64_t* t,
                                    int64_t n_t, const float* coef, int steps, float w, float* out, float* hist, int64_t B,
                                    int64_t elems_per_seq, int64_t elem_offset, bool advance, cudaStream_t st) {
  DITTO_REQUIRE(elems_per_seq % 4 == 0 && elem_offset % 4 == 0, DITTO_E_UNSUPPORTED, "cfg_multistep_update_rng: elems_per_seq % 4");
  const int64_t total_vec = B * elems_per_seq / 4;
  if (total_vec == 0) return advance ? launch_step_advance(rng, t, n_t, st) : 0;
  const int64_t want = ceil_div(total_vec, 256 * 4);
  const unsigned blocks = static_cast<unsigned>(std::min<int64_t>(round_up(want, 148), 148 * 32));
  ProfScope prof(PC_CFG_UPDATE, st, 0.0, static_cast<double>(total_vec) * 16 * (5 + (eps_u ? 1 : 0)));
  cfg_multistep_update_rng_kernel<<<blocks, 256, 0, st>>>(
      reinterpret_cast<const float4*>(eps_c), reinterpret_cast<const float4*>(eps_u), reinterpret_cast<const float4*>(x), rng, t,
      n_t, coef, steps, w, reinterpret_cast<float4*>(out), reinterpret_cast<float4*>(hist), elems_per_seq / 4, total_vec,
      elem_offset / 4, advance ? 1 : 0);
  DITTO_LAUNCH_CHECK();
  return 0;
}

// =====================================================================================================
// CFG combine + update with known frames (replacement conditioning: a speech prompt or an infilled span; the imputation
// of Song et al. 2021, score SDE, i.e. RePaint without its resampling loop), one pass.  A frame flagged in `mask` is
// the known latent p re-noised to the level of this step's output,
//     x_out = a p + s z,   coef_known[t] = {a, s} = {sqrt(abar_next), sqrt(1 - abar_next)}   (last visited step: {1, 0} -> p)
// with z the normal the update draws (or is given) for that element, so the draw counter and its bookkeeping are those of
// the plain update.  Every other frame takes the DDPM-form (MULTISTEP = false) or multistep update through the same device
// helpers as cfg_ddpm_update(_rng)_kernel / cfg_multistep_update(_rng)_kernel, so it rounds exactly as they do.  A frame is
// H/4 consecutive float4s (6 warps at H = 768), so the branch is uniform per warp when H % 128 == 0.  A known frame reads
// the mask byte, p and (supplied noise) z -- no eps, x or hist -- and leaves hist as it was: 8 B / element with drawn noise
// (12 with supplied z) against 16-28 B for an unknown one.  All loads are issued before the noise is drawn.
// =====================================================================================================
__device__ __forceinline__ float known_value(float p, float z, float a, float s) { return __fmaf_rn(s, z, __fmul_rn(a, p)); }

template <bool MULTISTEP, bool RNG>
__global__ void __launch_bounds__(256)
    cfg_update_known_kernel(const float4* __restrict__ eps_c, const float4* __restrict__ eps_u, const float4* __restrict__ x,
                            const float4* __restrict__ z, unsigned long long* rng, int64_t* t, int64_t n_t,
                            const float* __restrict__ coef, const float* __restrict__ coef_known, int steps, float w,
                            float4* __restrict__ out, float4* __restrict__ hist, const float4* __restrict__ known,
                            const uint8_t* __restrict__ mask, int64_t vec_per_seq, int64_t vec_per_frame, int64_t total_vec,
                            int64_t vec_offset, int advance) {
  unsigned long long seed = 0ull, draw = 0ull;
  if (RNG) {
    seed = rng[0];
    draw = rng[1];
  }
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < total_vec;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int64_t seq = i / vec_per_seq;
    if (mask[i / vec_per_frame] != 0) {
      int64_t tt = t[seq];
      tt = tt < 0 ? 0 : (tt >= steps ? steps - 1 : tt);
      const float a = coef_known[tt * 2 + 0], s = coef_known[tt * 2 + 1];
      const float4 pv = known[i];
      const float4 zv = RNG ? philox_normal4(seed, draw, static_cast<unsigned long long>(vec_offset + i)) : z[i];
      out[i] = make_float4(known_value(pv.x, zv.x, a, s), known_value(pv.y, zv.y, a, s), known_value(pv.z, zv.z, a, s),
                           known_value(pv.w, zv.w, a, s));
      continue;
    }
    if (MULTISTEP) {
      const MultistepRow c = multistep_row(coef, t, seq, steps);
      float4 e = eps_c[i];
      if (eps_u != nullptr) {
        const float4 u = eps_u[i];
        e = make_float4(cfg_combine(e.x, u.x, w), cfg_combine(e.y, u.y, w), cfg_combine(e.z, u.z, w), cfg_combine(e.w, u.w, w));
      }
      const float4 xv = x[i];
      float4 zv = RNG ? make_float4(0.f, 0.f, 0.f, 0.f) : z[i];
      const float4 h = multistep_hist(hist, i, c.c4);
      if (RNG) zv = philox_normal4(seed, draw, static_cast<unsigned long long>(vec_offset + i));
      multistep_store(c, xv, e, zv, h, out, hist, i);
    } else {
      int64_t tt = t[seq];
      tt = tt < 0 ? 0 : (tt >= steps ? steps - 1 : tt);
      const float c1 = coef[tt * 3 + 0], c2 = coef[tt * 3 + 1], c3 = coef[tt * 3 + 2];
      float4 e = eps_c[i];
      if (eps_u != nullptr) {
        const float4 u = eps_u[i];
        e = make_float4(cfg_combine(e.x, u.x, w), cfg_combine(e.y, u.y, w), cfg_combine(e.z, u.z, w), cfg_combine(e.w, u.w, w));
      }
      const float4 xv = x[i];
      const float4 zv = RNG ? philox_normal4(seed, draw, static_cast<unsigned long long>(vec_offset + i)) : z[i];
      out[i] = make_float4(ddpm_update(xv.x, e.x, zv.x, c1, c2, c3), ddpm_update(xv.y, e.y, zv.y, c1, c2, c3),
                           ddpm_update(xv.z, e.z, zv.z, c1, c2, c3), ddpm_update(xv.w, e.w, zv.w, c1, c2, c3));
    }
  }
  if (RNG && advance) last_block_advances(rng, t, n_t, draw);
}

// only while profiling (which synchronises anyway and is never captured), so a step graph never sees the copy
int64_t profiled_nonzero(const uint8_t* mask, int64_t n, cudaStream_t st) {
  cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
  if (!g_prof_enabled || cudaStreamIsCapturing(st, &cs) != cudaSuccess || cs != cudaStreamCaptureStatusNone) return 0;
  std::vector<uint8_t> h(static_cast<size_t>(n));
  if (cudaMemcpyAsync(h.data(), mask, static_cast<size_t>(n), cudaMemcpyDeviceToHost, st) != cudaSuccess ||
      cudaStreamSynchronize(st) != cudaSuccess)
    return 0;
  int64_t k = 0;
  for (uint8_t v : h) k += v != 0;
  return k;
}

int launch_cfg_update_known(const float* eps_c, const float* eps_u, const float* x, const float* z, unsigned long long* rng, int64_t* t,
                            int64_t n_t, const float* coef, const float* coef_known, int steps, float w, float* out, float* hist,
                            const float* known, const uint8_t* mask, int64_t B, int64_t T, int64_t H, int64_t elem_offset, bool advance,
                            cudaStream_t st) {
  DITTO_REQUIRE(H % 4 == 0 && elem_offset % 4 == 0, DITTO_E_UNSUPPORTED, "cfg_update_known: H % 4 and element offset % 4");
  const bool draw = rng != nullptr, ms = hist != nullptr;
  const int64_t vec_per_frame = H / 4, total_vec = B * T * vec_per_frame;
  if (total_vec == 0) return (draw && advance) ? launch_step_advance(rng, t, n_t, st) : 0;
  const int64_t want = ceil_div(total_vec, 256 * 4);
  const unsigned blocks = static_cast<unsigned>(std::min<int64_t>(round_up(want, 148), 148 * 32));
  // bytes moved: 16 B per float4 of every stream a frame touches, plus one mask byte per frame
  const int64_t known_vec = profiled_nonzero(mask, B * T, st) * vec_per_frame;
  const double unknown_streams = (ms ? 5 : 3) + (eps_u ? 1 : 0) + (draw ? 0 : 1), known_streams = 2 + (draw ? 0 : 1);
  ProfScope prof(PC_CFG_UPDATE, st, 0.0,
                 16.0 * (static_cast<double>(total_vec - known_vec) * unknown_streams + static_cast<double>(known_vec) * known_streams) +
                     static_cast<double>(B * T));
  const float4 *ec = reinterpret_cast<const float4*>(eps_c), *eu = reinterpret_cast<const float4*>(eps_u);
  const float4 *xv = reinterpret_cast<const float4*>(x), *zv = reinterpret_cast<const float4*>(z);
  const float4* kv = reinterpret_cast<const float4*>(known);
  float4 *o = reinterpret_cast<float4*>(out), *h = reinterpret_cast<float4*>(hist);
  const int64_t vps = T * vec_per_frame, voff = elem_offset / 4;
  const int adv = advance ? 1 : 0;
  if (ms && draw)
    cfg_update_known_kernel<true, true><<<blocks, 256, 0, st>>>(ec, eu, xv, zv, rng, t, n_t, coef, coef_known, steps, w, o, h, kv, mask,
                                                                vps, vec_per_frame, total_vec, voff, adv);
  else if (ms)
    cfg_update_known_kernel<true, false><<<blocks, 256, 0, st>>>(ec, eu, xv, zv, rng, t, n_t, coef, coef_known, steps, w, o, h, kv, mask,
                                                                 vps, vec_per_frame, total_vec, voff, adv);
  else if (draw)
    cfg_update_known_kernel<false, true><<<blocks, 256, 0, st>>>(ec, eu, xv, zv, rng, t, n_t, coef, coef_known, steps, w, o, h, kv, mask,
                                                                 vps, vec_per_frame, total_vec, voff, adv);
  else
    cfg_update_known_kernel<false, false><<<blocks, 256, 0, st>>>(ec, eu, xv, zv, rng, t, n_t, coef, coef_known, steps, w, o, h, kv,
                                                                  mask, vps, vec_per_frame, total_vec, voff, adv);
  DITTO_LAUNCH_CHECK();
  return 0;
}

// the bookkeeping alone (ragged batches: their per-group update kernels run concurrently, so none of them can own it)
__global__ void step_advance_kernel(unsigned long long* rng, int64_t* t, int64_t n_t) {
  for (int64_t i = threadIdx.x; i < n_t; i += blockDim.x) t[i] -= 1;
  if (threadIdx.x == 0 && rng != nullptr) rng[1] += 1ull;
}
int launch_step_advance(unsigned long long* rng, int64_t* t, int64_t n_t, cudaStream_t st) {
  step_advance_kernel<<<1, 256, 0, st>>>(rng, t, n_t);
  DITTO_LAUNCH_CHECK();
  return 0;
}

// out[i] = the normal the update kernel draws for element elem_offset + i at the current draw counter (tests, and a
// stand-alone randn for callers that want the library's stream)
__global__ void randn_kernel(const unsigned long long* __restrict__ rng, int64_t vec_offset, float* __restrict__ out, int64_t n) {
  const unsigned long long seed = rng[0], draw = rng[1];
  const int64_t nv = (n + 3) / 4;
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < nv; i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const float4 z = philox_normal4(seed, draw, static_cast<unsigned long long>(vec_offset + i));
    if (4 * i + 3 < n) {
      *reinterpret_cast<float4*>(out + 4 * i) = z;
    } else {
      const float zz[4] = {z.x, z.y, z.z, z.w};
      for (int j = 0; 4 * i + j < n; ++j) out[4 * i + j] = zz[j];
    }
  }
}
int launch_randn(const unsigned long long* rng, int64_t elem_offset, float* out, int64_t n, cudaStream_t st) {
  DITTO_REQUIRE(elem_offset % 4 == 0 && (reinterpret_cast<uintptr_t>(out) & 15) == 0, DITTO_E_BADARG, "randn: offset % 4 and 16-B aligned output");
  if (n <= 0) return 0;
  const unsigned blocks = static_cast<unsigned>(std::min<int64_t>(round_up(ceil_div(n, 1024), 148), 148 * 32));
  randn_kernel<<<blocks, 256, 0, st>>>(rng, elem_offset / 4, out, n);
  DITTO_LAUNCH_CHECK();
  return 0;
}

// RotaryEmbedding.apply_rope (DiT.py:61-72) on its own: out = t cos(pos) + rotate_half(t) sin(pos); t [batch, T, heads, d],
// pos [T, d] fp32 ANGLES (what RotaryEmbedding.forward returns; both halves are read, as the reference does)
__global__ void rope_angles_kernel(const float* __restrict__ t, const float* __restrict__ pos, float* __restrict__ out, int64_t total,
                                   int T, int heads, int d) {
  const int half = d >> 1;
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < total; i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int j = static_cast<int>(i % d);
    const int64_t r = i / d;                               // (batch, T, head)
    const int p = static_cast<int>((r / heads) % T);
    const float a = pos[static_cast<int64_t>(p) * d + j];
    const float rot = j < half ? -t[i + half] : t[i - half];  // cat(-x2, x1)
    out[i] = t[i] * cosf(a) + rot * sinf(a);
  }
}
int launch_rope_angles(const float* t, const float* pos, float* out, int64_t batch, int T, int heads, int d, cudaStream_t st) {
  const int64_t total = batch * T * heads * d;
  if (total <= 0) return 0;
  const unsigned blocks = static_cast<unsigned>(std::min<int64_t>(ceil_div(total, 256), 148 * 32));
  ProfScope prof(PC_ROPE, st, 0.0, static_cast<double>(total) * 12);
  rope_angles_kernel<<<blocks, 256, 0, st>>>(t, pos, out, total, T, heads, d);
  DITTO_LAUNCH_CHECK();
  return 0;
}

// coef table from the host-provided schedule (device arithmetic mirrors torch: 1/sqrt(a), (1-a)/sqrt(1-acp), sqrt(b))
__global__ void schedule_coef_kernel(const float* __restrict__ betas, const float* __restrict__ alphas,
                                     const float* __restrict__ acp, float* __restrict__ coef, int steps) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= steps) return;
  coef[i * 3 + 0] = __fdiv_rn(1.0f, __fsqrt_rn(alphas[i]));
  coef[i * 3 + 1] = __fdiv_rn(__fsub_rn(1.0f, alphas[i]), __fsqrt_rn(__fsub_rn(1.0f, acp[i])));
  coef[i * 3 + 2] = i > 0 ? __fsqrt_rn(betas[i]) : 0.0f;
}
int launch_schedule_coef(const float* betas, const float* alphas, const float* acp, float* coef, int steps, cudaStream_t st) {
  schedule_coef_kernel<<<static_cast<unsigned>(ceil_div(steps, 128)), 128, 0, st>>>(betas, alphas, acp, coef, steps);
  DITTO_LAUNCH_CHECK();
  return 0;
}

// q_sample with the reference's buffer (betas stored as "alphas_cumprod"): sqrt(b_t) x0 + sqrt(1-b_t) noise
__global__ void q_sample_kernel(const float4* __restrict__ x0, const float4* __restrict__ noise, const int64_t* __restrict__ t,
                                const float* __restrict__ buf, int steps, float4* __restrict__ out, int64_t vec_per_seq,
                                int64_t total_vec) {
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < total_vec;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int64_t seq = i / vec_per_seq;
    int64_t tt = t[seq];
    tt = tt < 0 ? 0 : (tt >= steps ? steps - 1 : tt);
    const float a = __fsqrt_rn(buf[tt]), b = __fsqrt_rn(__fsub_rn(1.0f, buf[tt]));
    const float4 xv = x0[i], nv = noise[i];
    out[i] = make_float4(__fadd_rn(__fmul_rn(a, xv.x), __fmul_rn(b, nv.x)), __fadd_rn(__fmul_rn(a, xv.y), __fmul_rn(b, nv.y)),
                         __fadd_rn(__fmul_rn(a, xv.z), __fmul_rn(b, nv.z)), __fadd_rn(__fmul_rn(a, xv.w), __fmul_rn(b, nv.w)));
  }
}
int launch_q_sample(const float* x0, const float* noise, const int64_t* t, const float* buf, int steps, float* out, int64_t B,
                    int64_t elems_per_seq, cudaStream_t st) {
  DITTO_REQUIRE(elems_per_seq % 4 == 0, DITTO_E_UNSUPPORTED, "q_sample: elems_per_seq % 4");
  const int64_t total_vec = B * elems_per_seq / 4;
  if (total_vec == 0) return 0;
  const unsigned blocks = static_cast<unsigned>(std::min<int64_t>(round_up(ceil_div(total_vec, 1024), 148), 148 * 32));
  q_sample_kernel<<<blocks, 256, 0, st>>>(reinterpret_cast<const float4*>(x0), reinterpret_cast<const float4*>(noise), t, buf,
                                          steps, reinterpret_cast<float4*>(out), elems_per_seq / 4, total_vec);
  DITTO_LAUNCH_CHECK();
  return 0;
}

}  // namespace ditto
