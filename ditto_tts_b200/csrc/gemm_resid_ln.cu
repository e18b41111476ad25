// fc2 GEMM + bias + fp32 residual + the LayerNorm that follows, in one kernel (reference: src/components/DiT.py:152-155
// `x = residual + mlp_fc2(...)` followed by the next block's `norm1`, DiT.py:105):
//
//     h  <- h + A W^T + b                 (fp32, in place; A = bf16 hidden activations [M, K], W = [N, K])
//     u  <- LayerNorm(h) gamma + beta     (bf16 operand of the next QKV GEMM)      or   u <- bf16(h)   (gamma == nullptr)
//
// Why a cluster: a 256-column accumulator tile is all of a row that fits next to a second (double-buffered) tile in TMEM,
// but LayerNorm needs statistics over the whole row (N = 768 = three tiles).  So the n_tiles cta_group::2 pairs that
// compute the n_tiles column tiles of the SAME 256 rows form one cluster (2 n_tiles CTAs; 6 for the repo-default hidden
// size): every epilogue warp sends the (sum, sum of squares) of its 128-column slab of each row to the CTAs holding the
// other columns of that row (st.async + complete_tx on their mbarrier, as flash_attn768 does for norm2), the result h is
// parked in its accumulator columns (tcgen05.st), and a second sweep normalises it from TMEM.  The statistics are those
// of the fp32 values that were stored (same arithmetic as the stand-alone layernorm_kernel).  The epilogue of tile i runs
// under the main loop of tile i + 1 (two accumulator buffers), which for K = 3072 is 48 k-blocks long -- the two sweeps
// are hidden, and the four LayerNorm launches between the blocks (110 MB of HBM traffic each at C2) disappear.
//
// Main loop = tc_gemm_pair_kernel (gemm_tc.cu): UMMA 256 x 256 x 16 over an SM pair, each CTA loads its 128 rows of A and
// half of the B tile, 6-stage TMA ring, persistent over row blocks: cluster c takes row blocks c, c + #clusters, ...
// Weight rows are packed in the `perm4` order (accumulator column 8 kb + 2 q + e of a 64-column block = output column
// 16 (kb / 2) + 4 q + 2 (kb % 2) + e), so a thread owns four consecutive outputs: 16-byte residual accesses, 8-byte bf16 stores.
#include "common.cuh"
#include "kernels.cuh"

namespace ditto {
namespace {

constexpr int RL_BM = 128, RL_BN = 256, RL_BK = 64;
constexpr int RL_THREADS = 384;
constexpr int RL_EPI_WARP0 = 4, RL_EPI_WARPS = 8;
constexpr int RL_STAGES = 6;
constexpr int RL_A_BYTES = RL_BM * RL_BK * 2;          // 16 KiB
constexpr int RL_B_BYTES = (RL_BN / 2) * RL_BK * 2;    // 16 KiB: this CTA's half of the B tile
constexpr int RL_STAGE_BYTES = RL_A_BYTES + RL_B_BYTES;
constexpr int RL_MAX_NT = 4;                           // column tiles per row = pairs per cluster (cluster size <= 8)
constexpr int RL_OFF_BAR = RL_STAGES * RL_STAGE_BYTES;
constexpr int RL_BAR_BYTES = 256;
constexpr int RL_OFF_STAT = RL_OFF_BAR + RL_BAR_BYTES;
constexpr int RL_STAT_BYTES = 2 * (2 * RL_MAX_NT) * RL_BM * 8;   // [tile parity][slab][row] (sum, sum of squares)
constexpr int RL_SMEM_BYTES = RL_OFF_STAT + RL_STAT_BYTES + 1024;
static_assert(RL_SMEM_BYTES <= 232448, "exceeds the 227 KiB shared memory of an sm_100 CTA");
constexpr int RL_TMEM_COLS = 512;

struct RlDev {
  int M, N, K;
  int n_tiles, m_pairs, num_kb;
  const float* bias;                 // [N], output-column order
  float* h; long long ldh;           // [M, N] fp32 output; also the residual (in place) unless `resid` is given
  const float* resid; long long ldr; int resid_mod;   // optional separate residual, row r reads resid[r % resid_mod] (0: r)
  const float* gamma; const float* beta;   // nullptr: no normalisation
  bf16* u; long long ldu;            // [M, N] bf16 output (may be nullptr when gamma == nullptr)
  float inv_n;
};

__global__ void __launch_bounds__(RL_THREADS, 1)
    tc_gemm_resid_ln_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_b, const RlDev p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw_addr = smem_u32(smem_raw);
  uint8_t* smem = smem_raw + ((1024u - (raw_addr & 1023u)) & 1023u);
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + RL_OFF_BAR);   // leader's copy in use: bytes of both CTAs
  uint64_t* empty_bar = full_bar + RL_STAGES;                            // multicast commit to both CTAs of the pair
  uint64_t* tmem_full = empty_bar + RL_STAGES;                           // [2] multicast commit
  uint64_t* tmem_empty = tmem_full + 2;                                  // [2] leader's copy: epilogue warps of both CTAs
  uint64_t* stat_bar = tmem_empty + 2;                                   // [2] own: row statistics of every slab landed
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(stat_bar + 2);
  static_assert((2 * RL_STAGES + 6) * 8 + 4 <= RL_BAR_BYTES, "barrier block too small");
  float2* stat_x = reinterpret_cast<float2*>(smem + RL_OFF_STAT);        // [2][2 n_tiles][128]

  const int warp = warp_id_uniform();
  const int lane = threadIdx.x & 31;
  const uint32_t rank = __shfl_sync(0xffffffffu, cluster_ctarank(), 0);
  const int a = static_cast<int>(rank & 1u);          // which 128 rows of the 256-row block; 0 = pair leader
  const int n_blk = static_cast<int>(rank >> 1);      // this pair's column tile
  const int csize = 2 * p.n_tiles;
  const int num_clusters = gridDim.x / csize;
  const int cluster_id = blockIdx.x / csize;
  const uint16_t pair_mask = static_cast<uint16_t>(3u << (rank & ~1u));
  const int parts = 2 * p.n_tiles;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmap_a);
    tma_prefetch_desc(&tmap_b);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < RL_STAGES; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
    for (int s = 0; s < 2; ++s) {
      mbar_init(&tmem_full[s], 1);
      mbar_init(&tmem_empty[s], 2 * RL_EPI_WARPS);
      mbar_init(&stat_bar[s], 1);
    }
    fence_barrier_init();
  }
  if (warp == 2) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_ptr)), "n"(RL_TMEM_COLS) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
  }
  __syncwarp();
  tcgen05_fence_before();
  cluster_sync_all();
  tcgen05_fence_after();
  const uint32_t tmem_base = *tmem_ptr;

  if (warp == 0) {
    // ---------------- TMA producer ----------------
    regs_shrink_ctrl();
    const bool leader = elect_one();
    int stage = 0;
    uint32_t phase = 0;
    for (int m_pair = cluster_id; m_pair < p.m_pairs; m_pair += num_clusters) {
      const int m0 = m_pair * 2 * RL_BM + a * RL_BM;
      const int n0 = n_blk * RL_BN + a * (RL_BN / 2);
      for (int kb = 0; kb < p.num_kb; ++kb) {
        mbar_wait(&empty_bar[stage], phase ^ 1u);
        if (leader) {
          uint8_t* sa = smem + stage * RL_STAGE_BYTES;
          if (a == 0) mbar_expect_tx(&full_bar[stage], 2 * RL_STAGE_BYTES);
          tma_load_4d_2sm(&tmap_a, &full_bar[stage], sa, kb * RL_BK, m0, 0, 0);
          tma_load_4d_2sm(&tmap_b, &full_bar[stage], sa + RL_A_BYTES, kb * RL_BK, n0, 0, 0);
        }
        __syncwarp();
        if (++stage == RL_STAGES) { stage = 0; phase ^= 1u; }
      }
    }
  } else if (warp == 1) {
    // ---------------- MMA issuer (pair leader) ----------------
    regs_shrink_ctrl();
    if (a == 0) {
      const bool leader = elect_one();
      constexpr uint32_t idesc = umma_idesc_bf16(2 * RL_BM, RL_BN, false, false);
      const uint64_t da0 = umma_smem_desc(smem_u32(smem), 16, 1024);
      const uint64_t db0 = umma_smem_desc(smem_u32(smem) + RL_A_BYTES, 16, 1024);
      int stage = 0, as = 0;
      uint32_t phase = 0, aphase = 0;
      for (int m_pair = cluster_id; m_pair < p.m_pairs; m_pair += num_clusters) {
        mbar_wait(&tmem_empty[as], aphase ^ 1u);
        tcgen05_fence_after();
        const uint32_t d_tmem = tmem_base + static_cast<uint32_t>(as * RL_BN);
        for (int kb = 0; kb < p.num_kb; ++kb) {
          mbar_wait(&full_bar[stage], phase);
          tcgen05_fence_after();
          if (leader) {
            const uint64_t so = static_cast<uint64_t>((stage * RL_STAGE_BYTES) >> 4);
#pragma unroll
            for (int k = 0; k < RL_BK / 16; ++k)
              umma_bf16_2sm(d_tmem, da0 + so + ((k * 32) >> 4), db0 + so + ((k * 32) >> 4), idesc, (kb | k) != 0 ? 1u : 0u);
            umma_commit_2sm_mc(&empty_bar[stage], pair_mask);
          }
          __syncwarp();
          if (++stage == RL_STAGES) { stage = 0; phase ^= 1u; }
        }
        if (leader) umma_commit_2sm_mc(&tmem_full[as], pair_mask);
        __syncwarp();
        if (++as == 2) { as = 0; aphase ^= 1u; }
      }
    }
  } else if (warp >= RL_EPI_WARP0) {
    // ---------------- epilogue: residual update, row statistics, LayerNorm ----------------
    regs_grow_epi();
    const int ew = warp - RL_EPI_WARP0;
    const int quarter = warp & 3, half_sel = ew >> 2;
    const int g = lane >> 2, q = lane & 3;
    const bool writer = q == 0;
    const bool norm = p.gamma != nullptr;
    const int colw = n_blk * RL_BN + half_sel * 128 + q * 4;   // this thread's first output column of chunk 0, group 0
    const int part = n_blk * 2 + half_sel;                     // this warp's slab index in the row statistics
    int as = 0;
    uint32_t aphase = 0, it = 0;
    for (int m_pair = cluster_id; m_pair < p.m_pairs; m_pair += num_clusters, ++it) {
      const int row_cta = m_pair * 2 * RL_BM + a * RL_BM;      // first row of this CTA
      const int r0 = row_cta + quarter * 32 + g;               // rows r0, r0 + 8, r0 + 16, r0 + 24
      const uint32_t t_lane = tmem_base + (static_cast<uint32_t>(quarter * 32) << 16) + static_cast<uint32_t>(as * RL_BN + half_sel * 128);
      const uint32_t par = it & 1u;
      float* h0 = p.h + static_cast<long long>(r0) * p.ldh + colw;
      bf16* u0 = p.u ? p.u + static_cast<long long>(r0) * p.ldu + colw : nullptr;
      bool ok[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) ok[i] = r0 + 8 * i < p.M;
      // one step = (hh, cb): 16 rows (r0 + 16 hh, + 8) x 64 columns (cb); residual of the next step requested one step ahead
      float4 f0[8], f1[8];
      // residual rows: the output rows themselves (in place), or rows of a separate tensor that repeats with period resid_mod
      // (x_skip is shared by the conditional / unconditional halves of a CFG batch)
      const float* rrow[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int rr = r0 + 8 * i;
        rrow[i] = p.resid == nullptr ? p.h + static_cast<long long>(rr) * p.ldh + colw
                                     : p.resid + static_cast<long long>(p.resid_mod > 0 ? rr % p.resid_mod : rr) * p.ldr + colw;
      }
      auto load_res = [&](int hh, int cb, float4(&f)[8]) {
        const float* ra = rrow[2 * hh] + cb * 64;
        const float* rb = rrow[2 * hh + 1] + cb * 64;
#pragma unroll
        for (int jj = 0; jj < 4; ++jj) {
          f[jj] = ok[2 * hh] ? *reinterpret_cast<const float4*>(ra + jj * 16) : make_float4(0.f, 0.f, 0.f, 0.f);
          f[4 + jj] = ok[2 * hh + 1] ? *reinterpret_cast<const float4*>(rb + jj * 16) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
      };
      load_res(0, 0, f0);
      load_res(0, 1, f1);
      if (norm && ew == 0 && lane == 0) mbar_expect_tx(&stat_bar[par], static_cast<uint32_t>(parts * RL_BM * 8));
      mbar_wait(&tmem_full[as], aphase);
      tcgen05_fence_after();
      // row statistics of this thread's 32 values of each row: sums of v - K and (v - K)^2, K = its first value (common.cuh)
      float sm[4] = {0.f, 0.f, 0.f, 0.f}, sq[4] = {0.f, 0.f, 0.f, 0.f}, kk[4];
      auto sweep1 = [&](int hh, int cb, const float4(&f)[8]) {
        uint32_t o[32];
        tmem_ld_16x64(t_lane + (static_cast<uint32_t>(16 * hh) << 16) + cb * 64, o);
        float4 bs[4];
#pragma unroll
        for (int jj = 0; jj < 4; ++jj) bs[jj] = __ldg(reinterpret_cast<const float4*>(p.bias + colw + cb * 64 + jj * 16));
        float* oa = h0 + static_cast<long long>(16 * hh) * p.ldh + cb * 64;
        float* ob = oa + 8 * p.ldh;
        const bool okA = ok[2 * hh], okB = ok[2 * hh + 1];
        tmem_ld_wait();
#pragma unroll
        for (int jj = 0; jj < 4; ++jj) {   // accumulator 8-column blocks 2 jj, 2 jj + 1 = output columns 16 jj + 4 q .. + 3
          const int k0 = 2 * jj, k1 = 2 * jj + 1;
          float4 vA, vB;
          vA.x = (__uint_as_float(o[4 * k0]) + bs[jj].x) + f[jj].x;
          vA.y = (__uint_as_float(o[4 * k0 + 1]) + bs[jj].y) + f[jj].y;
          vA.z = (__uint_as_float(o[4 * k1]) + bs[jj].z) + f[jj].z;
          vA.w = (__uint_as_float(o[4 * k1 + 1]) + bs[jj].w) + f[jj].w;
          vB.x = (__uint_as_float(o[4 * k0 + 2]) + bs[jj].x) + f[4 + jj].x;
          vB.y = (__uint_as_float(o[4 * k0 + 3]) + bs[jj].y) + f[4 + jj].y;
          vB.z = (__uint_as_float(o[4 * k1 + 2]) + bs[jj].z) + f[4 + jj].z;
          vB.w = (__uint_as_float(o[4 * k1 + 3]) + bs[jj].w) + f[4 + jj].w;
          if (okA) *reinterpret_cast<float4*>(oa + jj * 16) = vA;
          if (okB) *reinterpret_cast<float4*>(ob + jj * 16) = vB;
          if (norm) {
            if (cb == 0 && jj == 0) { kk[2 * hh] = vA.x; kk[2 * hh + 1] = vB.x; }
            const float4 dA = make_float4(vA.x - kk[2 * hh], vA.y - kk[2 * hh], vA.z - kk[2 * hh], vA.w - kk[2 * hh]);
            const float4 dB = make_float4(vB.x - kk[2 * hh + 1], vB.y - kk[2 * hh + 1], vB.z - kk[2 * hh + 1], vB.w - kk[2 * hh + 1]);
            sm[2 * hh] += (dA.x + dA.y) + (dA.z + dA.w);
            sq[2 * hh] = fmaf(dA.x, dA.x, fmaf(dA.y, dA.y, fmaf(dA.z, dA.z, fmaf(dA.w, dA.w, sq[2 * hh]))));
            sm[2 * hh + 1] += (dB.x + dB.y) + (dB.z + dB.w);
            sq[2 * hh + 1] = fmaf(dB.x, dB.x, fmaf(dB.y, dB.y, fmaf(dB.z, dB.z, fmaf(dB.w, dB.w, sq[2 * hh + 1]))));
            o[4 * k0] = __float_as_uint(vA.x); o[4 * k0 + 1] = __float_as_uint(vA.y);
            o[4 * k1] = __float_as_uint(vA.z); o[4 * k1 + 1] = __float_as_uint(vA.w);
            o[4 * k0 + 2] = __float_as_uint(vB.x); o[4 * k0 + 3] = __float_as_uint(vB.y);
            o[4 * k1 + 2] = __float_as_uint(vB.z); o[4 * k1 + 3] = __float_as_uint(vB.w);
          } else if (u0 != nullptr) {   // plain bf16 copy of the updated residual stream
            bf16* ua = u0 + static_cast<long long>(16 * hh) * p.ldu + cb * 64 + jj * 16;
            if (okA) *reinterpret_cast<uint2*>(ua) = make_uint2(pack_bf16x2(vA.x, vA.y), pack_bf16x2(vA.z, vA.w));
            if (okB) *reinterpret_cast<uint2*>(ua + 8 * p.ldu) = make_uint2(pack_bf16x2(vB.x, vB.y), pack_bf16x2(vB.z, vB.w));
          }
        }
        if (norm) tmem_st_16x64(t_lane + (static_cast<uint32_t>(16 * hh) << 16) + cb * 64, o);
      };
      sweep1(0, 0, f0); load_res(1, 0, f0);
      sweep1(0, 1, f1); load_res(1, 1, f1);
      sweep1(1, 0, f0);
      sweep1(1, 1, f1);
      if (norm) {
        tmem_st_wait();
        // this warp's slab partials (mean, M2) of its 32 rows -> every CTA that holds columns of these rows (same a, every pair)
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const float2 st = ln_quad_merge(ln_partial(kk[i], sm[i], sq[i], 1.0f / 32.f), 32.f);
          sm[i] = st.x; sq[i] = st.y;
        }
        if (writer) {
          const uint32_t slot = smem_u32(stat_x + (par * parts + part) * RL_BM + quarter * 32 + g);
          const uint32_t bar = smem_u32(&stat_bar[par]);
          for (int pr = 0; pr < p.n_tiles; ++pr) {
            const uint32_t dst_rank = static_cast<uint32_t>(2 * pr + a);
            const uint32_t rs = mapa_shared(slot, dst_rank), rb = mapa_shared(bar, dst_rank);
#pragma unroll
            for (int i = 0; i < 4; ++i) st_async_f32x2(rs + i * 8 * 8, sm[i], sq[i], rb);
          }
        }
        mbar_wait(&stat_bar[par], (it >> 1) & 1u);
        float mean[4], rstd[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {   // parts of 128 values each: mean of the means, then M2 = sum M2_c + 128 sum (mean_c - mean)^2
          const float2* sx = stat_x + par * parts * RL_BM + quarter * 32 + g + 8 * i;
          float s = 0.f;
          for (int c = 0; c < parts; ++c) s += sx[c * RL_BM].x;
          const float m = s * (128.f * p.inv_n);
          float m2 = 0.f, dd = 0.f;
          for (int c = 0; c < parts; ++c) {
            const float2 v = sx[c * RL_BM];
            m2 += v.y;
            dd = fmaf(v.x - m, v.x - m, dd);
          }
          mean[i] = m;
          rstd[i] = rsqrtf(fmaxf(fmaf(128.f, dd, m2), 0.f) * p.inv_n + 1e-5f);
        }
        // ---------------- sweep 2: u = LayerNorm(h) gamma + beta, bf16, 8-byte stores ----------------
#pragma unroll
        for (int step = 0; step < 4; ++step) {
          const int hh = step >> 1, cb = step & 1;
          uint32_t o[32];
          tmem_ld_16x64(t_lane + (static_cast<uint32_t>(16 * hh) << 16) + cb * 64, o);
          float4 gm[4], bt[4];
#pragma unroll
          for (int jj = 0; jj < 4; ++jj) {
            gm[jj] = __ldg(reinterpret_cast<const float4*>(p.gamma + colw + cb * 64 + jj * 16));
            bt[jj] = __ldg(reinterpret_cast<const float4*>(p.beta + colw + cb * 64 + jj * 16));
          }
          const float2 aA2 = make_float2(rstd[2 * hh], rstd[2 * hh]), cA2 = make_float2(-mean[2 * hh] * rstd[2 * hh], -mean[2 * hh] * rstd[2 * hh]);
          const float2 aB2 = make_float2(rstd[2 * hh + 1], rstd[2 * hh + 1]),
                       cB2 = make_float2(-mean[2 * hh + 1] * rstd[2 * hh + 1], -mean[2 * hh + 1] * rstd[2 * hh + 1]);
          bf16* ua = u0 + static_cast<long long>(16 * hh) * p.ldu + cb * 64;
          bf16* ub = ua + 8 * p.ldu;
          const bool okA = ok[2 * hh], okB = ok[2 * hh + 1];
          tmem_ld_wait();
#pragma unroll
          for (int jj = 0; jj < 4; ++jj) {
            const int k0 = 2 * jj, k1 = 2 * jj + 1;
            // (o - mean) rstd gamma + beta as two packed FMAs per column pair: o a + c with a = rstd, c = -mean rstd, then * gamma + beta
            const float2 g01 = make_float2(gm[jj].x, gm[jj].y), g23 = make_float2(gm[jj].z, gm[jj].w);
            const float2 b01 = make_float2(bt[jj].x, bt[jj].y), b23 = make_float2(bt[jj].z, bt[jj].w);
            const float2 yA0 = __ffma2_rn(__ffma2_rn(make_float2(__uint_as_float(o[4 * k0]), __uint_as_float(o[4 * k0 + 1])), aA2, cA2), g01, b01);
            const float2 yA1 = __ffma2_rn(__ffma2_rn(make_float2(__uint_as_float(o[4 * k1]), __uint_as_float(o[4 * k1 + 1])), aA2, cA2), g23, b23);
            const float2 yB0 = __ffma2_rn(__ffma2_rn(make_float2(__uint_as_float(o[4 * k0 + 2]), __uint_as_float(o[4 * k0 + 3])), aB2, cB2), g01, b01);
            const float2 yB1 = __ffma2_rn(__ffma2_rn(make_float2(__uint_as_float(o[4 * k1 + 2]), __uint_as_float(o[4 * k1 + 3])), aB2, cB2), g23, b23);
            uint2 wA, wB;
            wA.x = pack_bf16x2(yA0.x, yA0.y);
            wA.y = pack_bf16x2(yA1.x, yA1.y);
            wB.x = pack_bf16x2(yB0.x, yB0.y);
            wB.y = pack_bf16x2(yB1.x, yB1.y);
            if (okA) *reinterpret_cast<uint2*>(ua + jj * 16) = wA;
            if (okB) *reinterpret_cast<uint2*>(ub + jj * 16) = wB;
          }
        }
      }
      tcgen05_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive_leader(&tmem_empty[as]);
      if (++as == 2) { as = 0; aphase ^= 1u; }
    }
  } else {
    regs_shrink_ctrl();   // warps 2 and 3 idle; the whole warpgroup has to execute the setmaxnreg
  }

  __syncwarp();
  tcgen05_fence_before();
  cluster_sync_all();   // nobody leaves while a peer may still write statistics into it / signal its barriers
  if (warp == 2) {
    tcgen05_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(RL_TMEM_COLS) : "memory");
  }
}

}  // namespace

bool gemm_resid_ln_supported(int N, int K) { return N > 0 && N % RL_BN == 0 && N / RL_BN <= RL_MAX_NT && K > 0 && K % 8 == 0; }

// source row of packed weight row r (the `perm4` order inside every 64-row block)
int gemm_resid_ln_weight_row(int r) {
  const int blk = r / 64, c = r % 64;
  const int kb = c / 8, q = (c % 8) / 2, e = c % 2;
  return blk * 64 + 16 * (kb / 2) + 4 * q + 2 * (kb % 2) + e;
}

bool gemm_resid_ln_schedulable(int N) {
  return N > 0 && N % RL_BN == 0 && N / RL_BN <= RL_MAX_NT && tc_gemm_init() == 0 &&
         max_active_clusters(reinterpret_cast<const void*>(tc_gemm_resid_ln_kernel), 2 * (N / RL_BN), RL_THREADS, RL_SMEM_BYTES) > 0;
}

int launch_gemm_resid_ln(const GemmResidLnParams& q, cudaStream_t st) {
  DITTO_TRY(tc_gemm_init());
  DITTO_REQUIRE(q.A && q.W && q.h && q.bias && q.M > 0, DITTO_E_BADARG, "gemm_resid_ln: null argument");
  DITTO_REQUIRE(gemm_resid_ln_supported(q.N, q.K), DITTO_E_UNSUPPORTED, "gemm_resid_ln: N must be 256, 512, 768 or 1024 and K a multiple of 8");
  DITTO_REQUIRE(q.gamma == nullptr || (q.beta != nullptr && q.u != nullptr), DITTO_E_BADARG, "gemm_resid_ln: LayerNorm needs gamma, beta and u");
  DITTO_REQUIRE(q.resid == nullptr || (q.ldr % 4 == 0 && (reinterpret_cast<uintptr_t>(q.resid) & 15) == 0 && q.resid_mod >= 0 && q.resid_mod < (1ll << 31)),
                DITTO_E_BADARG, "gemm_resid_ln: separate residual must be 16-byte aligned with a row stride that is a multiple of 4");
  DITTO_REQUIRE(q.ldh % 4 == 0 && (q.u == nullptr || q.ldu % 4 == 0) && (reinterpret_cast<uintptr_t>(q.h) & 15) == 0 &&
                    (reinterpret_cast<uintptr_t>(q.u) & 7) == 0 && (reinterpret_cast<uintptr_t>(q.bias) & 15) == 0 &&
                    (reinterpret_cast<uintptr_t>(q.gamma) & 15) == 0 && (reinterpret_cast<uintptr_t>(q.beta) & 15) == 0,
                DITTO_E_BADARG, "gemm_resid_ln: h / bias / gamma / beta must be 16-byte aligned with strides that keep rows aligned");
  RlDev p;
  p.M = q.M; p.N = q.N; p.K = q.K;
  p.n_tiles = q.N / RL_BN;
  p.m_pairs = static_cast<int>(ceil_div(q.M, 2 * RL_BM));
  p.num_kb = static_cast<int>(ceil_div(q.K, RL_BK));
  p.bias = q.bias; p.h = q.h; p.ldh = q.ldh; p.gamma = q.gamma; p.beta = q.beta; p.u = q.u; p.ldu = q.ldu;
  p.resid = q.resid; p.ldr = q.ldr; p.resid_mod = static_cast<int>(q.resid_mod);
  p.inv_n = 1.0f / static_cast<float>(q.N);
  const int csize = 2 * p.n_tiles;
  const void* fn = reinterpret_cast<const void*>(tc_gemm_resid_ln_kernel);
  DITTO_REQUIRE(max_active_clusters(fn, csize, RL_THREADS, RL_SMEM_BYTES) > 0, DITTO_E_UNSUPPORTED,
                "gemm_resid_ln: this cluster size cannot be scheduled on the device");
  TcOperand A, B;
  A.ptr = q.A; A.rows = q.M; A.cols = q.K; A.ld = q.lda;
  B.ptr = q.W; B.rows = q.N; B.cols = q.K; B.ld = q.ldw;
  CUtensorMap ma, mb;
  DITTO_TRY(tc_make_map(&ma, A, 1, 1, RL_BK, RL_BM));
  DITTO_TRY(tc_make_map(&mb, B, 1, 1, RL_BK, RL_BN / 2));
  const double rows = static_cast<double>(q.M);
  ProfScope prof(q.tag, st, 2.0 * rows * q.N * static_cast<double>(q.K),
                 rows * (2.0 * q.K + q.N * (8.0 + (q.u ? 2.0 : 0.0))) + 2.0 * q.N * static_cast<double>(q.K));
  void* args[3] = {&ma, &mb, &p};
  return launch_clusters(fn, csize, RL_THREADS, RL_SMEM_BYTES, p.m_pairs, args, st);
}

}  // namespace ditto
