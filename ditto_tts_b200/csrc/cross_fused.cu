// Fused cross-attention block of the folded single-head path (reference: src/components/DiT.py:141-151 -> torch
// nn.MultiheadAttention math path, then norm3):
//
//     h   <- h + softmax(alpha * u (K Wq)^T + sbias) (V Wo^T) + bo          (one utterance's S <= 64 text tokens)
//     u3  <- LayerNorm(h) * gamma3 + beta3                                     (bf16 operand of the gated-MLP GEMM)
//
// in ONE kernel per layer instead of scores+softmax -> P (HBM) -> P.V GEMM with residual epilogue -> LayerNorm: the scores
// and the probabilities never leave the SM, and the residual stream is read once and written once per block instead of
// being re-read by a separate LayerNorm launch.  The kernel is an HBM stream over u (bf16), h (fp32, in place) and u3
// (bf16): 12 B per element of h -> 221 MB per launch at C2 (24 000 x 768).
//
// Per CTA (640 threads, persistent over 128-row tiles; a tile never crosses an utterance):
//   warp 0   TMA producer of the MMA operands: u tile [128 x H] and K-fold [64 x H] through a 2-stage ring (64-column
//            k-blocks, 128-B swizzle); per output half-chunk one V-fold box [64 k x 64 n] (MN-major operand, ring of 3)
//   warp 1   MMA issuer (whole warp on warp-uniform values, one elected lane issues):  scores S[128 x 64] = U Kf^T (tcgen05.mma, fp32 in TMEM, two buffers; the NEXT tile's scores are
//            issued right after the current tile's P.V, so their operand stream overlaps the rest of the epilogue without
//            sitting in front of the P.V);  O chunk c [128 x 128] = P[128 x 64] Vf[64 x 128c..] as two N = 64 MMAs into a
//            ring of three 128-column TMEM buffers
//   warps 2, 3  movers: the residual stream goes global <-> shared memory by TMA only (4 staging buffers of 128 rows x 64
//            fp32 columns; warp 2 loads as soon as a buffer is free, warp 3 stores and frees): no LSU wavefronts are spent
//            on HBM traffic -- the first version of this kernel moved h with 8-byte register accesses (8 wavefronts per warp
//            instruction) and was LSU-bound at 117 us
//   warps 4-19  (4 per TMEM lane quarter) the first 8: softmax on the accumulator fragments (tcgen05.ld.16x256b), probabilities
//            written as the bf16 K-major A operand into shared memory (128-B swizzle by hand);  all 16: pass 0, O + bias +
//            residual in place in the staging buffer (-> TMA store to h) with packed f32x2 running row sums;  row statistics
//            exchanged through shared memory;  pass 1 over the rows just written (TMA re-load, L2 hits): normalise,
//            gamma/beta, bf16 in place (-> TMA store to u3)
// TMEM: columns [0, 384) O ring, [384, 512) two score buffers.  Optional deferred norm2 of the query operand (ln_stat).
// Measured (profiles/README.md): 63-70 us per launch at C2 against 104 us for the three kernels it replaces; the tile loop is
// bound by the latency of its 24 staging jobs per tile (96 KiB of loads in flight per SM), not by bytes or instructions.
#include <algorithm>
#include <cstdlib>

#include "common.cuh"
#include "kernels.cuh"

namespace ditto {
namespace {

constexpr int XF_THREADS = 640;            // 4 control warps + 16 softmax / epilogue warps
constexpr int XF_EPI_WARP0 = 4;
constexpr int XF_EPI_WARPS = 16;          // 4 per TMEM lane quarter: 4 warps per scheduler hide the TMEM / shared-memory latencies
constexpr int XF_SM_WARPS = 8;            // of which the first 8 also do the softmax (16 rows x 64 score columns each)
// setmaxnreg moves registers inside the CTA's own pool only: what the control warps release is all the epilogue warps can
// take, on top of the launch allocation of 96 per thread (640 threads)
constexpr int XF_REGS_LAUNCH = 96, XF_REGS_CTRL = 56, XF_REGS_EPI = 104;
static_assert(128 * XF_REGS_CTRL + 32 * XF_EPI_WARPS * XF_REGS_EPI <= XF_THREADS * XF_REGS_LAUNCH, "register re-distribution exceeds the CTA pool");
constexpr int XF_BM = 128;          // rows per tile
constexpr int XF_BK = 64;           // k-block (one 128-B swizzle span of bf16)
constexpr int XF_NS = 64;           // score columns (text tokens, padded)
constexpr int XF_CH = 128;          // output columns per TMEM chunk
constexpr int XF_HC = 64;           // output columns per staged half-chunk (two 32-column fp32 slabs)
constexpr int XF_STAGES = 2;
constexpr int XF_A_BYTES = XF_BM * XF_BK * 2;   // 16 KiB
constexpr int XF_B_BYTES = XF_NS * XF_BK * 2;   //  8 KiB
constexpr int XF_STAGE_BYTES = XF_A_BYTES + XF_B_BYTES;
constexpr int XF_MAX_H = 768;
constexpr int XF_P_BYTES = XF_BM * XF_NS * 2;   // 16 KiB
constexpr int XF_VF_BOX = XF_NS * 64 * 2;      //  8 KiB: V-fold [64 k-rows x 64 n] box of one output half-chunk
constexpr int XF_VF_RING = 3;
constexpr int XF_VF_BYTES = XF_VF_RING * XF_VF_BOX;
constexpr int XF_NB = 4;                        // staging buffers for the residual stream
constexpr int XF_SLAB_BYTES = XF_BM * 32 * 4;   // 16 KiB: 128 rows x 32 fp32 columns (one TMA box)
constexpr int XF_HBUF_BYTES = 2 * XF_SLAB_BYTES;
constexpr int XF_OFF_P = XF_STAGES * XF_STAGE_BYTES;
constexpr int XF_OFF_VF = XF_OFF_P + XF_P_BYTES;
constexpr int XF_OFF_HB = XF_OFF_VF + XF_VF_BYTES;
constexpr int XF_OFF_BAR = XF_OFF_HB + XF_NB * XF_HBUF_BYTES;
constexpr int XF_BAR_BYTES = 512;
constexpr int XF_OFF_STAT = XF_OFF_BAR + XF_BAR_BYTES;
constexpr int XF_STAT_BYTES = 2 * XF_BM * 4 * 8;  // [tile parity][row][column quarter] (sum, sum of squares)
constexpr int XF_SMEM_BYTES = XF_OFF_STAT + XF_STAT_BYTES + 1024 /*align slack*/;
static_assert(XF_SMEM_BYTES <= 232448, "exceeds the 227 KiB shared memory of an sm_100 CTA");
static_assert(XF_OFF_P % 1024 == 0 && XF_OFF_VF % 1024 == 0 && XF_OFF_HB % 1024 == 0 && XF_STAGE_BYTES % 1024 == 0,
              "swizzled operands need 1024-B alignment");
constexpr int XF_TMEM_COLS = 512;
constexpr int XF_O_BUFS = 3;
constexpr int XF_S_COL0 = XF_O_BUFS * XF_CH;  // 384

struct XfDev {
  int n_seq, T, S, H;
  int rt;                                     // rows per tile (<= 128, multiple of 8): the TMA boxes carry rt rows, the MMA computes 128
  int m_tiles, num_tiles, num_kb, num_ch, num_hc;
  float alpha2;                               // alpha * log2(e)
  const float* sbias; long long sb_seq;       // [n_seq, sb_seq] additive score bias
  const float* out_bias;                      // [H]
  const float* gamma; const float* beta;      // LayerNorm after the block
  float inv_h;
  const float2* ln_stat; int ln_parts; const float* ln_c;   // deferred LayerNorm of the query operand (nullptr: off)
  const uint8_t* skip_seq;                    // [n_seq] sequences whose tiles are not processed (nullptr: none)
};

// first tile at or after `tile` (stepping over the grid) that this launch processes.  Every role walks the same tiles, and
// the iteration counters that drive the barrier phases count processed tiles only.
__device__ __forceinline__ int xf_next_tile(const XfDev& p, int tile, int step) {
  if (p.skip_seq != nullptr)
    while (tile < p.num_tiles && __ldg(p.skip_seq + tile / p.m_tiles) != 0) tile += step;
  return tile;
}

__device__ __forceinline__ void epi_bar_sync() { asm volatile("bar.sync 1, %0;" ::"n"(32 * XF_EPI_WARPS) : "memory"); }
// the four warps that share a TMEM lane quarter (= the same 32 tile rows): named barriers 2..5
__device__ __forceinline__ void quarter_bar_sync(int quarter) { asm volatile("bar.sync %0, 128;" ::"r"(2 + quarter) : "memory"); }
__device__ __forceinline__ void xf_regs_ctrl() { asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(XF_REGS_CTRL)); }
__device__ __forceinline__ void xf_regs_epi() { asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(XF_REGS_EPI)); }
__device__ __forceinline__ void tmem_ld_16x16(uint32_t taddr, uint32_t (&r)[8]) {  // 16 lanes x 16 fp32 columns, fragment layout
  asm volatile("tcgen05.ld.sync.aligned.16x256b.x2.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
               : "r"(taddr)
               : "memory");
}
// shared -> global tiled store (bulk async-group completion); out-of-range rows are clipped by the TMA unit
__device__ __forceinline__ void tma_store_4d(const CUtensorMap* m, const void* smem, int c0, int c1, int c2, int c3) {
  asm volatile("cp.async.bulk.tensor.4d.global.shared::cta.bulk_group [%0, {%2, %3, %4, %5}], [%1];" ::"l"(reinterpret_cast<uint64_t>(m)),
               "r"(smem_u32(smem)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
               : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void bulk_wait() { asm volatile("cp.async.bulk.wait_group %0;" ::"n"(N) : "memory"); }
template <int N>  // ... only until the sources have been READ (the shared-memory buffers may be reused)
__device__ __forceinline__ void bulk_wait_read() { asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory"); }

__global__ void __launch_bounds__(XF_THREADS, 1)
    cross_fused_kernel(const __grid_constant__ CUtensorMap tmap_u, const __grid_constant__ CUtensorMap tmap_kf,
                       const __grid_constant__ CUtensorMap tmap_vf, const __grid_constant__ CUtensorMap tmap_h,
                       const __grid_constant__ CUtensorMap tmap_uo, const XfDev p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw_addr = smem_u32(smem_raw);
  uint8_t* smem = smem_raw + ((1024u - (raw_addr & 1023u)) & 1023u);
  uint8_t* p_smem = smem + XF_OFF_P;
  uint8_t* vf_smem = smem + XF_OFF_VF;
  uint8_t* hbuf = smem + XF_OFF_HB;
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + XF_OFF_BAR);
  uint64_t* empty_bar = full_bar + XF_STAGES;
  uint64_t* s_full = empty_bar + XF_STAGES;   // [2] scores accumulator complete        (MMA -> epilogue)
  uint64_t* s_empty = s_full + 2;             // [2] scores accumulator read            (epilogue -> MMA)
  uint64_t* p_full = s_empty + 2;             //     probabilities in shared memory     (epilogue -> MMA)
  uint64_t* vf_full = p_full + 1;             // [3] V-fold box landed                  (TMA -> MMA)
  uint64_t* vf_empty = vf_full + XF_VF_RING;  // [3] its MMAs retired                   (MMA -> TMA)
  uint64_t* o_full = vf_empty + XF_VF_RING;   // [3] output chunk complete              (MMA -> epilogue)
  uint64_t* o_empty = o_full + XF_O_BUFS;     // [3] output chunk read                  (epilogue -> MMA)
  uint64_t* hin_full = o_empty + XF_O_BUFS;   // [NB] residual half-chunk landed        (mover TMA -> epilogue)
  uint64_t* hout_full = hin_full + XF_NB;     // [NB] result half-chunk in place        (epilogue -> mover)
  uint64_t* hfree = hout_full + XF_NB;        // [NB] staging buffer reusable           (storer -> loader)
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(hfree + XF_NB);
  float2* stat = reinterpret_cast<float2*>(smem + XF_OFF_STAT);
  static_assert((2 * XF_STAGES + 2 + 2 + 1 + 2 * XF_VF_RING + 2 * XF_O_BUFS + 3 * XF_NB) * 8 + 4 <= XF_BAR_BYTES, "barrier block too small");

  const int warp = warp_id_uniform();   // control warps run on warp-uniform values, one elected lane issues (common.cuh: elect_one)
  const int lane = threadIdx.x & 31;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmap_u);
    tma_prefetch_desc(&tmap_kf);
    tma_prefetch_desc(&tmap_vf);
    tma_prefetch_desc(&tmap_h);
    tma_prefetch_desc(&tmap_uo);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < XF_STAGES; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init(&s_full[s], 1);
      mbar_init(&s_empty[s], XF_SM_WARPS);
    }
    mbar_init(p_full, XF_SM_WARPS);
    for (int s = 0; s < XF_VF_RING; ++s) {
      mbar_init(&vf_full[s], 1);
      mbar_init(&vf_empty[s], 1);
    }
    for (int s = 0; s < XF_O_BUFS; ++s) {
      mbar_init(&o_full[s], 1);
      mbar_init(&o_empty[s], XF_EPI_WARPS);
    }
    for (int s = 0; s < XF_NB; ++s) {
      mbar_init(&hin_full[s], 1);
      mbar_init(&hout_full[s], XF_EPI_WARPS);
      mbar_init(&hfree[s], 1);
    }
    fence_barrier_init();
  }
  if (warp == 2) tmem_alloc<XF_TMEM_COLS>(tmem_ptr);
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem_base = *tmem_ptr;
  const int first = blockIdx.x, step = gridDim.x;

  if (warp == 0) {
    // =========================== TMA producer: MMA operands ===========================
    xf_regs_ctrl();
    {
      const bool leader = elect_one();
      int stage = 0;
      uint32_t phase = 0;
      uint32_t vc = 0;  // V-fold boxes loaded so far
      const uint32_t stage_tx = static_cast<uint32_t>(p.rt) * (XF_BK * 2) + XF_B_BYTES;
      auto load_scores_operands = [&](int tile) {
        const int seq = tile / p.m_tiles, mb = tile - seq * p.m_tiles;
        for (int kb = 0; kb < p.num_kb; ++kb) {
          mbar_wait(&empty_bar[stage], phase ^ 1u);
          if (leader) {
            uint8_t* sa = smem + stage * XF_STAGE_BYTES;
            mbar_expect_tx(&full_bar[stage], stage_tx);
            tma_load_4d(&tmap_u, &full_bar[stage], sa, kb * XF_BK, mb * p.rt, 0, seq);
            tma_load_4d(&tmap_kf, &full_bar[stage], sa + XF_A_BYTES, kb * XF_BK, 0, 0, seq);  // rows >= S: zero-filled
          }
          __syncwarp();
          if (++stage == XF_STAGES) { stage = 0; phase ^= 1u; }
        }
      };
      // same order as the MMA issuer consumes: scores(0), then per tile its P.V boxes followed by scores(next tile)
      const int tile0 = xf_next_tile(p, first, step);
      if (tile0 < p.num_tiles) load_scores_operands(tile0);
      for (int tile = tile0; tile < p.num_tiles;) {
        const int seq = tile / p.m_tiles;
        const int next = xf_next_tile(p, tile + step, step);
        for (int hc = 0; hc < p.num_hc; ++hc, ++vc) {
          const uint32_t vs = vc % XF_VF_RING;
          mbar_wait(&vf_empty[vs], ((vc / XF_VF_RING) & 1u) ^ 1u);  // the MMAs that read this box have retired
          if (leader) {
            mbar_expect_tx(&vf_full[vs], XF_VF_BOX);
            // [64 k-rows x 64 n] box, n contiguous (MN-major operand); rows >= Sp zero-filled
            tma_load_4d(&tmap_vf, &vf_full[vs], vf_smem + vs * XF_VF_BOX, hc * XF_HC, 0, 0, seq);
          }
          __syncwarp();
        }
        if (next < p.num_tiles) load_scores_operands(next);
        tile = next;
      }
    }
  } else if (warp == 1) {
    // =========================== MMA issuer (single thread) ===========================
    xf_regs_ctrl();
    {
      const bool leader = elect_one();
      constexpr uint32_t idesc_s = umma_idesc_bf16(XF_BM, XF_NS, false, false);
      constexpr uint32_t idesc_o = umma_idesc_bf16(XF_BM, XF_HC, false, true);
      const uint64_t ds0 = umma_smem_desc(smem_u32(smem), 16, 1024);               // ring slot 0, K-major
      const uint64_t dp0 = umma_smem_desc(smem_u32(p_smem), 16, 1024);
      const uint64_t dv0 = umma_smem_desc(smem_u32(vf_smem), XF_VF_BOX, 1024);     // MN-major V-fold box 0
      int stage = 0;
      uint32_t phase = 0;
      auto issue_scores = [&](uint32_t j) {  // scores of this CTA's j-th tile into score buffer j & 1
        const uint32_t sb = j & 1u;
        mbar_wait(&s_empty[sb], ((j >> 1) & 1u) ^ 1u);
        tcgen05_fence_after();
        const uint32_t d_tmem = tmem_base + XF_S_COL0 + sb * XF_NS;
        for (int kb = 0; kb < p.num_kb; ++kb) {
          mbar_wait(&full_bar[stage], phase);
          tcgen05_fence_after();
          if (leader) {
            const uint64_t da = ds0 + static_cast<uint64_t>((stage * XF_STAGE_BYTES) >> 4);
#pragma unroll
            for (int k = 0; k < XF_BK / 16; ++k)
              umma_bf16(d_tmem, da + ((k * 32) >> 4), da + ((XF_A_BYTES + k * 32) >> 4), idesc_s, (kb | k) != 0 ? 1u : 0u);
            umma_commit(&empty_bar[stage]);
          }
          __syncwarp();
          if (++stage == XF_STAGES) { stage = 0; phase ^= 1u; }
        }
        if (leader) umma_commit(&s_full[sb]);
        __syncwarp();
      };
      uint32_t it = 0, oc = 0, vc = 0;
      const int tile0 = xf_next_tile(p, first, step);
      if (tile0 < p.num_tiles) issue_scores(0);
      for (int tile = tile0; tile < p.num_tiles; ++it) {
        const int next = xf_next_tile(p, tile + step, step);
        mbar_wait(p_full, it & 1u);
        for (int hc = 0; hc < p.num_hc; ++hc, ++vc) {
          const uint32_t ob = oc % XF_O_BUFS, vs = vc % XF_VF_RING;
          mbar_wait(&vf_full[vs], (vc / XF_VF_RING) & 1u);
          if ((hc & 1) == 0) mbar_wait(&o_empty[ob], ((oc / XF_O_BUFS) & 1u) ^ 1u);
          tcgen05_fence_after();
          if (leader) {
            const uint32_t d_tmem = tmem_base + ob * XF_CH + (hc & 1) * XF_HC;
            const uint64_t dv = dv0 + static_cast<uint64_t>((vs * XF_VF_BOX) >> 4);
#pragma unroll
            for (int k = 0; k < XF_NS / 16; ++k)
              umma_bf16(d_tmem, dp0 + ((k * 32) >> 4), dv + ((k * (16 * 128)) >> 4), idesc_o, k != 0 ? 1u : 0u);
            umma_commit(&vf_empty[vs]);  // the box (and, after the last one, P) may be overwritten once these MMAs retire
            if (hc & 1) umma_commit(&o_full[ob]);
          }
          __syncwarp();
          if (hc & 1) ++oc;
        }
        // the next tile's scores AFTER this tile's P.V (the issuer is sequential: ahead of the P.V they would put their
        // operand stream on the critical path); they still overlap the rest of this tile's epilogue
        if (next < p.num_tiles) issue_scores(it + 1);
        tile = next;
      }
    }
  } else if (warp == 2 || warp == 3) {
    // =========================== movers: residual stream global <-> shared by TMA ===========================
    // job j = (tile, pass, half-chunk): pass 0 loads h (fp32) and stores h + attention; pass 1 re-loads the updated rows
    // (L2 hits) and stores LayerNorm(h) as bf16.  Buffer j % NB.  Two threads so that the TMA issue latency of the loads
    // and of the stores is not paid in one serial chain: warp 2 loads (as soon as a buffer is free), warp 3 stores and
    // frees the buffers.
    xf_regs_ctrl();
    {
      const bool leader = elect_one();
      const int tile0 = xf_next_tile(p, first, step);
      int my_tiles = 0;
      if (p.skip_seq == nullptr) my_tiles = first < p.num_tiles ? (p.num_tiles - 1 - first) / step + 1 : 0;
      else for (int t = tile0; t < p.num_tiles; t = xf_next_tile(p, t + step, step)) ++my_tiles;
      const int jobs_per_tile = 2 * p.num_hc;
      const int J = my_tiles * jobs_per_tile;
      // tile of this CTA's ti-th processed tile: a cursor per caller, every caller asks for non-decreasing ti
      struct Cursor { int ti, tile; };
      auto tile_at = [&](Cursor& cur, int ti) {
        for (; cur.ti < ti; ++cur.ti) cur.tile = xf_next_tile(p, cur.tile + step, step);
        return cur.tile;
      };
      Cursor jc{0, tile0};
      auto job_coords = [&](int j, int& seq, int& row, int& pass, int& hc) {
        const int ti = j / jobs_per_tile, r = j - ti * jobs_per_tile;
        const int tile = tile_at(jc, ti);
        seq = tile / p.m_tiles;
        row = (tile - seq * p.m_tiles) * p.rt;
        pass = r / p.num_hc;
        hc = r - pass * p.num_hc;
      };
      if (warp == 2) {
        for (int j = 0; j < J; ++j) {
          int seq, row, pass, hc;
          job_coords(j, seq, row, pass, hc);
          const int b = j % XF_NB;
          mbar_wait(&hfree[b], ((j / XF_NB) & 1u) ^ 1u);   // the store that last used this buffer has read it
          if (leader) {
            uint8_t* buf = hbuf + b * XF_HBUF_BYTES;
            mbar_expect_tx(&hin_full[b], static_cast<uint32_t>(p.rt) * 256);  // two slabs of rt rows x 128 B
            tma_load_4d(&tmap_h, &hin_full[b], buf, hc * XF_HC, row, 0, seq);
            tma_load_4d(&tmap_h, &hin_full[b], buf + XF_SLAB_BYTES, hc * XF_HC + 32, row, 0, seq);
          }
          __syncwarp();
        }
      } else {
        for (int j = 0; j < J; ++j) {
          const int b = j % XF_NB;
          mbar_wait(&hout_full[b], (j / XF_NB) & 1u);
          int seq, row, pass, hc;
          job_coords(j, seq, row, pass, hc);
          if (leader) {   // bulk async-groups belong to the issuing thread: commit / wait on the same lane
            const uint8_t* buf = hbuf + b * XF_HBUF_BYTES;
            if (pass == 0) {
              tma_store_4d(&tmap_h, buf, hc * XF_HC, row, 0, seq);
              tma_store_4d(&tmap_h, buf + XF_SLAB_BYTES, hc * XF_HC + 32, row, 0, seq);
            } else {
              tma_store_4d(&tmap_uo, buf, hc * XF_HC, row, 0, seq);
            }
            bulk_commit();
            const int jn = j - 1 + XF_NB;  // the job that takes over the buffer of job j - 1
            if (j >= 1 && jn < J) {
              bulk_wait_read<1>();  // every store but the one just issued has read its source
              // a pass-1 job re-loads what pass-0 job jn - num_hc stored, num_hc - NB + 1 groups before the newest one:
              // that store must have COMPLETED (be visible), not just have read its source
              if ((jn % jobs_per_tile) >= p.num_hc) {
                if (p.num_hc - XF_NB + 1 > 8) bulk_wait<8>();
                else bulk_wait<1>();
              }
              mbar_arrive(&hfree[(j - 1) % XF_NB]);
            }
          }
          __syncwarp();
        }
        if (leader) bulk_wait<0>();
        __syncwarp();
      }
    }
  } else if (warp >= XF_EPI_WARP0) {
    // =========================== softmax + epilogue ===========================
    xf_regs_epi();
    const int ew = warp - XF_EPI_WARP0;
    const int quarter = warp & 3;   // TMEM lanes [32 quarter, +32)
    const int sub = ew >> 2;        // softmax (sub < 2): 16-row half of the quarter; output: 16-column quarter of the half-chunk
    const int g = lane >> 2, q = lane & 3, q2 = q * 2;
    const bool writer = q == 0;
    uint32_t it = 0, oc = 0, job = 0;
    for (int tile = xf_next_tile(p, first, step); tile < p.num_tiles; tile = xf_next_tile(p, tile + step, step), ++it) {
      const int seq = tile / p.m_tiles;
      const uint32_t sb = it & 1u;
      // ---------------- softmax of the 128 x 64 score tile -> bf16 probabilities in shared memory ----------------
      if (sub < 2) {
        const int trow = quarter * 32 + sub * 16;
        const float* bias = p.sbias + seq * p.sb_seq;
        float2 bb[8];
#pragma unroll
        for (int kb = 0; kb < 8; ++kb) {
          const int c = kb * 8 + q2;
          bb[kb].x = c < p.S ? __ldg(bias + c) * 1.4426950408889634f : 0.f;
          bb[kb].y = c + 1 < p.S ? __ldg(bias + c + 1) * 1.4426950408889634f : 0.f;
        }
        // deferred LayerNorm of the query rows: s' = aX acc + (nX c + bias log2e); (alpha2, 0) without it
        float aA = p.alpha2, nA = 0.f, aB = p.alpha2, nB = 0.f;
        float2 cc[8];
#pragma unroll
        for (int kb = 0; kb < 8; ++kb) cc[kb] = make_float2(0.f, 0.f);
        if (p.ln_stat != nullptr) {
          const float* lnc = p.ln_c + seq * p.sb_seq;
#pragma unroll
          for (int kb = 0; kb < 8; ++kb) {
            const int c = kb * 8 + q2;
            cc[kb].x = c < p.S ? __ldg(lnc + c) : 0.f;
            cc[kb].y = c + 1 < p.S ? __ldg(lnc + c + 1) : 0.f;
          }
          const int mbt = tile - seq * p.m_tiles;
          const int lrA = mbt * p.rt + trow + g;            // row inside the utterance
#pragma unroll
          for (int half = 0; half < 2; ++half) {
            const int lr = lrA + half * 8;
            float sm = 0.f, sq = 0.f;
            if (lr < p.T) {
              const float2* sp2 = p.ln_stat + (static_cast<long long>(seq) * p.T + lr) * p.ln_parts;
              for (int c = 0; c < p.ln_parts; ++c) {
                const float2 v = __ldg(sp2 + c);
                sm += v.x; sq += v.y;
              }
            }
            const float mean = sm * p.inv_h;
            const float rstd = rsqrtf(fmaxf(fmaf(-mean, mean, sq * p.inv_h), 0.f) + 1e-5f);
            if (half == 0) { aA = rstd * p.alpha2; nA = -mean * aA; }
            else { aB = rstd * p.alpha2; nB = -mean * aB; }
          }
        }
        mbar_wait(&s_full[sb], (it >> 1) & 1u);
        tcgen05_fence_after();
        uint32_t r[32];
        tmem_ld_16x64(tmem_base + (static_cast<uint32_t>(trow) << 16) + XF_S_COL0 + sb * XF_NS, r);
        tmem_ld_wait();
        tcgen05_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&s_empty[sb]);  // the scores are in registers: the buffer may take tile it + 2
        float mA = -INFINITY, mB = -INFINITY;
#pragma unroll
        for (int kb = 0; kb < 8; ++kb) {  // s' = (alpha acc + bias) log2 e, in place in r; padded columns -> -inf
          const int c = kb * 8 + q2;
          const float a0 = c < p.S ? fmaf(aA, __uint_as_float(r[4 * kb]), fmaf(nA, cc[kb].x, bb[kb].x)) : -INFINITY;
          const float a1 = c + 1 < p.S ? fmaf(aA, __uint_as_float(r[4 * kb + 1]), fmaf(nA, cc[kb].y, bb[kb].y)) : -INFINITY;
          const float b0 = c < p.S ? fmaf(aB, __uint_as_float(r[4 * kb + 2]), fmaf(nB, cc[kb].x, bb[kb].x)) : -INFINITY;
          const float b1 = c + 1 < p.S ? fmaf(aB, __uint_as_float(r[4 * kb + 3]), fmaf(nB, cc[kb].y, bb[kb].y)) : -INFINITY;
          r[4 * kb] = __float_as_uint(a0); r[4 * kb + 1] = __float_as_uint(a1);
          r[4 * kb + 2] = __float_as_uint(b0); r[4 * kb + 3] = __float_as_uint(b1);
          mA = fmaxf(mA, fmaxf(a0, a1));
          mB = fmaxf(mB, fmaxf(b0, b1));
        }
        mA = quad_max(mA);
        mB = quad_max(mB);
        float sumA = 0.f, sumB = 0.f;
#pragma unroll
        for (int kb = 0; kb < 8; ++kb) {
          const float a0 = ex2_approx(__uint_as_float(r[4 * kb]) - mA), a1 = ex2_approx(__uint_as_float(r[4 * kb + 1]) - mA);
          const float b0 = ex2_approx(__uint_as_float(r[4 * kb + 2]) - mB), b1 = ex2_approx(__uint_as_float(r[4 * kb + 3]) - mB);
          r[4 * kb] = __float_as_uint(a0); r[4 * kb + 1] = __float_as_uint(a1);   // exp2(-inf) = 0 for the padded columns
          r[4 * kb + 2] = __float_as_uint(b0); r[4 * kb + 3] = __float_as_uint(b1);
          sumA += a0 + a1;
          sumB += b0 + b1;
        }
        const float iA = 1.0f / quad_sum(sumA), iB = 1.0f / quad_sum(sumB);
        // K-major A operand, 128-B swizzle: row r at r * 128 B, its 16-B chunk kb stored at chunk position kb ^ (r & 7)
        const int rA = trow + g, rB = rA + 8;
        uint8_t* pa = p_smem + rA * 128 + q2 * 2;
        uint8_t* pb = p_smem + rB * 128 + q2 * 2;
#pragma unroll
        for (int kb = 0; kb < 8; ++kb) {
          *reinterpret_cast<uint32_t*>(pa + ((kb ^ (rA & 7)) << 4)) =
              pack_bf16x2(__uint_as_float(r[4 * kb]) * iA, __uint_as_float(r[4 * kb + 1]) * iA);
          *reinterpret_cast<uint32_t*>(pb + ((kb ^ (rB & 7)) << 4)) =
              pack_bf16x2(__uint_as_float(r[4 * kb + 2]) * iB, __uint_as_float(r[4 * kb + 3]) * iB);
        }
        fence_proxy_async_smem();  // generic-proxy writes -> visible to the tensor core's async-proxy reads
        __syncwarp();
        if (lane == 0) mbar_arrive(p_full);
      }
      // ---------------- pass 0: h <- h + O + bo, half-chunk by half-chunk in the staging buffers; row statistics -------
      // This warp: tile rows lrow0 + hh * 16 + g (+ 8), columns sub * 16 + kbl * 8 + q2 (+ 1) of the 64-column half-chunk.
      // fp32 slab (32 columns) in shared memory, TMA 128-B swizzle: row r at r * 128 B, 16-B chunk j at position j ^ (r & 7).
      const int lrow0 = quarter * 32;
      const int slab_sel = sub >> 1, jbase = (sub & 1) * 4 + (q >> 1);   // 32-column slab, first 16-B chunk of this thread
      // [hh][A|B] packed sums of v - K and (v - K)^2, K = this thread's first value of the row (nk = -K; common.cuh)
      float2 sm2[4], sq2[4], nk[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) sm2[j] = sq2[j] = nk[j] = make_float2(0.f, 0.f);
      uint32_t ob = 0;
      float2 b2N[2];
#pragma unroll
      for (int kbl = 0; kbl < 2; ++kbl) b2N[kbl] = __ldg(reinterpret_cast<const float2*>(p.out_bias + sub * 16 + q2 + kbl * 8));
#pragma unroll 1
      for (int hc = 0; hc < p.num_hc; ++hc, ++job) {
        const uint32_t b = job % XF_NB;
        uint8_t* slab = hbuf + b * XF_HBUF_BYTES + slab_sel * XF_SLAB_BYTES + (q & 1) * 8;
        const int col0 = hc * XF_HC + sub * 16 + q2;
        float2 b2[2];
#pragma unroll
        for (int kbl = 0; kbl < 2; ++kbl) b2[kbl] = b2N[kbl];
        if (hc + 1 < p.num_hc) {
#pragma unroll
          for (int kbl = 0; kbl < 2; ++kbl) b2N[kbl] = __ldg(reinterpret_cast<const float2*>(p.out_bias + col0 + XF_HC + kbl * 8));
        }
        if ((hc & 1) == 0) {
          ob = oc % XF_O_BUFS;
          mbar_wait(&o_full[ob], (oc / XF_O_BUFS) & 1u);
          tcgen05_fence_after();
        }
        mbar_wait(&hin_full[b], (job / XF_NB) & 1u);
        uint32_t r[2][8];
        float2 rsA[2][2], rsB[2][2];
#pragma unroll
        for (int hh = 0; hh < 2; ++hh) {  // every load of the job first (TMEM and shared memory), then the arithmetic
          const int rA = lrow0 + hh * 16 + g, rB = rA + 8;
          tmem_ld_16x16(tmem_base + (static_cast<uint32_t>(lrow0 + hh * 16) << 16) + ob * XF_CH + (hc & 1) * XF_HC + sub * 16, r[hh]);
#pragma unroll
          for (int kbl = 0; kbl < 2; ++kbl) {
            const int j = jbase + kbl * 2;
            rsA[hh][kbl] = *reinterpret_cast<const float2*>(slab + rA * 128 + ((j ^ (rA & 7)) << 4));
            rsB[hh][kbl] = *reinterpret_cast<const float2*>(slab + rB * 128 + ((j ^ (rB & 7)) << 4));
          }
        }
        tmem_ld_wait();
#pragma unroll
        for (int hh = 0; hh < 2; ++hh) {
          const int rA = lrow0 + hh * 16 + g, rB = rA + 8;
#pragma unroll
          for (int kbl = 0; kbl < 2; ++kbl) {
            const int j = jbase + kbl * 2;
            const float2 vA = __fadd2_rn(__fadd2_rn(make_float2(__uint_as_float(r[hh][4 * kbl]), __uint_as_float(r[hh][4 * kbl + 1])), b2[kbl]),
                                         rsA[hh][kbl]);
            const float2 vB = __fadd2_rn(__fadd2_rn(make_float2(__uint_as_float(r[hh][4 * kbl + 2]), __uint_as_float(r[hh][4 * kbl + 3])), b2[kbl]),
                                         rsB[hh][kbl]);
            if (hc == 0 && kbl == 0) { nk[2 * hh] = make_float2(-vA.x, -vA.x); nk[2 * hh + 1] = make_float2(-vB.x, -vB.x); }
            const float2 dA = __fadd2_rn(vA, nk[2 * hh]), dB = __fadd2_rn(vB, nk[2 * hh + 1]);
            sm2[2 * hh] = __fadd2_rn(sm2[2 * hh], dA);
            sq2[2 * hh] = __ffma2_rn(dA, dA, sq2[2 * hh]);
            sm2[2 * hh + 1] = __fadd2_rn(sm2[2 * hh + 1], dB);
            sq2[2 * hh + 1] = __ffma2_rn(dB, dB, sq2[2 * hh + 1]);
            *reinterpret_cast<float2*>(slab + rA * 128 + ((j ^ (rA & 7)) << 4)) = vA;   // in place: one owner per element
            *reinterpret_cast<float2*>(slab + rB * 128 + ((j ^ (rB & 7)) << 4)) = vB;
          }
        }
        fence_proxy_async_smem();  // the TMA store reads these generic-proxy writes
        if (hc & 1) tcgen05_fence_before();
        __syncwarp();
        if (lane == 0) {
          mbar_arrive(&hout_full[b]);
          if (hc & 1) mbar_arrive(&o_empty[ob]);
        }
        if (hc & 1) ++oc;
      }
      // ---------------- row statistics: the four column quarters of a row live in four warps ----------------
      // partials (mean, M2): a thread has 4 num_hc values of a row, a quad 16 num_hc, a warp's quarter H / 4
      float2* sp = stat + (it & 1u) * (XF_BM * 4);
      const float n_t = static_cast<float>(4 * p.num_hc);
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float2 st = ln_quad_merge(ln_partial(-nk[j].x, sm2[j].x + sm2[j].y, sq2[j].x + sq2[j].y, 1.0f / n_t), n_t);
        if (writer) sp[(lrow0 + (j >> 1) * 16 + g + (j & 1) * 8) * 4 + sub] = st;
      }
      epi_bar_sync();
      float mean[4], rstd[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int lr = lrow0 + (j >> 1) * 16 + g + (j & 1) * 8;
        const float4 a = *reinterpret_cast<const float4*>(sp + lr * 4), c = *reinterpret_cast<const float4*>(sp + lr * 4 + 2);
        const float2 st = ln_merge(ln_merge(make_float2(a.x, a.y), make_float2(a.z, a.w), 4.f * n_t),
                                   ln_merge(make_float2(c.x, c.y), make_float2(c.z, c.w), 4.f * n_t), 8.f * n_t);
        mean[j] = st.x;
        rstd[j] = rsqrtf(fmaxf(st.y, 0.f) * p.inv_h + 1e-5f);
      }
      // ---------------- pass 1: LayerNorm of the updated rows -> bf16, written over the staging buffer ----------------
      // bf16 box in shared memory: row r at r * 128 B (64 columns), 16-B chunk j (8 columns) at position j ^ (r & 7)
      float2 gmN[2], btN[2];
#pragma unroll
      for (int kbl = 0; kbl < 2; ++kbl) {
        gmN[kbl] = __ldg(reinterpret_cast<const float2*>(p.gamma + sub * 16 + q2 + kbl * 8));
        btN[kbl] = __ldg(reinterpret_cast<const float2*>(p.beta + sub * 16 + q2 + kbl * 8));
      }
#pragma unroll 1
      for (int hc = 0; hc < p.num_hc; ++hc, ++job) {
        const uint32_t b = job % XF_NB;
        uint8_t* buf = hbuf + b * XF_HBUF_BYTES;
        const uint8_t* slab = buf + slab_sel * XF_SLAB_BYTES + (q & 1) * 8;
        const int col0 = hc * XF_HC + sub * 16 + q2;
        float2 gm[2], bt[2];
#pragma unroll
        for (int kbl = 0; kbl < 2; ++kbl) { gm[kbl] = gmN[kbl]; bt[kbl] = btN[kbl]; }
        if (hc + 1 < p.num_hc) {  // gamma / beta of the next half-chunk: their L2 latency (the L1 is almost all shared memory) hides behind this job
#pragma unroll
          for (int kbl = 0; kbl < 2; ++kbl) {
            gmN[kbl] = __ldg(reinterpret_cast<const float2*>(p.gamma + col0 + XF_HC + kbl * 8));
            btN[kbl] = __ldg(reinterpret_cast<const float2*>(p.beta + col0 + XF_HC + kbl * 8));
          }
        }
        mbar_wait(&hin_full[b], (job / XF_NB) & 1u);
        float2 v[2][4];
#pragma unroll
        for (int hh = 0; hh < 2; ++hh) {
          const int rA = lrow0 + hh * 16 + g, rB = rA + 8;
#pragma unroll
          for (int kbl = 0; kbl < 2; ++kbl) {
            const int j = jbase + kbl * 2;
            v[hh][2 * kbl] = *reinterpret_cast<const float2*>(slab + rA * 128 + ((j ^ (rA & 7)) << 4));
            v[hh][2 * kbl + 1] = *reinterpret_cast<const float2*>(slab + rB * 128 + ((j ^ (rB & 7)) << 4));
          }
        }
        // the bf16 result of rows r overwrites bytes of the fp32 slab-0 data of the SAME rows only, which the four warps of this
        // lane quarter read: once those have their values in registers the buffer may be overwritten
        quarter_bar_sync(quarter);
#pragma unroll
        for (int hh = 0; hh < 2; ++hh) {
          const int rA = lrow0 + hh * 16 + g, rB = rA + 8;
          const float mA = mean[2 * hh], iA = rstd[2 * hh], mB = mean[2 * hh + 1], iB = rstd[2 * hh + 1];
#pragma unroll
          for (int kbl = 0; kbl < 2; ++kbl) {
            const int j = sub * 2 + kbl;
            const float2 a = v[hh][2 * kbl], c = v[hh][2 * kbl + 1];
            *reinterpret_cast<uint32_t*>(buf + rA * 128 + ((j ^ (rA & 7)) << 4) + q * 4) =
                pack_bf16x2(fmaf((a.x - mA) * iA, gm[kbl].x, bt[kbl].x), fmaf((a.y - mA) * iA, gm[kbl].y, bt[kbl].y));
            *reinterpret_cast<uint32_t*>(buf + rB * 128 + ((j ^ (rB & 7)) << 4) + q * 4) =
                pack_bf16x2(fmaf((c.x - mB) * iB, gm[kbl].x, bt[kbl].x), fmaf((c.y - mB) * iB, gm[kbl].y, bt[kbl].y));
          }
        }
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) mbar_arrive(&hout_full[b]);
      }
    }
  } else {
    xf_regs_ctrl();  // warp 2 idles after the TMEM allocation; the whole warpgroup has to execute the setmaxnreg
  }

  __syncwarp();
  tcgen05_fence_before();
  __syncthreads();
  if (warp == 2) {
    tcgen05_fence_after();
    tmem_dealloc<XF_TMEM_COLS>(tmem_base);
  }
}

typedef CUresult (*XfEncodeFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                               const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                               CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
XfEncodeFn g_xf_encode = nullptr;

// fp32 residual stream as a 4-D map (cols, rows of one utterance, 1, utterance): box 32 x 128, 128-B swizzle
int make_map_h(CUtensorMap* m, float* h, int64_t n_seq, int64_t T, int H, int box_rows) {
  if (g_xf_encode == nullptr) {
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult qres;
    DITTO_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres));
    DITTO_REQUIRE(fn != nullptr && qres == cudaDriverEntryPointSuccess, DITTO_E_CUDA, "cuTensorMapEncodeTiled not available");
    g_xf_encode = reinterpret_cast<XfEncodeFn>(fn);
  }
  DITTO_REQUIRE((reinterpret_cast<uintptr_t>(h) & 15) == 0, DITTO_E_BADARG, "cross_fused: h must be 16-B aligned");
  cuuint64_t dims[4] = {static_cast<cuuint64_t>(H), static_cast<cuuint64_t>(T), 1, static_cast<cuuint64_t>(n_seq)};
  cuuint64_t strides[3] = {static_cast<cuuint64_t>(H) * 4, static_cast<cuuint64_t>(T) * H * 4, static_cast<cuuint64_t>(T) * H * 4};
  cuuint32_t box[4] = {32, static_cast<cuuint32_t>(box_rows), 1, 1};
  cuuint32_t estr[4] = {1, 1, 1, 1};
  CUresult r = g_xf_encode(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, h, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                           CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cross_fused: cuTensorMapEncodeTiled (fp32) failed with CUresult " + std::to_string(static_cast<int>(r)));
    return DITTO_E_CUDA;
  }
  return 0;
}

}  // namespace

bool cross_fused_supported(int64_t T, int64_t S, int H, int heads) {
  // H >= 4 half-chunks: the mover re-loads a row block only after the store that produced it has completed (NB <= H / 64)
  return heads == 1 && S >= 1 && S <= XF_NS && H % XF_CH == 0 && H >= XF_NB * XF_HC && H <= XF_MAX_H && T >= 1;
}

int launch_cross_fused(const CrossFusedParams& q, cudaStream_t st) {
  DITTO_TRY(tc_gemm_init());
  DITTO_REQUIRE(cross_fused_supported(q.T, q.S, q.H, 1), DITTO_E_UNSUPPORTED, "cross_fused: unsupported shape");
  DITTO_REQUIRE(q.u && q.kfold && q.vfold && q.sbias && q.out_bias && q.h && q.gamma && q.beta && q.u_out, DITTO_E_BADARG,
                "cross_fused: null argument");
  DITTO_REQUIRE(q.n_seq >= 1 && q.Sp >= q.S && q.Sp % 8 == 0, DITTO_E_BADARG, "cross_fused: bad sizes");
  DeviceState* ds = device_state();
  if (ds == nullptr) return DITTO_E_CUDA;
  if (!ds->xf_attr) {  // per device
    DITTO_CUDA(cudaFuncSetAttribute(cross_fused_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, XF_SMEM_BYTES));
    ds->xf_attr = true;
  }
  TcOperand U, Kf, Vf, Uo;
  U.ptr = q.u; U.rows = q.T; U.cols = q.H; U.ld = q.H; U.s_outer = q.T * q.H;
  Kf.ptr = q.kfold; Kf.rows = q.S; Kf.cols = q.H; Kf.ld = q.H; Kf.s_outer = q.kf_seq;
  Vf.ptr = q.vfold; Vf.rows = q.Sp; Vf.cols = q.H; Vf.ld = q.H; Vf.s_outer = q.vf_seq;
  Uo.ptr = q.u_out; Uo.rows = q.T; Uo.cols = q.H; Uo.ld = q.H; Uo.s_outer = q.T * q.H;
  // Rows per tile: the MMAs always compute 128 rows, the TMA boxes (and so the HBM traffic) carry `rt` of them.  Measured at
  // C2 (profiles/README.md): 128 / 96 / 88 rows all take ~70 us and 64 rows 90 us -- the tile loop is bound by the latency of
  // its 24 staging jobs per tile, not by their bytes, so fewer, larger tiles win; the xf_rows debug option overrides for experiments.
  const int sms = tc_num_sms();
  int rt = XF_BM;
  if (g_opt.xf_rows >= 8 && g_opt.xf_rows <= XF_BM && g_opt.xf_rows % 8 == 0) rt = g_opt.xf_rows;
  CUtensorMap mu, mk, mv, mh, mo;
  DITTO_TRY(tc_make_map(&mu, U, 1, q.n_seq, XF_BK, rt));
  DITTO_TRY(tc_make_map(&mk, Kf, 1, q.n_seq, XF_BK, XF_NS));
  DITTO_TRY(tc_make_map(&mv, Vf, 1, q.n_seq, 64, XF_NS));
  DITTO_TRY(tc_make_map(&mo, Uo, 1, q.n_seq, XF_HC, rt));
  DITTO_TRY(make_map_h(&mh, q.h, q.n_seq, q.T, q.H, rt));
  XfDev p;
  p.n_seq = static_cast<int>(q.n_seq); p.T = static_cast<int>(q.T); p.S = static_cast<int>(q.S); p.H = q.H;
  p.rt = rt;
  p.m_tiles = static_cast<int>(ceil_div(q.T, rt));
  const int64_t tiles = static_cast<int64_t>(p.m_tiles) * q.n_seq;
  DITTO_REQUIRE(tiles < (1ll << 31), DITTO_E_UNSUPPORTED, "cross_fused: too many tiles");
  p.num_tiles = static_cast<int>(tiles);
  p.num_kb = q.H / XF_BK;
  p.num_ch = q.H / XF_CH;
  p.num_hc = q.H / XF_HC;
  p.alpha2 = q.alpha * 1.4426950408889634f;
  p.sbias = q.sbias; p.sb_seq = q.sb_seq;
  p.out_bias = q.out_bias;
  p.gamma = q.gamma; p.beta = q.beta;
  p.inv_h = 1.0f / static_cast<float>(q.H);
  p.ln_stat = q.ln_stat; p.ln_parts = q.ln_parts; p.ln_c = q.ln_c;
  p.skip_seq = q.skip_seq;
  if (q.ln_stat != nullptr) DITTO_REQUIRE(q.ln_parts > 0 && q.ln_c != nullptr, DITTO_E_BADARG, "cross_fused: deferred LayerNorm arguments");
  // flops: both contractions; bytes: u read, h read + write, u3 write (the HBM stream that bounds the kernel)
  const double rows = static_cast<double>(q.n_seq - (q.skip_seq ? profiled_nonzero(q.skip_seq, q.n_seq, st) : 0)) * q.T;
  ProfScope prof(q.tag, st, 4.0 * rows * q.S * q.H, rows * q.H * 12.0);
  const int grid = static_cast<int>(std::min<int64_t>(sms, tiles));
  cross_fused_kernel<<<grid, XF_THREADS, XF_SMEM_BYTES, st>>>(mu, mk, mv, mh, mo, p);
  DITTO_LAUNCH_CHECK();
  return 0;
}

}  // namespace ditto
