// Flash-style self-attention for the repo-default single head of 768 (reference: src/components/DiT.py:117-139 on the
// config src/utils/Config.py:109-111), fused with the residual add and the LayerNorm that follows (norm2, DiT.py:143):
//
//     h  <- h + softmax(alpha q k^T) v          (no out_proj: DiT.py:137-139)
//     u  <- LayerNorm(h) * gamma2 + beta2       (bf16 operand of the cross-attention kernel)
//
// in ONE kernel: neither the scores nor the probabilities touch HBM (the two-kernel formulation writes and re-reads the
// unnormalised bf16 P, 72 MB per layer at C2, and a third launch re-reads h for the LayerNorm).
//
// Why a cluster of two CTAs: an fp32 128 x 768 output accumulator is 768 TMEM columns, the SM has 512.  The two CTAs of a
// cluster work on the SAME 128 query rows; CTA r owns output columns [384 r, 384 r + 384) (384 TMEM columns) next to one
// 128-column score tile = 512 columns exactly.  The score tiles are split by KEYS: CTA r computes S(j) = Q K_j^T and its
// softmax for the key tiles j = r, r + 2, ... only, and hands the bf16 probability tile to its peer through distributed
// shared memory (one 32 KiB cp.async.bulk shared::cta -> shared::cluster per tile, completion on the peer's mbarrier), so
// no contraction is done twice and each CTA streams only half of the Q / K operand traffic -- the kernel is bound by the
// L2 -> SM operand feed (~44 B/clk/SM), not by the tensor pipe (first version, every CTA computing all score tiles:
// 137 us per layer at C2 with the tensor pipe 33 % busy and 1.2 GB delivered to the SMs).
//
// Online softmax with ONE reference per row shared by both CTAs (both accumulate every P tile into their own O half, so a
// tile's reference must be the one their accumulators are scaled to): tile 0 fixes r = rowmax; the owner of tile j moves it
// only when the tile's maximum exceeds r by more than 2^8 ("lazy rescale"), and sends its decision r_j (128 floats, st.async
// + complete_tx) to the peer before it exponentiates.  Whoever sees r change multiplies its O rows in TMEM by 2^(r_old - r_new)
// (tcgen05.ld / tcgen05.st, after the previous P.V has retired) before the tile's P.V may be issued.  P = 2^(s - r) <= 256 is
// exact enough in bf16 (same relative precision at any scale); l and O accumulate in fp32; the result is O / l.
//
// Per CTA (384 threads, persistent over (utterance, 128-query tile) items):
//   warp 0   TMA producer, ONE ring of four 32 KiB slots fed in exactly the order the MMA issuer consumes it:
//            score stages  Q[128 x 64] + K[128 keys x 64]   (12 per OWN key tile; head dim streamed in 64-wide chunks)
//            P.V stages    V[32 keys x 384] as six MN-major [32 x 64] boxes (4 per key tile, every tile)
//   warp 1   MMA issuer:  S(own_0) { [S(next own)] P.V(j) }  -- the next own score tile is issued before the P.V of the
//            current one, so its MMAs run under the softmax
//   warp 2   probability courier: own tile written -> one bulk copy into the peer's landing buffer
//   warps 4-11  softmax of the own tiles (warp = 16 rows, accumulator fragments via tcgen05.ld.16x256b, quad reductions), P
//            written as the bf16 K-major A operand (128-B swizzle by hand); reference bookkeeping for the peer's tiles;
//            epilogue: O / l + h -> h (fp32, 16-byte accesses through the v-column order `out_perm4` of the QKV epilogue),
//            row statistics, h kept in TMEM, statistics exchanged with the peer CTA, second sweep writes LayerNorm(h) as bf16
//   (control warps run on warp-uniform values with one elected lane issuing, see common.cuh: elect_one)
// TMEM: [0, 384) O, [384, 512) S.
#include <algorithm>

#include "common.cuh"
#include "kernels.cuh"

namespace ditto {
namespace {

constexpr int F7_THREADS = 384;
constexpr int F7_EPI_WARP0 = 4;
constexpr int F7_EPI_WARPS = 8;
constexpr int F7_BM = 128, F7_BN = 128, F7_BK = 64;
constexpr int F7_D = 768;             // head dim == hidden
constexpr int F7_DH = F7_D / 2;       // output columns per CTA
constexpr int F7_KCH = F7_D / F7_BK;  // 12 head-dim chunks per score tile
constexpr int F7_VKEYS = 32;          // keys per P.V stage
constexpr int F7_VST = F7_BN / F7_VKEYS;  // 4 P.V stages per key tile
constexpr int F7_VBOX = F7_VKEYS * 128;   // 4 KiB: [32 keys x 64 n] bf16, n contiguous
constexpr int F7_STAGES = 4;
constexpr int F7_STAGE_BYTES = 32768;
constexpr int F7_QK_BYTES = F7_BM * F7_BK * 2;  // 16 KiB each for the Q and the K chunk
constexpr int F7_V_BYTES = (F7_DH / 64) * F7_VBOX;  // 24 KiB
constexpr int F7_P_BYTES = F7_BM * F7_BN * 2;   // 32 KiB (two K-major 64-key sub-tiles)
constexpr int F7_OFF_POWN = F7_STAGES * F7_STAGE_BYTES;        // probabilities of the tile this CTA owns
constexpr int F7_OFF_PLAND = F7_OFF_POWN + F7_P_BYTES;         // landing buffer for the peer's tile
constexpr int F7_OFF_BAR = F7_OFF_PLAND + F7_P_BYTES;
constexpr int F7_BAR_BYTES = 256;
constexpr int F7_OFF_XCH = F7_OFF_BAR + F7_BAR_BYTES;
// written by the peer CTA (st.async): [2][128] softmax references, [2][128] partial row sums, [2][128][2] LayerNorm partials
constexpr int F7_XCH_HDR = 0, F7_XCH_L = 2 * F7_BM * 4, F7_XCH_STAT = 4 * F7_BM * 4;
constexpr int F7_XCH_BYTES = 4 * F7_BM * 4 + 2 * F7_BM * 8;
constexpr int F7_SMEM_BYTES = F7_OFF_XCH + F7_XCH_BYTES + 1024;
static_assert(F7_SMEM_BYTES <= 232448, "exceeds the 227 KiB shared memory of an sm_100 CTA");
static_assert(F7_V_BYTES <= F7_STAGE_BYTES && 2 * F7_QK_BYTES == F7_STAGE_BYTES, "ring slot too small");
static_assert(F7_KCH % F7_STAGES == 0 && F7_VST == F7_STAGES, "every tile must start at ring slot 0");
constexpr int F7_TMEM_COLS = 512;
constexpr int F7_S_COL = F7_DH;       // 384
constexpr float F7_TAU = 8.0f;        // lazy-rescale threshold, log2 units

struct F7Dev {
  unsigned long long* trace;
  int n_seq, T;
  int m_tiles, k_tiles, num_items;
  float alpha2;                       // alpha * log2(e)
  float* h;                           // [n_seq * T, 768] fp32 residual stream, updated in place
  const float* gamma; const float* beta;
  bf16* u_out;                        // [n_seq * T, 768] LayerNorm(h) (nullptr: no LayerNorm stage)
  int force_rescale;                  // tests: move the reference whenever a tile raises a row maximum
};

__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(F7_THREADS, 1)
    flash_attn768_kernel(const __grid_constant__ CUtensorMap tmap_q, const __grid_constant__ CUtensorMap tmap_k,
                         const __grid_constant__ CUtensorMap tmap_v, const F7Dev p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw_addr = smem_u32(smem_raw);
  uint8_t* smem = smem_raw + ((1024u - (raw_addr & 1023u)) & 1023u);
  uint8_t* p_own = smem + F7_OFF_POWN;
  uint8_t* p_land = smem + F7_OFF_PLAND;
  uint64_t* ring_full = reinterpret_cast<uint64_t*>(smem + F7_OFF_BAR);
  uint64_t* ring_empty = ring_full + F7_STAGES;
  uint64_t* s_full = ring_empty + F7_STAGES;     // score tile complete                         (MMA -> softmax)
  uint64_t* s_empty = s_full + 1;                // score tile read                             (softmax -> MMA)
  uint64_t* p_full = s_empty + 1;                // own probabilities written                   (softmax -> MMA, courier)
  uint64_t* p_free = p_full + 1;                 // own buffer reusable: P.V of BOTH CTAs retired (2 arrivals: local + peer's commit)
  uint64_t* land_full = p_free + 1;              // peer's probabilities landed                 (peer's courier, complete_tx)
  uint64_t* accept = land_full + 1;              // [2] reference of a peer tile adopted        (softmax -> MMA)
  uint64_t* pv_done = accept + 2;                // [4] P.V of tile (global index mod 4) retired (MMA -> softmax: pacing, TMEM rescale)
  uint64_t* o_full = pv_done + 4;                // O complete                                  (MMA -> epilogue)
  uint64_t* o_empty = o_full + 1;                // O drained                                   (epilogue -> MMA)
  uint64_t* hdr_bar = o_empty + 1;               // [2] peer's reference decision landed        (st.async complete_tx)
  uint64_t* l_bar = hdr_bar + 2;                 // [2] peer's partial row sums landed
  uint64_t* stat_bar = l_bar + 2;                // [2] peer's LayerNorm partials landed
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(stat_bar + 2);
  static_assert((2 * F7_STAGES + 13 + 6) * 8 + 4 <= F7_BAR_BYTES, "barrier block too small");
  float* hdr_x = reinterpret_cast<float*>(smem + F7_OFF_XCH + F7_XCH_HDR);     // [2][128]
  float* l_x = reinterpret_cast<float*>(smem + F7_OFF_XCH + F7_XCH_L);         // [2][128]
  float* stat_x = reinterpret_cast<float*>(smem + F7_OFF_XCH + F7_XCH_STAT);   // [2][128][2]

  const int warp = warp_id_uniform();
  const int lane = threadIdx.x & 31;
  const uint32_t rank = __shfl_sync(0xffffffffu, cluster_ctarank(), 0);   // which half of the output columns / which key tiles
  const uint32_t peer = rank ^ 1u;
  const int num_clusters = gridDim.x >> 1;
  const int first = blockIdx.x >> 1;
  const int KT = p.k_tiles;
  const int c = static_cast<int>(rank);

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmap_q);
    tma_prefetch_desc(&tmap_k);
    tma_prefetch_desc(&tmap_v);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < F7_STAGES; ++s) { mbar_init(&ring_full[s], 1); mbar_init(&ring_empty[s], 1); }
    mbar_init(s_full, 1);
    mbar_init(s_empty, F7_EPI_WARPS);
    mbar_init(p_full, F7_EPI_WARPS);
    mbar_init(p_free, 2);
    mbar_init(land_full, 1);
    mbar_init(&accept[0], F7_EPI_WARPS);
    mbar_init(&accept[1], F7_EPI_WARPS);
    for (int s = 0; s < 4; ++s) mbar_init(&pv_done[s], 1);
    mbar_init(o_full, 1);
    mbar_init(o_empty, F7_EPI_WARPS);
    for (int s = 0; s < 2; ++s) { mbar_init(&hdr_bar[s], 1); mbar_init(&l_bar[s], 1); mbar_init(&stat_bar[s], 1); }
    fence_barrier_init();
  }
  if (warp == 2) tmem_alloc<F7_TMEM_COLS>(tmem_ptr);
  tcgen05_fence_before();
  __syncthreads();
  cluster_sync_all();   // the peer's barriers exist before the first st.async / bulk copy / commit reaches them
  tcgen05_fence_after();
  const uint32_t tmem_base = *tmem_ptr;
  const long long t_sync = DITTO_F7_TRACE ? clock64() : 0;   // the cluster barrier released both CTAs at (about) the same moment

  if (warp == 0) {
    // =========================== TMA producer (whole warp, one elected lane issues) ===========================
    // Every score tile takes 12 and every P.V tile 4 ring slots, so each starts at slot 0: slot indices are compile-time
    // constants and the barrier phase flips once per group of four.
    regs_shrink_ctrl();
    const bool leader = elect_one();
    F7Tr tr; tr.init(p.trace, c, 2, first == 0 && leader, t_sync);
    uint32_t phase = 0;
    for (int item = first; item < p.num_items; item += num_clusters) {
      const int qt = item % p.m_tiles, seq = item / p.m_tiles;
      auto load_s = [&](int j) {
#pragma unroll 1
        for (int c4 = 0; c4 < F7_KCH / F7_STAGES; ++c4) {
#pragma unroll
          for (int s = 0; s < F7_STAGES; ++s) {
            mbar_wait(&ring_empty[s], phase ^ 1u);
            if (leader) {
              uint8_t* sb = smem + s * F7_STAGE_BYTES;
              mbar_expect_tx(&ring_full[s], 2 * F7_QK_BYTES);
              tma_load_4d(&tmap_q, &ring_full[s], sb, (c4 * F7_STAGES + s) * F7_BK, qt * F7_BM, 0, seq);   // rows >= T: zero-filled
              tma_load_4d(&tmap_k, &ring_full[s], sb + F7_QK_BYTES, (c4 * F7_STAGES + s) * F7_BK, j * F7_BN, 0, seq);
            }
            __syncwarp();
          }
          phase ^= 1u;
        }
        tr.ev(30, j);
      };
      auto load_v = [&](int j) {
#pragma unroll
        for (int s = 0; s < F7_VST; ++s) {
          mbar_wait(&ring_empty[s], phase ^ 1u);
          if (leader) {
            uint8_t* sb = smem + s * F7_STAGE_BYTES;
            mbar_expect_tx(&ring_full[s], F7_V_BYTES);
#pragma unroll
            for (int b = 0; b < F7_DH / 64; ++b)  // [32 key-rows x 64 n] boxes, n contiguous (MN-major operand)
              tma_load_4d(&tmap_v, &ring_full[s], sb + b * F7_VBOX, c * F7_DH + b * 64, j * F7_BN + s * F7_VKEYS, 0, seq);
          }
          __syncwarp();
        }
        phase ^= 1u;
        tr.ev(31, j);
      };
      // same order as the MMA issuer: the first own score tile, then per key tile [the next own score tile] and the P.V
      if (c < KT) load_s(c);
      for (int j = 0; j < KT; ++j) {
        if ((j & 1) == c && j + 2 < KT) load_s(j + 2);
        load_v(j);
      }
    }
  } else if (warp == 1) {
    // =========================== MMA issuer (whole warp, one elected lane issues) ===========================
    regs_shrink_ctrl();
    const bool leader = elect_one();
    constexpr uint32_t idesc_s = umma_idesc_bf16(F7_BM, F7_BN, false, false);
    constexpr uint32_t idesc_o256 = umma_idesc_bf16(F7_BM, 256, false, true);
    constexpr uint32_t idesc_o128 = umma_idesc_bf16(F7_BM, 128, false, true);
    // descriptors of ring slot 0 / the P buffers; everything else is these plus a compile-time constant (the 14-bit address
    // field counts 16-byte units and cannot carry: shared memory ends below 256 KiB)
    // ONE runtime value: the K-major descriptor of ring slot 0.  The MN-major V descriptor differs only in the LBO field
    // (bits 16-29: 4 KiB between the 64-column boxes instead of 16 B), the P buffers only in the address field.
    const uint64_t dq0 = umma_smem_desc(smem_u32(smem), 16, 1024);
    constexpr uint64_t kToV = static_cast<uint64_t>((F7_VBOX >> 4) - 1) << 16;
    constexpr uint64_t kToPOwn = F7_OFF_POWN >> 4, kToPLand = F7_OFF_PLAND >> 4;
    const uint16_t peer_mask = static_cast<uint16_t>(1u << peer);
    uint32_t phase = 0;
    uint32_t it = 0, sc = 0, oc = 0, rc = 0, pvi = 0;   // items, own score tiles, own / peer probability tiles consumed, P.V issued
    F7Tr tr; tr.init(p.trace, c, 0, first == 0 && leader, t_sync);
    auto issue_s = [&]() {
      mbar_wait(s_empty, (sc & 1u) ^ 1u);
      tcgen05_fence_after();
      tr.ev(1, sc);
      long long fw = 0;
#pragma unroll 1
      for (int c4 = 0; c4 < F7_KCH / F7_STAGES; ++c4) {
#pragma unroll
        for (int s = 0; s < F7_STAGES; ++s) {
          if (DITTO_F7_TRACE && tr.b) { const long long w0 = clock64(); mbar_wait(&ring_full[s], phase); fw += clock64() - w0; }
          else mbar_wait(&ring_full[s], phase);
          tcgen05_fence_after();
          if (leader) {
#pragma unroll
            for (int k = 0; k < F7_BK / 16; ++k)
              umma_bf16(tmem_base + F7_S_COL, dq0 + ((s * F7_STAGE_BYTES + k * 32) >> 4),
                        dq0 + ((s * F7_STAGE_BYTES + F7_QK_BYTES + k * 32) >> 4), idesc_s, (c4 | s | k) != 0 ? 1u : 0u);
            umma_commit(&ring_empty[s]);
          }
          __syncwarp();
        }
        phase ^= 1u;
      }
      if (leader) umma_commit(s_full);
      __syncwarp();
      tr.ev(2, sc);
      tr.val(6, sc, fw);
      ++sc;
    };
    auto issue_pv = [&](int j) {
      const bool own = (j & 1) == c;
      if (own) {
        mbar_wait(p_full, oc & 1u);
      } else {
        if (leader) mbar_expect_tx(land_full, F7_P_BYTES);   // arm this tile's landing (the copy may already be on its way)
        __syncwarp();
        mbar_wait(land_full, rc & 1u);
        mbar_wait(&accept[rc & 1u], (rc >> 1) & 1u);          // ... and its reference has been adopted (O rescaled if it moved)
      }
      if (j == 0) mbar_wait(o_empty, (it & 1u) ^ 1u);         // the previous item's O has been drained
      tcgen05_fence_after();
      tr.ev(3, j);
      long long fw = 0;
      const uint64_t dp = dq0 + (own ? kToPOwn : kToPLand);
#pragma unroll
      for (int s = 0; s < F7_VST; ++s) {
        if (DITTO_F7_TRACE && tr.b) { const long long w0 = clock64(); mbar_wait(&ring_full[s], phase); fw += clock64() - w0; }
        else mbar_wait(&ring_full[s], phase);
        tcgen05_fence_after();
        if (leader) {
#pragma unroll
          for (int k = 0; k < F7_VKEYS / 16; ++k) {
            const int key16 = s * (F7_VKEYS / 16) + k;                 // 16-key step inside the 128-key tile
            const uint64_t da = dp + (((key16 >> 2) * (F7_BM * 128) + (key16 & 3) * 32) >> 4);
            const uint32_t acc = (j | s | k) != 0 ? 1u : 0u;
            umma_bf16(tmem_base, da, dq0 + (kToV + ((s * F7_STAGE_BYTES + k * (16 * 128)) >> 4)), idesc_o256, acc);
            umma_bf16(tmem_base + 256, da, dq0 + (kToV + ((s * F7_STAGE_BYTES + 4 * F7_VBOX + k * (16 * 128)) >> 4)), idesc_o128, acc);
          }
          umma_commit(&ring_empty[s]);
        }
        __syncwarp();
      }
      phase ^= 1u;
      if (leader) {
        umma_commit(&pv_done[pvi & 3u]);
        // the tile's buffer in its OWNER is reusable once both CTAs' P.V have retired
        if (own) umma_commit(p_free);
        else umma_commit_mc(p_free, peer_mask);
      }
      __syncwarp();
      tr.ev(4, j);
      tr.val(7, j, fw);
      if (own) ++oc; else ++rc;
      ++pvi;
    };
    for (int item = first; item < p.num_items; item += num_clusters, ++it) {
      if (c < KT) issue_s();
      for (int j = 0; j < KT; ++j) {
        if ((j & 1) == c && j + 2 < KT) issue_s();   // the next own score tile runs under this tile's softmax
        issue_pv(j);
      }
      if (leader) umma_commit(o_full);
      __syncwarp();
      tr.ev(5, it);
    }
  } else if (warp == 2) {
    // =========================== probability courier ===========================
    regs_shrink_ctrl();
    const bool leader = elect_one();
    const uint32_t dst = mapa_shared(smem_u32(p_land), peer), src = smem_u32(p_own), bar = mapa_shared(smem_u32(land_full), peer);
    uint32_t oc = 0;
    for (int item = first; item < p.num_items; item += num_clusters)
      for (int j = c; j < KT; j += 2, ++oc) {
        mbar_wait(p_full, oc & 1u);     // written + fence.proxy.async by the softmax warps; the peer's landing buffer is free:
        if (leader) bulk_copy_to_peer(dst, src, F7_P_BYTES, bar);   // p_free (awaited before the tile was written) includes the peer's P.V
        __syncwarp();
      }
  } else if (warp >= F7_EPI_WARP0) {
    // =========================== softmax + epilogue ===========================
    regs_grow_epi();
    const int ew = warp - F7_EPI_WARP0;
    const int quarter = warp & 3, hsel = ew >> 2;
    const int g = lane >> 2, q = lane & 3, q2 = q * 2;
    const int trow = quarter * 32 + hsel * 16;     // this warp's 16 rows: trow + g, trow + g + 8
    const int rA = trow + g, rB = rA + 8;
    const uint32_t t_lane = tmem_base + (static_cast<uint32_t>(trow) << 16);
    const bool writer = q == 0;
    const int col_half = c * F7_DH;
    uint32_t it = 0, sc = 0, oc = 0, rc = 0, pvc = 0;   // items, own score tiles, own / peer tiles, P.V issued (all tiles)
    F7Tr tr; tr.init(p.trace, c, 1, first == 0 && ew == 0 && lane == 0, t_sync);
    // multiply this warp's O rows by (fA, fB): the previous P.V (global index pvc - 1) must have retired, the next one waits
    // for this warp.  (pv_done cycles through four barriers and every tile first waits for P.V(pvc - 4): a parity wait is
    // only unambiguous while the barrier is at most one completion behind -- or ahead.)
    auto rescale_o = [&](float fA, float fB) {
      mbar_wait(&pv_done[(pvc - 1) & 3u], ((pvc - 1) >> 2) & 1u);
      tcgen05_fence_after();
#pragma unroll 1
      for (int cb = 0; cb < F7_DH / 64; ++cb) {
        uint32_t o[32];
        tmem_ld_16x64(t_lane + cb * 64, o);
        tmem_ld_wait();
#pragma unroll
        for (int kb = 0; kb < 8; ++kb) {
          o[4 * kb] = __float_as_uint(__uint_as_float(o[4 * kb]) * fA);
          o[4 * kb + 1] = __float_as_uint(__uint_as_float(o[4 * kb + 1]) * fA);
          o[4 * kb + 2] = __float_as_uint(__uint_as_float(o[4 * kb + 2]) * fB);
          o[4 * kb + 3] = __float_as_uint(__uint_as_float(o[4 * kb + 3]) * fB);
        }
        tmem_st_16x64(t_lane + cb * 64, o);
      }
      tmem_st_wait();
      tcgen05_fence_before();
    };
    for (int item = first; item < p.num_items; item += num_clusters, ++it) {
      const int qt = item % p.m_tiles, seq = item / p.m_tiles;
      const int lrowA = qt * F7_BM + rA;                         // row inside the utterance
      const bool okA = lrowA < p.T, okB = lrowA + 8 < p.T;
      const long long growA = static_cast<long long>(seq) * p.T + lrowA;
      float* hA = p.h + growA * F7_D + col_half + q * 4;         // this thread's first output column of a 64-column chunk
      float* hB = hA + 8 * F7_D;
      // residual rows of this warp -> L2 while the tile computes (16 rows x 384 columns = 192 lines of 128 B)
      for (int i = lane; i < 16 * (F7_DH * 4 / 128); i += 32) {
        const int r = i / (F7_DH * 4 / 128), l = i - r * (F7_DH * 4 / 128);
        if (qt * F7_BM + trow + r < p.T)
          prefetch_l2(p.h + (static_cast<long long>(seq) * p.T + qt * F7_BM + trow + r) * F7_D + col_half + l * 32);
      }
      float refA = 0.f, refB = 0.f;                              // softmax references (log2 domain) shared by both CTAs
      float2 lA2 = make_float2(0.f, 0.f), lB2 = make_float2(0.f, 0.f);   // row sums of the OWN tiles relative to the references
      uint32_t s0[32], s1[32];
      bool have_s = false;   // the next own score tile is already in registers (loaded while waiting for the peer's reference)
      auto load_scores = [&]() {
        mbar_wait(s_full, sc & 1u);
        tcgen05_fence_after();
        tmem_ld_16x64(t_lane + F7_S_COL, s0);
        tmem_ld_16x64(t_lane + F7_S_COL + 64, s1);
        tmem_ld_wait();
        tcgen05_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(s_empty);                     // the scores are in registers: the next own S may be issued
        tr.ev(10, sc);
        ++sc;
        have_s = true;
      };
      for (int j = 0; j < KT; ++j, ++pvc) {
        // pacing: never more than four tiles ahead of the tensor pipe (keeps every parity wait below unambiguous, and the
        // accept / header barriers from completing twice before they are consumed)
        if (pvc >= 4) mbar_wait(&pv_done[pvc & 3u], ((pvc >> 2) - 1) & 1u);
        tr.ev(20, j);
        if ((j & 1) != c) {
          // ---------------- a tile of the peer: adopt its reference ----------------
          // first take the next own score tile out of TMEM: it needs no reference yet, and the tensor pipe gets the buffer back
          if (j + 1 < KT && !have_s) load_scores();
          const uint32_t slot = rc & 1u;
          if (ew == 0 && lane == 0) mbar_expect_tx(&hdr_bar[slot], F7_BM * 4);
          mbar_wait(&hdr_bar[slot], (rc >> 1) & 1u);
          tr.ev(11, j);
          const float nA = hdr_x[slot * F7_BM + rA], nB = hdr_x[slot * F7_BM + rB];
          if (j > 0) {
            const bool upA = nA != refA, upB = nB != refB;
            if (__any_sync(0xffffffffu, upA || upB)) {
              const float fA = upA ? ex2_approx(refA - nA) : 1.0f, fB = upB ? ex2_approx(refB - nB) : 1.0f;
              lA2.x *= fA; lA2.y *= fA; lB2.x *= fB; lB2.y *= fB;
              rescale_o(fA, fB);
            }
          }
          refA = nA; refB = nB;
          __syncwarp();
          if (lane == 0) mbar_arrive(&accept[slot]);
          ++rc;
          continue;
        }
        // ---------------- an own tile: scores -> reference decision -> probabilities ----------------
        if (!have_s) load_scores();
        have_s = false;
        // tile maximum (raw accumulators; alpha2 > 0 is applied once)
        const int c0 = j * F7_BN + q2;                            // key column of r[0]
        const bool full = j * F7_BN + F7_BN <= p.T;
        float mA = -INFINITY, mB = -INFINITY;
        if (full) {
#pragma unroll
          for (int kb = 0; kb < 8; ++kb) {
            mA = fmaxf(mA, fmaxf(fmaxf(__uint_as_float(s0[4 * kb]), __uint_as_float(s0[4 * kb + 1])),
                                 fmaxf(__uint_as_float(s1[4 * kb]), __uint_as_float(s1[4 * kb + 1]))));
            mB = fmaxf(mB, fmaxf(fmaxf(__uint_as_float(s0[4 * kb + 2]), __uint_as_float(s0[4 * kb + 3])),
                                 fmaxf(__uint_as_float(s1[4 * kb + 2]), __uint_as_float(s1[4 * kb + 3]))));
          }
        } else {
#pragma unroll
          for (int kb = 0; kb < 8; ++kb) {
            const int cc = c0 + kb * 8;
            if (cc < p.T) { mA = fmaxf(mA, __uint_as_float(s0[4 * kb])); mB = fmaxf(mB, __uint_as_float(s0[4 * kb + 2])); }
            if (cc + 1 < p.T) { mA = fmaxf(mA, __uint_as_float(s0[4 * kb + 1])); mB = fmaxf(mB, __uint_as_float(s0[4 * kb + 3])); }
            if (cc + 64 < p.T) { mA = fmaxf(mA, __uint_as_float(s1[4 * kb])); mB = fmaxf(mB, __uint_as_float(s1[4 * kb + 2])); }
            if (cc + 65 < p.T) { mA = fmaxf(mA, __uint_as_float(s1[4 * kb + 1])); mB = fmaxf(mB, __uint_as_float(s1[4 * kb + 3])); }
          }
        }
        mA = quad_max(mA) * p.alpha2;   // every key tile has at least one valid key (KT = ceil(T / 128)): finite
        mB = quad_max(mB) * p.alpha2;
        // lazy rescale: tile 0 fixes the reference; later it only moves when the tile's maximum exceeds it by more than 2^TAU
        const bool upA = j > 0 && (mA > refA + F7_TAU || (p.force_rescale && mA > refA));
        const bool upB = j > 0 && (mB > refB + F7_TAU || (p.force_rescale && mB > refB));
        const float nA = (j == 0 || upA) ? mA : refA, nB = (j == 0 || upB) ? mB : refB;
        if (writer) {   // tell the peer first: its own next tile (and its accumulator) waits for this decision
          const uint32_t slot = oc & 1u;
          const uint32_t dsta = mapa_shared(smem_u32(hdr_x + slot * F7_BM + rA), peer);
          const uint32_t barr = mapa_shared(smem_u32(&hdr_bar[slot]), peer);
          st_async_f32(dsta, nA, barr);
          st_async_f32(dsta + 8 * 4, nB, barr);
        }
        tr.ev(12, j);
        if (__any_sync(0xffffffffu, upA || upB)) {
          const float fA = upA ? ex2_approx(refA - nA) : 1.0f, fB = upB ? ex2_approx(refB - nB) : 1.0f;
          lA2.x *= fA; lA2.y *= fA; lB2.x *= fB; lB2.y *= fB;
          rescale_o(fA, fB);
        }
        refA = nA; refB = nB;
        // P = exp2(alpha2 s - ref) -> shared memory (K-major A operand, 128-B swizzle), row sums
        mbar_wait(p_free, (oc & 1u) ^ 1u);   // both CTAs' P.V of the previous own tile have retired (and the copy with them)
        tr.ev(13, j);
#pragma unroll
        for (int cb = 0; cb < 2; ++cb) {
          const uint32_t(&r)[32] = cb == 0 ? s0 : s1;
          uint8_t* pa = p_own + cb * (F7_BM * 128) + rA * 128 + q2 * 2;
          uint8_t* pbp = p_own + cb * (F7_BM * 128) + rB * 128 + q2 * 2;
#pragma unroll
          for (int kb = 0; kb < 8; ++kb) {
            float2 eA = make_float2(ex2_approx(fmaf(__uint_as_float(r[4 * kb]), p.alpha2, -refA)),
                                    ex2_approx(fmaf(__uint_as_float(r[4 * kb + 1]), p.alpha2, -refA)));
            float2 eB = make_float2(ex2_approx(fmaf(__uint_as_float(r[4 * kb + 2]), p.alpha2, -refB)),
                                    ex2_approx(fmaf(__uint_as_float(r[4 * kb + 3]), p.alpha2, -refB)));
            if (!full) {   // keys past the sequence contribute nothing
              const int cc = c0 + cb * 64 + kb * 8;
              if (cc >= p.T) { eA.x = 0.f; eB.x = 0.f; }
              if (cc + 1 >= p.T) { eA.y = 0.f; eB.y = 0.f; }
            }
            lA2 = __fadd2_rn(lA2, eA);
            lB2 = __fadd2_rn(lB2, eB);
            *reinterpret_cast<uint32_t*>(pa + ((kb ^ (rA & 7)) << 4)) = pack_bf16x2(eA.x, eA.y);
            *reinterpret_cast<uint32_t*>(pbp + ((kb ^ (rB & 7)) << 4)) = pack_bf16x2(eB.x, eB.y);
          }
        }
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) mbar_arrive(p_full);
        tr.ev(14, j);
        ++oc;
      }
      // ---------------- total row sums: own partial + the peer's (both relative to the final references) ----------------
      float lA = quad_sum(lA2.x + lA2.y), lB = quad_sum(lB2.x + lB2.y);
      const uint32_t par = it & 1u;
      if (ew == 0 && lane == 0) mbar_expect_tx(&l_bar[par], F7_BM * 4);
      if (writer) {
        const uint32_t dsta = mapa_shared(smem_u32(l_x + par * F7_BM + rA), peer);
        const uint32_t barr = mapa_shared(smem_u32(&l_bar[par]), peer);
        st_async_f32(dsta, lA, barr);
        st_async_f32(dsta + 8 * 4, lB, barr);
      }
      // ---------------- epilogue sweep 1: h <- O / l + h (fp32, in place), row statistics, h kept in TMEM ----------------
      float4 f0[8], f1[8];   // residual of two 64-column chunks in flight (rows A: [0, 4), rows B: [4, 8))
      auto load_res = [&](int cb, float4(&f)[8]) {
#pragma unroll
        for (int jj = 0; jj < 4; ++jj) {
          f[jj] = okA ? *reinterpret_cast<const float4*>(hA + cb * 64 + jj * 16) : make_float4(0.f, 0.f, 0.f, 0.f);
          f[4 + jj] = okB ? *reinterpret_cast<const float4*>(hB + cb * 64 + jj * 16) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
      };
      load_res(0, f0);       // both requested before the waits below: their L2 latency hides behind the exchange / the last P.V
      load_res(1, f1);
      mbar_wait(&l_bar[par], (it >> 1) & 1u);
      tr.ev(15, it);
      lA += l_x[par * F7_BM + rA];
      lB += l_x[par * F7_BM + rB];
      const float iA = 1.0f / lA, iB = 1.0f / lB;
      mbar_wait(o_full, it & 1u);
      tcgen05_fence_after();
      tr.ev(16, it);
      // row statistics of this thread's 96 values of rows A and B: sums of v - K and (v - K)^2, K = its first value (common.cuh)
      float smA = 0.f, sqA = 0.f, smB = 0.f, sqB = 0.f, kA = 0.f, kB = 0.f;
      auto sweep1 = [&](int cb, const float4(&f)[8]) {
        uint32_t o[32];
        tmem_ld_16x64(t_lane + cb * 64, o);
        tmem_ld_wait();
#pragma unroll
        for (int jj = 0; jj < 4; ++jj) {   // accumulator 8-column blocks 2 jj, 2 jj + 1 = output columns 16 jj + 4 q .. + 3
          const int k0 = 2 * jj, k1 = 2 * jj + 1;
          float4 vA, vB;
          vA.x = fmaf(iA, __uint_as_float(o[4 * k0]), f[jj].x);
          vA.y = fmaf(iA, __uint_as_float(o[4 * k0 + 1]), f[jj].y);
          vA.z = fmaf(iA, __uint_as_float(o[4 * k1]), f[jj].z);
          vA.w = fmaf(iA, __uint_as_float(o[4 * k1 + 1]), f[jj].w);
          vB.x = fmaf(iB, __uint_as_float(o[4 * k0 + 2]), f[4 + jj].x);
          vB.y = fmaf(iB, __uint_as_float(o[4 * k0 + 3]), f[4 + jj].y);
          vB.z = fmaf(iB, __uint_as_float(o[4 * k1 + 2]), f[4 + jj].z);
          vB.w = fmaf(iB, __uint_as_float(o[4 * k1 + 3]), f[4 + jj].w);
          if (okA) *reinterpret_cast<float4*>(hA + cb * 64 + jj * 16) = vA;
          if (okB) *reinterpret_cast<float4*>(hB + cb * 64 + jj * 16) = vB;
          if (cb == 0 && jj == 0) { kA = vA.x; kB = vB.x; }
          const float4 dA = make_float4(vA.x - kA, vA.y - kA, vA.z - kA, vA.w - kA);
          const float4 dB = make_float4(vB.x - kB, vB.y - kB, vB.z - kB, vB.w - kB);
          smA += (dA.x + dA.y) + (dA.z + dA.w);
          sqA = fmaf(dA.x, dA.x, fmaf(dA.y, dA.y, fmaf(dA.z, dA.z, fmaf(dA.w, dA.w, sqA))));
          smB += (dB.x + dB.y) + (dB.z + dB.w);
          sqB = fmaf(dB.x, dB.x, fmaf(dB.y, dB.y, fmaf(dB.z, dB.z, fmaf(dB.w, dB.w, sqB))));
          o[4 * k0] = __float_as_uint(vA.x); o[4 * k0 + 1] = __float_as_uint(vA.y);
          o[4 * k1] = __float_as_uint(vA.z); o[4 * k1 + 1] = __float_as_uint(vA.w);
          o[4 * k0 + 2] = __float_as_uint(vB.x); o[4 * k0 + 3] = __float_as_uint(vB.y);
          o[4 * k1 + 2] = __float_as_uint(vB.z); o[4 * k1 + 3] = __float_as_uint(vB.w);
        }
        if (p.u_out != nullptr) tmem_st_16x64(t_lane + cb * 64, o);
      };
#pragma unroll 1
      for (int cb = 0; cb < F7_DH / 64; cb += 2) {
        sweep1(cb, f0);
        if (cb + 2 < F7_DH / 64) load_res(cb + 2, f0);
        sweep1(cb + 1, f1);
        if (cb + 3 < F7_DH / 64) load_res(cb + 3, f1);
      }
      tr.ev(17, it);
      if (p.u_out != nullptr) {
        tmem_st_wait();
        // ---------------- LayerNorm statistics: this CTA has 384 of the 768 columns; the peer has the rest ----------------
        // partials (mean, M2) of this CTA's 384 columns; the peer's are merged in below
        const float2 pA = ln_quad_merge(ln_partial(kA, smA, sqA, 1.0f / (F7_DH / 4)), F7_DH / 4);
        const float2 pB = ln_quad_merge(ln_partial(kB, smB, sqB, 1.0f / (F7_DH / 4)), F7_DH / 4);
        if (ew == 0 && lane == 0) mbar_expect_tx(&stat_bar[par], F7_BM * 8);
        if (writer) {
          const uint32_t slot = mapa_shared(smem_u32(stat_x + (par * F7_BM + rA) * 2), peer);
          const uint32_t bar = mapa_shared(smem_u32(&stat_bar[par]), peer);
          st_async_f32(slot, pA.x, bar);
          st_async_f32(slot + 4, pA.y, bar);
          st_async_f32(slot + 8 * 8, pB.x, bar);
          st_async_f32(slot + 8 * 8 + 4, pB.y, bar);
        }
        mbar_wait(&stat_bar[par], (it >> 1) & 1u);
        tr.ev(18, it);
        const float2 xA = *reinterpret_cast<const float2*>(stat_x + (par * F7_BM + rA) * 2);
        const float2 xB = *reinterpret_cast<const float2*>(stat_x + (par * F7_BM + rB) * 2);
        const float inv_h = 1.0f / static_cast<float>(F7_D);
        const float2 stA = ln_merge(pA, xA, F7_DH), stB = ln_merge(pB, xB, F7_DH);
        const float meanA = stA.x, meanB = stB.x;
        const float rsA = rsqrtf(fmaxf(stA.y, 0.f) * inv_h + 1e-5f);
        const float rsB = rsqrtf(fmaxf(stB.y, 0.f) * inv_h + 1e-5f);
        // ---------------- sweep 2: u = LayerNorm(h) gamma + beta, bf16, 8-byte stores ----------------
        bf16* uA = p.u_out + growA * F7_D + col_half + q * 4;
        bf16* uB = uA + 8 * F7_D;
        const float* gp = p.gamma + col_half + q * 4;
        const float* bp = p.beta + col_half + q * 4;
#pragma unroll 1
        for (int cb = 0; cb < F7_DH / 64; ++cb) {
          uint32_t o[32];
          tmem_ld_16x64(t_lane + cb * 64, o);
          float4 gm[4], bt[4];
#pragma unroll
          for (int jj = 0; jj < 4; ++jj) {
            gm[jj] = __ldg(reinterpret_cast<const float4*>(gp + cb * 64 + jj * 16));
            bt[jj] = __ldg(reinterpret_cast<const float4*>(bp + cb * 64 + jj * 16));
          }
          tmem_ld_wait();
#pragma unroll
          for (int jj = 0; jj < 4; ++jj) {
            const int k0 = 2 * jj, k1 = 2 * jj + 1;
            uint2 wA, wB;
            wA.x = pack_bf16x2(fmaf((__uint_as_float(o[4 * k0]) - meanA) * rsA, gm[jj].x, bt[jj].x),
                               fmaf((__uint_as_float(o[4 * k0 + 1]) - meanA) * rsA, gm[jj].y, bt[jj].y));
            wA.y = pack_bf16x2(fmaf((__uint_as_float(o[4 * k1]) - meanA) * rsA, gm[jj].z, bt[jj].z),
                               fmaf((__uint_as_float(o[4 * k1 + 1]) - meanA) * rsA, gm[jj].w, bt[jj].w));
            wB.x = pack_bf16x2(fmaf((__uint_as_float(o[4 * k0 + 2]) - meanB) * rsB, gm[jj].x, bt[jj].x),
                               fmaf((__uint_as_float(o[4 * k0 + 3]) - meanB) * rsB, gm[jj].y, bt[jj].y));
            wB.y = pack_bf16x2(fmaf((__uint_as_float(o[4 * k1 + 2]) - meanB) * rsB, gm[jj].z, bt[jj].z),
                               fmaf((__uint_as_float(o[4 * k1 + 3]) - meanB) * rsB, gm[jj].w, bt[jj].w));
            if (okA) *reinterpret_cast<uint2*>(uA + cb * 64 + jj * 16) = wA;
            if (okB) *reinterpret_cast<uint2*>(uB + cb * 64 + jj * 16) = wB;
          }
        }
      }
      tcgen05_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(o_empty);
      tr.ev(19, it);
    }
  } else {
    regs_shrink_ctrl();  // warp 3 idles; the whole warpgroup has to execute the setmaxnreg
  }

  __syncwarp();
  tcgen05_fence_before();
  __syncthreads();
  cluster_sync_all();   // nobody leaves while the peer may still write into this CTA / signal its barriers
  if (warp == 2) {
    tcgen05_fence_after();
    tmem_dealloc<F7_TMEM_COLS>(tmem_base);
  }
}

}  // namespace

bool flash768_supported(int H, int heads, int T) { return heads == 1 && H == F7_D && T >= 1; }

// four-CTA clusters (two cta_group::2 pairs, K / V loaded once per pair) when 256-row query tiles fit the sequence length
bool flash768_picks_quad(int T) {
  return g_opt.flash768_quad != 1 && T >= 1 && (g_opt.flash768_quad == 2 || flash768_quad_preferred(T)) && flash768_quad_schedulable();
}

int launch_flash768(const Flash768Params& q, cudaStream_t st) {
  if (flash768_picks_quad(q.T)) return launch_flash768_quad(q, st);
  DITTO_TRY(tc_gemm_init());
  DITTO_REQUIRE(q.const_flag == nullptr, DITTO_E_UNSUPPORTED, "flash768: constant-text rows need the four-CTA kernel");
  DITTO_REQUIRE(flash768_supported(q.H, 1, q.T), DITTO_E_UNSUPPORTED, "flash768: single head of 768 only");
  DITTO_REQUIRE(q.qkv && q.h && q.n_seq >= 1 && q.ld % 8 == 0 && q.ld >= 3 * F7_D, DITTO_E_BADARG, "flash768: bad argument");
  DITTO_REQUIRE(q.u_out == nullptr || (q.gamma && q.beta), DITTO_E_BADARG, "flash768: LayerNorm output needs gamma and beta");
  DITTO_REQUIRE((reinterpret_cast<uintptr_t>(q.h) & 15) == 0 && (reinterpret_cast<uintptr_t>(q.u_out) & 7) == 0, DITTO_E_BADARG,
                "flash768: h must be 16-byte, u 8-byte aligned");
  DeviceState* ds = device_state();
  if (ds == nullptr) return DITTO_E_CUDA;
  DITTO_REQUIRE(ds->num_sms >= 2, DITTO_E_UNSUPPORTED, "flash768: needs an SM pair");
  if (!ds->f768_attr) {  // per device
    DITTO_CUDA(cudaFuncSetAttribute(flash_attn768_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, F7_SMEM_BYTES));
    ds->f768_attr = true;
  }
  TcOperand Q, K, V;
  Q.ptr = q.qkv; Q.rows = q.T; Q.cols = F7_D; Q.ld = q.ld; Q.s_outer = static_cast<int64_t>(q.T) * q.ld;
  K = Q; K.ptr = q.qkv + F7_D;
  V = Q; V.ptr = q.qkv + 2 * F7_D;
  CUtensorMap mq, mk, mv;
  DITTO_TRY(tc_make_map(&mq, Q, 1, q.n_seq, F7_BK, F7_BM));
  DITTO_TRY(tc_make_map(&mk, K, 1, q.n_seq, F7_BK, F7_BN));
  DITTO_TRY(tc_make_map(&mv, V, 1, q.n_seq, 64, F7_VKEYS));
  F7Dev p;
  p.n_seq = static_cast<int>(q.n_seq); p.T = q.T;
  p.m_tiles = static_cast<int>(ceil_div(q.T, F7_BM));
  p.k_tiles = static_cast<int>(ceil_div(q.T, F7_BN));
  const int64_t items = static_cast<int64_t>(p.m_tiles) * q.n_seq;
  DITTO_REQUIRE(items < (1ll << 31), DITTO_E_UNSUPPORTED, "flash768: too many work items");
  p.num_items = static_cast<int>(items);
  p.alpha2 = q.alpha * 1.4426950408889634f;
  p.h = q.h; p.gamma = q.gamma; p.beta = q.beta; p.u_out = q.u_out;
  p.force_rescale = q.force_rescale ? 1 : 0;
  p.trace = DITTO_F7_TRACE ? tc_gemm_debug_counters() : nullptr;
  // algorithmic flops: 4 T^2 d per utterance (the second Q K^T of the cluster is not counted); bytes: q, k, v read once, h
  // read + written, u written
  const double rows = static_cast<double>(q.n_seq) * q.T;
  ProfScope prof(q.tag, st, 4.0 * q.T * static_cast<double>(q.T) * F7_D * q.n_seq, rows * F7_D * (6.0 + 8.0 + (q.u_out ? 2.0 : 0.0)));
  const int clusters = static_cast<int>(std::min<int64_t>(ds->num_sms / 2, items));
  flash_attn768_kernel<<<2 * clusters, F7_THREADS, F7_SMEM_BYTES, st>>>(mq, mk, mv, p);
  DITTO_LAUNCH_CHECK();
  return 0;
}

}  // namespace ditto
