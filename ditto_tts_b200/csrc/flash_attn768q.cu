// Flash-style self-attention for the single head of 768 + residual + norm2 -- FOUR-CTA cluster version of flash_attn768.cu
// (same arithmetic, same softmax-reference protocol; reference: src/components/DiT.py:117-139, :143).
//
// Why: flash_attn768_kernel is bound by the L2 -> SM operand feed, not by the tensor pipe (ncu, C2: tensor pipe 29 % busy,
// 33 B/clk/SM delivered): per 128 query rows it streams Q six times (once per key tile), K once and V once = 3.4 MiB for
// 18 k tensor cycles.  Here a cluster covers 256 query rows with TWO cta_group::2 pairs:
//
//     rank = 2 c + a      a = row group (query rows 128 a .. 128 a + 127 of the item; a = 0 is the pair leader)
//                         c = output-column half [384 c, 384 c + 384) and parity of the key tiles whose scores the pair owns
//
// Pair c issues UMMA 256 x N x 16 over both SMs: every K chunk and every V block is loaded ONCE PER PAIR (each CTA fetches
// half of the B operand), so the K / V traffic per query row is halved; Q (the A operand) stays per CTA.  Per 128 query
// rows: 2.2 MiB instead of 3.4.  Everything else is the protocol of flash_attn768.cu with "the peer" = the CTA of the same
// row group in the other pair (rank ^ 2): score tiles split by key parity, bf16 probability tiles handed over by one
// 32 KiB DSMEM bulk copy, ONE softmax reference per row chained through st.async headers with lazy rescale, partial row
// sums and LayerNorm statistics exchanged the same way.
//
// Barriers.  The MMA issuer exists only in the pair leader, so everything it waits for lives in the LEADER's shared memory
// and is signalled by both CTAs of the pair (remote mbarrier.arrive.release.cluster); everything it signals is a
// tcgen05.commit multicast to both CTAs.  Per CTA (384 threads):
//   warp 0   TMA producer: ring of six 24 KiB slots in the order the issuer consumes them
//            score stage  Q[128 rows x 64] + K[64 keys x 64]  (this CTA's half of the 128-key chunk), 12 per own key tile
//            P.V stage    V[64 keys x 192 columns] as three MN-major [64 x 64] boxes (this CTA's part of the pair's 384
//                         output columns: 128 of the N = 256 block + 64 of the N = 128 block), 2 per key tile
//   warp 1   MMA issuer (leader CTA only)
//   warp 2   probability courier: own tile written -> bulk copy into the landing buffer of rank ^ 2
//   warp 3   landing relay: the peer's tile has landed in THIS CTA -> arrive on the leader's land_ready
//   warps 4-11  softmax / reference chain / epilogue, exactly as in flash_attn768.cu
// TMEM per CTA: [0, 384) O (own 128 rows x the pair's 384 columns), [384, 512) S (own 128 rows x 128 keys).
#include "common.cuh"
#include "kernels.cuh"

namespace ditto {
namespace {

constexpr int Q7_THREADS = 384;
constexpr int Q7_EPI_WARP0 = 4;
constexpr int Q7_EPI_WARPS = 8;
constexpr int Q7_BM = 128, Q7_BN = 128, Q7_BK = 64;
constexpr int Q7_D = 768;
constexpr int Q7_DH = Q7_D / 2;       // output columns per pair
constexpr int Q7_KCH = Q7_D / Q7_BK;  // 12 head-dim chunks per score tile
constexpr int Q7_VKEYS = 64;          // keys per P.V stage
constexpr int Q7_VST = Q7_BN / Q7_VKEYS;   // 2 P.V stages per key tile
constexpr int Q7_VBOX = Q7_VKEYS * 128;    // 8 KiB: [64 keys x 64 n] bf16, n contiguous
constexpr int Q7_STAGES = 6;
constexpr int Q7_Q_BYTES = Q7_BM * Q7_BK * 2;        // 16 KiB
constexpr int Q7_K_BYTES = (Q7_BN / 2) * Q7_BK * 2;  // 8 KiB: this CTA's 64 keys of the chunk
constexpr int Q7_V_BYTES = 3 * Q7_VBOX;              // 24 KiB
constexpr int Q7_STAGE_BYTES = 24576;
static_assert(Q7_Q_BYTES + Q7_K_BYTES == Q7_STAGE_BYTES && Q7_V_BYTES == Q7_STAGE_BYTES, "both stage kinds fill a ring slot");
constexpr int Q7_P_BYTES = Q7_BM * Q7_BN * 2;   // 32 KiB (two K-major 64-key sub-tiles)
constexpr int Q7_OFF_POWN = Q7_STAGES * Q7_STAGE_BYTES;
constexpr int Q7_OFF_PLAND = Q7_OFF_POWN + Q7_P_BYTES;
constexpr int Q7_OFF_BAR = Q7_OFF_PLAND + Q7_P_BYTES;
constexpr int Q7_BAR_BYTES = 512;
constexpr int Q7_OFF_XCH = Q7_OFF_BAR + Q7_BAR_BYTES;
constexpr int Q7_XCH_HDR = 0, Q7_XCH_L = 2 * Q7_BM * 4, Q7_XCH_STAT = 4 * Q7_BM * 4;
constexpr int Q7_XCH_BYTES = 4 * Q7_BM * 4 + 2 * Q7_BM * 8;
constexpr int Q7_OFF_CROW = Q7_OFF_XCH + Q7_XCH_BYTES;   // [2][384] fp32: a constant-text item's row, this CTA's column half
constexpr int Q7_SMEM_BYTES = Q7_OFF_CROW + 2 * Q7_DH * 4 + 1024;
static_assert(Q7_SMEM_BYTES <= 232448, "exceeds the 227 KiB shared memory of an sm_100 CTA");
static_assert(Q7_OFF_POWN % 1024 == 0, "operand buffers must be 1024-byte aligned (128-B swizzle atoms)");
constexpr int Q7_TMEM_COLS = 512;
constexpr int Q7_S_COL = Q7_DH;       // 384
constexpr float Q7_TAU = 8.0f;

struct Q7Dev {
  unsigned long long* trace;
  int n_seq, T;
  int Tk;                             // keys per sequence (self-attention: T; cross-attention: text tokens S)
  int m_tiles, k_tiles, num_items;    // m_tiles: 256-row query tiles per utterance
  const float* kbias; long long kb_seq;   // CROSS: additive score bias per key [n_seq, kb_seq] (already scaled; folded k-bias)
  const float* obias;                 // CROSS: output bias [768] (cross_attn.out_proj.bias); KONST: constant rows [n_seq][768]
  float alpha2;
  float* h;
  const float* gamma; const float* beta;
  bf16* u_out;
  int force_rescale;
  int dbg;   // always 0: kept only because removing its tests below makes ptxas spill more in the epilogue (slower)
  // constant-text sequences (Flash768Params::const_flag); self-attention: norm3, which replaces norm2 for them.  (Few new
  // fields, at the end: a larger parameter block costs the plain self-attention kernel spills.)
  const uint8_t* const_flag; const float* gamma_c; const float* beta_c;
};

// first item at or after `item` (stepping over the grid) that this launch processes: the cross-attention kernel skips the
// items of constant-text sequences, whose output the self-attention kernel has already added.  Every role walks the same
// items, so the barrier phases (counted per processed item) agree.
template <bool CROSS>
__device__ __forceinline__ int q7_next_item(const Q7Dev& p, int item, int step) {
  if (CROSS && p.const_flag != nullptr)
    while (item < p.num_items && __ldg(p.const_flag + item / p.m_tiles) != 0) item += step;
  return item;
}

// CROSS = false: self-attention (q, k, v = column thirds of the QKV GEMM output).  CROSS = true: the folded cross-attention
// of a single-head model with 64 < S <= 256 text tokens (DiT.py:141-151 -> torch MHA math path):
//   h <- h + softmax(alpha u (K Wq)^T + kbias) (V Wo^T) + bo ;  u <- LayerNorm(h) gamma3 + beta3
// q = u (norm2 output, overwritten in place with norm3's), k = K-fold [S, 768], v = V-fold [Sp, 768] in the perm4 column order.
// KONST (self-attention only): the launch carries constant-text sequences (Q7Dev::const_flag); a separate instantiation, so
// that the plain self-attention kernel keeps its registers.
template <bool CROSS, bool KONST = false>
__global__ void __launch_bounds__(Q7_THREADS, 1)
    flash_attn768q_kernel(const __grid_constant__ CUtensorMap tmap_q, const __grid_constant__ CUtensorMap tmap_k,
                          const __grid_constant__ CUtensorMap tmap_v, const Q7Dev p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw_addr = smem_u32(smem_raw);
  uint8_t* smem = smem_raw + ((1024u - (raw_addr & 1023u)) & 1023u);
  uint8_t* p_own = smem + Q7_OFF_POWN;
  uint8_t* p_land = smem + Q7_OFF_PLAND;
  // (L) = the pair leader's copy is the one in use, both CTAs of the pair arrive on it; (B) = signalled in both CTAs by a
  // multicast commit, each CTA waits on its own copy; (own) = CTA-local
  uint64_t* ring_full = reinterpret_cast<uint64_t*>(smem + Q7_OFF_BAR);   // (L) operands of both CTAs landed
  uint64_t* ring_empty = ring_full + Q7_STAGES;  // (B) slot consumed
  uint64_t* s_full = ring_empty + Q7_STAGES;     // (B) score tile complete
  uint64_t* s_empty = s_full + 1;                // (L) score tile read by the softmax warps of both CTAs
  uint64_t* p_full = s_empty + 1;                // (L) own probabilities written in both CTAs
  uint64_t* p_ready = p_full + 1;                // (own) own probabilities written here                    (-> courier)
  uint64_t* p_free = p_ready + 1;                // (B) own buffer reusable: P.V of BOTH pairs retired (2 commits)
  uint64_t* land_full = p_free + 1;              // (own) peer's probabilities landed here (complete_tx)   (-> relay)
  uint64_t* land_ready = land_full + 1;          // (L) ... in both CTAs of the pair (2 arrivals)
  uint64_t* accept = land_ready + 1;             // (L) [2] reference of a peer tile adopted by both CTAs
  uint64_t* pv_done = accept + 2;                // (B) [4] P.V of tile (global index mod 4) retired
  uint64_t* o_full = pv_done + 4;                // (B) O complete
  uint64_t* o_empty = o_full + 1;                // (L) O drained in both CTAs
  uint64_t* hdr_bar = o_empty + 1;               // (own) [2] peer's reference decision landed (st.async complete_tx)
  uint64_t* l_bar = hdr_bar + 2;                 // (own) [2] peer's partial row sums landed
  uint64_t* stat_bar = l_bar + 2;                // (own) [2] peer's LayerNorm partials landed
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(stat_bar + 2);
  static_assert((2 * Q7_STAGES + 21) * 8 + 4 <= Q7_BAR_BYTES, "barrier block too small");
  float* hdr_x = reinterpret_cast<float*>(smem + Q7_OFF_XCH + Q7_XCH_HDR);     // [2][128]
  float* l_x = reinterpret_cast<float*>(smem + Q7_OFF_XCH + Q7_XCH_L);         // [2][128]
  float* stat_x = reinterpret_cast<float*>(smem + Q7_OFF_XCH + Q7_XCH_STAT);   // [2][128][2]

  const int warp = warp_id_uniform();
  const int lane = threadIdx.x & 31;
  const uint32_t rank = __shfl_sync(0xffffffffu, cluster_ctarank(), 0);
  const int a = static_cast<int>(rank & 1u);        // row group; 0 = pair leader
  const int c = static_cast<int>(rank >> 1);        // column half / key-tile parity
  const uint32_t peer = rank ^ 2u;                  // same rows, other column half
  const int num_clusters = gridDim.x >> 2;
  const int first = blockIdx.x >> 2;
  const int KT = p.k_tiles;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmap_q);
    tma_prefetch_desc(&tmap_k);
    tma_prefetch_desc(&tmap_v);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < Q7_STAGES; ++s) { mbar_init(&ring_full[s], 1); mbar_init(&ring_empty[s], 1); }
    mbar_init(s_full, 1);
    mbar_init(s_empty, 2 * Q7_EPI_WARPS);
    mbar_init(p_full, 2 * Q7_EPI_WARPS);
    mbar_init(p_ready, Q7_EPI_WARPS);
    mbar_init(p_free, 2);
    mbar_init(land_full, 1);
    mbar_init(land_ready, 2);
    mbar_init(&accept[0], 2 * Q7_EPI_WARPS);
    mbar_init(&accept[1], 2 * Q7_EPI_WARPS);
    for (int s = 0; s < 4; ++s) mbar_init(&pv_done[s], 1);
    mbar_init(o_full, 1);
    mbar_init(o_empty, 2 * Q7_EPI_WARPS);
    for (int s = 0; s < 2; ++s) { mbar_init(&hdr_bar[s], 1); mbar_init(&l_bar[s], 1); mbar_init(&stat_bar[s], 1); }
    fence_barrier_init();
  }
  if (warp == 2) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_ptr)), "n"(Q7_TMEM_COLS) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
  }
  __syncwarp();
  tcgen05_fence_before();
  __syncthreads();
  cluster_sync_all();   // every CTA's barriers exist and TMEM is allocated on all four SMs
  tcgen05_fence_after();
  const uint32_t tmem_base = *tmem_ptr;
  if ((p.dbg >> 8) != 0 && (first & 1)) {   // timing experiment: odd clusters start late (units of 2048 clocks)
    const long long t_go = clock64() + (static_cast<long long>(p.dbg >> 8) << 11);
    while (clock64() < t_go) {}
  }
  const long long t_sync = DITTO_F7_TRACE ? clock64() : 0;

  if (warp == 0) {
    // =========================== TMA producer ===========================
    regs_shrink_ctrl();
    const bool leader = elect_one();
    F7Tr tr; tr.init(p.trace, rank, 2, first == 0 && leader, t_sync);
    int stage = 0;
    uint32_t phase = 0;
    for (int item = q7_next_item<CROSS>(p, first, num_clusters); item < p.num_items; item = q7_next_item<CROSS>(p, item + num_clusters, num_clusters)) {
      const int qt = item % p.m_tiles, seq = item / p.m_tiles;
      const int q_row0 = qt * (2 * Q7_BM) + a * Q7_BM;
      auto load_s = [&](int j) {
#pragma unroll 1
        for (int ch = 0; ch < Q7_KCH; ++ch) {
          mbar_wait(&ring_empty[stage], phase ^ 1u);
          if (leader) {
            uint8_t* sb = smem + stage * Q7_STAGE_BYTES;
            if (a == 0) mbar_expect_tx(&ring_full[stage], 2 * Q7_STAGE_BYTES);
            tma_load_4d_2sm(&tmap_q, &ring_full[stage], sb, ch * Q7_BK, q_row0, 0, seq);   // rows >= T: zero-filled
            tma_load_4d_2sm(&tmap_k, &ring_full[stage], sb + Q7_Q_BYTES, ch * Q7_BK, j * Q7_BN + a * (Q7_BN / 2), 0, seq);
          }
          __syncwarp();
          if (++stage == Q7_STAGES) { stage = 0; phase ^= 1u; }
        }
        tr.ev(30, j);
      };
      auto load_v = [&](int j) {
#pragma unroll 1
        for (int s = 0; s < Q7_VST; ++s) {
          mbar_wait(&ring_empty[stage], phase ^ 1u);
          if (leader) {
            uint8_t* sb = smem + stage * Q7_STAGE_BYTES;
            const int key0 = j * Q7_BN + s * Q7_VKEYS;
            if (a == 0) mbar_expect_tx(&ring_full[stage], 2 * Q7_STAGE_BYTES);
            // this CTA's half of the pair's B operand: 128 of the first 256 output columns, 64 of the last 128
            tma_load_4d_2sm(&tmap_v, &ring_full[stage], sb, c * Q7_DH + a * 128, key0, 0, seq);
            tma_load_4d_2sm(&tmap_v, &ring_full[stage], sb + Q7_VBOX, c * Q7_DH + a * 128 + 64, key0, 0, seq);
            tma_load_4d_2sm(&tmap_v, &ring_full[stage], sb + 2 * Q7_VBOX, c * Q7_DH + 256 + a * 64, key0, 0, seq);
          }
          __syncwarp();
          if (++stage == Q7_STAGES) { stage = 0; phase ^= 1u; }
        }
        tr.ev(31, j);
      };
      if (c < KT) load_s(c);
      for (int j = 0; j < KT; ++j) {
        if ((j & 1) == c && j + 2 < KT) load_s(j + 2);
        load_v(j);
      }
    }
  } else if (warp == 1) {
    // =========================== MMA issuer (pair leader only) ===========================
    regs_shrink_ctrl();
    if (a == 0) {
      const bool leader = elect_one();
      constexpr uint32_t idesc_s = umma_idesc_bf16(2 * Q7_BM, Q7_BN, false, false);
      constexpr uint32_t idesc_o256 = umma_idesc_bf16(2 * Q7_BM, 256, false, true);
      constexpr uint32_t idesc_o128 = umma_idesc_bf16(2 * Q7_BM, 128, false, true);
      const uint64_t dk0 = umma_smem_desc(smem_u32(smem), 16, 1024);          // K-major operands (Q, K, P)
      const uint64_t dv0 = umma_smem_desc(smem_u32(smem), Q7_VBOX, 1024);     // MN-major V: 8 KiB between 64-column boxes
      constexpr uint64_t kToPOwn = Q7_OFF_POWN >> 4, kToPLand = Q7_OFF_PLAND >> 4;
      const uint16_t own_mask = static_cast<uint16_t>(3u << (2 * c)), peer_mask = static_cast<uint16_t>(3u << (2 * (c ^ 1)));
      int stage = 0;
      uint32_t phase = 0;
      uint32_t it = 0, sc = 0, oc = 0, rc = 0, pvi = 0;
      F7Tr tr; tr.init(p.trace, rank, 0, first == 0 && leader, t_sync);
      auto issue_s = [&]() {
        mbar_wait(s_empty, (sc & 1u) ^ 1u);
        tcgen05_fence_after();
        tr.ev(1, sc);
        long long fw = 0;
#pragma unroll 1
        for (int ch = 0; ch < Q7_KCH; ++ch) {
          if (DITTO_F7_TRACE && tr.b) { const long long w0 = clock64(); mbar_wait(&ring_full[stage], phase); fw += clock64() - w0; }
          else mbar_wait(&ring_full[stage], phase);
          tcgen05_fence_after();
          if (leader) {
            const uint64_t so = static_cast<uint64_t>((stage * Q7_STAGE_BYTES) >> 4);
#pragma unroll
            for (int k = 0; k < Q7_BK / 16; ++k)
              umma_bf16_2sm(tmem_base + Q7_S_COL, dk0 + so + ((k * 32) >> 4), dk0 + so + ((Q7_Q_BYTES + k * 32) >> 4), idesc_s,
                            (ch | k) != 0 ? 1u : 0u);
            umma_commit_2sm_mc(&ring_empty[stage], own_mask);
          }
          __syncwarp();
          if (++stage == Q7_STAGES) { stage = 0; phase ^= 1u; }
        }
        if (leader) umma_commit_2sm_mc(s_full, own_mask);
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
          mbar_wait(land_ready, rc & 1u);                       // the peer pair's tile landed in both CTAs
          mbar_wait(&accept[rc & 1u], (rc >> 1) & 1u);          // ... and its reference has been adopted by both
        }
        if (j == 0) mbar_wait(o_empty, (it & 1u) ^ 1u);        // the previous item's O has been drained
        tcgen05_fence_after();
        tr.ev(3, j);
        long long fw = 0;
        const uint64_t dp = dk0 + (own ? kToPOwn : kToPLand);
#pragma unroll 1
        for (int s = 0; s < Q7_VST; ++s) {
          if (DITTO_F7_TRACE && tr.b) { const long long w0 = clock64(); mbar_wait(&ring_full[stage], phase); fw += clock64() - w0; }
          else mbar_wait(&ring_full[stage], phase);
          tcgen05_fence_after();
          if (leader) {
            const uint64_t so = static_cast<uint64_t>((stage * Q7_STAGE_BYTES) >> 4);
#pragma unroll
            for (int k = 0; k < Q7_VKEYS / 16; ++k) {
              const int key16 = s * (Q7_VKEYS / 16) + k;                 // 16-key step inside the 128-key tile
              const uint64_t da = dp + (((key16 >> 2) * (Q7_BM * 128) + (key16 & 3) * 32) >> 4);
              const uint32_t acc = (j | s | k) != 0 ? 1u : 0u;
              umma_bf16_2sm(tmem_base, da, dv0 + so + ((k * (16 * 128)) >> 4), idesc_o256, acc);
              umma_bf16_2sm(tmem_base + 256, da, dv0 + so + ((2 * Q7_VBOX + k * (16 * 128)) >> 4), idesc_o128, acc);
            }
            umma_commit_2sm_mc(&ring_empty[stage], own_mask);
          }
          __syncwarp();
          tr.ev(8 + s, j);
          if (++stage == Q7_STAGES) { stage = 0; phase ^= 1u; }
        }
        if (leader) {
          umma_commit_2sm_mc(&pv_done[pvi & 3u], own_mask);
          // the tile's buffers in its OWNER pair are reusable once both pairs' P.V have retired
          umma_commit_2sm_mc(p_free, own ? own_mask : peer_mask);
        }
        __syncwarp();
        tr.ev(4, j);
        tr.val(7, j, fw);
        if (own) ++oc; else ++rc;
        ++pvi;
      };
      for (int item = q7_next_item<CROSS>(p, first, num_clusters); item < p.num_items;
           item = q7_next_item<CROSS>(p, item + num_clusters, num_clusters), ++it) {
        if (c < KT) issue_s();
        for (int j = 0; j < KT; ++j) {
          if ((j & 1) == c && j + 2 < KT) issue_s();
          issue_pv(j);
        }
        if (leader) umma_commit_2sm_mc(o_full, own_mask);
        __syncwarp();
        tr.ev(5, it);
      }
    }
  } else if (warp == 2) {
    // =========================== probability courier ===========================
    regs_shrink_ctrl();
    const bool leader = elect_one();
    const uint32_t dst = mapa_shared(smem_u32(p_land), peer), src = smem_u32(p_own), bar = mapa_shared(smem_u32(land_full), peer);
    uint32_t oc = 0;
    for (int item = q7_next_item<CROSS>(p, first, num_clusters); item < p.num_items; item = q7_next_item<CROSS>(p, item + num_clusters, num_clusters))
      for (int j = c; j < KT; j += 2, ++oc) {
        mbar_wait(p_ready, oc & 1u);   // written + fence.proxy.async by this CTA's softmax warps; the peer's landing buffer is
        if (leader) bulk_copy_to_peer(dst, src, Q7_P_BYTES, bar);   // free: p_free (awaited before the tile was written)
        __syncwarp();                                                  // includes the peer pair's P.V of the previous tile
      }
  } else if (warp == 3) {
    // =========================== landing relay ===========================
    regs_shrink_ctrl();
    uint32_t rc = 0;
    for (int item = q7_next_item<CROSS>(p, first, num_clusters); item < p.num_items; item = q7_next_item<CROSS>(p, item + num_clusters, num_clusters))
      for (int j = c ^ 1; j < KT; j += 2, ++rc) {
        if (lane == 0) {
          mbar_expect_tx(land_full, Q7_P_BYTES);   // arm this tile's landing (the copy may already be on its way)
          mbar_wait(land_full, rc & 1u);
          mbar_arrive_leader(land_ready);
        }
        __syncwarp();
      }
  } else {
    // =========================== softmax + epilogue ===========================
    regs_grow_epi();
    const int ew = warp - Q7_EPI_WARP0;
    const int quarter = warp & 3, hsel = ew >> 2;
    const int g = lane >> 2, q = lane & 3, q2 = q * 2;
    const int trow = quarter * 32 + hsel * 16;
    const int rA = trow + g, rB = rA + 8;
    const uint32_t t_lane = tmem_base + (static_cast<uint32_t>(trow) << 16);
    const bool writer = q == 0;
    const int col_half = c * Q7_DH;
    uint32_t it = 0, sc = 0, oc = 0, rc = 0, pvc = 0;
    F7Tr tr; tr.init(p.trace, rank, 1, first == 0 && ew == 0 && lane == 0, t_sync);
    auto rescale_o = [&](float fA, float fB) {
      tr.ev(25, static_cast<int>(pvc));
      mbar_wait(&pv_done[(pvc - 1) & 3u], ((pvc - 1) >> 2) & 1u);
      tcgen05_fence_after();
#pragma unroll 1
      for (int cb = 0; cb < Q7_DH / 64; ++cb) {
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
    for (int item = q7_next_item<CROSS>(p, first, num_clusters); item < p.num_items;
         item = q7_next_item<CROSS>(p, item + num_clusters, num_clusters), ++it) {
      const int qt = item % p.m_tiles, seq = item / p.m_tiles;
      const int row0 = qt * (2 * Q7_BM) + a * Q7_BM;               // first row of this CTA inside the utterance
      // a constant-text sequence (warp-uniform, per item): sweep 1 adds its constant cross-attention output row the way
      // CROSS adds the output bias, sweep 2 applies norm3 instead of norm2
      const bool konst = KONST && __ldg(p.const_flag + seq) != 0;
      // the row goes to shared memory once per item (two buffers by item parity: a warp fills the next item's only after
      // every epilogue warp has passed this item's barrier, i.e. finished the previous item's sweep 1)
      float* crow = reinterpret_cast<float*>(smem + Q7_OFF_CROW) + (it & 1u) * Q7_DH;
      if (KONST) {
        if (konst)
          for (int i = ew * 32 + lane; i < Q7_DH / 4; i += Q7_EPI_WARPS * 32)
            reinterpret_cast<float4*>(crow)[i] = __ldg(reinterpret_cast<const float4*>(p.obias + seq * Q7_D + col_half) + i);
        asm volatile("bar.sync 1, %0;" ::"n"(Q7_EPI_WARPS * 32) : "memory");
      }
      const int lrowA = row0 + rA;
      const bool okA = lrowA < p.T, okB = lrowA + 8 < p.T;
      const long long growA = static_cast<long long>(seq) * p.T + lrowA;
      float* hA = p.h + growA * Q7_D + col_half + q * 4;
      float* hB = hA + 8 * Q7_D;
      // residual rows of this warp -> L2 while the tiles compute (16 rows x 384 columns = 192 lines of 128 B); issued after
      // the first own tile's probabilities are out, not before: the score tile of this item is already waiting
      auto prefetch_residual = [&]() {
        if (p.dbg & 16) return;
        for (int i = lane; i < 16 * (Q7_DH * 4 / 128); i += 32) {
          const int r = i / (Q7_DH * 4 / 128), l = i - r * (Q7_DH * 4 / 128);
          if (row0 + trow + r < p.T)
            prefetch_l2(p.h + (static_cast<long long>(seq) * p.T + row0 + trow + r) * Q7_D + col_half + l * 32);
        }
      };
      if (c >= KT) prefetch_residual();
      tr.ev(24, it);
      float refA = 0.f, refB = 0.f;
      float2 lA2 = make_float2(0.f, 0.f), lB2 = make_float2(0.f, 0.f);
      uint32_t s0[32], s1[32];
      bool have_s = false;
      auto load_scores = [&]() {
        mbar_wait(s_full, sc & 1u);
        tcgen05_fence_after();
        tmem_ld_16x64(t_lane + Q7_S_COL, s0);
        tmem_ld_16x64(t_lane + Q7_S_COL + 64, s1);
        tmem_ld_wait();
        tcgen05_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive_leader(s_empty);
        tr.ev(10, sc);
        ++sc;
        have_s = true;
      };
      for (int j = 0; j < KT; ++j, ++pvc) {
        if (pvc >= 4) mbar_wait(&pv_done[pvc & 3u], ((pvc >> 2) - 1) & 1u);
        tr.ev(20, j);
        if ((j & 1) != c) {
          // ---------------- a tile of the peer pair: adopt its reference ----------------
          if (j + 1 < KT && !have_s) load_scores();
          const uint32_t slot = rc & 1u;
          if (ew == 0 && lane == 0) mbar_expect_tx(&hdr_bar[slot], Q7_BM * 4);
          if (!(p.dbg & 1)) mbar_wait(&hdr_bar[slot], (rc >> 1) & 1u);
          tr.ev(11, j);
          const float nA = hdr_x[slot * Q7_BM + rA], nB = hdr_x[slot * Q7_BM + rB];
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
          if (lane == 0) mbar_arrive_leader(&accept[slot]);
          ++rc;
          continue;
        }
        // ---------------- an own tile: scores -> reference decision -> probabilities ----------------
        if (!have_s) load_scores();
        have_s = false;
        const int c0 = j * Q7_BN + q2;
        const bool full = j * Q7_BN + Q7_BN <= p.Tk;
        const float a2 = CROSS ? 1.0f : p.alpha2;   // CROSS: the accumulators are turned into alpha2 s + bias first
        if (CROSS) {
          const float* kbp = p.kbias + static_cast<long long>(seq) * p.kb_seq;
#pragma unroll
          for (int kb = 0; kb < 8; ++kb) {
            const int cc = c0 + kb * 8;
            const float b0 = cc < p.Tk ? __ldg(kbp + cc) * 1.4426950408889634f : 0.f;
            const float b1 = cc + 1 < p.Tk ? __ldg(kbp + cc + 1) * 1.4426950408889634f : 0.f;
            const float b2 = cc + 64 < p.Tk ? __ldg(kbp + cc + 64) * 1.4426950408889634f : 0.f;
            const float b3 = cc + 65 < p.Tk ? __ldg(kbp + cc + 65) * 1.4426950408889634f : 0.f;
            s0[4 * kb] = __float_as_uint(fmaf(__uint_as_float(s0[4 * kb]), p.alpha2, b0));
            s0[4 * kb + 1] = __float_as_uint(fmaf(__uint_as_float(s0[4 * kb + 1]), p.alpha2, b1));
            s0[4 * kb + 2] = __float_as_uint(fmaf(__uint_as_float(s0[4 * kb + 2]), p.alpha2, b0));
            s0[4 * kb + 3] = __float_as_uint(fmaf(__uint_as_float(s0[4 * kb + 3]), p.alpha2, b1));
            s1[4 * kb] = __float_as_uint(fmaf(__uint_as_float(s1[4 * kb]), p.alpha2, b2));
            s1[4 * kb + 1] = __float_as_uint(fmaf(__uint_as_float(s1[4 * kb + 1]), p.alpha2, b3));
            s1[4 * kb + 2] = __float_as_uint(fmaf(__uint_as_float(s1[4 * kb + 2]), p.alpha2, b2));
            s1[4 * kb + 3] = __float_as_uint(fmaf(__uint_as_float(s1[4 * kb + 3]), p.alpha2, b3));
          }
        }
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
            if (cc < p.Tk) { mA = fmaxf(mA, __uint_as_float(s0[4 * kb])); mB = fmaxf(mB, __uint_as_float(s0[4 * kb + 2])); }
            if (cc + 1 < p.Tk) { mA = fmaxf(mA, __uint_as_float(s0[4 * kb + 1])); mB = fmaxf(mB, __uint_as_float(s0[4 * kb + 3])); }
            if (cc + 64 < p.Tk) { mA = fmaxf(mA, __uint_as_float(s1[4 * kb])); mB = fmaxf(mB, __uint_as_float(s1[4 * kb + 2])); }
            if (cc + 65 < p.Tk) { mA = fmaxf(mA, __uint_as_float(s1[4 * kb + 1])); mB = fmaxf(mB, __uint_as_float(s1[4 * kb + 3])); }
          }
        }
        mA = quad_max(mA) * a2;
        mB = quad_max(mB) * a2;
        const bool upA = j > 0 && (mA > refA + Q7_TAU || (p.force_rescale && mA > refA));
        const bool upB = j > 0 && (mB > refB + Q7_TAU || (p.force_rescale && mB > refB));
        const float nA = (j == 0 || upA) ? mA : refA, nB = (j == 0 || upB) ? mB : refB;
        if (writer) {
          const uint32_t slot = oc & 1u;
          const uint32_t dsta = mapa_shared(smem_u32(hdr_x + slot * Q7_BM + rA), peer);
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
        mbar_wait(p_free, (oc & 1u) ^ 1u);
        tr.ev(13, j);
#pragma unroll
        for (int cb = 0; cb < 2; ++cb) {
          const uint32_t(&r)[32] = cb == 0 ? s0 : s1;
          uint8_t* pa = p_own + cb * (Q7_BM * 128) + rA * 128 + q2 * 2;
          uint8_t* pbp = p_own + cb * (Q7_BM * 128) + rB * 128 + q2 * 2;
#pragma unroll
          for (int kb = 0; kb < 8; ++kb) {
            float2 eA = make_float2(ex2_approx(fmaf(__uint_as_float(r[4 * kb]), a2, -refA)),
                                    ex2_approx(fmaf(__uint_as_float(r[4 * kb + 1]), a2, -refA)));
            float2 eB = make_float2(ex2_approx(fmaf(__uint_as_float(r[4 * kb + 2]), a2, -refB)),
                                    ex2_approx(fmaf(__uint_as_float(r[4 * kb + 3]), a2, -refB)));
            if (!full) {
              const int cc = c0 + cb * 64 + kb * 8;
              if (cc >= p.Tk) { eA.x = 0.f; eB.x = 0.f; }
              if (cc + 1 >= p.Tk) { eA.y = 0.f; eB.y = 0.f; }
            }
            lA2 = __fadd2_rn(lA2, eA);
            lB2 = __fadd2_rn(lB2, eB);
            *reinterpret_cast<uint32_t*>(pa + ((kb ^ (rA & 7)) << 4)) = pack_bf16x2(eA.x, eA.y);
            *reinterpret_cast<uint32_t*>(pbp + ((kb ^ (rB & 7)) << 4)) = pack_bf16x2(eB.x, eB.y);
          }
        }
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) {
          mbar_arrive(p_ready);
          mbar_arrive_leader(p_full);
        }
        tr.ev(14, j);
        if (j == c) prefetch_residual();
        ++oc;
      }
      // ---------------- total row sums ----------------
      float lA = quad_sum(lA2.x + lA2.y), lB = quad_sum(lB2.x + lB2.y);
      const uint32_t par = it & 1u;
      if (ew == 0 && lane == 0) mbar_expect_tx(&l_bar[par], Q7_BM * 4);
      if (writer) {
        const uint32_t dsta = mapa_shared(smem_u32(l_x + par * Q7_BM + rA), peer);
        const uint32_t barr = mapa_shared(smem_u32(&l_bar[par]), peer);
        st_async_f32(dsta, lA, barr);
        st_async_f32(dsta + 8 * 4, lB, barr);
      }
      // ---------------- epilogue sweep 1: h <- O / l + h, row statistics, h kept in TMEM ----------------
      float4 f0[8], f1[8], f2[8];   // residual of three 64-column chunks in flight (rows A: [0, 4), rows B: [4, 8))
      auto load_res = [&](int cb, float4(&f)[8]) {
#pragma unroll
        for (int jj = 0; jj < 4; ++jj) {
          f[jj] = (okA && !(p.dbg & 2)) ? *reinterpret_cast<const float4*>(hA + cb * 64 + jj * 16) : make_float4(0.f, 0.f, 0.f, 0.f);
          f[4 + jj] = (okB && !(p.dbg & 2)) ? *reinterpret_cast<const float4*>(hB + cb * 64 + jj * 16) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
      };
      tr.ev(26, it);
      load_res(0, f0);
      load_res(1, f1);
      load_res(2, f2);
      tr.ev(27, it);
      mbar_wait(&l_bar[par], (it >> 1) & 1u);
      tr.ev(15, it);
      lA += l_x[par * Q7_BM + rA];
      lB += l_x[par * Q7_BM + rB];
      const float iA = 1.0f / lA, iB = 1.0f / lB;
      mbar_wait(o_full, it & 1u);
      tcgen05_fence_after();
      tr.ev(16, it);
      // row statistics of this thread's 96 values of rows A and B: sums of v - K and (v - K)^2, K = its first value (common.cuh)
      float smA = 0.f, sqA = 0.f, smB = 0.f, sqB = 0.f, kA = 0.f, kB = 0.f;
      auto sweep1 = [&](int cb, const float4(&f)[8]) {
        uint32_t o[32];
        tmem_ld_16x64(t_lane + cb * 64, o);
        float4 ob[4];
        if (CROSS) {
#pragma unroll
          for (int jj = 0; jj < 4; ++jj) ob[jj] = __ldg(reinterpret_cast<const float4*>(p.obias + col_half + q * 4 + cb * 64 + jj * 16));
        }
        tmem_ld_wait();
        tr.ev(21, cb);
#pragma unroll
        for (int jj = 0; jj < 4; ++jj) {
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
          if (konst) ob[jj] = *reinterpret_cast<const float4*>(crow + q * 4 + cb * 64 + jj * 16);
          if (CROSS || konst) {   // + out_proj bias (the torch MHA output projection, folded into V) / constant row
            vA.x += ob[jj].x; vA.y += ob[jj].y; vA.z += ob[jj].z; vA.w += ob[jj].w;
            vB.x += ob[jj].x; vB.y += ob[jj].y; vB.z += ob[jj].z; vB.w += ob[jj].w;
          }
          if (okA && !(p.dbg & 4)) *reinterpret_cast<float4*>(hA + cb * 64 + jj * 16) = vA;
          if (okB && !(p.dbg & 4)) *reinterpret_cast<float4*>(hB + cb * 64 + jj * 16) = vB;
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
        tr.ev(22, cb);
      };
      static_assert(Q7_DH / 64 == 6, "two rounds of three chunks");
      sweep1(0, f0); load_res(3, f0);
      sweep1(1, f1); load_res(4, f1);
      sweep1(2, f2); load_res(5, f2);
      sweep1(3, f0);
      sweep1(4, f1);
      sweep1(5, f2);
      tr.ev(17, it);
      if (p.u_out != nullptr) {
        tmem_st_wait();
        // partials (mean, M2) of this CTA's 384 columns; the peer's are merged in below
        const float2 pA = ln_quad_merge(ln_partial(kA, smA, sqA, 1.0f / (Q7_DH / 4)), Q7_DH / 4);
        const float2 pB = ln_quad_merge(ln_partial(kB, smB, sqB, 1.0f / (Q7_DH / 4)), Q7_DH / 4);
        if (ew == 0 && lane == 0) mbar_expect_tx(&stat_bar[par], Q7_BM * 8);
        if (writer) {
          const uint32_t slot = mapa_shared(smem_u32(stat_x + (par * Q7_BM + rA) * 2), peer);
          const uint32_t bar = mapa_shared(smem_u32(&stat_bar[par]), peer);
          st_async_f32(slot, pA.x, bar);
          st_async_f32(slot + 4, pA.y, bar);
          st_async_f32(slot + 8 * 8, pB.x, bar);
          st_async_f32(slot + 8 * 8 + 4, pB.y, bar);
        }
        mbar_wait(&stat_bar[par], (it >> 1) & 1u);
        tr.ev(18, it);
        const float2 xA = *reinterpret_cast<const float2*>(stat_x + (par * Q7_BM + rA) * 2);
        const float2 xB = *reinterpret_cast<const float2*>(stat_x + (par * Q7_BM + rB) * 2);
        const float inv_h = 1.0f / static_cast<float>(Q7_D);
        const float2 stA = ln_merge(pA, xA, Q7_DH), stB = ln_merge(pB, xB, Q7_DH);
        const float meanA = stA.x, meanB = stB.x;
        const float rsA = rsqrtf(fmaxf(stA.y, 0.f) * inv_h + 1e-5f);
        const float rsB = rsqrtf(fmaxf(stB.y, 0.f) * inv_h + 1e-5f);
        const float2 aA2 = make_float2(rsA, rsA), cA2 = make_float2(-meanA * rsA, -meanA * rsA);
        const float2 aB2 = make_float2(rsB, rsB), cB2 = make_float2(-meanB * rsB, -meanB * rsB);
        bf16* uA = p.u_out + growA * Q7_D + col_half + q * 4;
        bf16* uB = uA + 8 * Q7_D;
        const float* gp = (konst ? p.gamma_c : p.gamma) + col_half + q * 4;
        const float* bp = (konst ? p.beta_c : p.beta) + col_half + q * 4;
        // the TMEM load of chunk cb + 1 is in flight while chunk cb is normalised and stored (tcgen05.wait::ld waits for every
        // outstanding load, so the next load is issued right after the wait and consumed one iteration later)
        auto sweep2 = [&](int cb, const uint32_t(&o)[32]) {
          float4 gm[4], bt[4];
#pragma unroll
          for (int jj = 0; jj < 4; ++jj) {
            gm[jj] = __ldg(reinterpret_cast<const float4*>(gp + cb * 64 + jj * 16));
            bt[jj] = __ldg(reinterpret_cast<const float4*>(bp + cb * 64 + jj * 16));
          }
          tr.ev(23, cb);
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
            if (okA && !(p.dbg & 8)) *reinterpret_cast<uint2*>(uA + cb * 64 + jj * 16) = wA;
            if (okB && !(p.dbg & 8)) *reinterpret_cast<uint2*>(uB + cb * 64 + jj * 16) = wB;
          }
        };
        {
          uint32_t o0[32], o1[32];
          tmem_ld_16x64(t_lane, o0);
          tmem_ld_wait();
#pragma unroll 1
          for (int cb = 0; cb < Q7_DH / 64; cb += 2) {
            tmem_ld_16x64(t_lane + (cb + 1) * 64, o1);
            sweep2(cb, o0);
            tmem_ld_wait();
            if (cb + 2 < Q7_DH / 64) tmem_ld_16x64(t_lane + (cb + 2) * 64, o0);
            sweep2(cb + 1, o1);
            tmem_ld_wait();
          }
        }
      }
      tcgen05_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive_leader(o_empty);
      tr.ev(19, it);
    }
  }

  __syncwarp();
  tcgen05_fence_before();
  __syncthreads();
  cluster_sync_all();   // nobody leaves while another CTA may still write into it / signal its barriers / read its operands
  if (warp == 2) {
    tcgen05_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(Q7_TMEM_COLS) : "memory");
  }
}

}  // namespace

// The four-CTA kernel pays when 256-row query tiles do not pad much more than 128-row tiles would (T = 750: 768 = 768).
bool flash768_quad_preferred(int T) { return round_up(T, 2 * Q7_BM) * 100 <= round_up(T, Q7_BM) * 120; }

bool flash768_quad_schedulable() {
  if (tc_gemm_init() != 0) return false;
  return max_active_clusters(reinterpret_cast<const void*>(flash_attn768q_kernel<false>), 4, Q7_THREADS, Q7_SMEM_BYTES) > 0;
}

int launch_flash768_quad(const Flash768Params& q, cudaStream_t st) {
  DITTO_TRY(tc_gemm_init());
  DITTO_REQUIRE(flash768_supported(q.H, 1, q.T), DITTO_E_UNSUPPORTED, "flash768: single head of 768 only");
  const bool cross = q.kfold != nullptr;
  DITTO_REQUIRE(q.qkv && q.h && q.n_seq >= 1 && q.ld % 8 == 0 && q.ld >= (cross ? 1 : 3) * Q7_D, DITTO_E_BADARG, "flash768: bad argument");
  DITTO_REQUIRE(!cross || (q.vfold && q.kbias && q.out_bias && q.Tk >= 1 && q.Tk <= 256 && q.vf_rows >= q.Tk && q.kb_seq >= q.Tk &&
                           q.kf_seq % 8 == 0 && q.vf_seq % 8 == 0 && (reinterpret_cast<uintptr_t>(q.out_bias) & 15) == 0),
                DITTO_E_BADARG, "flash768 (cross-attention): folded keys / values, score bias and output bias for 1..256 text tokens");
  DITTO_REQUIRE(q.u_out == nullptr || (q.gamma && q.beta), DITTO_E_BADARG, "flash768: LayerNorm output needs gamma and beta");
  DITTO_REQUIRE(q.const_flag == nullptr || cross ||
                    (q.u_out && q.const_row && q.gamma_c && q.beta_c && (reinterpret_cast<uintptr_t>(q.const_row) & 15) == 0),
                DITTO_E_BADARG, "flash768 (constant text): 16-byte aligned constant rows, norm3 and a LayerNorm output");
  DITTO_REQUIRE((reinterpret_cast<uintptr_t>(q.h) & 15) == 0 && (reinterpret_cast<uintptr_t>(q.u_out) & 7) == 0, DITTO_E_BADARG,
                "flash768: h must be 16-byte, u 8-byte aligned");
  const void* fn = !cross ? (q.const_flag ? reinterpret_cast<const void*>(flash_attn768q_kernel<false, true>)
                                          : reinterpret_cast<const void*>(flash_attn768q_kernel<false>))
                          : reinterpret_cast<const void*>(flash_attn768q_kernel<true>);
  DITTO_REQUIRE(max_active_clusters(fn, 4, Q7_THREADS, Q7_SMEM_BYTES) > 0, DITTO_E_UNSUPPORTED,
                "flash768: four-CTA clusters cannot be scheduled on this device");
  TcOperand Q, K, V;
  Q.ptr = q.qkv; Q.rows = q.T; Q.cols = Q7_D; Q.ld = q.ld; Q.s_outer = static_cast<int64_t>(q.T) * q.ld;
  K = Q; K.ptr = q.qkv + Q7_D;
  V = Q; V.ptr = q.qkv + 2 * Q7_D;
  if (cross) {
    K.ptr = q.kfold; K.rows = q.Tk; K.ld = Q7_D; K.s_outer = q.kf_seq;
    V.ptr = q.vfold; V.rows = q.Tk; V.ld = Q7_D; V.s_outer = q.vf_seq;   // rows past Tk: zero-filled by TMA
  }
  CUtensorMap mq, mk, mv;
  DITTO_TRY(tc_make_map(&mq, Q, 1, q.n_seq, Q7_BK, Q7_BM));
  DITTO_TRY(tc_make_map(&mk, K, 1, q.n_seq, Q7_BK, Q7_BN / 2));
  DITTO_TRY(tc_make_map(&mv, V, 1, q.n_seq, 64, Q7_VKEYS));
  Q7Dev p;
  p.n_seq = static_cast<int>(q.n_seq); p.T = q.T;
  p.Tk = cross ? q.Tk : q.T;
  p.kbias = q.kbias; p.kb_seq = q.kb_seq; p.obias = cross ? q.out_bias : q.const_row;
  p.m_tiles = static_cast<int>(ceil_div(q.T, 2 * Q7_BM));
  p.k_tiles = static_cast<int>(ceil_div(p.Tk, Q7_BN));
  const int64_t items = static_cast<int64_t>(p.m_tiles) * q.n_seq;
  DITTO_REQUIRE(items < (1ll << 31), DITTO_E_UNSUPPORTED, "flash768: too many work items");
  p.num_items = static_cast<int>(items);
  p.alpha2 = q.alpha * 1.4426950408889634f;
  p.h = q.h; p.gamma = q.gamma; p.beta = q.beta; p.u_out = q.u_out;
  p.const_flag = q.const_flag; p.gamma_c = q.gamma_c; p.beta_c = q.beta_c;
  p.force_rescale = q.force_rescale ? 1 : 0;
  p.dbg = 0;
  p.trace = DITTO_F7_TRACE ? tc_gemm_debug_counters() : nullptr;
  // the cross-attention kernel does no work for the skipped sequences (profiler byte / flop counts over the processed ones)
  const double n_run = static_cast<double>(q.n_seq - (cross && q.const_flag ? profiled_nonzero(q.const_flag, q.n_seq, st) : 0));
  const double rows = n_run * q.T;
  ProfScope prof(q.tag, st, 4.0 * q.T * static_cast<double>(p.Tk) * Q7_D * n_run,
                 rows * Q7_D * ((cross ? 2.0 : 6.0) + 8.0 + (q.u_out ? 2.0 : 0.0)) + (cross ? 4.0 * n_run * static_cast<double>(p.Tk) * Q7_D : 0.0));
  void* args[4] = {&mq, &mk, &mv, &p};
  return launch_clusters(fn, 4, Q7_THREADS, Q7_SMEM_BYTES, items, args, st);
}

}  // namespace ditto
