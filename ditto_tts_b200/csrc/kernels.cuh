// Internal launcher interface shared by the translation units of libditto_b200.
#pragma once
#include <algorithm>

#include "common.cuh"

namespace ditto {

// ---- developer options (ditto_debug_option): A/B switches of the kernels, all 0 = the product path.  The library never
// reads the environment; tools / tests set these through the C-ABI before creating an engine.
struct DebugOptions {
  // cross_fused.cu
  int xf_rows = 0;
  // engine.cu (read by ditto_engine_create)
  int no_defer_ln = 0, no_flash = 0, no_flash768 = 0, no_fused_cross = 0, defer_ln2 = 0, rope_generic = 0, glu_generic = 0,
      no_pv_perm4 = 0, side_streams = -1;
  // flash_attn768.cu (read at launch time): 1 = always the two-CTA kernel, 2 = the four-CTA kernel whenever it is supported
  int flash768_quad = 0;
  // engine.cu: fc2 + residual + next block's norm1 as separate launches (GEMM, LayerNorm) instead of gemm_resid_ln.cu
  int no_fc2_ln = 0;
  // engine.cu: cross-attention with 64 < S <= 256 text tokens as scores+softmax / P.V / LayerNorm launches instead of flash_attn768q<CROSS>
  int no_cross_flash = 0;
  // engine.cu (read by ditto_engine_create): sequences with constant text rows go through the cross-attention kernel too
  int no_const_text = 0;
};
extern DebugOptions g_opt;

// ---- per-device one-time state (kernel attributes are per device: an engine on cuda:1 must not reuse cuda:0's set-up)
struct DeviceState {
  bool tc_init = false, xf_attr = false, fa_attr = false, f768_attr = false;
  int num_sms = 0;
};
DeviceState* device_state();  // state of the CURRENT device (nullptr + error set when cudaGetDevice fails)
// Co-resident clusters of `csize` CTAs (`threads` threads, `smem_bytes` of dynamic shared memory each) of the kernel `func`
// on the current device, queried once per (device, kernel, cluster size); sets the kernel's shared-memory attribute.
// <= 0: clusters of this size cannot be scheduled.
int max_active_clusters(const void* func, int csize, int threads, int smem_bytes);
// Persistent launch of `func` (the kernel strides over its work items by the number of clusters): grid = csize x
// min(co-resident clusters, work_items); csize == 1 is a plain launch of one CTA per SM.  args: the kernel's parameters.
int launch_clusters(const void* func, int csize, int threads, int smem_bytes, int64_t work_items, void** args, cudaStream_t st);

// ---- elementwise.cu ----------------------------------------------------------------------------------
int launch_cast_bf16(const float* x, bf16* y, int64_t n, cudaStream_t st);
// text [n_seq, S, D] fp32 -> y (bf16 when y_bf16, else fp32) with rows s >= len[seq] (device, [n_seq]) set to zero
int launch_stage_text(const float* x, void* y, bool y_bf16, const int* len, int64_t n_seq, int S, int D, cudaStream_t st);
int launch_fill_i32(int* y, int v, int64_t n, cudaStream_t st);
int launch_pack_rows(const float* x, bf16* y, float* bias_out, const float* bias_in, const int* perm, int rows, int K,
                     cudaStream_t st, const float* gamma = nullptr, const float* beta = nullptr, float* csum = nullptr);
int launch_rowsum_bf16(const bf16* x, float* out, int64_t groups, int S, int Sp, int K, cudaStream_t st);
int launch_layernorm(const float* x, const float* gamma, const float* beta, void* y, bool out_bf16, int64_t rows, int H,
                     cudaStream_t st);
int launch_adaln_ln(const float* x, int64_t n_x, const float* time_table, const float* text_mod, const int64_t* t,
                    int steps, const float* gamma, const float* beta, float* h, void* u, bool u_bf16, bf16* xcast,
                    int64_t n_seq, int T, int H, cudaStream_t st, float2* stat = nullptr, bool xcast_all = false,
                    int* row_pos = nullptr);
int launch_rope_table(const float* inv_freq, float* cos_t, float* sin_t, float* freq_out, int max_T, int half, int head_dim,
                      cudaStream_t st);
int launch_rope(void* qkv, bool is_bf16, int64_t ld, const float* cos_t, const float* sin_t, int64_t rows, int seq_T,
                int H, int head_dim, cudaStream_t st);
// col_len (optional): row r has min(cols, col_len[r / rows_per_len]) valid columns, the rest get probability 0
int launch_softmax(const float* s, int64_t lds, void* p, bool p_bf16, int64_t ldp, int64_t rows, int cols, cudaStream_t st,
                   const int* col_len = nullptr, int64_t rows_per_len = 1);
int launch_geglu_f32(const float* a, const float* g, float* out, int64_t n, cudaStream_t st);
int launch_silu(float* x, int64_t n, cudaStream_t st);
// len (optional, device [n]): masked text, sequence seq uses its first len[seq] rows only (mean over them; score bias -inf
// past them; constant flag from them)
int launch_mean_silu(const float* text, float* out, int64_t n, int S, int D, cudaStream_t st, const int* len = nullptr);
int launch_fold_bias(const bf16* kv, int64_t ld, const float* bq, float* sb, int64_t n, int S, int Sp, int heads, int d, float scale,
                     cudaStream_t st, const int* len = nullptr);
// constant text (all S rows of a sequence's text_emb [n, S, D] bitwise equal): flag[seq] (written when flag != nullptr) and,
// for every sequence, crow[seq] = vfold[seq][0] + bo in the plain column order (vf_perm4: vfold columns in the perm4 order)
int launch_const_text(const float* text, int64_t n, int S, int D, const bf16* vfold, int64_t vf_seq, bool vf_perm4, const float* bo,
                      uint8_t* flag, float* crow, int H, cudaStream_t st, const int* len = nullptr);
// number of nonzero bytes of flags[0, n) for the profiler's byte counts; 0 without synchronising unless profiling (which
// synchronises anyway and is never captured)
int64_t profiled_nonzero(const uint8_t* flags, int64_t n, cudaStream_t st);
// One sampler update over B sequences of `per` elements: eps = eps_u + w (eps_c - eps_u) (eps_u == null: eps = eps_c), then
//   DDPM form (hist == null, coef [steps, 3] = {c1, c2, c3}):  x_out = c1 (x - c2 eps) + c3 z
//   multistep (hist != null, coef [steps, 6] = {c1, c2, c3, c4, d1, d2}, DPM-Solver++(2M)): the same + c4 hist, then
//     hist <- d1 (x - d2 eps); hist is read only on rows with c4 != 0
// with the row t[seq] of the table.  Noise: supplied z, or (rng != null) drawn in the kernel (Philox4x32-10 + Box-Muller from
// rng = {seed, draw counter, ticket, -}) at element elem_offset + i; neither: no noise term.  advance (needs rng): the last
// block to finish adds 1 to the draw counter and subtracts 1 from t[0 .. n_t).  Known frames (replacement conditioning, speech
// prompt / infilling; mask != null): every `frame` elements share one mask byte, and a frame with mask != 0 becomes a p + s z
// with {a, s} = coef_known[t] and p = known.  Per sequence (w_seq / seeds non-null): the scale w_seq[seq] instead of w, and
// (with rng) the key seeds[seq] instead of rng[0], the element counted from the sequence's first element instead of
// elem_offset + i.
struct CfgUpdateParams {
  const float* eps_c = nullptr; const float* eps_u = nullptr; const float* x = nullptr;
  const float* z = nullptr; unsigned long long* rng = nullptr;
  int64_t* t = nullptr; int64_t n_t = 0;   // t is written only with advance
  const float* coef = nullptr; const float* coef_known = nullptr; int steps = 0; float w = 0.f;
  float* out = nullptr; float* hist = nullptr;
  const float* known = nullptr; const uint8_t* mask = nullptr;
  int64_t B = 0, per = 0, frame = 0, elem_offset = 0;
  bool advance = false;
  const unsigned long long* seeds = nullptr; const float* w_seq = nullptr;
};
int launch_cfg_update(const CfgUpdateParams& p, cudaStream_t st);
int launch_step_advance(unsigned long long* rng, int64_t* t, int64_t n_t, cudaStream_t st);
int launch_randn(const unsigned long long* rng, int64_t elem_offset, float* out, int64_t n, cudaStream_t st);
// x_T of B utterances: rows row0[b] .. row0[b + 1] - 1 of out [rows, H] get draw 2^64 - 1 under seeds[b] (row0 [B + 1], device)
int launch_randn_latents(const unsigned long long* seeds, const int64_t* row0, int64_t B, int64_t H, float* out, cudaStream_t st);
int launch_rope_angles(const float* t, const float* pos, float* out, int64_t batch, int T, int heads, int d, cudaStream_t st);
int launch_schedule_coef(const float* betas, const float* alphas, const float* acp, float* coef, int steps, cudaStream_t st);
int launch_q_sample(const float* x0, const float* noise, const int64_t* t, const float* buf, int steps, float* out, int64_t B,
                    int64_t elems_per_seq, cudaStream_t st);

// ---- gemm_f32.cu -------------------------------------------------------------------------------------
struct SgemmParams {
  const float* A = nullptr; int64_t lda = 0, sA_inner = 0, sA_outer = 0;
  const float* B = nullptr; int64_t ldb = 0, sB_inner = 0, sB_outer = 0;
  float* C = nullptr;       int64_t ldc = 0, sC_inner = 0, sC_outer = 0;
  const float* resid = nullptr; int64_t ldr = 0, sR_inner = 0, sR_outer = 0;
  const float* bias = nullptr;
  float alpha = 1.f;
  int M = 0, N = 0, K = 0;
  int batch_inner = 1, batch_outer = 1;
  bool b_is_nk = true;  // B [N,K] (x W^T) else B [K,N]
};
int launch_sgemm(const SgemmParams& p, cudaStream_t st);

// ---- gemm_tc.cu (tcgen05 / TMEM / TMA) ---------------------------------------------------------------
enum TcEpilogue { TC_EPI_STORE = 0, TC_EPI_GEGLU = 1, TC_EPI_QKV_ROPE = 2 };

// 2-D operand view with two batch levels; strides in ELEMENTS (bf16).  rows x cols with `cols` contiguous.
struct TcOperand {
  const bf16* ptr = nullptr;
  int64_t rows = 0, cols = 0, ld = 0;
  int64_t s_inner = 0, s_outer = 0;  // batch strides; 0 => operand shared by every batch item
};

struct TcGemmParams {
  // C[b] (M x N) = alpha * A[b] (M x K) @ B[b]^T  where B is [N, K] (b_kn == false) or [K, N] (b_kn == true)
  TcOperand A, B;
  bool b_kn = false;
  int M = 0, N = 0, K = 0;
  int batch_inner = 1, batch_outer = 1;
  int epilogue = TC_EPI_STORE;
  int tag = PC_TC_OTHER;                       // profiling class (call site)
  float alpha = 1.f;
  const float* bias = nullptr;                 // [N], indexed by GEMM column
  int64_t sb_inner = 0, sb_outer = 0;          // optional per-batch-item bias (element strides)
  void* out = nullptr; bool out_bf16 = false;  // [M, ldo] per batch item
  int64_t ldo = 0, so_inner = 0, so_outer = 0;
  const float* resid = nullptr;                // fp32, added after bias
  int64_t ldr = 0, sr_inner = 0, sr_outer = 0;
  int64_t resid_row_mod = 0;                   // >0: residual row = row % resid_row_mod (x_skip shared by CFG branches)
  bf16* out2 = nullptr; int64_t ldo2 = 0;      // optional bf16 copy of the (fp32) result, batch strides as `out`
  // TC_EPI_QKV_ROPE
  const float* rope_freq = nullptr;            // [d/2] inv_freq (required): cos/sin are computed in the epilogue
  int rope_half = 0, rope_pd = 0, seq_T = 0, hidden = 0;
  const int* rope_pos = nullptr;               // optional [M] row -> position table (ragged batches) instead of row % seq_T
  // weight rows additionally permuted inside every 64-row block (GEMM column kb*8 + 2q + e = output column q*16 + kb*2 + e):
  // lean epilogue with 16-byte stores; needs rope_pd == 128, rope_freq, no deferred LayerNorm, N % 256 == 0, hidden % 256 == 0
  bool rope_perm16 = false;
  // TC_EPI_GEGLU: [fc1; gate] rows packed in the store-friendly order of geglu_epilogue_fast (gemm_tc.cu) instead of [a16 | g16]
  bool glu_perm16 = false;
  // TC_EPI_STORE, fp32 + residual: the B operand's columns are stored so that accumulator column 8 kb + 2 q + e of a 64-column
  // block is output column 16 (kb / 2) + 4 q + 2 (kb % 2) + e -> 16-byte residual loads / result stores (self-attention P.V)
  bool out_perm4 = false;
  // optional per-row scale 1 / sum_c row_lsum[row*row_lparts + c] applied to the accumulator (softmax normalisation of an
  // unnormalised P operand, see launch_tc_scores_softmax); batch strides in elements
  const float* row_lsum = nullptr; int row_lparts = 0; int64_t sl_inner = 0, sl_outer = 0;
  // Deferred LayerNorm (see DevParams in gemm_tc.cu).
  //  producer (STORE with fp32 residual, even N): stat_out[(outer * stat_rows_outer + row) * stat_parts + inner *
  //    ceil(N / 128) + slab] = (sum, sum of squares) of the 128-column slab of the stored row; stat_parts must equal
  //    batch_inner * ceil(N / 128)
  //  consumer (QKV_ROPE / GEGLU, unbatched): ln_stat [M, ln_parts] as written by a producer over rows of width ln_width;
  //    ln_c [N] = row sums of the gamma-scaled weight; `bias` must already contain W beta
  float2* stat_out = nullptr; int stat_parts = 0; int64_t stat_rows_outer = 0;
  const float2* ln_stat = nullptr; int ln_parts = 0; int ln_width = 0; const float* ln_c = nullptr;
};
int launch_tc_gemm(const TcGemmParams& p, cudaStream_t st);

// Fused attention scores + softmax: P[b] = softmax_rows(alpha * Q[b] K[b]^T + bias[b]) written as bf16, the fp32 scores
// never leave the SM (TMEM).  One thread-block CLUSTER per 128 query rows: CTA r owns key columns [256 r, 256 r + 256)
// and the row maxima are exchanged through distributed shared memory.  Cluster size 1: P is normalised in the kernel.
// Cluster size > 1: P holds exp(s - rowmax) (in (0, 1]) and lpart[row][r] the partial row sums; the P.V GEMM divides by
// their sum through TcGemmParams::row_lsum.  Columns [N, npad) of P are zero-filled.
struct TcScoresSoftmaxParams {
  TcOperand Q, Km;                              // [M, K] and [N, K] per batch item, K contiguous
  int M = 0, N = 0, K = 0;
  int batch_inner = 1, batch_outer = 1;
  float alpha = 1.f;
  const float* bias = nullptr; int64_t sb_inner = 0, sb_outer = 0;  // optional additive score bias per key column
  bf16* P = nullptr; int64_t ldp = 0, sp_inner = 0, sp_outer = 0;
  int npad = 0;                                 // zero-fill bound (multiple of 2, >= N)
  float* lpart = nullptr; int64_t sl_inner = 0, sl_outer = 0;  // [M, csize] per batch item; required when csize > 1
  // optional [batch_outer] valid key count of each outer batch item (masked text): columns [col_len[b], N) get probability 0
  const int* col_len = nullptr;
  // deferred LayerNorm of Q (needs bias): statistics row = outer batch index * M + query row; ln_c strided like bias
  const float2* ln_stat = nullptr; int ln_parts = 0; int ln_width = 0; const float* ln_c = nullptr;
  int tag = PC_TC_OTHER;
};
int tc_scores_softmax_csize(int N);             // cluster size the kernel will use for N key columns (0: unsupported)
int launch_tc_scores_softmax(const TcScoresSoftmaxParams& p, cudaStream_t st);
// ---- cross_fused.cu: folded single-head cross-attention + residual + the LayerNorm that follows, one kernel -------------
struct CrossFusedParams {
  const bf16* u = nullptr;                     // [n_seq * T, H] LayerNorm-2 output (query operand)
  const bf16* kfold = nullptr; int64_t kf_seq = 0;   // [n_seq, S, H]  K Wq,  element stride between sequences
  const bf16* vfold = nullptr; int64_t vf_seq = 0;   // [n_seq, Sp, H] V Wo^T (rows >= S zero)
  const float* sbias = nullptr; int64_t sb_seq = 0;  // [n_seq, Sp] additive score bias
  const float* out_bias = nullptr;             // [H] cross_attn.out_proj.bias
  float* h = nullptr;                          // [n_seq * T, H] residual stream, updated in place
  const float* gamma = nullptr; const float* beta = nullptr;  // the next LayerNorm (norm3)
  bf16* u_out = nullptr;                       // [n_seq * T, H] its bf16 output (may alias u)
  // deferred norm2: u is the raw bf16 residual stream, kfold carries gamma2, sbias carries the beta2 term; the scores are
  // rstd (u kfold^T) - rstd mean c + sbias with (sum, sum of squares) partials ln_stat[row * ln_parts + part] over H columns
  const float2* ln_stat = nullptr; int ln_parts = 0; const float* ln_c = nullptr;  // ln_c [n_seq, Sp] like sbias
  // [n_seq]: tiles of sequences with skip_seq[seq] != 0 are not processed (constant text: the self-attention kernel has
  // already added their constant cross-attention output and written norm3); nullptr: every tile
  const uint8_t* skip_seq = nullptr;
  int64_t n_seq = 0, T = 0, S = 0, Sp = 0; int H = 0;
  float alpha = 1.f;
  int tag = PC_TC_OTHER;
};
bool cross_fused_supported(int64_t T, int64_t S, int H, int heads);
int launch_cross_fused(const CrossFusedParams& p, cudaStream_t st);

// ---- flash_attn.cu: self-attention for head_dim 64 without materialised scores (two passes over the keys) ---------------
struct FlashAttnParams {
  TcOperand Q, Km, V;                          // [Tq, d], [Tk, d], [Tk, d] per (head, utterance): s_inner = head stride, s_outer = utterance stride
  int64_t n_seq = 0; int heads = 0, d = 0, Tq = 0, Tk = 0;
  float alpha = 1.f;
  float* out = nullptr; const float* resid = nullptr;   // fp32 [n_seq, Tq, ld]; head h = columns [d h, d h + d); may alias
  int64_t ldo = 0, o_seq = 0, ldr = 0, r_seq = 0;
  int tag = PC_TC_OTHER;
};
bool flash_attn_supported(int d, int Tq, int Tk);
int launch_flash_attn(const FlashAttnParams& p, cudaStream_t st);

// ---- flash_attn768.cu: self-attention for ONE head of 768 + residual + the LayerNorm that follows, one kernel ---------
struct Flash768Params {
  const bf16* qkv = nullptr; int64_t ld = 0;   // [n_seq * T, ld]: q at column 0, k at 768 (both rotated), v at 1536 in the out_perm4 column order
  int64_t n_seq = 0; int T = 0; int H = 0;
  float alpha = 1.f;
  float* h = nullptr;                          // [n_seq * T, 768] fp32 residual stream, updated in place
  const float* gamma = nullptr; const float* beta = nullptr;   // LayerNorm after the attention (norm2)
  bf16* u_out = nullptr;                       // [n_seq * T, 768] its bf16 output; nullptr: no LayerNorm stage
  // cross-attention mode (four-CTA kernel only; kfold != nullptr): qkv = the query operand u [n_seq * T, ld] (its first 768
  // columns), keys / values = the folded text projections of ditto_text_context, one score bias per key, an output bias
  const bf16* kfold = nullptr; int64_t kf_seq = 0;                  // [n_seq][Tk, 768]         K Wq
  const bf16* vfold = nullptr; int64_t vf_seq = 0; int vf_rows = 0; // [n_seq][vf_rows, 768]    V Wo^T, columns in the perm4 order, zero rows past Tk
  int Tk = 0;                                                       // text tokens (<= 256)
  const float* kbias = nullptr; int64_t kb_seq = 0;                 // [n_seq][kb_seq] additive score bias (already scaled)
  const float* out_bias = nullptr;                                  // [768]
  // constant text (four-CTA kernel only).  Self-attention: sequences with const_flag[seq] != 0 get h <- h + attn + const_row[seq]
  // and u <- LayerNorm(h) gamma_c + beta_c (norm3: their cross-attention output is the constant row, so the cross-attention
  // section is done here).  Cross-attention: items of flagged sequences are skipped.  nullptr: off
  const uint8_t* const_flag = nullptr;
  const float* const_row = nullptr;                                 // [n_seq][768] fp32, plain column order
  const float* gamma_c = nullptr; const float* beta_c = nullptr;
  bool force_rescale = false;                 // tests: take the online-softmax rescale path whenever a tile raises the maximum
  int tag = PC_TC_OTHER;
};
bool flash768_supported(int H, int heads, int T);
int launch_flash768(const Flash768Params& p, cudaStream_t st);   // picks the two- or the four-CTA kernel
bool flash768_quad_preferred(int T);
bool flash768_picks_quad(int T);   // launch_flash768 takes the four-CTA kernel at this length (constant-text rows need it)
bool flash768_quad_schedulable();   // four-CTA clusters fit the current device (else the two-CTA kernel is used)
int launch_flash768_quad(const Flash768Params& p, cudaStream_t st);   // flash_attn768q.cu

// ---- gemm_resid_ln.cu: h += A W^T + b (fp32, in place) and u = LayerNorm(h) gamma + beta (bf16) in one cluster kernel ----
struct GemmResidLnParams {
  const bf16* A = nullptr; int64_t lda = 0;     // [M, K] bf16
  const bf16* W = nullptr; int64_t ldw = 0;     // [N, K] bf16, rows in the perm4 order (gemm_resid_ln_weight_row)
  const float* bias = nullptr;                  // [N], plain column order
  float* h = nullptr; int64_t ldh = 0;          // [M, N] fp32 residual stream, updated in place (or the output when `resid` is set)
  const float* resid = nullptr; int64_t ldr = 0; int64_t resid_mod = 0;   // optional separate residual: row r reads resid[r % resid_mod] (0: row r)
  const float* gamma = nullptr; const float* beta = nullptr;   // LayerNorm after the update; gamma == nullptr: u = bf16(h)
  bf16* u = nullptr; int64_t ldu = 0;           // [M, N] bf16 output (optional when gamma == nullptr)
  int M = 0, N = 0, K = 0;
  int tag = PC_TC_OTHER;
};
bool gemm_resid_ln_supported(int N, int K);
bool gemm_resid_ln_schedulable(int N);   // clusters of 2 N / 256 CTAs fit the current device
int gemm_resid_ln_weight_row(int packed_row);   // source row of a packed weight row
int launch_gemm_resid_ln(const GemmResidLnParams& p, cudaStream_t st);

int tc_gemm_init();  // resolves cuTensorMapEncodeTiled, sets kernel attributes
// 4-D bf16 tensor map (cols, rows, inner batch, outer batch) with a (box_cols, box_rows, 1, 1) box, 128-B swizzle, zero OOB fill
int tc_make_map(CUtensorMap* m, const TcOperand& op, int64_t n_inner, int64_t n_outer, int box_cols, int box_rows);
int tc_num_sms();
void tc_gemm_set_debug_counters(unsigned long long* dev_ptr);  // ditto_debug_set_counters
unsigned long long* tc_gemm_debug_counters();

}  // namespace ditto
