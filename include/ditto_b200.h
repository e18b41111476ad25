/*
 * ditto_b200.h -- C-ABI of the B200-native DiTTo-TTS denoiser hot path (libditto_b200.so).
 *
 * The reference (Tikai7/DiTTO-TTS) is pure Python/PyTorch and has NO FFI / plugin layer
 * (SURVEY.md section 8b): its boundary for this path is the nn.Module call signatures
 *     DiTTO.forward(x, text_emb, t)                 src/model/DiTTO.py:66-94
 *     GlobalAdaLN.forward / DiT.forward             src/components/DiT.py:25-40, 100-157
 *     SpeechGenerator.__p_sample/__sample_latents   src/model/SpeechGenerator.py:131-164
 * Each entry point below names the reference code it replaces.  The Python host
 * (ditto_tts_b200/model.py, sampler.py) binds these with ctypes; INTEGRATION.md shows the stub a
 * reference maintainer would add.
 *
 * Conventions
 *   - plain pointers and sizes only; every tensor pointer is a DEVICE pointer (sm_100a, B200),
 *     fp32 contiguous row-major unless stated; `stream` is a cudaStream_t passed as void*.
 *   - the caller allocates outputs, the text context and the workspace (query the *_bytes functions);
 *     hot-path calls never allocate, never synchronise, and are CUDA-graph capturable.
 *   - return value: 0 = ok, <0 = error (DITTO_E_*); ditto_last_error() gives the message for the
 *     calling thread.  Nothing throws across the ABI.  There is NO CPU fallback.
 */
#ifndef DITTO_B200_H_
#define DITTO_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DITTO_ABI_VERSION 1

enum {
  DITTO_OK = 0,
  DITTO_E_BADARG = -1,      /* null pointer, negative size, unknown key, wrong numel        */
  DITTO_E_UNSUPPORTED = -2, /* shape outside what the kernels cover (see DESIGN.md)         */
  DITTO_E_CUDA = -3,        /* a CUDA runtime/driver call failed; message has the code      */
  DITTO_E_STATE = -4,       /* engine not finalized / weights missing                      */
  DITTO_E_WORKSPACE = -5    /* workspace or context buffer too small                       */
};

/* arithmetic mode of the engine (BASELINE.json: fp32 bar 1e-4, bf16 bar 2e-2 vs the fp32 reference) */
enum {
  DITTO_PREC_FP32 = 0, /* CUDA-core fp32 FMA GEMMs/attention: correctness path                  */
  DITTO_PREC_BF16 = 1  /* tcgen05 bf16 tensor-core GEMMs, fp32 accumulate / residual / statistics */
};

/* optional features of the bf16 path (bit mask in ditto_config_t.flags); 0 = the plain composition */
enum {
  DITTO_F_FUSED_ROPE = 1 << 0, /* RoPE fused into the QKV GEMM epilogue (column-permuted weights) */
  DITTO_F_FOLD_CROSS = 1 << 1, /* fold cross-attn q/out projections into the per-utterance text K/V */
  DITTO_F_FUSED_ATTN = 1 << 2, /* scores + softmax in one cluster kernel (fp32 scores never leave TMEM)   */
  DITTO_F_BLOCKS_ONLY = 1 << 4, /* the engine holds DiT blocks only (keys "blocks.i.*"): a stand-alone components/DiT.py module;
                                   ditto_dit_block / ditto_text_context work, ditto_forward / ditto_p_sample do not        */
  DITTO_F_DEFER_LN = 1 << 3    /* block LayerNorms (DiT.py:105,143,151) folded into the neighbouring GEMMs: the producer
                                  epilogue emits bf16(h) + per-row partial (sum, sum of squares), gamma/beta live in the
                                  consumer's weights/bias and its epilogue applies rstd / mean (needs DITTO_F_FUSED_ROPE)  */
};

/* Shapes of one DiTTO instance == ctor arguments of the reference, src/model/DiTTO.py:10-19
 * (ConfigDiTTO defaults: src/utils/Config.py:109-116). */
typedef struct ditto_config {
  int32_t hidden_dim;      /* H, multiple of 8                                   */
  int32_t num_layers;      /* L                                                  */
  int32_t num_heads;       /* h, H % h == 0, (H/h) even                          */
  int32_t time_dim;        /* width of t_embedding / time_embed                  */
  int32_t text_dim;        /* must equal hidden_dim (nn.MultiheadAttention kdim) */
  int32_t diffusion_steps; /* rows of t_embedding and of the sampler tables      */
  int32_t precision;       /* DITTO_PREC_*                                       */
  int32_t max_seq_len;     /* RoPE table rows to precompute (T <= max_seq_len)   */
  int32_t flags;           /* DITTO_F_*                                          */
  int32_t reserved[7];
} ditto_config_t;

typedef struct ditto_engine ditto_engine_t; /* opaque */

/* ---- library ---------------------------------------------------------------------------------------- */
int32_t ditto_abi_version(void);
const char* ditto_last_error(void);
/* number of kernels this library has launched in this process (bench.py's gpu_launches claim) */
int64_t ditto_kernel_launch_count(void);

/* Opt-in per-kernel-class timing with CUDA events on the launching stream (bench.py's roofline numbers).
 * start: reset + enable; stop: device-synchronise, accumulate, disable.  Not for use under graph capture.
 * get: launches, summed duration [ms], summed algorithmic flops and bytes of class i. */
int32_t ditto_profile_start(void);
int32_t ditto_profile_stop(void);
int32_t ditto_profile_num_classes(void);
const char* ditto_profile_class_name(int32_t i);
int32_t ditto_profile_get(int32_t i, int64_t* launches, double* total_ms, double* flops, double* bytes);
/* Developer diagnostics of the paired tcgen05 GEMM: `counters` = 5 zero-initialised device uint64 (NULL = off) that
 * receive SM clock cycles summed over CTA pairs: [0] MMA issuer waiting for operands, [1] waiting for a drained
 * accumulator, [2] MMA issuer total; [3] TMA producer waiting for a free ring slot, [4] TMA producer total. */
int32_t ditto_debug_set_counters(uint64_t* counters);
/* Developer A/B switches of the kernels (tools/, tests/; all 0 = the product path, "reset" restores that).  The library
 * never reads the environment.  Engine-level options are sampled by ditto_engine_create.  Names: DESIGN.md section 9. */
int32_t ditto_debug_option(const char* name, int32_t value);

/* ---- engine life cycle == DiTTO.__init__ + load_state_dict (src/model/DiTTO.py:10-64) -------------- */
int32_t ditto_engine_create(const ditto_config_t* cfg, ditto_engine_t** out);
int32_t ditto_engine_destroy(ditto_engine_t* e);
/* Copy one state_dict tensor (reference key name, SURVEY.md 8b) from device fp32 memory into the engine.
 * Keys starting with "nac." and the dead "blocks.i.attn.out_proj.*" / "*.inv_freq" / "alphas_cumprod"
 * entries are accepted and ignored. */
int32_t ditto_engine_load_weight(ditto_engine_t* e, const char* key, const float* data, int64_t numel, void* stream);
/* Sampler tables betas/alphas/alphas_cumprod [diffusion_steps] fp32, computed by the host exactly as
 * src/model/SpeechGenerator.py:70-72 does. */
int32_t ditto_engine_load_schedule(ditto_engine_t* e, const float* betas, const float* alphas,
                                   const float* alphas_cumprod, int64_t steps, void* stream);
/* Sampler variants (SURVEY.md 8f row 4): replace the update table the schedule produced.  coef [diffusion_steps, 3] fp32
 * (device), row t = {c1, c2, c3} of   x_out = c1 (x - c2 eps) + c3 z   -- the form of SpeechGenerator.py:143-145, which
 * also expresses DDIM(eta) and DDPM over a strided sub-sequence of timesteps (rows that are never visited may hold
 * anything).  The host computes the rows (ditto_tts_b200/schedules.py); load_schedule restores the reference's table. */
int32_t ditto_engine_load_update_table(ditto_engine_t* e, const float* coef, int64_t steps, void* stream);
/* Multistep sampler (DPM-Solver++(2M), Lu et al. 2022 Alg. 2; eta > 0: its SDE variant).  coef6 [diffusion_steps, 6] fp32
 * (device), row t = {c1, c2, c3, c4, d1, d2} of
 *     x_out = c1 (x - c2 eps) + c3 z + c4 hist        hist <- d1 (x - d2 eps)   (= the x0 prediction of the step)
 * where hist carries the previous step's x0 prediction across steps (and CUDA-graph replays).  Rows with c4 == 0 (first-
 * order steps) do not read hist.  Held in its own engine buffer, next to the DDPM-form table, until replaced; the host
 * computes it (schedules.dpmpp_2m_coef).  DITTO_E_STATE without a loaded schedule, DITTO_E_BADARG if steps != diffusion_steps. */
int32_t ditto_engine_load_multistep_table(ditto_engine_t* e, const float* coef6, int64_t steps, void* stream);
/* Known frames (speech prompt, infilling; ditto_*_known below).  coef2 [diffusion_steps, 2] fp32 (device), row t =
 * {sqrt(abar_next), sqrt(1 - abar_next)}: the noise level of the OUTPUT of the step that starts at t, abar taken from the
 * sampler's own schedule (abar_next = 1 on the last visited step: row {1, 0}).  Held in its own engine buffer until replaced;
 * the host computes it (schedules.known_coef).  DITTO_E_STATE without a loaded schedule, DITTO_E_BADARG if
 * steps != diffusion_steps. */
int32_t ditto_engine_load_known_table(ditto_engine_t* e, const float* coef2, int64_t steps, void* stream);
/* Pack weights (bf16 copies, interleaved [fc1;gate], permuted QKV), build the per-step modulation table
 * time_mlp(SiLU(time_embed(t_embedding))) [steps, 2H] (DiTTO.py:75-76 + DiT.py:30) and the RoPE cos/sin
 * tables (DiT.py:46-59).  Synchronises the stream. */
int32_t ditto_engine_finalize(ditto_engine_t* e, void* stream);

/* ---- sizes ------------------------------------------------------------------------------------------ */
int64_t ditto_text_context_bytes(const ditto_engine_t* e, int64_t n_seq, int64_t S);
int64_t ditto_workspace_bytes(const ditto_engine_t* e, int64_t n_seq, int64_t T, int64_t S);

/* ---- hot path --------------------------------------------------------------------------------------- */
/* Step-invariant text work for n_seq sequences: mean-pooled text modulation text_mlp(SiLU(mean_S(text)))
 * (DiT.py:27,31) and every layer's cross-attention K/V projection (DiT.py:144-148 -> torch MHA in_proj).
 * text_emb [n_seq, S, text_dim].  ctx: caller buffer of ditto_text_context_bytes(). */
int32_t ditto_text_context(ditto_engine_t* e, const float* text_emb, int64_t n_seq, int64_t S, void* ctx,
                           void* workspace, int64_t workspace_bytes, void* stream);

/* eps_hat = DiTTO.forward(x, text_emb, t)   (src/model/DiTTO.py:66-94)
 * x [n_x, T, H]; sequence i of n_seq reads x[i % n_x] (n_seq % n_x == 0; CFG: n_seq = 2 n_x shares x
 * between the conditional and unconditional branch); t [n_seq] int64 (device); out [n_seq, T, H]. */
int32_t ditto_forward(ditto_engine_t* e, const float* x, int64_t n_x, const void* ctx, const int64_t* t,
                      int64_t n_seq, int64_t T, int64_t S, float* out, void* workspace,
                      int64_t workspace_bytes, void* stream);

/* Fused classifier-free-guidance combine + DDPM ancestral update (SpeechGenerator.py:137-147):
 *   eps = eps_u + w (eps_c - eps_u)           (eps_u == NULL: eps = eps_c, the reference's no-guidance case)
 *   x_out = 1/sqrt(alpha_t) (x - (1-alpha_t)/sqrt(1-acp_t) eps) + [t>0] sqrt(beta_t) z
 * all [B, T*H] fp32; t [B] int64 (device); z == NULL: no noise term.  x_out may alias x. */
int32_t ditto_cfg_ddpm_update(ditto_engine_t* e, const float* eps_c, const float* eps_u, const float* x,
                              const float* z, const int64_t* t, float guidance_scale, float* x_out,
                              int64_t B, int64_t elems_per_seq, void* stream);

/* One sampler iteration == SpeechGenerator.__p_sample (SpeechGenerator.py:131-147) with the CFG
 * extension: ditto_forward on n_seq = (guided ? 2B : B) sequences sharing x, then ditto_cfg_ddpm_update.
 * ctx holds [cond(B); uncond(B)] when guided.  t [n_seq] int64.  eps_scratch [n_seq, T, H]. */
int32_t ditto_p_sample(ditto_engine_t* e, const float* x, const void* ctx, const int64_t* t, const float* z,
                       int32_t guided, float guidance_scale, int64_t B, int64_t T, int64_t S,
                       float* eps_scratch, float* x_out, void* workspace, int64_t workspace_bytes,
                       void* stream);

/* The same with the step's noise z = randn_like(x) (SpeechGenerator.py:145) drawn INSIDE the fused update kernel: Philox4x32-10
 * + Box-Muller, element i of draw k of seed s always gets the same normal.  rng: device uint64[4] = {seed, draw counter,
 * 0 (ticket, owned by the kernel), reserved}; t is read-write here.  advance != 0: when the update is done the kernel adds 1 to
 * the draw counter and subtracts 1 from every t[i] (i < n_seq) -- the bookkeeping of `for t_val in reversed(range(steps))`
 * (SpeechGenerator.py:161-162) -- so that ONE captured CUDA graph of this call can be replayed step after step and contains
 * kernels of this library only. */
int32_t ditto_p_sample_rng(ditto_engine_t* e, const float* x, const void* ctx, int64_t* t, uint64_t* rng, int32_t guided,
                           float guidance_scale, int64_t B, int64_t T, int64_t S, float* eps_scratch, float* x_out,
                           void* workspace, int64_t workspace_bytes, int32_t advance, void* stream);
/* ditto_cfg_ddpm_update with in-kernel noise; t [n_t] (n_t >= B; all n_t entries are decremented when advance != 0). */
int32_t ditto_cfg_ddpm_update_rng(ditto_engine_t* e, const float* eps_c, const float* eps_u, const float* x, uint64_t* rng,
                                  int64_t* t, int64_t n_t, float guidance_scale, float* x_out, int64_t B,
                                  int64_t elems_per_seq, int32_t advance, void* stream);
/* out[i] = the N(0,1) sample the update kernels draw for element elem_offset + i at the current {seed, draw counter}
 * (elem_offset % 4 == 0, out 16-B aligned): stand-alone randn on the library's stream of numbers; parity tests. */
int32_t ditto_randn(const uint64_t* rng, int64_t elem_offset, float* out, int64_t n, void* stream);

/* Multistep forms of the four calls above: the same arguments plus hist [B, T, H] (ragged: packed like x, [sum n_x*T, H]),
 * read on second-order rows and overwritten with this step's x0 prediction; the update reads ditto_engine_load_multistep_table's
 * table (DITTO_E_STATE before one was loaded).  One launch per step, like their DDPM-form twins; x_out may alias x.  A row
 * with c4 == 0 gives x_out bit-identical to ditto_cfg_ddpm_update(_rng) with (c1, c2, c3). */
int32_t ditto_cfg_multistep_update(ditto_engine_t* e, const float* eps_c, const float* eps_u, const float* x,
                                   const float* z, const int64_t* t, float guidance_scale, float* x_out, float* hist,
                                   int64_t B, int64_t elems_per_seq, void* stream);
int32_t ditto_cfg_multistep_update_rng(ditto_engine_t* e, const float* eps_c, const float* eps_u, const float* x, uint64_t* rng,
                                       int64_t* t, int64_t n_t, float guidance_scale, float* x_out, float* hist, int64_t B,
                                       int64_t elems_per_seq, int32_t advance, void* stream);
int32_t ditto_p_sample_multistep(ditto_engine_t* e, const float* x, const void* ctx, const int64_t* t, const float* z,
                                 int32_t guided, float guidance_scale, int64_t B, int64_t T, int64_t S,
                                 float* eps_scratch, float* x_out, float* hist, void* workspace, int64_t workspace_bytes,
                                 void* stream);
int32_t ditto_p_sample_multistep_rng(ditto_engine_t* e, const float* x, const void* ctx, int64_t* t, uint64_t* rng,
                                     int32_t guided, float guidance_scale, int64_t B, int64_t T, int64_t S,
                                     float* eps_scratch, float* x_out, float* hist, void* workspace,
                                     int64_t workspace_bytes, int32_t advance, void* stream);

/* Known frames: replacement conditioning (the imputation of Song et al. 2021, score SDE) for a speech prompt
 * (known_mask[b, :P] = 1) or an infilled span.  known [B, T, H] holds the given latents p, known_mask [B, T] uint8 (nonzero =
 * known).  Frames that are not known take exactly the update of the calls above (bit-identical: the DDPM-form table, or with
 * hist != NULL the multistep table); a known frame becomes
 *     x_out = a p + s z,     {a, s} = the row t of ditto_engine_load_known_table's table
 * where z is the normal the update uses for that element.  Known frames read neither eps, x nor hist and leave hist as it was.
 * Exactly one of z (supplied noise [B, T, H]) or rng (in-kernel noise, as ditto_p_sample_rng) is non-NULL; advance != 0
 * needs rng.  DITTO_E_STATE without a known table (or, with hist, without a multistep table).  One launch per step, like the
 * calls above; x_out may alias x.  t [n_t] (n_t >= B) is read-write when advance != 0. */
int32_t ditto_cfg_update_known(ditto_engine_t* e, const float* eps_c, const float* eps_u, const float* x, const float* z,
                               uint64_t* rng, int64_t* t, int64_t n_t, float guidance_scale, float* x_out, float* hist,
                               const float* known, const uint8_t* known_mask, int64_t B, int64_t T, int32_t advance,
                               void* stream);
/* ditto_p_sample / _rng / _multistep(_rng) with known frames: the forward on (guided ? 2B : B) sequences sharing x (the
 * known frames are seen by both CFG branches), then ditto_cfg_update_known. */
int32_t ditto_p_sample_known(ditto_engine_t* e, const float* x, const void* ctx, int64_t* t, const float* z, uint64_t* rng,
                             int32_t guided, float guidance_scale, int64_t B, int64_t T, int64_t S, float* eps_scratch,
                             float* x_out, float* hist, const float* known, const uint8_t* known_mask, void* workspace,
                             int64_t workspace_bytes, int32_t advance, void* stream);

/* DiTTO.q_sample (DiTTO.py:106-126) with the reference's betas-as-alphas_cumprod buffer. */
int32_t ditto_q_sample(ditto_engine_t* e, const float* x_start, const float* noise, const int64_t* t,
                       float* out, int64_t B, int64_t elems_per_seq, void* stream);

/* ---- ragged (mixed-length) batches: BASELINE.json config 5 ------------------------------------------------
 * The reference has no padding masks (DiT.py:131-148 attends over every frame it is given), so utterances of different
 * length must run UNPADDED to match it.  A ragged batch is a list of groups of equal-length sequences; x, z, x_out are
 * packed group after group ([sum n_x*T, H]), t/out/eps_scratch likewise in sequence order ([sum n_seq], [sum n_seq*T, H]).
 * Row-wise work (LayerNorm, QKV/GLU/fc2/projection GEMMs) runs once over all packed rows; AdaLN modulation, RoPE
 * positions and both attentions run per group.  Each group has its own text context (ditto_text_context on its n_seq
 * sequences, S tokens each). */
typedef struct ditto_seq_group {
  int64_t n_seq;   /* sequences in the group; CFG: n_x conditional then n_x unconditional                 */
  int64_t n_x;     /* distinct latents: sequence i reads the group's x[i % n_x]  (n_seq % n_x == 0)      */
  int64_t T;       /* latent frames of every sequence of the group                                      */
  int64_t S;       /* text tokens of every sequence of the group                                        */
  const void* ctx; /* device buffer filled by ditto_text_context(e, text[n_seq,S,text_dim], n_seq, S, ...) */
} ditto_seq_group_t;
int64_t ditto_workspace_bytes_ragged(const ditto_engine_t* e, const ditto_seq_group_t* groups, int64_t n_groups);
/* DiTTO.forward (DiTTO.py:66-94) on every sequence of the ragged batch, each at its own length. */
int32_t ditto_forward_ragged(ditto_engine_t* e, const float* x, const ditto_seq_group_t* groups, int64_t n_groups,
                             const int64_t* t, float* out, void* workspace, int64_t workspace_bytes, void* stream);
/* __p_sample (SpeechGenerator.py:131-147) + CFG on a ragged batch; guided: every group has n_seq == 2 n_x. */
int32_t ditto_p_sample_ragged(ditto_engine_t* e, const float* x, const ditto_seq_group_t* groups, int64_t n_groups,
                              const int64_t* t, const float* z, int32_t guided, float guidance_scale,
                              float* eps_scratch, float* x_out, void* workspace, int64_t workspace_bytes, void* stream);

/* ditto_p_sample_ragged with in-kernel noise (element offset = position in the packed latent buffer) and, with advance != 0,
 * the t / draw-counter bookkeeping in a one-block kernel after the per-group updates.  t [sum n_seq] is read-write. */
int32_t ditto_p_sample_ragged_rng(ditto_engine_t* e, const float* x, const ditto_seq_group_t* groups, int64_t n_groups,
                                  int64_t* t, uint64_t* rng, int32_t guided, float guidance_scale, float* eps_scratch,
                                  float* x_out, void* workspace, int64_t workspace_bytes, int32_t advance, void* stream);
/* Multistep forms of the two ragged calls (hist packed like x; each group's update runs on its fork stream). */
int32_t ditto_p_sample_ragged_multistep(ditto_engine_t* e, const float* x, const ditto_seq_group_t* groups, int64_t n_groups,
                                        const int64_t* t, const float* z, int32_t guided, float guidance_scale,
                                        float* eps_scratch, float* x_out, float* hist, void* workspace,
                                        int64_t workspace_bytes, void* stream);
int32_t ditto_p_sample_ragged_multistep_rng(ditto_engine_t* e, const float* x, const ditto_seq_group_t* groups, int64_t n_groups,
                                            int64_t* t, uint64_t* rng, int32_t guided, float guidance_scale,
                                            float* eps_scratch, float* x_out, float* hist, void* workspace,
                                            int64_t workspace_bytes, int32_t advance, void* stream);
/* The ragged calls with known frames (ditto_p_sample_known): known packed like x, known_mask uint8 [sum n_x*T] (one byte per
 * packed latent row); noise offsets are packed positions, each group's update runs on its fork stream and advance != 0
 * runs the bookkeeping in a one-block kernel after them. */
int32_t ditto_p_sample_ragged_known(ditto_engine_t* e, const float* x, const ditto_seq_group_t* groups, int64_t n_groups,
                                    int64_t* t, const float* z, uint64_t* rng, int32_t guided, float guidance_scale,
                                    float* eps_scratch, float* x_out, float* hist, const float* known,
                                    const uint8_t* known_mask, void* workspace, int64_t workspace_bytes, int32_t advance,
                                    void* stream);

/* ---- block-level operators: the component signatures of src/components/DiT.py ------------------------------- */
/* DiT.forward(x, text_emb, time_emb, rotary_pos) (DiT.py:100-157) for block `layer` of the engine: x [n_seq, T, H] -> out
 * [n_seq, T, H] (may alias x).  time_emb is ignored by the reference block (DiT.py:100: never read); rotary_pos is the
 * engine's own table = RotaryEmbedding.forward(T) (DiT.py:56-59).  ctx: ditto_text_context of the block's text_emb. */
int32_t ditto_dit_block(ditto_engine_t* e, int32_t layer, const float* x, const void* ctx, int64_t n_seq, int64_t T,
                        int64_t S, float* out, void* workspace, int64_t workspace_bytes, void* stream);
/* The three sections of that block on their own, each from its LayerNorm to its residual add, same arguments as
 * ditto_dit_block (SURVEY 8b: ditto_attn_self / ditto_attn_cross):
 *   ditto_attn_self   x + merge_heads(softmax(rope(q) rope(k)^T / sqrt(d)) v),  q|k|v = norm1(x) attn.in_proj     DiT.py:103-139
 *   ditto_attn_cross  x + MHA(norm2(x), text, text) (torch math path, out_proj applied)                         DiT.py:141-148
 *   ditto_gated_mlp   x + fc2(GELU_erf(fc1(u)) * sigmoid(gate(u))),  u = norm3(x)                               DiT.py:150-155
 * They run the same kernels as the block (flash-style attention, folded / fused cross-attention, GLU GEMM + fc2 cluster GEMM);
 * ditto_dit_block == the three in this order. */
int32_t ditto_attn_self(ditto_engine_t* e, int32_t layer, const float* x, const void* ctx, int64_t n_seq, int64_t T,
                        int64_t S, float* out, void* workspace, int64_t workspace_bytes, void* stream);
int32_t ditto_attn_cross(ditto_engine_t* e, int32_t layer, const float* x, const void* ctx, int64_t n_seq, int64_t T,
                         int64_t S, float* out, void* workspace, int64_t workspace_bytes, void* stream);
int32_t ditto_gated_mlp(ditto_engine_t* e, int32_t layer, const float* x, const void* ctx, int64_t n_seq, int64_t T,
                        int64_t S, float* out, void* workspace, int64_t workspace_bytes, void* stream);
/* GlobalAdaLN.forward(x, time_emb, text_emb) (DiT.py:25-40), no engine needed: x [n_seq, T, H], time_emb [n_seq, time_dim],
 * text_emb [n_seq, S, text_dim]; w_time [2H, time_dim], b_time [2H] = time_mlp.1.*; w_text [2H, text_dim], b_text [2H] =
 * text_mlp.1.*; out [n_seq, T, H] (may alias x). */
int64_t ditto_adaln_workspace_bytes(int64_t n_seq, int64_t H, int64_t time_dim, int64_t text_dim);
int32_t ditto_adaln(const float* x, const float* time_emb, const float* text_emb, const float* w_time, const float* b_time,
                    const float* w_text, const float* b_text, float* out, int64_t n_seq, int64_t T, int64_t S, int64_t H,
                    int64_t time_dim, int64_t text_dim, void* workspace, int64_t workspace_bytes, void* stream);
/* RotaryEmbedding.apply_rope(pos, t) (DiT.py:52-54,61-72): out = t cos(pos) + rotate_half(t) sin(pos); t, out
 * [batch, T, heads, head_dim], pos [T, head_dim] fp32 angles (RotaryEmbedding.forward's return value). */
int32_t ditto_rope(const float* t, const float* pos, float* out, int64_t batch, int64_t T, int64_t heads, int64_t head_dim,
                   void* stream);

/* The attention core of DiT.forward for ONE head of 768 (DiT.py:117-139: softmax(alpha q k^T) v, no out_proj) + residual
 * + the LayerNorm that follows (norm2, DiT.py:143) in one kernel; bf16 operands, fp32 accumulation / softmax / statistics.
 * qkv [n_seq * T, ld] bf16: q at column 0 and k at column 768 (both already rotated), v at column 1536 with its columns in
 * the order the fused QKV epilogue stores them: position 64 b + 8 kb + 2 q + e (kb < 8, q < 4, e < 2) holds column
 * 64 b + 16 (kb / 2) + 4 q + 2 (kb % 2) + e.  h [n_seq * T, 768] fp32 in/out; u_out bf16 = LayerNorm(h) gamma + beta, or NULL.
 * flags bit 0: take the online-softmax rescale path whenever a key tile raises a row maximum (tests). */
int32_t ditto_attn_self768(const void* qkv, int64_t ld, int64_t n_seq, int64_t T, float alpha, float* h, const float* gamma,
                           const float* beta, void* u_out, int32_t flags, void* stream);

/* ---- single operators (unit-tested against the oracle; also usable on their own) --------------------- */
/* y = LayerNorm(x) * gamma + beta over the last dim (eps 1e-5, biased variance; DiT.py:84,89,94).
 * gamma/beta may be NULL (no affine, DiT.py:23).  out_bf16 != 0: y is written as bf16. */
int32_t ditto_layernorm(const float* x, const float* gamma, const float* beta, void* y, int32_t out_bf16,
                        int64_t rows, int64_t H, void* stream);
/* C[b] = alpha * A[b] @ op(B[b]) (+ bias) (+ resid), fp32 CUDA-core path.  A [M,K] lda; b_is_nk: B [N,K]
 * (y = x W^T, F.linear) else B [K,N].  batch strides in elements. */
int32_t ditto_gemm_f32(const float* A, int64_t lda, int64_t strideA, const float* B, int64_t ldb,
                       int64_t strideB, int32_t b_is_nk, float* C, int64_t ldc, int64_t strideC,
                       const float* bias, const float* resid, float alpha, int64_t M, int64_t N, int64_t K,
                       int64_t batch, void* stream);
/* C = alpha * A @ W^T (+bias) (+resid) with bf16 operands on tcgen05 tensor cores, fp32 accumulation in
 * TMEM.  A [M,K] bf16 (lda), W [N,K] bf16 (ldw); out fp32 or bf16 (out_bf16).  K % 8 == 0. */
int32_t ditto_gemm_bf16(const void* A, int64_t lda, const void* W, int64_t ldw, void* C, int64_t ldc,
                        int32_t out_bf16, const float* bias, const float* resid, int64_t ldr, float alpha,
                        int64_t M, int64_t N, int64_t K, void* stream);
/* The gated MLP's second linear with what follows it, in one cluster kernel (csrc/gemm_resid_ln.cu; reference
 * src/components/DiT.py:152-155 `x = residual + mlp_fc2(...)` and the next block's `norm1`, DiT.py:105):
 *   h <- h + A W^T + bias          (fp32, in place; A [M,K] bf16, W [N,K] bf16)
 *   u <- LayerNorm(h) gamma + beta (bf16; eps 1e-5, biased variance)   -- gamma == NULL: u <- bf16(h), u may be NULL
 * N in {256, 512, 768, 1024}, K % 8 == 0.  W holds the rows of the nn.Linear weight in the order
 * ditto_gemm_resid_ln_weight_row(r) -> source row of packed row r (a fixed permutation inside every 64-row block that
 * makes a thread's accumulators four consecutive outputs); bias / gamma / beta / h / u are in plain column order. */
int32_t ditto_gemm_resid_ln_weight_row(int32_t packed_row);
int32_t ditto_gemm_resid_ln(const void* A, int64_t lda, const void* W, int64_t ldw, const float* bias, float* h, int64_t ldh,
                            const float* gamma, const float* beta, void* u, int64_t ldu, int64_t M, int64_t N, int64_t K,
                            void* stream);
/* fp32 -> bf16 (round to nearest even) */
int32_t ditto_cast_bf16(const float* x, void* y, int64_t n, void* stream);

/* ---- hand-off steps either side of the sampling loop (fp32, like the reference) ----------------------- */
/* |c|^2 of every codebook row: torch.sum(self.codebook**2, dim=1), VectorQuantizer.py:37.  codebook [codes, dim] ->
 * sqnorm [codes].  Step-invariant: compute once per codebook. */
int32_t ditto_vq_code_sqnorm(const float* codebook, int64_t codes, int64_t dim, float* sqnorm, void* stream);
/* VectorQuantizer.forward (VectorQuantizer.py:22-43): indices = argmin_k (|z|^2 - 2 z.c_k + |c_k|^2), fp32, lowest index
 * on ties.  latents [batch, frames, dim]; indices int64 [batch, repeat_channels, frames]: repeat_channels > 1 writes the
 * same index to every channel, which is what quantising latents.unsqueeze(1).repeat(1, C, 1, 1) gives
 * (SpeechGenerator.py:117-118) without the C-fold work.  A general [B, C, T, dim] input is batch = B*C, repeat 1. */
int32_t ditto_vq_encode(const float* latents, int64_t batch, int64_t frames, int64_t dim, const float* codebook,
                        int64_t codes, const float* code_sqnorm, int64_t repeat_channels, int64_t* indices,
                        void* stream);
/* audio_latents[:, :, :max_frames].mean(dim=1) (TrainDiTTO.py:70-71, :113-114): latents [batch, channels, frames, dim]
 * -> out [batch, min(frames, max_frames), dim].  dim % 4 == 0. */
int32_t ditto_pool_latents(const float* latents, int64_t batch, int64_t channels, int64_t frames, int64_t dim,
                           int64_t max_frames, float* out, void* stream);
/* nn.MSELoss() (TrainDiTTO.py:51,87,126): loss[0] = mean((a - b)^2) over n elements; deterministic two-stage
 * reduction, workspace of ditto_mse_workspace_bytes() (8-byte aligned). */
int64_t ditto_mse_workspace_bytes(void);
int32_t ditto_mse_loss(const float* a, const float* b, int64_t n, float* loss, void* workspace,
                       int64_t workspace_bytes, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* DITTO_B200_H_ */
