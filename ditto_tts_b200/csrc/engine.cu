// C-ABI entry points (include/ditto_b200.h) and the host-side orchestration of one DiTTO forward / sampler step.
// Semantics follow the reference line by line (citations: src/model/DiTTO.py, src/components/DiT.py,
// src/model/SpeechGenerator.py of Tikai7/DiTTO-TTS); the arithmetic runs in the kernels of this library only.
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <mutex>
#include <vector>

#include "kernels.cuh"

namespace ditto {

// ---------------------------------------------------------------------------------------------------
// error plumbing
// ---------------------------------------------------------------------------------------------------
static thread_local std::string t_last_error;
std::atomic<long long> g_launches{0};
DebugOptions g_opt;
void set_error(const std::string& msg) { t_last_error = msg; }
int cuda_fail(cudaError_t err, const char* what, const char* file, int line) {
  t_last_error = std::string("CUDA error ") + std::to_string(static_cast<int>(err)) + " (" + cudaGetErrorString(err) + ") at " +
                 what + " [" + file + ":" + std::to_string(line) + "]";
  return DITTO_E_CUDA;
}

// ---------------------------------------------------------------------------------------------------
// opt-in profiler: one CUDA event pair per launcher call, accumulated per class on ditto_profile_stop()
// ---------------------------------------------------------------------------------------------------
bool g_prof_enabled = false;
namespace {
struct ProfRec { int cls; cudaEvent_t a, b; double flops, bytes; };
std::vector<ProfRec> g_prof_recs;
struct ProfAcc { long long launches = 0; double ms = 0, flops = 0, bytes = 0; };
ProfAcc g_prof_acc[PC_COUNT];
const char* kProfNames[PC_COUNT] = {"tc_gemm.proj_in", "tc_gemm.qkv_rope", "tc_gemm.self_scores", "tc_gemm.self_pv", "tc_gemm.cross_q",
                                    "tc_gemm.cross_scores", "tc_gemm.cross_pv", "tc_gemm.cross_out", "tc_gemm.glu", "tc_gemm.fc2",
                                    "tc_gemm.proj_out", "tc_gemm.text_kv", "tc_gemm.other", "sgemm_f32", "layernorm", "adaln_ln",
                                    "rope", "softmax", "cfg_ddpm_update", "elementwise", "tc_gemm.cross_fused_ln", "tc_gemm.flash_attn",
                                    "tc_gemm.flash768_ln", "tc_gemm.cross_flash_ln"};
}  // namespace
ProfScope::ProfScope(int cls, cudaStream_t stream, double flops, double bytes) : st(stream) {
  if (!g_prof_enabled) return;
  ProfRec r;
  r.cls = cls; r.flops = flops; r.bytes = bytes;
  if (cudaEventCreate(&r.a) != cudaSuccess || cudaEventCreate(&r.b) != cudaSuccess) return;
  cudaEventRecord(r.a, st);
  g_prof_recs.push_back(r);
  slot = static_cast<int>(g_prof_recs.size()) - 1;
}
ProfScope::~ProfScope() {
  if (slot >= 0) cudaEventRecord(g_prof_recs[slot].b, st);
}

// bump allocator over a caller buffer; with base == nullptr it only measures
struct Arena {
  char* base;
  size_t off = 0;
  explicit Arena(void* b) : base(static_cast<char*>(b)) {}
  template <typename T>
  T* take(int64_t n) {
    off = (off + 255) & ~static_cast<size_t>(255);
    T* p = base ? reinterpret_cast<T*>(base + off) : nullptr;
    off += static_cast<size_t>(n) * sizeof(T);
    return p;
  }
};

struct LayerPack {
  bf16 *w_qkv = nullptr, *wc_in = nullptr, *wc_o = nullptr, *w_glu = nullptr, *w_fc2 = nullptr;
  bf16* wc_o_p4 = nullptr;   // cross_attn.out_proj rows in the perm4 order of gemm_resid_ln.cu (fc2_ln engines; wc_o stays plain for the fold)
  float *b_qkv = nullptr, *b_glu = nullptr;  // permuted / interleaved copies
  // deferred LayerNorm (DITTO_F_DEFER_LN): w_qkv / w_glu carry gamma1 / gamma3, b_* carry W beta, c_* = row sums of the
  // scaled bf16 weights; wq_g / bq_g = cross-attention query projection with gamma2 / beta2 folded in (folded cross path)
  float *c_qkv = nullptr, *c_glu = nullptr, *bq_g = nullptr;
  bf16* wq_g = nullptr;
};

}  // namespace ditto

using namespace ditto;

struct ditto_engine {
  ditto_config_t cfg;
  int H = 0, L = 0, heads = 0, d = 0, half = 0, Td = 0, Xd = 0, steps = 0, maxT = 0;
  bool bf16_mode = false, fused_rope = false, finalized = false, have_schedule = false;
  bool blocks_only = false;  // DITTO_F_BLOCKS_ONLY: a stack of DiT blocks without the DiTTO wrapper (stand-alone DiT modules)
  int device = -1;           // CUDA device the engine was created on (kernel attributes / SM count are per device)
  int rope_pd = 0;
  bool glu_perm16 = false;  // [fc1; gate] rows packed for the lean GEGLU epilogue (TcGemmParams::glu_perm16)
  bool pv_perm4 = false;    // v columns stored in the order the float4 P.V epilogue wants (TcGemmParams::out_perm4)
  bool qkv_perm16 = false;  // QKV weight rows also permuted inside 64-row blocks for the lean RoPE epilogue (TcGemmParams::rope_perm16)
  bool cross_flash = false; // folded cross-attention with 64 < S <= 256 text tokens through flash_attn768q<CROSS> (+ residual + norm3)
  bool fc2_ln = false;      // fc2 + residual + the next block's norm1 in one cluster kernel (gemm_resid_ln.cu); w_fc2 rows in perm4 order
  bool flash768 = false;    // one head of 768 (repo default): self-attention + residual + norm2 in one cluster kernel (flash_attn768.cu)
  bool flash_attn = true;   // head_dim 64: self-attention without materialised scores (flash_attn.cu); DITTO_NO_FLASH=1 disables
  bool defer_ln2 = false;   // norm2 only: row statistics from the self-attention P.V epilogue, LayerNorm folded into cross_fused's scores
  bool fused_cross = true;  // folded cross-attention + residual + norm3 in one kernel (cross_fused.cu); DITTO_NO_FUSED_CROSS=1 disables
  bool fused_attn = false;  // scores + softmax fused (cluster kernel); falls back per call when a row needs > 16 tiles
  bool fold_cross = false;  // cross-attn q/out projections folded into the per-utterance text K/V (heads == 1 only)
  bool defer_ln = false;    // block LayerNorms folded into the neighbouring GEMM epilogues (no LayerNorm launches)
  bool const_text = true;   // sequences with constant text rows: constant cross-attention output added by the self-attention kernel
  int pv_transpose = 0;  // debug: use the transposed-V operand instead of the MN-major descriptor
  bool rope_table_in_epilogue = false;  // debug (DITTO_ROPE_TABLE=1): fused RoPE reads the cos/sin tables instead of computing them
  std::map<std::string, int64_t> expected;  // key -> numel
  std::map<std::string, float*> w;          // device fp32 copies (owned)
  std::vector<void*> owned;                 // everything else cudaMalloc'ed by the engine
  float *time_table = nullptr, *rope_cos = nullptr, *rope_sin = nullptr, *rope_freq = nullptr, *coef = nullptr, *qs_buf = nullptr;
  float* coef_ms = nullptr;  // [steps, 6] multistep update table (ditto_engine_load_multistep_table); null until loaded
  float* coef_known = nullptr;  // [steps, 2] re-noising table of known frames (ditto_engine_load_known_table); null until loaded
  bf16 *w_in16 = nullptr, *w_out16 = nullptr;
  bf16* w_out_p4 = nullptr;   // proj_out rows in the perm4 order of gemm_resid_ln.cu (fc2_ln engines)
  std::vector<LayerPack> layers;
  // ragged batches: the per-group launches (small attention kernels) are spread over side streams so that groups overlap
  // on the GPU; fork/join with events, which CUDA-graph capture turns into parallel branches.  The mutex serialises the
  // ENQUEUE of ragged forwards from different host threads (the fork event is re-recorded by every call).
  static constexpr int kSide = 8;
  cudaStream_t side[kSide] = {};
  cudaEvent_t ev_fork = nullptr, ev_join[kSide] = {};
  int n_side = 0;
  std::recursive_mutex fork_mutex;

  const float* W(const std::string& k) const {
    auto it = w.find(k);
    return it == w.end() ? nullptr : it->second;
  }
  const float* LW(int i, const char* name) const { return W("blocks." + std::to_string(i) + "." + name); }
};

namespace ditto {

static int dev_alloc(ditto_engine* e, void** p, size_t bytes) {
  DITTO_CUDA(cudaMalloc(p, bytes ? bytes : 16));
  e->owned.push_back(*p);
  return 0;
}

static void build_expected(ditto_engine* e) {
  const int64_t H = e->H, Td = e->Td, Xd = e->Xd, St = e->steps;
  auto& m = e->expected;
  if (!e->blocks_only) {
    m["t_embedding.weight"] = St * Td;
    m["time_embed.0.weight"] = Td * Td; m["time_embed.0.bias"] = Td;
    m["time_embed.2.weight"] = Td * Td; m["time_embed.2.bias"] = Td;
    m["ada_ln.time_mlp.1.weight"] = 2 * H * Td; m["ada_ln.time_mlp.1.bias"] = 2 * H;
    m["ada_ln.text_mlp.1.weight"] = 2 * H * Xd; m["ada_ln.text_mlp.1.bias"] = 2 * H;
    m["proj_in.weight"] = H * H; m["proj_in.bias"] = H;
    m["proj_out.weight"] = H * H; m["proj_out.bias"] = H;
  }
  for (int i = 0; i < e->L; ++i) {
    const std::string p = "blocks." + std::to_string(i) + ".";
    for (const char* n : {"norm1", "norm2", "norm3"}) { m[p + n + ".weight"] = H; m[p + n + ".bias"] = H; }
    m[p + "attn.in_proj_weight"] = 3 * H * H; m[p + "attn.in_proj_bias"] = 3 * H;
    m[p + "cross_attn.in_proj_weight"] = 3 * H * H; m[p + "cross_attn.in_proj_bias"] = 3 * H;
    m[p + "cross_attn.out_proj.weight"] = H * H; m[p + "cross_attn.out_proj.bias"] = H;
    m[p + "mlp_fc1.weight"] = 4 * H * H; m[p + "mlp_fc1.bias"] = 4 * H;
    m[p + "gate.weight"] = 4 * H * H; m[p + "gate.bias"] = 4 * H;
    m[p + "mlp_fc2.weight"] = 4 * H * H; m[p + "mlp_fc2.bias"] = H;
  }
  m["rotary.inv_freq"] = e->half;  // optional
}

static bool ignorable_key(const std::string& k) {
  if (k.rfind("nac.", 0) == 0) return true;
  if (k == "alphas_cumprod") return true;  // the sampler tables come through ditto_engine_load_schedule
  if (k.size() > 9 && k.compare(k.size() - 9, 9, ".inv_freq") == 0 && k != "rotary.inv_freq") return true;
  if (k.find(".attn.out_proj.") != std::string::npos) return true;  // dead weights (DiT.py:137-139 never applies them)
  return false;
}

// simple fp32 GEMM helper: C[M,N] = alpha * A[M,K] @ W[N,K]^T + bias (+resid)
static int sgemm_nt(const float* A, int64_t lda, const float* Wt, int64_t ldw, float* C, int64_t ldc, const float* bias,
                    const float* resid, int64_t ldr, float alpha, int M, int N, int K, cudaStream_t st) {
  SgemmParams p;
  p.A = A; p.lda = lda; p.B = Wt; p.ldb = ldw; p.C = C; p.ldc = ldc; p.bias = bias; p.resid = resid; p.ldr = ldr;
  p.alpha = alpha; p.M = M; p.N = N; p.K = K; p.b_is_nk = true;
  return launch_sgemm(p, st);
}

// bf16 tensor-core helper: out = alpha * A[M,K] @ W[N,K]^T (+bias) (+resid)
static int tc_nt(const bf16* A, int64_t lda, const bf16* Wt, int64_t ldw, void* out, bool out_bf16, int64_t ldo,
                 const float* bias, const float* resid, int64_t ldr, int64_t resid_row_mod, bf16* out2, int64_t ldo2,
                 int M, int N, int K, cudaStream_t st, int tag = PC_TC_OTHER, float2* stat_out = nullptr, int stat_parts = 0) {
  TcGemmParams p;
  p.tag = tag;
  p.stat_out = stat_out; p.stat_parts = stat_parts;
  p.A.ptr = A; p.A.rows = M; p.A.cols = K; p.A.ld = lda;
  p.B.ptr = Wt; p.B.rows = N; p.B.cols = K; p.B.ld = ldw;
  p.M = M; p.N = N; p.K = K;
  p.bias = bias; p.out = out; p.out_bf16 = out_bf16; p.ldo = ldo;
  p.resid = resid; p.ldr = ldr; p.resid_row_mod = resid_row_mod; p.out2 = out2; p.ldo2 = ldo2;
  return launch_tc_gemm(p, st);
}

struct CtxLayout {
  float* text_mod = nullptr;  // [n, 2H]
  void* kv0 = nullptr;        // layer 0 K|V [n*S, 2H] (bf16 or fp32); layers are kv_stride bytes apart
  size_t kv_stride = 0;
  // folded cross-attention (bf16 path, DITTO_F_FOLD_CROSS): per layer
  //   kfold [n, heads, S, H]   = K_h Wq_h           (scores = u . kfold^T + sbias)
  //   vfold [n, heads*Sp, H]   = V_h Wo_h^T         (out = P . vfold + bo), zero rows for s >= S
  //   sbias [n, heads, Sp] f32 = sqrt(1/d) K_h bq_h
  //   cvec  [n, heads, Sp] f32 = row sums of the gamma2-scaled kfold (deferred LayerNorm only), strided like sbias
  // and, single head only, for sequences whose S text rows are all equal (the unconditional CFG half, S = 1):
  //   cflag [n] u8             = 1 when they are (cross-attention output = vfold[0] + bo for every query row)
  //   crow  [n, H] f32         = vfold[seq][0] + bo, plain column order, per layer
  bf16 *kfold0 = nullptr, *vfold0 = nullptr;
  float *sbias0 = nullptr, *cvec0 = nullptr, *crow0 = nullptr;
  uint8_t* cflag = nullptr;
  size_t kfold_stride = 0, vfold_stride = 0, sbias_stride = 0, crow_stride = 0;  // elements between layers
  size_t total = 0;
};
static bool fold_active(const ditto_engine* e, int64_t S) {
  // folding trades the two M x H x H projections for (heads*S)-wide products: only worth it when heads*S << H
  return e->bf16_mode && e->fold_cross && e->heads * round_up(S, 8) * 2 <= e->H;
}
// LN2 is folded into the cross-attention scores only on the folded path with a single key tile (fused scores kernel)
static bool fold_ln_active(const ditto_engine* e, int64_t S) {
  const bool want = e->defer_ln || (e->defer_ln2 && cross_fused_supported(1, S, e->H, e->heads));
  return want && fold_active(e, S) && tc_scores_softmax_csize(static_cast<int>(S)) == 1;
}
// text lengths the fused single-key-tile kernel (cross_fused.cu, S <= 64) does not cover go through the flash-style kernel
// (up to two key tiles); the V fold of such a context is built in that kernel's column order
static bool cross_flash_active(const ditto_engine* e, int64_t S) {
  return e->cross_flash && e->fused_cross && e->heads == 1 && S <= 256 && fold_active(e, S) && !cross_fused_supported(1, S, e->H, e->heads);
}
static CtxLayout ctx_layout(const ditto_engine* e, void* base, int64_t n, int64_t S) {
  Arena a(base);
  CtxLayout c;
  c.text_mod = a.take<float>(n * 2 * e->H);
  const int64_t kv_elems = n * S * 2 * e->H;
  a.take<char>(0);
  const size_t kv_bytes = ((static_cast<size_t>(kv_elems) * (e->bf16_mode ? 2 : 4)) + 255) & ~static_cast<size_t>(255);
  c.kv0 = a.take<char>(static_cast<int64_t>(kv_bytes) * e->L);
  c.kv_stride = kv_bytes;
  if (fold_active(e, S)) {
    const int64_t Sp = round_up(S, 8);
    c.kfold_stride = static_cast<size_t>(n * e->heads * S * e->H);
    c.vfold_stride = static_cast<size_t>(n * e->heads * Sp * e->H);
    c.sbias_stride = static_cast<size_t>(n * e->heads * Sp);
    c.kfold0 = a.take<bf16>(static_cast<int64_t>(c.kfold_stride) * e->L);
    c.vfold0 = a.take<bf16>(static_cast<int64_t>(c.vfold_stride) * e->L);
    c.sbias0 = a.take<float>(static_cast<int64_t>(c.sbias_stride) * e->L);
    if (e->defer_ln || e->defer_ln2) c.cvec0 = a.take<float>(static_cast<int64_t>(c.sbias_stride) * e->L);
    if (e->heads == 1) {
      c.crow_stride = static_cast<size_t>(n * e->H);
      c.cflag = a.take<uint8_t>(n);
      c.crow0 = a.take<float>(static_cast<int64_t>(c.crow_stride) * e->L);
    }
  }
  c.total = a.off + 256;
  return c;
}

// One group of equal-length sequences of a (possibly ragged) batch, with its offsets into the packed buffers.
struct SeqGroup {
  int64_t n = 0, n_x = 0, T = 0, S = 0;
  const void* ctx = nullptr;
  int64_t row0 = 0;    // first row of the group in the packed [M, *] activations (sequence layout)
  int64_t xrow0 = 0;   // first row of the group's latents in the packed x / z / x_out buffers
  int64_t seq0 = 0;    // index of the group's first sequence (t, per-sequence tables)
  int64_t p_off = 0;   // element offset of the group's score / P scratch
  int64_t l_off = 0;   // element offset of the group's partial-denominator scratch
  int64_t vt_off = 0;  // element offset of the transposed-V scratch (debug fallback)
};

struct Workspace {
  float *h = nullptr, *xskip = nullptr, *scores = nullptr;
  void *u = nullptr, *qkv = nullptr, *P = nullptr, *qc = nullptr, *oc = nullptr, *hid = nullptr, *xb16 = nullptr;
  float *fc1 = nullptr, *gate = nullptr;  // fp32 path only
  bf16* vt = nullptr;                     // transposed-V fallback
  float* lpart = nullptr;                 // [n*heads, T, ceil(Tp/256)] partial softmax denominators (fused attention)
  float2* lnstat = nullptr;               // [M, ln_parts] per-row partial (sum, sum of squares) of h (deferred LayerNorm)
  int ln_parts_h = 0, ln_parts_attn = 0;  // parts written by an N = H producer / by the per-head P.V producer
  float* tmp_small = nullptr;             // [n, Xd] pooled text
  bf16* text16 = nullptr;                 // [n*S, Xd]
  int* row_pos = nullptr;                 // [M] position of each packed row inside its sequence (ragged batches: RoPE)
  int64_t M = 0;                          // packed rows: sum over groups of n * T
  size_t total = 0;
};
// Lays the workspace out for `ng` groups and fills in the groups' offsets.  Token-wise buffers are sized by the packed
// row count; the attention scratch is the sum over groups (so groups may run concurrently).
static Workspace ws_layout(const ditto_engine* e, void* base, SeqGroup* gs, int ng) {
  Arena a(base);
  Workspace w;
  const int64_t H = e->H;
  const int es = e->bf16_mode ? 2 : 4;
  int64_t M = 0, Mx = 0, seqs = 0, p_el = 0, l_el = 0, vt_el = 0, n_tot = 0, text_el = 0;
  for (int i = 0; i < ng; ++i) {
    SeqGroup& g = gs[i];
    const int64_t ldp = std::max(round_up(g.T, 8), round_up(g.S, 8));
    g.row0 = M; g.xrow0 = Mx; g.seq0 = seqs; g.p_off = p_el; g.l_off = l_el; g.vt_off = vt_el;
    M += g.n * g.T; Mx += g.n_x * g.T; seqs += g.n;
    p_el += round_up(g.n * e->heads * g.T * ldp, 128);
    l_el += round_up(g.n * e->heads * g.T * ceil_div(ldp, 256), 64);
    vt_el += round_up(g.n * e->heads * e->d * ldp, 128);
    n_tot = std::max(n_tot, g.n);
    text_el = std::max(text_el, g.n * g.S);
  }
  w.M = M;
  w.h = a.take<float>(M * H);
  w.xskip = a.take<float>(M * H);
  w.u = a.take<char>(M * H * es);
  w.xb16 = a.take<char>(M * H * 2);
  w.qkv = a.take<char>(M * 3 * H * es);
  w.scores = a.take<float>(p_el);
  w.P = e->bf16_mode ? static_cast<void*>(a.take<bf16>(p_el)) : static_cast<void*>(w.scores);
  w.qc = a.take<char>(M * H * es);
  w.oc = a.take<char>(M * H * es);
  w.hid = a.take<char>(M * 4 * H * es);
  if (!e->bf16_mode) {
    w.fc1 = a.take<float>(M * 4 * H);
    w.gate = a.take<float>(M * 4 * H);
  } else if (e->pv_transpose) {
    w.vt = a.take<bf16>(vt_el);
  }
  if (e->bf16_mode) w.lpart = a.take<float>(l_el);
  w.ln_parts_h = static_cast<int>(ceil_div(H, 128));
  w.ln_parts_attn = static_cast<int>(e->heads * ceil_div(e->d, 128));
  if (e->defer_ln || e->defer_ln2) w.lnstat = a.take<float2>(M * std::max(w.ln_parts_h, w.ln_parts_attn));
  w.tmp_small = a.take<float>(n_tot * e->Xd);
  w.text16 = a.take<bf16>(text_el * e->Xd);
  if (ng > 1) w.row_pos = a.take<int>(M);
  w.total = a.off + 256;
  return w;
}
static Workspace ws_layout(const ditto_engine* e, void* base, int64_t n, int64_t T, int64_t S) {
  SeqGroup g;
  g.n = n; g.n_x = n; g.T = T; g.S = S;
  return ws_layout(e, base, &g, 1);
}

}  // namespace ditto

// ---------------------------------------------------------------------------------------------------
// attention cores (materialised scores; see DESIGN.md for the roofline discussion)
// ---------------------------------------------------------------------------------------------------
namespace ditto {

// bf16: scores = alpha * Q K^T (tcgen05) -> softmax -> P V (tcgen05, V as MN-major operand) (+ fp32 residual)
static int attention_bf16(ditto_engine* e, const Workspace& w, const bf16* q, int64_t ldq, int64_t q_seq_stride, const bf16* k,
                          int64_t ldk, int64_t k_seq_stride, const bf16* v, int64_t ldv, int64_t v_seq_stride, int64_t n, int Tq,
                          int Tk, float alpha, void* out, bool out_bf16, int64_t ldo, int64_t o_seq_stride, const float* resid,
                          cudaStream_t st, bool cross, bf16* out2 = nullptr, float2* stat_out = nullptr) {
  const int d = e->d, heads = e->heads;
  if (e->flash_attn && !cross && !out_bf16 && resid != nullptr && out2 == nullptr && stat_out == nullptr && flash_attn_supported(d, Tq, Tk)) {
    FlashAttnParams f;
    f.Q.ptr = q; f.Q.rows = Tq; f.Q.cols = d; f.Q.ld = ldq; f.Q.s_inner = d; f.Q.s_outer = q_seq_stride;
    f.Km.ptr = k; f.Km.rows = Tk; f.Km.cols = d; f.Km.ld = ldk; f.Km.s_inner = d; f.Km.s_outer = k_seq_stride;
    f.V.ptr = v; f.V.rows = Tk; f.V.cols = d; f.V.ld = ldv; f.V.s_inner = d; f.V.s_outer = v_seq_stride;
    f.n_seq = n; f.heads = heads; f.d = d; f.Tq = Tq; f.Tk = Tk; f.alpha = alpha;
    f.out = static_cast<float*>(out); f.resid = resid; f.ldo = ldo; f.o_seq = o_seq_stride; f.ldr = ldo; f.r_seq = o_seq_stride;
    f.tag = PC_FLASH_ATTN;
    return launch_flash_attn(f, st);
  }
  const int64_t ldp = round_up(Tk, 8);
  const int csize = e->fused_attn ? tc_scores_softmax_csize(Tk) : 0;
  if (csize > 0) {
    // flash-style: P = exp(s - rowmax) straight from TMEM (normalised in the kernel when one tile holds the row)
    TcScoresSoftmaxParams f;
    f.Q.ptr = q; f.Q.rows = Tq; f.Q.cols = d; f.Q.ld = ldq; f.Q.s_inner = d; f.Q.s_outer = q_seq_stride;
    f.Km.ptr = k; f.Km.rows = Tk; f.Km.cols = d; f.Km.ld = ldk; f.Km.s_inner = d; f.Km.s_outer = k_seq_stride;
    f.M = Tq; f.N = Tk; f.K = d; f.batch_inner = heads; f.batch_outer = static_cast<int>(n);
    f.alpha = alpha;
    f.P = static_cast<bf16*>(w.P); f.ldp = ldp; f.sp_inner = static_cast<int64_t>(Tq) * ldp;
    f.sp_outer = static_cast<int64_t>(heads) * Tq * ldp; f.npad = static_cast<int>(ldp);
    f.lpart = w.lpart; f.sl_inner = static_cast<int64_t>(Tq) * csize; f.sl_outer = static_cast<int64_t>(heads) * Tq * csize;
    f.tag = cross ? PC_TC_CROSS_SCORES : PC_TC_SELF_SCORES;
    DITTO_TRY(launch_tc_scores_softmax(f, st));
  } else {
    TcGemmParams g;
    g.A.ptr = q; g.A.rows = Tq; g.A.cols = d; g.A.ld = ldq; g.A.s_inner = d; g.A.s_outer = q_seq_stride;
    g.B.ptr = k; g.B.rows = Tk; g.B.cols = d; g.B.ld = ldk; g.B.s_inner = d; g.B.s_outer = k_seq_stride;
    g.M = Tq; g.N = Tk; g.K = d; g.batch_inner = heads; g.batch_outer = static_cast<int>(n);
    g.alpha = alpha; g.out = w.scores; g.out_bf16 = false; g.ldo = ldp; g.so_inner = static_cast<int64_t>(Tq) * ldp;
    g.so_outer = static_cast<int64_t>(heads) * Tq * ldp;
    g.tag = cross ? PC_TC_CROSS_SCORES : PC_TC_SELF_SCORES;
    DITTO_TRY(launch_tc_gemm(g, st));
    DITTO_TRY(launch_softmax(w.scores, ldp, w.P, true, ldp, n * heads * Tq, Tk, st));
  }
  TcGemmParams o;
  o.A.ptr = static_cast<const bf16*>(w.P); o.A.rows = Tq; o.A.cols = Tk; o.A.ld = ldp; o.A.s_inner = static_cast<int64_t>(Tq) * ldp;
  o.A.s_outer = static_cast<int64_t>(heads) * Tq * ldp;
  if (e->pv_transpose && w.vt) {  // fallback operand: V^T [d, Tp] per (seq, head), keys contiguous
    DITTO_TRY(launch_transpose_v(v, ldv, w.vt, n, Tk, static_cast<int>(ldp), heads, d, st));
    o.B.ptr = w.vt; o.B.rows = d; o.B.cols = Tk; o.B.ld = ldp; o.B.s_inner = static_cast<int64_t>(d) * ldp;
    o.B.s_outer = static_cast<int64_t>(heads) * d * ldp;
    o.b_kn = false;
  } else {
    o.B.ptr = v; o.B.rows = Tk; o.B.cols = d; o.B.ld = ldv; o.B.s_inner = d; o.B.s_outer = v_seq_stride;
    o.b_kn = true;
  }
  o.M = Tq; o.N = d; o.K = Tk; o.batch_inner = heads; o.batch_outer = static_cast<int>(n);
  o.out = out; o.out_bf16 = out_bf16; o.ldo = ldo; o.so_inner = d; o.so_outer = o_seq_stride;
  o.resid = resid; o.ldr = ldo; o.sr_inner = d; o.sr_outer = o_seq_stride;
  if (csize > 1) {  // P is unnormalised: divide by the summed partial denominators in the epilogue
    o.row_lsum = w.lpart; o.row_lparts = csize; o.sl_inner = static_cast<int64_t>(Tq) * csize;
    o.sl_outer = static_cast<int64_t>(heads) * Tq * csize;
  }
  o.tag = cross ? PC_TC_CROSS_PV : PC_TC_SELF_PV;
  o.out_perm4 = e->pv_perm4 && !cross && !out_bf16 && resid != nullptr && out2 == nullptr && stat_out == nullptr && e->fused_rope;
  if (out2 != nullptr) { o.out2 = out2; o.ldo2 = ldo; }
  if (stat_out != nullptr) { o.stat_out = stat_out; o.stat_parts = w.ln_parts_attn; o.stat_rows_outer = Tq; }
  DITTO_TRY(launch_tc_gemm(o, st));
  return 0;
}

static int attention_f32(ditto_engine* e, const Workspace& w, const float* q, int64_t ldq, int64_t q_seq_stride, const float* k,
                         int64_t ldk, int64_t k_seq_stride, const float* v, int64_t ldv, int64_t v_seq_stride, int64_t n, int Tq,
                         int Tk, float alpha, float* out, int64_t ldo, int64_t o_seq_stride, const float* resid, cudaStream_t st) {
  const int d = e->d, heads = e->heads;
  const int64_t ldp = round_up(Tk, 8);
  SgemmParams g;
  g.A = q; g.lda = ldq; g.sA_inner = d; g.sA_outer = q_seq_stride;
  g.B = k; g.ldb = ldk; g.sB_inner = d; g.sB_outer = k_seq_stride; g.b_is_nk = true;
  g.C = w.scores; g.ldc = ldp; g.sC_inner = static_cast<int64_t>(Tq) * ldp; g.sC_outer = static_cast<int64_t>(heads) * Tq * ldp;
  g.alpha = alpha; g.M = Tq; g.N = Tk; g.K = d; g.batch_inner = heads; g.batch_outer = static_cast<int>(n);
  DITTO_TRY(launch_sgemm(g, st));
  DITTO_TRY(launch_softmax(w.scores, ldp, w.scores, false, ldp, n * heads * Tq, Tk, st));
  SgemmParams o;
  o.A = w.scores; o.lda = ldp; o.sA_inner = static_cast<int64_t>(Tq) * ldp; o.sA_outer = static_cast<int64_t>(heads) * Tq * ldp;
  o.B = v; o.ldb = ldv; o.sB_inner = d; o.sB_outer = v_seq_stride; o.b_is_nk = false;
  o.C = out; o.ldc = ldo; o.sC_inner = d; o.sC_outer = o_seq_stride;
  o.resid = resid; o.ldr = ldo; o.sR_inner = d; o.sR_outer = o_seq_stride;
  o.M = Tq; o.N = d; o.K = Tk; o.batch_inner = heads; o.batch_outer = static_cast<int>(n);
  DITTO_TRY(launch_sgemm(o, st));
  return 0;
}

// Workspace view of one group: the attention scratch pointers moved to the group's slice.
static Workspace group_view(const ditto_engine* e, const Workspace& w, const SeqGroup& g) {
  Workspace v = w;
  v.scores = w.scores ? w.scores + g.p_off : nullptr;
  v.P = e->bf16_mode ? static_cast<void*>(static_cast<bf16*>(w.P) + g.p_off) : static_cast<void*>(v.scores);
  v.lpart = w.lpart ? w.lpart + g.l_off : nullptr;
  v.vt = w.vt ? w.vt + g.vt_off : nullptr;
  return v;
}

// fork / join of the per-group launches over the engine's side streams (no-op for a single group)
struct Fork {
  ditto_engine* e; cudaStream_t st; int used = 0;
  Fork(ditto_engine* e_, cudaStream_t st_) : e(e_), st(st_) {}
  int begin(int ng) {
    used = (ng > 1) ? std::min(ng, e->n_side) : 0;
    if (used == 0) return 0;
    DITTO_CUDA(cudaEventRecord(e->ev_fork, st));
    for (int k = 0; k < used; ++k) DITTO_CUDA(cudaStreamWaitEvent(e->side[k], e->ev_fork, 0));
    return 0;
  }
  cudaStream_t stream(int gi) const { return used ? e->side[gi % used] : st; }
  int end() {
    for (int k = 0; k < used; ++k) {
      DITTO_CUDA(cudaEventRecord(e->ev_join[k], e->side[k]));
      DITTO_CUDA(cudaStreamWaitEvent(st, e->ev_join[k], 0));
    }
    used = 0;
    return 0;
  }
};

// One DiTTO forward over `ng` groups of equal-length sequences packed back to back (group-major, sequences of a group
// contiguous).  Everything that works on single rows (LayerNorm, the QKV / GLU / fc2 / projection GEMMs) runs ONCE over
// all packed rows; only what depends on sequence boundaries (AdaLN modulation, attention, RoPE positions) runs per group.
// ng == 1 is the uniform batch of ditto_forward (x shared between CFG branches through n_x).
// block_layer >= 0: ONE DiT block on its own (DiT.forward, DiT.py:100-157 -> ditto_dit_block): x [n, T, H] is the block's input
// residual stream, out its output; no AdaLN / proj_in / proj_out, t unused.
// block_stage (block_layer >= 0 only): 0 = the whole block; 1 / 2 / 3 = its self-attention / cross-attention / gated-MLP
// section alone, each from its own LayerNorm to its residual add (DiT.py:103-139 / :141-148 / :150-155).
static int forward_impl(ditto_engine* e, const float* x, const int64_t* t, SeqGroup* gs, int ng, float* out, void* workspace,
                        int64_t workspace_bytes, cudaStream_t st, int block_layer = -1, int block_stage = 0) {
  const int H = e->H, d = e->d;
  const bool block_only = block_layer >= 0;
  const int stage = block_only ? block_stage : 0;
  const bool do_self = stage == 0 || stage == 1, do_cross = stage == 0 || stage == 2, do_mlp = stage == 0 || stage == 3;
  const int l_begin = block_only ? block_layer : 0, l_end = block_only ? block_layer + 1 : e->L;
  Workspace w = ws_layout(e, workspace, gs, ng);
  const int64_t M = w.M;
  DITTO_REQUIRE(M < (1ll << 31) / 8, DITTO_E_UNSUPPORTED, "forward: batch too large for one call (split it)");
  DITTO_REQUIRE(static_cast<int64_t>(w.total) <= workspace_bytes, DITTO_E_WORKSPACE, "forward: workspace too small");
  const bool ragged = ng > 1;
  const bool b16 = e->bf16_mode;
  const float inv_sqrt_d = 1.0f / sqrtf(static_cast<float>(d));          // DiT.py:131-132: scores / sqrt(d)
  const float sqrt_inv_d = sqrtf(1.0f / static_cast<float>(d));          // torch MHA: q * sqrt(1/d)
  DITTO_REQUIRE(!(ragged && e->defer_ln), DITTO_E_UNSUPPORTED, "forward: ragged batches do not support DITTO_F_DEFER_LN");
  const SeqGroup& g0 = gs[0];
  std::unique_lock<std::recursive_mutex> fork_lock(e->fork_mutex, std::defer_lock);
  if (ragged && e->n_side > 0) fork_lock.lock();
  Fork fork(e, st);

  // deferred LayerNorm: `u` holds bf16(h) and w.lnstat the row statistics; ln1_parts = parts written by the last producer
  const bool dln = e->defer_ln;
  const bool dln2_all = dln && fold_ln_active(e, g0.S);  // LN2 feeds the folded scores kernel; the unfolded q projection needs a real LN
  int ln1_parts = 1;
  if (block_only) {
    DITTO_REQUIRE(!ragged && !dln, DITTO_E_UNSUPPORTED, "dit_block: uniform batches without DITTO_F_DEFER_LN only");
    DITTO_CUDA(cudaMemcpyAsync(w.h, x, static_cast<size_t>(M) * H * sizeof(float), cudaMemcpyDeviceToDevice, st));
    const char* nw = stage == 2 ? "norm2.weight" : stage == 3 ? "norm3.weight" : "norm1.weight";     // DiT.py:105 / :143 / :152
    const char* nb = stage == 2 ? "norm2.bias" : stage == 3 ? "norm3.bias" : "norm1.bias";
    // cross-attention alone with norm2 folded into the text context (K Wq diag(gamma2), score bias with beta2): there are no
    // row statistics from a self-attention before it, so the query operand is the normalised row without the affine part
    const bool affine = !(stage == 2 && fold_ln_active(e, g0.S));
    DITTO_TRY(launch_layernorm(w.h, affine ? e->LW(l_begin, nw) : nullptr, affine ? e->LW(l_begin, nb) : nullptr, w.u, b16, M, H, st));
  }
  // AdaLN + LN1 of block 0 (+ bf16 copy of x for proj_in)                 DiTTO.py:86, DiT.py:25-40,105
  DITTO_TRY(fork.begin(block_only ? 0 : ng));
  for (int gi = 0; gi < ng && !block_only; ++gi) {
    const SeqGroup& g = gs[gi];
    CtxLayout c = ctx_layout(e, const_cast<void*>(g.ctx), g.n, g.S);
    const int es = b16 ? 2 : 4;
    // ragged: the bf16 copy of x is written for EVERY sequence (sequence layout) so that proj_in / proj_out stay single GEMMs
    bf16* xc = b16 ? static_cast<bf16*>(w.xb16) + (ragged ? g.row0 : g.xrow0) * H : nullptr;
    DITTO_TRY(launch_adaln_ln(x + g.xrow0 * H, g.n_x, e->time_table, c.text_mod, t + g.seq0, e->steps, e->LW(0, "norm1.weight"),
                              e->LW(0, "norm1.bias"), w.h + g.row0 * H, static_cast<char*>(w.u) + g.row0 * H * es, b16, xc, g.n,
                              static_cast<int>(g.T), H, fork.stream(gi), dln ? w.lnstat : nullptr, ragged,
                              ragged ? w.row_pos + g.row0 : nullptr));
  }
  DITTO_TRY(fork.end());
  // x_skip = proj_in(x): once per distinct x (uniform batch) / per packed row (ragged)      DiTTO.py:83
  if (block_only) {
  } else if (b16) {
    const int Mp = static_cast<int>(ragged ? M : g0.n_x * g0.T);
    DITTO_TRY(tc_nt(static_cast<bf16*>(w.xb16), H, e->w_in16, H, w.xskip, false, H, e->W("proj_in.bias"), nullptr, 0, 0, nullptr, 0, Mp, H,
                    H, st, PC_TC_PROJ_IN));
  } else {
    for (int gi = 0; gi < ng; ++gi)  // fp32: x-layout rows, group by group
      DITTO_TRY(sgemm_nt(x + gs[gi].xrow0 * H, H, e->W("proj_in.weight"), H, w.xskip + gs[gi].xrow0 * H, H, e->W("proj_in.bias"), nullptr, 0,
                         1.f, static_cast<int>(gs[gi].n_x * gs[gi].T), H, H, st));
  }

  // the fused cross-attention kernel also produces norm3's output; the decision is taken GROUP BY GROUP (one utterance with
  // more than 64 text tokens must not push the whole ragged batch onto the three-kernel path): a group that does not
  // qualify runs the composition and its own norm3 LayerNorm
  const bool fuse_cross_any = b16 && e->fused_cross && !dln;
  auto fuse_cross_group = [&](const SeqGroup& g) {
    return fuse_cross_any && fold_active(e, g.S) && cross_fused_supported(g.T, g.S, H, e->heads);
  };
  for (int i = l_begin; i < l_end; ++i) {
    const LayerPack& lp = e->layers[i];
    const bool last = (i == l_end - 1);
    if (b16) {
      bf16* u = static_cast<bf16*>(w.u);
      bf16* qkv = static_cast<bf16*>(w.qkv);
      // ---- self-attention: QKV projection (+RoPE), softmax(QK^T/sqrt d)V, + residual (no out_proj)   DiT.py:103-139
      if (do_self) {
        TcGemmParams g;
        g.A.ptr = u; g.A.rows = M; g.A.cols = H; g.A.ld = H;
        g.B.ptr = lp.w_qkv; g.B.rows = 3 * H; g.B.cols = H; g.B.ld = H;
        g.M = static_cast<int>(M); g.N = 3 * H; g.K = H; g.bias = lp.b_qkv; g.out = qkv; g.out_bf16 = true; g.ldo = 3 * H;
        g.tag = PC_TC_QKV;
        if (e->fused_rope) {
          g.epilogue = TC_EPI_QKV_ROPE; g.rope_cos = e->rope_cos; g.rope_sin = e->rope_sin; g.rope_half = e->half;
          g.rope_freq = e->rope_table_in_epilogue ? nullptr : e->rope_freq;
          g.rope_pd = e->rope_pd; g.seq_T = static_cast<int>(g0.T); g.hidden = H;
          g.rope_pos = ragged ? w.row_pos : nullptr;
          g.rope_perm16 = e->qkv_perm16;
        }
        if (dln) { g.ln_stat = w.lnstat; g.ln_parts = ln1_parts; g.ln_width = H; g.ln_c = lp.c_qkv; }
        DITTO_TRY(launch_tc_gemm(g, st));
        if (!e->fused_rope)
          for (int gi = 0; gi < ng; ++gi)
            DITTO_TRY(launch_rope(qkv + gs[gi].row0 * 3 * H, true, 3 * H, e->rope_cos, e->rope_sin, gs[gi].n * gs[gi].T,
                                  static_cast<int>(gs[gi].T), H, d, st));
      }
      // per group (each on its own side stream when the batch is ragged): self-attention, LN2, cross-attention
      DITTO_TRY(fork.begin(ng));
      for (int gi = 0; gi < ng; ++gi) {
        const SeqGroup& grp = gs[gi];
        const Workspace wg = group_view(e, w, grp);
        const CtxLayout c = ctx_layout(e, const_cast<void*>(grp.ctx), grp.n, grp.S);
        const int64_t n = grp.n, T = grp.T, S = grp.S, Mg = n * T;
        cudaStream_t st = fork.stream(gi);  // shadows the caller's stream inside the group section
        bf16* q = qkv + grp.row0 * 3 * H;
        bf16* ug = u + grp.row0 * H;
        float* hg = w.h + grp.row0 * H;
        // norm2 deferred for this group (context built with the gamma2-folded K): whole-model DITTO_F_DEFER_LN, or norm2 only
        const bool dln2 = dln ? dln2_all : fold_ln_active(e, S) && do_self;   // the row statistics come from the self-attention
        float2* lnstat_g = w.lnstat ? w.lnstat + grp.row0 * std::max(w.ln_parts_h, w.ln_parts_attn) : nullptr;
        const bool self768 = do_self && e->flash768 && !dln2 && flash768_supported(H, e->heads, static_cast<int>(T));
        // constant-text sequences (all text rows equal: the unconditional CFG half, S = 1): their cross-attention output is one
        // row per layer, added by the self-attention kernel together with norm3; the cross-attention kernel skips them.  Only
        // where both sections run here and both kernels know the flags (four-CTA self-attention, folded fused cross-attention)
        const uint8_t* kflag = e->const_text && c.cflag != nullptr && do_cross && self768 && !dln && flash768_picks_quad(static_cast<int>(T)) &&
                                       (cross_flash_active(e, S) || fuse_cross_group(grp))
                                   ? c.cflag : nullptr;
        if (!do_self) {
          // stand-alone cross-attention / MLP section: u already holds that section's LayerNorm of the input
        } else if (self768) {
          // scores, softmax, P.V, + residual AND norm2 in one kernel: no S / P in HBM, no LayerNorm launch     DiT.py:117-143
          Flash768Params f;
          f.qkv = q; f.ld = 3 * H; f.n_seq = n; f.T = static_cast<int>(T); f.H = H; f.alpha = inv_sqrt_d; f.h = hg;
          f.gamma = e->LW(i, "norm2.weight"); f.beta = e->LW(i, "norm2.bias"); f.u_out = ug; f.tag = PC_FLASH768;
          if (kflag) {
            f.const_flag = kflag; f.const_row = c.crow0 + c.crow_stride * i;
            f.gamma_c = e->LW(i, "norm3.weight"); f.beta_c = e->LW(i, "norm3.bias");
          }
          DITTO_TRY(launch_flash768(f, st));
        } else {
          DITTO_TRY(attention_bf16(e, wg, q, 3 * H, T * 3 * H, q + H, 3 * H, T * 3 * H, q + 2 * H, 3 * H, T * 3 * H, n, static_cast<int>(T),
                                   static_cast<int>(T), inv_sqrt_d, hg, false, H, T * H, hg, st, false, dln2 ? ug : nullptr,
                                   dln2 ? lnstat_g : nullptr));
          // ---- cross-attention (torch MHA math path)                                                   DiT.py:141-148
          if (!dln2) DITTO_TRY(launch_layernorm(hg, e->LW(i, "norm2.weight"), e->LW(i, "norm2.bias"), ug, true, Mg, H, st));
        }
        if (!do_cross) continue;
        void* kv = static_cast<char*>(c.kv0) + c.kv_stride * i;
        bool norm3_done = false;   // a fused kernel of this group also wrote norm3's output
        if (fold_active(e, S)) {
          // scores = sqrt(1/d) (u Wq^T + bq) K^T == sqrt(1/d) u (K Wq)^T + sqrt(1/d) K bq ; out = P (V Wo^T) + bo
          const int heads = e->heads;
          const int64_t Sp = round_up(S, 8);
          if (!dln && cross_flash_active(e, S)) {
            // 64 < S <= 256: scores, online softmax, P (V Wo^T), + bo + residual AND norm3 in the flash-style cluster kernel
            Flash768Params f;
            f.qkv = ug; f.ld = H; f.n_seq = n; f.T = static_cast<int>(T); f.H = H; f.alpha = sqrt_inv_d; f.h = hg;
            f.kfold = c.kfold0 + c.kfold_stride * i; f.kf_seq = S * H; f.vfold = c.vfold0 + c.vfold_stride * i; f.vf_seq = Sp * H;
            f.vf_rows = static_cast<int>(Sp); f.Tk = static_cast<int>(S); f.kbias = c.sbias0 + c.sbias_stride * i; f.kb_seq = Sp;
            f.out_bias = e->LW(i, "cross_attn.out_proj.bias");
            f.gamma = e->LW(i, "norm3.weight"); f.beta = e->LW(i, "norm3.bias"); f.u_out = ug; f.tag = PC_CROSS_FLASH;
            f.const_flag = kflag;
            DITTO_TRY(launch_flash768_quad(f, st));
            continue;
          }
          if (fuse_cross_group(grp)) {
            // scores + softmax + P.V + out bias + residual + norm3 in one kernel (cross_fused.cu); u is overwritten with LN3(h)
            CrossFusedParams f;
            f.u = ug; f.kfold = c.kfold0 + c.kfold_stride * i; f.kf_seq = S * H; f.vfold = c.vfold0 + c.vfold_stride * i; f.vf_seq = Sp * H;
            f.sbias = c.sbias0 + c.sbias_stride * i; f.sb_seq = Sp; f.out_bias = e->LW(i, "cross_attn.out_proj.bias");
            f.h = hg; f.gamma = e->LW(i, "norm3.weight"); f.beta = e->LW(i, "norm3.bias"); f.u_out = ug;
            f.n_seq = n; f.T = T; f.S = S; f.Sp = Sp; f.H = H; f.alpha = sqrt_inv_d; f.tag = PC_TC_CROSS_FUSED; f.skip_seq = kflag;
            if (dln2) { f.ln_stat = lnstat_g; f.ln_parts = w.ln_parts_attn; f.ln_c = c.cvec0 + c.sbias_stride * i; }
            DITTO_TRY(launch_cross_fused(f, st));
            continue;
          }
          if (e->fused_attn && tc_scores_softmax_csize(static_cast<int>(S)) == 1) {
            TcScoresSoftmaxParams f;
            f.Q.ptr = ug; f.Q.rows = T; f.Q.cols = H; f.Q.ld = H; f.Q.s_inner = 0; f.Q.s_outer = T * H;
            f.Km.ptr = c.kfold0 + c.kfold_stride * i; f.Km.rows = S; f.Km.cols = H; f.Km.ld = H; f.Km.s_inner = S * H;
            f.Km.s_outer = static_cast<int64_t>(heads) * S * H;
            f.M = static_cast<int>(T); f.N = static_cast<int>(S); f.K = H; f.batch_inner = heads; f.batch_outer = static_cast<int>(n);
            f.alpha = sqrt_inv_d; f.bias = c.sbias0 + c.sbias_stride * i; f.sb_inner = Sp; f.sb_outer = heads * Sp;
            f.P = static_cast<bf16*>(wg.P); f.ldp = heads * Sp; f.sp_inner = Sp; f.sp_outer = T * heads * Sp; f.npad = static_cast<int>(Sp);
            f.tag = PC_TC_CROSS_SCORES;
            if (dln2) { f.ln_stat = lnstat_g; f.ln_parts = w.ln_parts_attn; f.ln_width = H; f.ln_c = c.cvec0 + c.sbias_stride * i; }
            DITTO_TRY(launch_tc_scores_softmax(f, st));
          } else {
            DITTO_REQUIRE(!dln2, DITTO_E_UNSUPPORTED, "forward: deferred LayerNorm needs the fused scores kernel on the folded cross path");
            TcGemmParams g;
            g.A.ptr = ug; g.A.rows = T; g.A.cols = H; g.A.ld = H; g.A.s_inner = 0; g.A.s_outer = T * H;
            g.B.ptr = c.kfold0 + c.kfold_stride * i; g.B.rows = S; g.B.cols = H; g.B.ld = H; g.B.s_inner = S * H;
            g.B.s_outer = static_cast<int64_t>(heads) * S * H;
            g.M = static_cast<int>(T); g.N = static_cast<int>(S); g.K = H; g.batch_inner = heads; g.batch_outer = static_cast<int>(n);
            g.alpha = sqrt_inv_d; g.bias = c.sbias0 + c.sbias_stride * i; g.sb_inner = Sp; g.sb_outer = heads * Sp;
            g.out = wg.scores; g.out_bf16 = false; g.ldo = heads * Sp; g.so_inner = Sp; g.so_outer = T * heads * Sp;
            g.tag = PC_TC_CROSS_SCORES;
            DITTO_TRY(launch_tc_gemm(g, st));
            DITTO_TRY(launch_softmax(wg.scores, Sp, wg.P, true, Sp, n * T * heads, static_cast<int>(S), st));
          }
          TcGemmParams o;
          o.A.ptr = static_cast<const bf16*>(wg.P); o.A.rows = T; o.A.cols = heads * Sp; o.A.ld = heads * Sp; o.A.s_outer = T * heads * Sp;
          o.B.ptr = c.vfold0 + c.vfold_stride * i; o.B.rows = heads * Sp; o.B.cols = H; o.B.ld = H; o.B.s_outer = heads * Sp * H;
          o.b_kn = true;
          o.M = static_cast<int>(T); o.N = H; o.K = static_cast<int>(heads * Sp); o.batch_inner = 1; o.batch_outer = static_cast<int>(n);
          o.bias = e->LW(i, "cross_attn.out_proj.bias");
          o.out = hg; o.out_bf16 = false; o.ldo = H; o.so_outer = T * H; o.resid = hg; o.ldr = H; o.sr_outer = T * H;
          o.tag = PC_TC_CROSS_PV;
          if (dln) { o.out2 = u; o.ldo2 = H; o.stat_out = w.lnstat; o.stat_parts = w.ln_parts_h; o.stat_rows_outer = T; }
          DITTO_TRY(launch_tc_gemm(o, st));
        } else {
          bf16* qc = static_cast<bf16*>(w.qc) + grp.row0 * H;
          bf16* oc = static_cast<bf16*>(w.oc) + grp.row0 * H;
          DITTO_TRY(tc_nt(ug, H, lp.wc_in, H, qc, true, H, e->LW(i, "cross_attn.in_proj_bias"), nullptr, 0, 0, nullptr, 0, static_cast<int>(Mg),
                          H, H, st, PC_TC_CROSS_Q));
          const bf16* kc = static_cast<const bf16*>(kv);
          DITTO_TRY(attention_bf16(e, wg, qc, H, T * H, kc, 2 * H, S * 2 * H, kc + H, 2 * H, S * 2 * H, n, static_cast<int>(T),
                                   static_cast<int>(S), sqrt_inv_d, oc, true, H, T * H, nullptr, st, true));
          if (e->fc2_ln && !dln) {
            // out_proj + bias + residual AND norm3 in one cluster kernel (gemm_resid_ln.cu)                 DiT.py:148-151
            GemmResidLnParams f;
            f.A = oc; f.lda = H; f.W = lp.wc_o_p4; f.ldw = H; f.bias = e->LW(i, "cross_attn.out_proj.bias"); f.h = hg; f.ldh = H;
            f.gamma = e->LW(i, "norm3.weight"); f.beta = e->LW(i, "norm3.bias"); f.u = ug; f.ldu = H;
            f.M = static_cast<int>(Mg); f.N = H; f.K = H; f.tag = PC_TC_CROSS_OUT;
            DITTO_TRY(launch_gemm_resid_ln(f, st));
            norm3_done = true;
          } else {
          DITTO_TRY(tc_nt(oc, H, lp.wc_o, H, hg, false, H, e->LW(i, "cross_attn.out_proj.bias"), hg, H, 0, dln ? u : nullptr, H,
                          static_cast<int>(Mg), H, H, st, PC_TC_CROSS_OUT, dln ? w.lnstat : nullptr, w.ln_parts_h));
          }
        }
        // norm3 of a group that did not take a fused kernel (which writes it itself)                      DiT.py:151
        if (!dln && !norm3_done) DITTO_TRY(launch_layernorm(hg, e->LW(i, "norm3.weight"), e->LW(i, "norm3.bias"), ug, true, Mg, H, st));
      }
      DITTO_TRY(fork.end());
      // ---- gated MLP                                                                                  DiT.py:150-155
      if (!do_mlp) continue;
      {
        TcGemmParams g;
        g.A.ptr = u; g.A.rows = M; g.A.cols = H; g.A.ld = H;
        g.B.ptr = lp.w_glu; g.B.rows = 8 * H; g.B.cols = H; g.B.ld = H;
        g.M = static_cast<int>(M); g.N = 8 * H; g.K = H; g.bias = lp.b_glu; g.out = w.hid; g.out_bf16 = true; g.ldo = 4 * H;
        g.epilogue = TC_EPI_GEGLU; g.glu_perm16 = e->glu_perm16;
        if (dln) { g.ln_stat = w.lnstat; g.ln_parts = w.ln_parts_h; g.ln_width = H; g.ln_c = lp.c_glu; }
        g.tag = PC_TC_GLU;
        DITTO_TRY(launch_tc_gemm(g, st));
      }
      if (e->fc2_ln) {
        // h += fc2(hid) + b and, in the same kernel, the operand of what follows: norm1 of the next block (DiT.py:105) or,
        // after the last block, the plain bf16 copy that proj_out reads
        GemmResidLnParams f;
        f.A = static_cast<bf16*>(w.hid); f.lda = 4 * H; f.W = lp.w_fc2; f.ldw = 4 * H; f.bias = e->LW(i, "mlp_fc2.bias");
        f.h = w.h; f.ldh = H; f.M = static_cast<int>(M); f.N = H; f.K = 4 * H; f.tag = PC_TC_FC2;
        if (last) { f.u = static_cast<bf16*>(w.xb16); f.ldu = H; }
        else { f.gamma = e->LW(i + 1, "norm1.weight"); f.beta = e->LW(i + 1, "norm1.bias"); f.u = u; f.ldu = H; }
        DITTO_TRY(launch_gemm_resid_ln(f, st));
      } else {
      DITTO_TRY(tc_nt(static_cast<bf16*>(w.hid), 4 * H, lp.w_fc2, 4 * H, w.h, false, H, e->LW(i, "mlp_fc2.bias"), w.h, H, 0,
                      last ? static_cast<bf16*>(w.xb16) : (dln ? u : nullptr), H, static_cast<int>(M), H, 4 * H, st, PC_TC_FC2,
                      (dln && !last) ? w.lnstat : nullptr, w.ln_parts_h));
      ln1_parts = w.ln_parts_h;
      if (!last && !dln)
        DITTO_TRY(launch_layernorm(w.h, e->LW(i + 1, "norm1.weight"), e->LW(i + 1, "norm1.bias"), u, true, M, H, st));
      }
    } else {
      float* u = static_cast<float*>(w.u);
      float* qkv = static_cast<float*>(w.qkv);
      float* qc = static_cast<float*>(w.qc);
      float* oc = static_cast<float*>(w.oc);
      if (do_self)
      DITTO_TRY(sgemm_nt(u, H, e->LW(i, "attn.in_proj_weight"), H, qkv, 3 * H, e->LW(i, "attn.in_proj_bias"), nullptr, 0, 1.f,
                         static_cast<int>(M), 3 * H, H, st));
      for (int gi = 0; gi < ng && do_self; ++gi) {
        const SeqGroup& g = gs[gi];
        const Workspace wg = group_view(e, w, g);
        float* q = qkv + g.row0 * 3 * H;
        float* hg = w.h + g.row0 * H;
        const int64_t T = g.T;
        DITTO_TRY(launch_rope(q, false, 3 * H, e->rope_cos, e->rope_sin, g.n * T, static_cast<int>(T), H, d, st));
        DITTO_TRY(attention_f32(e, wg, q, 3 * H, T * 3 * H, q + H, 3 * H, T * 3 * H, q + 2 * H, 3 * H, T * 3 * H, g.n, static_cast<int>(T),
                                static_cast<int>(T), inv_sqrt_d, hg, H, T * H, hg, st));
      }
      if (do_self && do_cross) DITTO_TRY(launch_layernorm(w.h, e->LW(i, "norm2.weight"), e->LW(i, "norm2.bias"), u, false, M, H, st));
      if (do_cross)
      DITTO_TRY(sgemm_nt(u, H, e->LW(i, "cross_attn.in_proj_weight"), H, qc, H, e->LW(i, "cross_attn.in_proj_bias"), nullptr, 0, 1.f,
                         static_cast<int>(M), H, H, st));
      for (int gi = 0; gi < ng && do_cross; ++gi) {
        const SeqGroup& g = gs[gi];
        const Workspace wg = group_view(e, w, g);
        const CtxLayout c = ctx_layout(e, const_cast<void*>(g.ctx), g.n, g.S);
        const float* kc = reinterpret_cast<const float*>(static_cast<const char*>(c.kv0) + c.kv_stride * i);
        const int64_t T = g.T, S = g.S;
        DITTO_TRY(attention_f32(e, wg, qc + g.row0 * H, H, T * H, kc, 2 * H, S * 2 * H, kc + H, 2 * H, S * 2 * H, g.n, static_cast<int>(T),
                                static_cast<int>(S), sqrt_inv_d, oc + g.row0 * H, H, T * H, nullptr, st));
      }
      if (do_cross)
      DITTO_TRY(sgemm_nt(oc, H, e->LW(i, "cross_attn.out_proj.weight"), H, w.h, H, e->LW(i, "cross_attn.out_proj.bias"), w.h, H, 1.f,
                         static_cast<int>(M), H, H, st));
      if (do_cross && do_mlp) DITTO_TRY(launch_layernorm(w.h, e->LW(i, "norm3.weight"), e->LW(i, "norm3.bias"), u, false, M, H, st));
      if (!do_mlp) continue;
      DITTO_TRY(sgemm_nt(u, H, e->LW(i, "mlp_fc1.weight"), H, w.fc1, 4 * H, e->LW(i, "mlp_fc1.bias"), nullptr, 0, 1.f, static_cast<int>(M),
                         4 * H, H, st));
      DITTO_TRY(sgemm_nt(u, H, e->LW(i, "gate.weight"), H, w.gate, 4 * H, e->LW(i, "gate.bias"), nullptr, 0, 1.f, static_cast<int>(M),
                         4 * H, H, st));
      DITTO_TRY(launch_geglu_f32(w.fc1, w.gate, static_cast<float*>(w.hid), M * 4 * H, st));
      DITTO_TRY(sgemm_nt(static_cast<float*>(w.hid), 4 * H, e->LW(i, "mlp_fc2.weight"), 4 * H, w.h, H, e->LW(i, "mlp_fc2.bias"), w.h, H, 1.f,
                         static_cast<int>(M), H, 4 * H, st));
      if (!last)
        DITTO_TRY(launch_layernorm(w.h, e->LW(i + 1, "norm1.weight"), e->LW(i + 1, "norm1.bias"), u, false, M, H, st));
    }
  }
  if (block_only) {
    DITTO_CUDA(cudaMemcpyAsync(out, w.h, static_cast<size_t>(M) * H * sizeof(float), cudaMemcpyDeviceToDevice, st));
    return 0;
  }
  // eps = x_skip + proj_out(h)                                              DiTTO.py:93-94
  if (b16 && e->fc2_ln && (reinterpret_cast<uintptr_t>(out) & 15) == 0) {
    GemmResidLnParams f;
    f.A = static_cast<bf16*>(w.xb16); f.lda = H; f.W = e->w_out_p4; f.ldw = H; f.bias = e->W("proj_out.bias"); f.h = out; f.ldh = H;
    f.resid = w.xskip; f.ldr = H; f.resid_mod = ragged ? 0 : g0.n_x * g0.T;
    f.M = static_cast<int>(M); f.N = H; f.K = H; f.tag = PC_TC_PROJ_OUT;
    DITTO_TRY(launch_gemm_resid_ln(f, st));
  } else if (b16) {
    DITTO_TRY(tc_nt(static_cast<bf16*>(w.xb16), H, e->w_out16, H, out, false, H, e->W("proj_out.bias"), w.xskip, H,
                    ragged ? 0 : g0.n_x * g0.T, nullptr, 0, static_cast<int>(M), H, H, st, PC_TC_PROJ_OUT));
  } else {
    // residual rows repeat with period n_x*T inside a group: one GEMM per run of n_x sequences
    for (int gi = 0; gi < ng; ++gi) {
      const SeqGroup& g = gs[gi];
      for (int64_t s0 = 0; s0 < g.n; s0 += g.n_x) {
        const int64_t r = g.row0 + s0 * g.T;
        DITTO_TRY(sgemm_nt(w.h + r * H, H, e->W("proj_out.weight"), H, out + r * H, H, e->W("proj_out.bias"), w.xskip + g.xrow0 * H, H, 1.f,
                           static_cast<int>(g.n_x * g.T), H, H, st));
      }
    }
  }
  return 0;
}

// uniform batch: one group
static int forward_impl(ditto_engine* e, const float* x, int64_t n_x, const void* ctx, const int64_t* t, int64_t n, int64_t T,
                        int64_t S, float* out, void* workspace, int64_t workspace_bytes, cudaStream_t st) {
  SeqGroup g;
  g.n = n; g.n_x = n_x; g.T = T; g.S = S; g.ctx = ctx;
  return forward_impl(e, x, t, &g, 1, out, workspace, workspace_bytes, st);
}

}  // namespace ditto

// =====================================================================================================
// C ABI
// =====================================================================================================
extern "C" {
#pragma GCC visibility push(default)

int32_t ditto_abi_version(void) { return DITTO_ABI_VERSION; }
const char* ditto_last_error(void) { return t_last_error.c_str(); }
int64_t ditto_kernel_launch_count(void) { return g_launches.load(); }

int32_t ditto_profile_start(void) {
  for (auto& r : g_prof_recs) { cudaEventDestroy(r.a); cudaEventDestroy(r.b); }
  g_prof_recs.clear();
  for (auto& a : g_prof_acc) a = ProfAcc();
  g_prof_enabled = true;
  return 0;
}
int32_t ditto_profile_stop(void) {
  g_prof_enabled = false;
  DITTO_CUDA(cudaDeviceSynchronize());
  for (auto& r : g_prof_recs) {
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, r.a, r.b) == cudaSuccess) {
      ProfAcc& a = g_prof_acc[r.cls];
      a.launches += 1; a.ms += ms; a.flops += r.flops; a.bytes += r.bytes;
    }
    cudaEventDestroy(r.a);
    cudaEventDestroy(r.b);
  }
  g_prof_recs.clear();
  return 0;
}
int32_t ditto_profile_num_classes(void) { return PC_COUNT; }
const char* ditto_profile_class_name(int32_t i) { return (i >= 0 && i < PC_COUNT) ? kProfNames[i] : ""; }
int32_t ditto_profile_get(int32_t i, int64_t* launches, double* total_ms, double* flops, double* bytes) {
  DITTO_REQUIRE(i >= 0 && i < PC_COUNT && launches && total_ms && flops && bytes, DITTO_E_BADARG, "profile_get: bad argument");
  *launches = g_prof_acc[i].launches; *total_ms = g_prof_acc[i].ms; *flops = g_prof_acc[i].flops; *bytes = g_prof_acc[i].bytes;
  return 0;
}

int32_t ditto_debug_set_counters(uint64_t* counters) {
  tc_gemm_set_debug_counters(reinterpret_cast<unsigned long long*>(counters));
  return 0;
}

int32_t ditto_engine_create(const ditto_config_t* cfg, ditto_engine_t** out) {
  DITTO_REQUIRE(cfg && out, DITTO_E_BADARG, "engine_create: null argument");
  DITTO_REQUIRE(cfg->hidden_dim > 0 && cfg->num_layers > 0 && cfg->num_heads > 0 && cfg->time_dim > 0 && cfg->diffusion_steps > 0,
                DITTO_E_BADARG, "engine_create: non-positive dimension");
  DITTO_REQUIRE(cfg->hidden_dim % cfg->num_heads == 0 && (cfg->hidden_dim / cfg->num_heads) % 2 == 0, DITTO_E_BADARG,
                "engine_create: hidden_dim must split into heads of even size");
  DITTO_REQUIRE(cfg->text_dim == cfg->hidden_dim, DITTO_E_UNSUPPORTED,
                "engine_create: text_dim must equal hidden_dim (nn.MultiheadAttention without kdim, DiT.py:90-91)");
  DITTO_REQUIRE(cfg->hidden_dim % 8 == 0 && cfg->hidden_dim <= 1024 && cfg->time_dim % 4 == 0, DITTO_E_UNSUPPORTED,
                "engine_create: need hidden_dim % 8 == 0, hidden_dim <= 1024, time_dim % 4 == 0");
  DITTO_REQUIRE(cfg->precision == DITTO_PREC_FP32 || cfg->precision == DITTO_PREC_BF16, DITTO_E_BADARG, "engine_create: precision");
  int ndev = 0;
  DITTO_CUDA(cudaGetDeviceCount(&ndev));
  DITTO_REQUIRE(ndev > 0, DITTO_E_CUDA, "engine_create: no CUDA device (there is no CPU fallback)");
  ditto_engine* e = new ditto_engine();
  e->cfg = *cfg;
  e->H = cfg->hidden_dim; e->L = cfg->num_layers; e->heads = cfg->num_heads; e->d = e->H / e->heads; e->half = e->d / 2;
  e->Td = cfg->time_dim; e->Xd = cfg->text_dim; e->steps = cfg->diffusion_steps;
  e->maxT = cfg->max_seq_len > 0 ? cfg->max_seq_len : 4096;
  e->bf16_mode = cfg->precision == DITTO_PREC_BF16;
  e->blocks_only = (cfg->flags & DITTO_F_BLOCKS_ONLY) != 0;
  if (cudaGetDevice(&e->device) != cudaSuccess) e->device = -1;
  if (e->bf16_mode) {
    if (e->bf16_mode && e->d % 8 != 0) {
      delete e;
      set_error("engine_create: bf16 path needs head_dim % 8 == 0 (16-byte TMA rows)");
      return DITTO_E_UNSUPPORTED;
    }
    int rc = tc_gemm_init();
    if (rc != 0) { delete e; return rc; }
    // RoPE pair distance inside a GEMM tile: largest of 128/64/32 dividing d/2 (d=768 -> 128, d=64 -> 32)
    for (int pd : {128, 64, 32})
      if (e->half % pd == 0 && e->H % (2 * pd) == 0) { e->rope_pd = pd; break; }
    e->fused_rope = (cfg->flags & DITTO_F_FUSED_ROPE) && e->rope_pd != 0;
    e->fold_cross = (cfg->flags & DITTO_F_FOLD_CROSS) != 0;
    e->fused_attn = (cfg->flags & DITTO_F_FUSED_ATTN) != 0;
    e->defer_ln = (cfg->flags & DITTO_F_DEFER_LN) != 0 && e->fused_rope && e->fused_attn;
    if (g_opt.no_defer_ln) e->defer_ln = false;
    if (g_opt.no_fused_attn) e->fused_attn = false;
    e->fused_cross = e->fused_attn;
    e->flash_attn = e->fused_attn;
    if (g_opt.no_flash) e->flash_attn = false;
    if (g_opt.no_fused_cross) e->fused_cross = false;
    e->const_text = !g_opt.no_const_text;
    e->defer_ln2 = !e->defer_ln && e->fused_cross && e->bf16_mode && e->heads == 1 && g_opt.defer_ln2 != 0;
    e->pv_transpose = g_opt.pv_transpose != 0;
    e->rope_table_in_epilogue = g_opt.rope_table != 0;
    e->glu_perm16 = !e->defer_ln && e->H % 32 == 0 && !g_opt.glu_generic;
    // no_rope_fast32: pair distance 32 (head_dim 64) through the generic epilogue
    const bool pd_ok = e->rope_pd == 128 || (e->rope_pd == 32 && !g_opt.no_rope_fast32);
    e->qkv_perm16 = e->fused_rope && pd_ok && !e->defer_ln && !e->rope_table_in_epilogue && e->H % 256 == 0 && !g_opt.rope_generic;
    e->pv_perm4 = e->qkv_perm16 && !e->pv_transpose && !e->defer_ln2 && e->d % 128 == 0 && !g_opt.no_pv_perm4;
    // needs the v columns in the 16-byte store order (pv_perm4) and the fused softmax machinery
    e->flash768 = e->fused_attn && e->pv_perm4 && !e->defer_ln && flash768_supported(e->H, e->heads, 1) && !g_opt.no_flash768;
    e->fc2_ln = !e->defer_ln && gemm_resid_ln_supported(e->H, 4 * e->H) && !g_opt.no_fc2_ln && gemm_resid_ln_schedulable(e->H);
    // needs the perm4-packed out-projection (packed with the fc2_ln weights) for the V fold and four-CTA clusters
    e->cross_flash = e->flash768 && e->fc2_ln && e->fold_cross && !e->defer_ln2 && !g_opt.no_cross_flash && flash768_quad_schedulable();
  }
  build_expected(e);
  e->layers.resize(e->L);
  int want_side = ditto_engine::kSide;
  if (g_opt.side_streams >= 0) want_side = std::min(ditto_engine::kSide, g_opt.side_streams);
  if (want_side > 0 && cudaEventCreateWithFlags(&e->ev_fork, cudaEventDisableTiming) == cudaSuccess) {
    for (int k = 0; k < want_side; ++k) {
      if (cudaStreamCreateWithFlags(&e->side[k], cudaStreamNonBlocking) != cudaSuccess ||
          cudaEventCreateWithFlags(&e->ev_join[k], cudaEventDisableTiming) != cudaSuccess)
        break;
      e->n_side = k + 1;
    }
  }
  *out = e;
  return 0;
}

int32_t ditto_engine_destroy(ditto_engine_t* e) {
  if (!e) return 0;
  for (int k = 0; k < ditto_engine::kSide; ++k) {
    if (e->side[k]) cudaStreamDestroy(e->side[k]);
    if (e->ev_join[k]) cudaEventDestroy(e->ev_join[k]);
  }
  if (e->ev_fork) cudaEventDestroy(e->ev_fork);
  for (auto& kv : e->w) cudaFree(kv.second);
  for (void* p : e->owned) cudaFree(p);
  delete e;
  return 0;
}

int32_t ditto_engine_load_weight(ditto_engine_t* e, const char* key, const float* data, int64_t numel, void* stream) {
  DITTO_REQUIRE(e && key && data, DITTO_E_BADARG, "load_weight: null argument");
  const std::string k(key);
  if (ignorable_key(k)) return 0;
  auto it = e->expected.find(k);
  if (it == e->expected.end()) {
    set_error("load_weight: unknown state_dict key '" + k + "'");
    return DITTO_E_BADARG;
  }
  if (it->second != numel) {
    set_error("load_weight: '" + k + "' has " + std::to_string(numel) + " elements, expected " + std::to_string(it->second));
    return DITTO_E_BADARG;
  }
  float*& dst = e->w[k];
  if (!dst) DITTO_CUDA(cudaMalloc(reinterpret_cast<void**>(&dst), static_cast<size_t>(numel) * sizeof(float)));
  DITTO_CUDA(cudaMemcpyAsync(dst, data, static_cast<size_t>(numel) * sizeof(float), cudaMemcpyDeviceToDevice,
                             static_cast<cudaStream_t>(stream)));
  e->finalized = false;
  return 0;
}

int32_t ditto_engine_load_schedule(ditto_engine_t* e, const float* betas, const float* alphas, const float* alphas_cumprod,
                                   int64_t steps, void* stream) {
  DITTO_REQUIRE(e && betas && alphas && alphas_cumprod, DITTO_E_BADARG, "load_schedule: null argument");
  DITTO_REQUIRE(steps == e->steps, DITTO_E_BADARG, "load_schedule: steps != diffusion_steps");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (!e->coef) {
    DITTO_TRY(dev_alloc(e, reinterpret_cast<void**>(&e->coef), sizeof(float) * 3 * steps));
    DITTO_TRY(dev_alloc(e, reinterpret_cast<void**>(&e->qs_buf), sizeof(float) * steps));
  }
  DITTO_TRY(launch_schedule_coef(betas, alphas, alphas_cumprod, e->coef, static_cast<int>(steps), st));
  // DiTTO.py:63-64: the module's "alphas_cumprod" buffer is cosine_beta_schedule(), i.e. the betas
  DITTO_CUDA(cudaMemcpyAsync(e->qs_buf, betas, sizeof(float) * steps, cudaMemcpyDeviceToDevice, st));
  e->have_schedule = true;
  return 0;
}

int32_t ditto_engine_load_update_table(ditto_engine_t* e, const float* coef, int64_t steps, void* stream) {
  DITTO_REQUIRE(e && coef, DITTO_E_BADARG, "load_update_table: null argument");
  DITTO_REQUIRE(steps == e->steps, DITTO_E_BADARG, "load_update_table: steps != diffusion_steps");
  DITTO_REQUIRE(e->have_schedule, DITTO_E_STATE, "load_update_table: call ditto_engine_load_schedule first (q_sample needs the betas)");
  DITTO_CUDA(cudaMemcpyAsync(e->coef, coef, sizeof(float) * 3 * steps, cudaMemcpyDeviceToDevice, static_cast<cudaStream_t>(stream)));
  return 0;
}

int32_t ditto_engine_load_multistep_table(ditto_engine_t* e, const float* coef6, int64_t steps, void* stream) {
  DITTO_REQUIRE(e && coef6, DITTO_E_BADARG, "load_multistep_table: null argument");
  DITTO_REQUIRE(steps == e->steps, DITTO_E_BADARG, "load_multistep_table: steps != diffusion_steps");
  DITTO_REQUIRE(e->have_schedule, DITTO_E_STATE, "load_multistep_table: call ditto_engine_load_schedule first");
  if (!e->coef_ms) DITTO_TRY(dev_alloc(e, reinterpret_cast<void**>(&e->coef_ms), sizeof(float) * 6 * steps));
  DITTO_CUDA(cudaMemcpyAsync(e->coef_ms, coef6, sizeof(float) * 6 * steps, cudaMemcpyDeviceToDevice, static_cast<cudaStream_t>(stream)));
  return 0;
}

int32_t ditto_engine_load_known_table(ditto_engine_t* e, const float* coef2, int64_t steps, void* stream) {
  DITTO_REQUIRE(e && coef2, DITTO_E_BADARG, "load_known_table: null argument");
  DITTO_REQUIRE(steps == e->steps, DITTO_E_BADARG, "load_known_table: steps != diffusion_steps");
  DITTO_REQUIRE(e->have_schedule, DITTO_E_STATE, "load_known_table: call ditto_engine_load_schedule first");
  if (!e->coef_known) DITTO_TRY(dev_alloc(e, reinterpret_cast<void**>(&e->coef_known), sizeof(float) * 2 * steps));
  DITTO_CUDA(cudaMemcpyAsync(e->coef_known, coef2, sizeof(float) * 2 * steps, cudaMemcpyDeviceToDevice, static_cast<cudaStream_t>(stream)));
  return 0;
}

int32_t ditto_engine_finalize(ditto_engine_t* e, void* stream) {
  DITTO_REQUIRE(e, DITTO_E_BADARG, "finalize: null engine");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  for (auto& kv : e->expected) {
    if (kv.first == "rotary.inv_freq") continue;
    if (!e->w.count(kv.first)) {
      set_error("finalize: missing weight '" + kv.first + "'");
      return DITTO_E_STATE;
    }
  }
  const int H = e->H, Td = e->Td, St = e->steps;
  int rc = 0;
  cudaError_t se = cudaSuccess;
  if (!e->blocks_only) {
  // ---- per-step modulation table: time_mlp(SiLU(time_embed(t_embedding[t])))  (DiTTO.py:75-76, DiT.py:30)
  if (!e->time_table) DITTO_TRY(dev_alloc(e, reinterpret_cast<void**>(&e->time_table), sizeof(float) * St * 2 * H));
  float *t1 = nullptr, *t2 = nullptr;
  DITTO_CUDA(cudaMalloc(reinterpret_cast<void**>(&t1), sizeof(float) * St * Td));
  DITTO_CUDA(cudaMalloc(reinterpret_cast<void**>(&t2), sizeof(float) * St * Td));
  rc = sgemm_nt(e->W("t_embedding.weight"), Td, e->W("time_embed.0.weight"), Td, t1, Td, e->W("time_embed.0.bias"), nullptr, 0,
                1.f, St, Td, Td, st);
  if (!rc) rc = launch_silu(t1, static_cast<int64_t>(St) * Td, st);
  if (!rc) rc = sgemm_nt(t1, Td, e->W("time_embed.2.weight"), Td, t2, Td, e->W("time_embed.2.bias"), nullptr, 0, 1.f, St, Td, Td, st);
  if (!rc) rc = launch_silu(t2, static_cast<int64_t>(St) * Td, st);
  if (!rc) rc = sgemm_nt(t2, Td, e->W("ada_ln.time_mlp.1.weight"), Td, e->time_table, 2 * H, e->W("ada_ln.time_mlp.1.bias"), nullptr,
                         0, 1.f, St, 2 * H, Td, st);
  se = cudaStreamSynchronize(st);
  cudaFree(t1);
  cudaFree(t2);
  if (rc) return rc;
  DITTO_CUDA(se);
  }
  // ---- RoPE tables (DiT.py:46-59)
  if (!e->rope_cos) {
    DITTO_TRY(dev_alloc(e, reinterpret_cast<void**>(&e->rope_cos), sizeof(float) * e->maxT * e->half));
    DITTO_TRY(dev_alloc(e, reinterpret_cast<void**>(&e->rope_sin), sizeof(float) * e->maxT * e->half));
    DITTO_TRY(dev_alloc(e, reinterpret_cast<void**>(&e->rope_freq), sizeof(float) * e->half));
  }
  DITTO_TRY(launch_rope_table(e->W("rotary.inv_freq"), e->rope_cos, e->rope_sin, e->rope_freq, e->maxT, e->half, e->d, st));

  // ---- bf16 packing
  if (e->bf16_mode) {
    auto cast_new = [&](const float* src, int64_t n, bf16** dst) -> int {
      if (!*dst) DITTO_TRY(dev_alloc(e, reinterpret_cast<void**>(dst), sizeof(bf16) * n));
      return launch_cast_bf16(src, *dst, n, st);
    };
    if (!e->blocks_only) {
      DITTO_TRY(cast_new(e->W("proj_in.weight"), static_cast<int64_t>(H) * H, &e->w_in16));
      DITTO_TRY(cast_new(e->W("proj_out.weight"), static_cast<int64_t>(H) * H, &e->w_out16));
      if (e->fc2_ln) {   // eps = x_skip + proj_out(h) through the float4-epilogue GEMM of gemm_resid_ln.cu (no LayerNorm stage)
        std::vector<int> perm(H);
        for (int r = 0; r < H; ++r) perm[r] = gemm_resid_ln_weight_row(r);
        int* d_perm = nullptr;
        DITTO_CUDA(cudaMalloc(reinterpret_cast<void**>(&d_perm), sizeof(int) * H));
        DITTO_CUDA(cudaMemcpyAsync(d_perm, perm.data(), sizeof(int) * H, cudaMemcpyHostToDevice, st));
        int rc2 = 0;
        if (!e->w_out_p4) rc2 = dev_alloc(e, reinterpret_cast<void**>(&e->w_out_p4), sizeof(bf16) * static_cast<int64_t>(H) * H);
        if (!rc2) rc2 = launch_pack_rows(e->W("proj_out.weight"), e->w_out_p4, nullptr, nullptr, d_perm, H, H, st, nullptr, nullptr, nullptr);
        cudaError_t se2 = cudaStreamSynchronize(st);
        cudaFree(d_perm);
        if (rc2) return rc2;
        DITTO_CUDA(se2);
      }
    }
    // row permutations (host-built, tiny)
    std::vector<int> glu_perm(8 * H), qkv_perm(3 * H);
    for (int r = 0; r < 8 * H; ++r) {
      const int blk = r / 32, i = r % 32;
      glu_perm[r] = i < 16 ? 16 * blk + i : 4 * H + 16 * blk + (i - 16);
    }
    for (int r = 0; r < 3 * H; ++r) qkv_perm[r] = r;
    if (e->fused_rope) {
      const int pd = e->rope_pd, half = e->half;
      for (int region = 0; region < 2; ++region)
        for (int lp = 0; lp < H; ++lp) {
          const int g = lp / (2 * pd), w = lp % (2 * pd);
          const int e0 = g * pd, head = e0 / half, j0 = e0 % half;
          const int x1 = head * 2 * half + j0 + (w % pd);
          qkv_perm[region * H + lp] = region * H + (w < pd ? x1 : x1 + half);
        }
    }
    if (e->glu_perm16) {  // 64-row block B: row kb*8 + 2q + e <- fc1 (kb%4 < 2) or gate row of output 32B + q*8 + ((kb/4)*2 + kb%2)*2 + e
      for (int r = 0; r < 8 * H; ++r) {
        const int blk = r / 64, c = r % 64;
        const int kb = c / 8, q = (c % 8) / 2, ee = c % 2;
        const int gi = kb / 4, kk = kb % 4;
        const int o = 32 * blk + q * 8 + (gi * 2 + (kk & 1)) * 2 + ee;
        glu_perm[r] = kk < 2 ? o : 4 * H + o;
      }
    }
    if (e->qkv_perm16) {  // GEMM column kb*8 + 2q + e of every 64-column block <- what stood at q*16 + kb*2 + e
      std::vector<int> base(qkv_perm);
      for (int r = 0; r < 3 * H; ++r) {
        const int blk = r / 64, c = r % 64;
        const int kb = c / 8, q = (c % 8) / 2, ee = c % 2;
        int l = q * 16 + kb * 2 + ee;   // storage position (inside the block) the lean QKV epilogue writes this accumulator to
        // pair distance 32 (q and k thirds): 8-column blocks kb < 4 are x1 elements q * 8 + kb * 2 + e, kb >= 4 their partners
        if (e->rope_pd == 32 && r < 2 * H) l = (kb < 4 ? 0 : 32) + q * 8 + (kb & 3) * 2 + ee;
        // v third with the float4 P.V epilogue: storage position l must hold logical column 16 (K / 2) + 4 Q + 2 (K % 2) + E,
        // where K, Q, E are the fragment coordinates of P.V accumulator column l
        if (e->pv_perm4 && r >= 2 * H) {
          const int K = l / 8, Q = (l % 8) / 2, E = l % 2;
          l = 16 * (K / 2) + 4 * Q + 2 * (K % 2) + E;
        }
        qkv_perm[r] = base[blk * 64 + l];
      }
    }
    int *d_glu = nullptr, *d_qkv = nullptr, *d_fc2 = nullptr;
    float* cat = nullptr;
    std::vector<int> fc2_perm(H);
    for (int r = 0; r < H; ++r) fc2_perm[r] = e->fc2_ln ? gemm_resid_ln_weight_row(r) : r;
    DITTO_CUDA(cudaMalloc(reinterpret_cast<void**>(&d_fc2), sizeof(int) * fc2_perm.size()));
    DITTO_CUDA(cudaMemcpyAsync(d_fc2, fc2_perm.data(), sizeof(int) * fc2_perm.size(), cudaMemcpyHostToDevice, st));
    DITTO_CUDA(cudaMalloc(reinterpret_cast<void**>(&d_glu), sizeof(int) * glu_perm.size()));
    DITTO_CUDA(cudaMalloc(reinterpret_cast<void**>(&d_qkv), sizeof(int) * qkv_perm.size()));
    DITTO_CUDA(cudaMalloc(reinterpret_cast<void**>(&cat), sizeof(float) * (8ll * H * H + 8 * H)));
    DITTO_CUDA(cudaMemcpyAsync(d_glu, glu_perm.data(), sizeof(int) * glu_perm.size(), cudaMemcpyHostToDevice, st));
    DITTO_CUDA(cudaMemcpyAsync(d_qkv, qkv_perm.data(), sizeof(int) * qkv_perm.size(), cudaMemcpyHostToDevice, st));
    float* cat_bias = cat + 8ll * H * H;
    rc = 0;
    for (int i = 0; i < e->L && !rc; ++i) {
      LayerPack& lp = e->layers[i];
      if (!lp.w_qkv) {
        rc = dev_alloc(e, reinterpret_cast<void**>(&lp.w_qkv), sizeof(bf16) * 3ll * H * H);
        if (!rc) rc = dev_alloc(e, reinterpret_cast<void**>(&lp.b_qkv), sizeof(float) * 3 * H);
        if (!rc) rc = dev_alloc(e, reinterpret_cast<void**>(&lp.w_glu), sizeof(bf16) * 8ll * H * H);
        if (!rc) rc = dev_alloc(e, reinterpret_cast<void**>(&lp.b_glu), sizeof(float) * 8 * H);
        if (!rc) rc = dev_alloc(e, reinterpret_cast<void**>(&lp.c_qkv), sizeof(float) * 3 * H);
        if (!rc) rc = dev_alloc(e, reinterpret_cast<void**>(&lp.c_glu), sizeof(float) * 8 * H);
        if (!rc) rc = dev_alloc(e, reinterpret_cast<void**>(&lp.wq_g), sizeof(bf16) * static_cast<int64_t>(H) * H);
        if (!rc) rc = dev_alloc(e, reinterpret_cast<void**>(&lp.bq_g), sizeof(float) * H);
        if (rc) break;
      }
      const bool dl = e->defer_ln;
      rc = launch_pack_rows(e->LW(i, "attn.in_proj_weight"), lp.w_qkv, lp.b_qkv, e->LW(i, "attn.in_proj_bias"), d_qkv, 3 * H, H, st,
                            dl ? e->LW(i, "norm1.weight") : nullptr, dl ? e->LW(i, "norm1.bias") : nullptr, lp.c_qkv);
      if (!rc && (dl || e->defer_ln2))
        rc = launch_pack_rows(e->LW(i, "cross_attn.in_proj_weight"), lp.wq_g, lp.bq_g, e->LW(i, "cross_attn.in_proj_bias"), nullptr, H, H, st,
                              e->LW(i, "norm2.weight"), e->LW(i, "norm2.bias"), nullptr);
      if (!rc) rc = cast_new(e->LW(i, "cross_attn.in_proj_weight"), 3ll * H * H, &lp.wc_in);
      if (!rc) rc = cast_new(e->LW(i, "cross_attn.out_proj.weight"), static_cast<int64_t>(H) * H, &lp.wc_o);
      if (!rc && e->fc2_ln) {
        if (!lp.wc_o_p4) rc = dev_alloc(e, reinterpret_cast<void**>(&lp.wc_o_p4), sizeof(bf16) * static_cast<int64_t>(H) * H);
        if (!rc) rc = launch_pack_rows(e->LW(i, "cross_attn.out_proj.weight"), lp.wc_o_p4, nullptr, nullptr, d_fc2, H, H, st, nullptr, nullptr, nullptr);
      }
      if (!rc && e->fc2_ln) {   // rows in the order the float4 residual + LayerNorm epilogue wants (gemm_resid_ln.cu)
        if (!lp.w_fc2) rc = dev_alloc(e, reinterpret_cast<void**>(&lp.w_fc2), sizeof(bf16) * 4ll * H * H);
        if (!rc) rc = launch_pack_rows(e->LW(i, "mlp_fc2.weight"), lp.w_fc2, nullptr, nullptr, d_fc2, H, 4 * H, st, nullptr, nullptr, nullptr);
      } else if (!rc) {
        rc = cast_new(e->LW(i, "mlp_fc2.weight"), 4ll * H * H, &lp.w_fc2);
      }
      if (rc) break;
      cudaMemcpyAsync(cat, e->LW(i, "mlp_fc1.weight"), sizeof(float) * 4ll * H * H, cudaMemcpyDeviceToDevice, st);
      cudaMemcpyAsync(cat + 4ll * H * H, e->LW(i, "gate.weight"), sizeof(float) * 4ll * H * H, cudaMemcpyDeviceToDevice, st);
      cudaMemcpyAsync(cat_bias, e->LW(i, "mlp_fc1.bias"), sizeof(float) * 4 * H, cudaMemcpyDeviceToDevice, st);
      cudaMemcpyAsync(cat_bias + 4 * H, e->LW(i, "gate.bias"), sizeof(float) * 4 * H, cudaMemcpyDeviceToDevice, st);
      rc = launch_pack_rows(cat, lp.w_glu, lp.b_glu, cat_bias, d_glu, 8 * H, H, st, dl ? e->LW(i, "norm3.weight") : nullptr,
                            dl ? e->LW(i, "norm3.bias") : nullptr, lp.c_glu);
    }
    se = cudaStreamSynchronize(st);
    cudaFree(d_glu);
    cudaFree(d_qkv);
    cudaFree(d_fc2);
    cudaFree(cat);
    if (rc) return rc;
    DITTO_CUDA(se);
  }
  DITTO_CUDA(cudaStreamSynchronize(st));
  e->finalized = true;
  return 0;
}

int64_t ditto_text_context_bytes(const ditto_engine_t* e, int64_t n_seq, int64_t S) {
  if (!e || n_seq <= 0 || S <= 0) return -1;
  return static_cast<int64_t>(ctx_layout(e, nullptr, n_seq, S).total);
}
int64_t ditto_workspace_bytes(const ditto_engine_t* e, int64_t n_seq, int64_t T, int64_t S) {
  if (!e || n_seq <= 0 || T <= 0 || S <= 0) return -1;
  return static_cast<int64_t>(ws_layout(e, nullptr, n_seq, T, S).total);
}

int32_t ditto_text_context(ditto_engine_t* e, const float* text_emb, int64_t n, int64_t S, void* ctx, void* workspace,
                           int64_t workspace_bytes, void* stream) {
  DITTO_REQUIRE(e && text_emb && ctx && workspace, DITTO_E_BADARG, "text_context: null argument");
  DITTO_REQUIRE(e->finalized, DITTO_E_STATE, "text_context: engine not finalized");
  DITTO_REQUIRE(n > 0 && S > 0, DITTO_E_BADARG, "text_context: empty input");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int H = e->H, Xd = e->Xd;
  // only the small tail of the workspace is needed here; lay it out with T = 1
  Workspace w = ws_layout(e, workspace, n, 1, S);
  DITTO_REQUIRE(static_cast<int64_t>(w.total) <= workspace_bytes, DITTO_E_WORKSPACE, "text_context: workspace too small");
  CtxLayout c = ctx_layout(e, ctx, n, S);
  // text modulation: text_mlp(SiLU(mean_S(text)))  (DiT.py:27,31)
  if (!e->blocks_only) {
    DITTO_TRY(launch_mean_silu(text_emb, w.tmp_small, n, static_cast<int>(S), Xd, st));
    DITTO_TRY(sgemm_nt(w.tmp_small, Xd, e->W("ada_ln.text_mlp.1.weight"), Xd, c.text_mod, 2 * H, e->W("ada_ln.text_mlp.1.bias"), nullptr,
                       0, 1.f, static_cast<int>(n), 2 * H, Xd, st));
  }
  // per-layer K|V = text @ in_proj[H:3H]^T + b  (torch MHA packed in_proj, rows H..3H)
  if (e->bf16_mode) DITTO_TRY(launch_cast_bf16(text_emb, w.text16, n * S * Xd, st));
  for (int i = 0; i < e->L; ++i) {
    void* kv = static_cast<char*>(c.kv0) + c.kv_stride * i;
    const float* bias = e->LW(i, "cross_attn.in_proj_bias") + H;
    if (e->bf16_mode) {
      DITTO_TRY(tc_nt(w.text16, Xd, e->layers[i].wc_in + static_cast<int64_t>(H) * H, H, kv, true, 2 * H, bias, nullptr, 0, 0, nullptr, 0,
                      static_cast<int>(n * S), 2 * H, Xd, st, PC_TC_TEXT_KV));
      if (fold_active(e, S)) {
        const int d = e->d, heads = e->heads;
        const int64_t Sp = round_up(S, 8);
        const bf16* kvb = static_cast<const bf16*>(kv);
        bf16* kf = c.kfold0 + c.kfold_stride * i;
        bf16* vf = c.vfold0 + c.vfold_stride * i;
        float* sb = c.sbias0 + c.sbias_stride * i;
        DITTO_CUDA(cudaMemsetAsync(vf, 0, c.vfold_stride * sizeof(bf16), st));
        // kfold[seq, h] (S x H) = K[seq][:, h*d:(h+1)*d] (S x d) @ Wq[h*d:(h+1)*d, :] (d x H, "KN" operand)
        TcGemmParams g;
        g.A.ptr = kvb; g.A.rows = S; g.A.cols = d; g.A.ld = 2 * H; g.A.s_inner = d; g.A.s_outer = S * 2 * H;
        // deferred LayerNorm: Wq diag(gamma2) instead of Wq, bq + Wq beta2 instead of bq, plus the row sums of the result
        const bool fln = fold_ln_active(e, S);
        g.B.ptr = fln ? e->layers[i].wq_g : e->layers[i].wc_in;
        g.B.rows = d; g.B.cols = H; g.B.ld = H; g.B.s_inner = static_cast<int64_t>(d) * H; g.B.s_outer = 0;
        g.b_kn = true;
        g.M = static_cast<int>(S); g.N = H; g.K = d; g.batch_inner = heads; g.batch_outer = static_cast<int>(n);
        g.out = kf; g.out_bf16 = true; g.ldo = H; g.so_inner = S * H; g.so_outer = static_cast<int64_t>(heads) * S * H;
        g.tag = PC_TC_TEXT_KV;
        DITTO_TRY(launch_tc_gemm(g, st));
        // vfold[seq, h*Sp + s, :] = V[seq][:, h*d:(h+1)*d] (S x d) @ Wo[:, h*d:(h+1)*d]^T
        TcGemmParams v;
        v.A.ptr = kvb + H; v.A.rows = S; v.A.cols = d; v.A.ld = 2 * H; v.A.s_inner = d; v.A.s_outer = S * 2 * H;
        v.B.ptr = cross_flash_active(e, S) ? e->layers[i].wc_o_p4 : e->layers[i].wc_o;   // output columns in the consumer's order
        v.B.rows = H; v.B.cols = d; v.B.ld = H; v.B.s_inner = d; v.B.s_outer = 0;
        v.M = static_cast<int>(S); v.N = H; v.K = d; v.batch_inner = heads; v.batch_outer = static_cast<int>(n);
        v.out = vf; v.out_bf16 = true; v.ldo = H; v.so_inner = Sp * H; v.so_outer = static_cast<int64_t>(heads) * Sp * H;
        v.tag = PC_TC_TEXT_KV;
        DITTO_TRY(launch_tc_gemm(v, st));
        DITTO_TRY(launch_fold_bias(kvb, 2 * H, fln ? e->layers[i].bq_g : e->LW(i, "cross_attn.in_proj_bias"), sb, n,
                                   static_cast<int>(S), static_cast<int>(Sp), heads, d, sqrtf(1.0f / static_cast<float>(d)), st));
        if (fln)
          DITTO_TRY(launch_rowsum_bf16(kf, c.cvec0 + c.sbias_stride * i, n * heads, static_cast<int>(S), static_cast<int>(Sp), H, st));
        if (c.cflag != nullptr)   // the flags once (layer 0), the constant rows of every layer
          DITTO_TRY(launch_const_text(text_emb, n, static_cast<int>(S), Xd, vf, Sp * H, cross_flash_active(e, S),
                                      e->LW(i, "cross_attn.out_proj.bias"), i == 0 ? c.cflag : nullptr, c.crow0 + c.crow_stride * i, H, st));
      }
    } else {
      DITTO_TRY(sgemm_nt(text_emb, Xd, e->LW(i, "cross_attn.in_proj_weight") + static_cast<int64_t>(H) * H, H, static_cast<float*>(kv),
                         2 * H, bias, nullptr, 0, 1.f, static_cast<int>(n * S), 2 * H, Xd, st));
    }
  }
  return 0;
}

int32_t ditto_forward(ditto_engine_t* e, const float* x, int64_t n_x, const void* ctx, const int64_t* t, int64_t n_seq, int64_t T,
                      int64_t S, float* out, void* workspace, int64_t workspace_bytes, void* stream) {
  DITTO_REQUIRE(e && x && ctx && t && out && workspace, DITTO_E_BADARG, "forward: null argument");
  DITTO_REQUIRE(e->finalized && !e->blocks_only, DITTO_E_STATE, "forward: engine not finalized (or a blocks-only engine)");
  DITTO_REQUIRE(n_seq > 0 && T > 0 && S > 0 && n_x > 0 && n_seq % n_x == 0, DITTO_E_BADARG, "forward: bad batch sizes");
  DITTO_REQUIRE(T <= e->maxT, DITTO_E_UNSUPPORTED, "forward: T exceeds max_seq_len of the engine");
  return forward_impl(e, x, n_x, ctx, t, n_seq, T, S, out, workspace, workspace_bytes, static_cast<cudaStream_t>(stream));
}

int32_t ditto_cfg_ddpm_update(ditto_engine_t* e, const float* eps_c, const float* eps_u, const float* x, const float* z,
                              const int64_t* t, float guidance_scale, float* x_out, int64_t B, int64_t elems_per_seq, void* stream) {
  DITTO_REQUIRE(e && eps_c && x && t && x_out, DITTO_E_BADARG, "cfg_ddpm_update: null argument");
  DITTO_REQUIRE(e->have_schedule, DITTO_E_STATE, "cfg_ddpm_update: schedule not loaded");
  DITTO_REQUIRE(B >= 0 && elems_per_seq >= 0, DITTO_E_BADARG, "cfg_ddpm_update: negative size");
  return launch_cfg_ddpm_update(eps_c, eps_u, x, z, t, e->coef, e->steps, guidance_scale, x_out, B, elems_per_seq,
                                static_cast<cudaStream_t>(stream));
}

// the update of one sampler step: the [steps, 3] DDPM-form table, or (hist != null) the [steps, 6] multistep table
static int launch_update(const ditto_engine* e, const float* eps_c, const float* eps_u, const float* x, const float* z, const int64_t* t,
                         float w, float* x_out, float* hist, int64_t B, int64_t per, cudaStream_t st) {
  if (hist) return launch_cfg_multistep_update(eps_c, eps_u, x, z, t, e->coef_ms, e->steps, w, x_out, hist, B, per, st);
  return launch_cfg_ddpm_update(eps_c, eps_u, x, z, t, e->coef, e->steps, w, x_out, B, per, st);
}
static int launch_update_rng(const ditto_engine* e, const float* eps_c, const float* eps_u, const float* x, uint64_t* rng, int64_t* t,
                             int64_t n_t, float w, float* x_out, float* hist, int64_t B, int64_t per, int64_t elem_offset, bool advance,
                             cudaStream_t st) {
  unsigned long long* r = reinterpret_cast<unsigned long long*>(rng);
  if (hist)
    return launch_cfg_multistep_update_rng(eps_c, eps_u, x, r, t, n_t, e->coef_ms, e->steps, w, x_out, hist, B, per, elem_offset, advance, st);
  return launch_cfg_ddpm_update_rng(eps_c, eps_u, x, r, t, n_t, e->coef, e->steps, w, x_out, B, per, elem_offset, advance, st);
}
// what every multistep entry point checks on top of its DDPM-form twin
static int require_multistep(const ditto_engine* e, const float* hist, const char* what) {
  DITTO_REQUIRE(e && hist, DITTO_E_BADARG, std::string(what) + ": null argument (hist)");
  DITTO_REQUIRE(e->coef_ms, DITTO_E_STATE, std::string(what) + ": no multistep table loaded (ditto_engine_load_multistep_table)");
  return 0;
}

static int32_t p_sample_impl(ditto_engine_t* e, const float* x, const void* ctx, const int64_t* t, const float* z, int32_t guided,
                             float guidance_scale, int64_t B, int64_t T, int64_t S, float* eps_scratch, float* x_out, float* hist,
                             void* workspace, int64_t workspace_bytes, void* stream) {
  DITTO_REQUIRE(e && x && ctx && t && eps_scratch && x_out && workspace, DITTO_E_BADARG, "p_sample: null argument");
  DITTO_REQUIRE(e->finalized && e->have_schedule && !e->blocks_only, DITTO_E_STATE, "p_sample: engine not finalized / schedule not loaded");
  DITTO_REQUIRE(B > 0 && T > 0 && S > 0 && T <= e->maxT, DITTO_E_BADARG, "p_sample: bad sizes");
  const int64_t n = guided ? 2 * B : B;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  DITTO_TRY(forward_impl(e, x, B, ctx, t, n, T, S, eps_scratch, workspace, workspace_bytes, st));
  const int64_t per = T * e->H;
  return launch_update(e, eps_scratch, guided ? eps_scratch + B * per : nullptr, x, z, t, guidance_scale, x_out, hist, B, per, st);
}

int32_t ditto_p_sample(ditto_engine_t* e, const float* x, const void* ctx, const int64_t* t, const float* z, int32_t guided,
                       float guidance_scale, int64_t B, int64_t T, int64_t S, float* eps_scratch, float* x_out, void* workspace,
                       int64_t workspace_bytes, void* stream) {
  return p_sample_impl(e, x, ctx, t, z, guided, guidance_scale, B, T, S, eps_scratch, x_out, nullptr, workspace, workspace_bytes, stream);
}

int32_t ditto_p_sample_multistep(ditto_engine_t* e, const float* x, const void* ctx, const int64_t* t, const float* z, int32_t guided,
                                 float guidance_scale, int64_t B, int64_t T, int64_t S, float* eps_scratch, float* x_out, float* hist,
                                 void* workspace, int64_t workspace_bytes, void* stream) {
  DITTO_TRY(require_multistep(e, hist, "p_sample_multistep"));
  return p_sample_impl(e, x, ctx, t, z, guided, guidance_scale, B, T, S, eps_scratch, x_out, hist, workspace, workspace_bytes, stream);
}

static int32_t p_sample_rng_impl(ditto_engine_t* e, const float* x, const void* ctx, int64_t* t, uint64_t* rng, int32_t guided,
                                 float guidance_scale, int64_t B, int64_t T, int64_t S, float* eps_scratch, float* x_out, float* hist,
                                 void* workspace, int64_t workspace_bytes, int32_t advance, void* stream) {
  DITTO_REQUIRE(e && x && ctx && t && rng && eps_scratch && x_out && workspace, DITTO_E_BADARG, "p_sample_rng: null argument");
  DITTO_REQUIRE(e->finalized && e->have_schedule && !e->blocks_only, DITTO_E_STATE, "p_sample_rng: engine not finalized / schedule not loaded");
  DITTO_REQUIRE(B > 0 && T > 0 && S > 0 && T <= e->maxT, DITTO_E_BADARG, "p_sample_rng: bad sizes");
  const int64_t n = guided ? 2 * B : B;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  DITTO_TRY(forward_impl(e, x, B, ctx, t, n, T, S, eps_scratch, workspace, workspace_bytes, st));
  const int64_t per = T * e->H;
  return launch_update_rng(e, eps_scratch, guided ? eps_scratch + B * per : nullptr, x, rng, t, n, guidance_scale, x_out, hist, B, per, 0,
                           advance != 0, st);
}

int32_t ditto_p_sample_rng(ditto_engine_t* e, const float* x, const void* ctx, int64_t* t, uint64_t* rng, int32_t guided,
                           float guidance_scale, int64_t B, int64_t T, int64_t S, float* eps_scratch, float* x_out, void* workspace,
                           int64_t workspace_bytes, int32_t advance, void* stream) {
  return p_sample_rng_impl(e, x, ctx, t, rng, guided, guidance_scale, B, T, S, eps_scratch, x_out, nullptr, workspace, workspace_bytes,
                           advance, stream);
}

int32_t ditto_p_sample_multistep_rng(ditto_engine_t* e, const float* x, const void* ctx, int64_t* t, uint64_t* rng, int32_t guided,
                                     float guidance_scale, int64_t B, int64_t T, int64_t S, float* eps_scratch, float* x_out, float* hist,
                                     void* workspace, int64_t workspace_bytes, int32_t advance, void* stream) {
  DITTO_TRY(require_multistep(e, hist, "p_sample_multistep_rng"));
  return p_sample_rng_impl(e, x, ctx, t, rng, guided, guidance_scale, B, T, S, eps_scratch, x_out, hist, workspace, workspace_bytes,
                           advance, stream);
}

int32_t ditto_cfg_ddpm_update_rng(ditto_engine_t* e, const float* eps_c, const float* eps_u, const float* x, uint64_t* rng, int64_t* t,
                                  int64_t n_t, float guidance_scale, float* x_out, int64_t B, int64_t elems_per_seq, int32_t advance,
                                  void* stream) {
  DITTO_REQUIRE(e && eps_c && x && t && rng && x_out, DITTO_E_BADARG, "cfg_ddpm_update_rng: null argument");
  DITTO_REQUIRE(e->have_schedule, DITTO_E_STATE, "cfg_ddpm_update_rng: schedule not loaded");
  DITTO_REQUIRE(B >= 0 && elems_per_seq >= 0 && n_t >= B, DITTO_E_BADARG, "cfg_ddpm_update_rng: bad sizes");
  return launch_cfg_ddpm_update_rng(eps_c, eps_u, x, reinterpret_cast<unsigned long long*>(rng), t, n_t, e->coef, e->steps, guidance_scale,
                                    x_out, B, elems_per_seq, 0, advance != 0, static_cast<cudaStream_t>(stream));
}

int32_t ditto_cfg_multistep_update(ditto_engine_t* e, const float* eps_c, const float* eps_u, const float* x, const float* z,
                                   const int64_t* t, float guidance_scale, float* x_out, float* hist, int64_t B, int64_t elems_per_seq,
                                   void* stream) {
  DITTO_REQUIRE(e && eps_c && x && t && x_out, DITTO_E_BADARG, "cfg_multistep_update: null argument");
  DITTO_REQUIRE(B >= 0 && elems_per_seq >= 0, DITTO_E_BADARG, "cfg_multistep_update: negative size");
  DITTO_TRY(require_multistep(e, hist, "cfg_multistep_update"));
  return launch_update(e, eps_c, eps_u, x, z, t, guidance_scale, x_out, hist, B, elems_per_seq, static_cast<cudaStream_t>(stream));
}

int32_t ditto_cfg_multistep_update_rng(ditto_engine_t* e, const float* eps_c, const float* eps_u, const float* x, uint64_t* rng,
                                       int64_t* t, int64_t n_t, float guidance_scale, float* x_out, float* hist, int64_t B,
                                       int64_t elems_per_seq, int32_t advance, void* stream) {
  DITTO_REQUIRE(e && eps_c && x && t && rng && x_out, DITTO_E_BADARG, "cfg_multistep_update_rng: null argument");
  DITTO_REQUIRE(B >= 0 && elems_per_seq >= 0 && n_t >= B, DITTO_E_BADARG, "cfg_multistep_update_rng: bad sizes");
  DITTO_TRY(require_multistep(e, hist, "cfg_multistep_update_rng"));
  return launch_update_rng(e, eps_c, eps_u, x, rng, t, n_t, guidance_scale, x_out, hist, B, elems_per_seq, 0, advance != 0,
                           static_cast<cudaStream_t>(stream));
}

// ---- known frames (speech prompt / infilling) -----------------------------------------------------------
// what every known-frame entry point checks before it launches anything
static int require_known(const ditto_engine* e, const float* z, const uint64_t* rng, const float* hist, const float* known,
                         const uint8_t* known_mask, int32_t advance, const char* what) {
  const std::string w(what);
  DITTO_REQUIRE(e && known && known_mask, DITTO_E_BADARG, w + ": null argument (known / known_mask)");
  DITTO_REQUIRE((z == nullptr) != (rng == nullptr), DITTO_E_BADARG, w + ": exactly one of z / rng (known frames need the step's noise)");
  DITTO_REQUIRE(!advance || rng, DITTO_E_BADARG, w + ": advance needs rng (in-kernel noise)");
  DITTO_REQUIRE(e->have_schedule, DITTO_E_STATE, w + ": schedule not loaded");
  DITTO_REQUIRE(e->coef_known, DITTO_E_STATE, w + ": no known table loaded (ditto_engine_load_known_table)");
  DITTO_REQUIRE(!hist || e->coef_ms, DITTO_E_STATE, w + ": no multistep table loaded (ditto_engine_load_multistep_table)");
  return 0;
}
// the update of one step with known frames: the DDPM-form table, or (hist != null) the multistep table
static int launch_update_known(const ditto_engine* e, const float* eps_c, const float* eps_u, const float* x, const float* z, uint64_t* rng,
                               int64_t* t, int64_t n_t, float w, float* x_out, float* hist, const float* known, const uint8_t* mask,
                               int64_t B, int64_t T, int64_t elem_offset, bool advance, cudaStream_t st) {
  return launch_cfg_update_known(eps_c, eps_u, x, z, reinterpret_cast<unsigned long long*>(rng), t, n_t, hist ? e->coef_ms : e->coef,
                                 e->coef_known, e->steps, w, x_out, hist, known, mask, B, T, e->H, elem_offset, advance, st);
}

int32_t ditto_cfg_update_known(ditto_engine_t* e, const float* eps_c, const float* eps_u, const float* x, const float* z, uint64_t* rng,
                               int64_t* t, int64_t n_t, float guidance_scale, float* x_out, float* hist, const float* known,
                               const uint8_t* known_mask, int64_t B, int64_t T, int32_t advance, void* stream) {
  DITTO_REQUIRE(e && eps_c && x && t && x_out, DITTO_E_BADARG, "cfg_update_known: null argument");
  DITTO_REQUIRE(B >= 0 && T >= 0 && (!rng || n_t >= B), DITTO_E_BADARG, "cfg_update_known: bad sizes");
  DITTO_TRY(require_known(e, z, rng, hist, known, known_mask, advance, "cfg_update_known"));
  return launch_update_known(e, eps_c, eps_u, x, z, rng, t, n_t, guidance_scale, x_out, hist, known, known_mask, B, T, 0, advance != 0,
                             static_cast<cudaStream_t>(stream));
}

int32_t ditto_p_sample_known(ditto_engine_t* e, const float* x, const void* ctx, int64_t* t, const float* z, uint64_t* rng, int32_t guided,
                             float guidance_scale, int64_t B, int64_t T, int64_t S, float* eps_scratch, float* x_out, float* hist,
                             const float* known, const uint8_t* known_mask, void* workspace, int64_t workspace_bytes, int32_t advance,
                             void* stream) {
  DITTO_REQUIRE(e && x && ctx && t && eps_scratch && x_out && workspace, DITTO_E_BADARG, "p_sample_known: null argument");
  DITTO_REQUIRE(e->finalized && !e->blocks_only, DITTO_E_STATE, "p_sample_known: engine not finalized");
  DITTO_REQUIRE(B > 0 && T > 0 && S > 0 && T <= e->maxT, DITTO_E_BADARG, "p_sample_known: bad sizes");
  DITTO_TRY(require_known(e, z, rng, hist, known, known_mask, advance, "p_sample_known"));
  const int64_t n = guided ? 2 * B : B;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  DITTO_TRY(forward_impl(e, x, B, ctx, t, n, T, S, eps_scratch, workspace, workspace_bytes, st));
  const int64_t per = T * e->H;
  return launch_update_known(e, eps_scratch, guided ? eps_scratch + B * per : nullptr, x, z, rng, t, n, guidance_scale, x_out, hist, known,
                             known_mask, B, T, 0, advance != 0, st);
}

int32_t ditto_randn(const uint64_t* rng, int64_t elem_offset, float* out, int64_t n, void* stream) {
  DITTO_REQUIRE(rng && out && n >= 0 && elem_offset >= 0, DITTO_E_BADARG, "randn: bad argument");
  return launch_randn(reinterpret_cast<const unsigned long long*>(rng), elem_offset, out, n, static_cast<cudaStream_t>(stream));
}

int32_t ditto_q_sample(ditto_engine_t* e, const float* x_start, const float* noise, const int64_t* t, float* out, int64_t B,
                       int64_t elems_per_seq, void* stream) {
  DITTO_REQUIRE(e && x_start && noise && t && out, DITTO_E_BADARG, "q_sample: null argument");
  DITTO_REQUIRE(e->have_schedule, DITTO_E_STATE, "q_sample: schedule not loaded");
  return launch_q_sample(x_start, noise, t, e->qs_buf, e->steps, out, B, elems_per_seq, static_cast<cudaStream_t>(stream));
}

// ---- ragged batches ------------------------------------------------------------------------------------
static int parse_groups(const ditto_engine_t* e, const ditto_seq_group_t* groups, int64_t n_groups, bool need_ctx,
                        std::vector<SeqGroup>& gs) {
  DITTO_REQUIRE(e && groups && n_groups > 0 && n_groups <= 4096, DITTO_E_BADARG, "ragged: bad group list");
  gs.resize(static_cast<size_t>(n_groups));
  for (int64_t i = 0; i < n_groups; ++i) {
    const ditto_seq_group_t& q = groups[i];
    DITTO_REQUIRE(q.n_seq > 0 && q.T > 0 && q.S > 0 && q.n_x > 0 && q.n_seq % q.n_x == 0, DITTO_E_BADARG, "ragged: bad group sizes");
    DITTO_REQUIRE(q.T <= e->maxT, DITTO_E_UNSUPPORTED, "ragged: T exceeds max_seq_len of the engine");
    DITTO_REQUIRE(!need_ctx || q.ctx != nullptr, DITTO_E_BADARG, "ragged: group without a text context");
    SeqGroup& g = gs[static_cast<size_t>(i)];
    g.n = q.n_seq; g.n_x = q.n_x; g.T = q.T; g.S = q.S; g.ctx = q.ctx;
  }
  return 0;
}

int64_t ditto_workspace_bytes_ragged(const ditto_engine_t* e, const ditto_seq_group_t* groups, int64_t n_groups) {
  std::vector<SeqGroup> gs;
  if (parse_groups(e, groups, n_groups, false, gs) != 0) return -1;
  return static_cast<int64_t>(ws_layout(e, nullptr, gs.data(), static_cast<int>(gs.size())).total);
}

int32_t ditto_forward_ragged(ditto_engine_t* e, const float* x, const ditto_seq_group_t* groups, int64_t n_groups, const int64_t* t,
                             float* out, void* workspace, int64_t workspace_bytes, void* stream) {
  DITTO_REQUIRE(e && x && t && out && workspace, DITTO_E_BADARG, "forward_ragged: null argument");
  DITTO_REQUIRE(e->finalized, DITTO_E_STATE, "forward_ragged: engine not finalized");
  std::vector<SeqGroup> gs;
  DITTO_TRY(parse_groups(e, groups, n_groups, true, gs));
  return forward_impl(e, x, t, gs.data(), static_cast<int>(gs.size()), out, workspace, workspace_bytes, static_cast<cudaStream_t>(stream));
}

static int32_t p_sample_ragged_impl(ditto_engine_t* e, const float* x, const ditto_seq_group_t* groups, int64_t n_groups, const int64_t* t,
                                    const float* z, int32_t guided, float guidance_scale, float* eps_scratch, float* x_out, float* hist,
                                    void* workspace, int64_t workspace_bytes, void* stream) {
  DITTO_REQUIRE(e && x && t && eps_scratch && x_out && workspace, DITTO_E_BADARG, "p_sample_ragged: null argument");
  DITTO_REQUIRE(e->finalized && e->have_schedule, DITTO_E_STATE, "p_sample_ragged: engine not finalized / schedule not loaded");
  std::vector<SeqGroup> gs;
  DITTO_TRY(parse_groups(e, groups, n_groups, true, gs));
  for (const SeqGroup& g : gs)
    DITTO_REQUIRE(g.n == (guided ? 2 : 1) * g.n_x, DITTO_E_BADARG, "p_sample_ragged: n_seq must be n_x (unguided) or 2 n_x (guided)");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  DITTO_TRY(forward_impl(e, x, t, gs.data(), static_cast<int>(gs.size()), eps_scratch, workspace, workspace_bytes, st));
  const int64_t H = e->H;
  std::unique_lock<std::recursive_mutex> fork_lock(e->fork_mutex, std::defer_lock);
  if (gs.size() > 1 && e->n_side > 0) fork_lock.lock();
  Fork fork(e, st);
  DITTO_TRY(fork.begin(static_cast<int>(gs.size())));
  for (size_t gi = 0; gi < gs.size(); ++gi) {  // offsets were filled in by the layout pass of forward_impl
    const SeqGroup& g = gs[gi];
    const int64_t per = g.T * H;
    const float* ec = eps_scratch + g.row0 * H;
    DITTO_TRY(launch_update(e, ec, guided ? ec + g.n_x * per : nullptr, x + g.xrow0 * H, z ? z + g.xrow0 * H : nullptr, t + g.seq0,
                            guidance_scale, x_out + g.xrow0 * H, hist ? hist + g.xrow0 * H : nullptr, g.n_x, per,
                            fork.stream(static_cast<int>(gi))));
  }
  DITTO_TRY(fork.end());
  return 0;
}

int32_t ditto_p_sample_ragged(ditto_engine_t* e, const float* x, const ditto_seq_group_t* groups, int64_t n_groups, const int64_t* t,
                              const float* z, int32_t guided, float guidance_scale, float* eps_scratch, float* x_out, void* workspace,
                              int64_t workspace_bytes, void* stream) {
  return p_sample_ragged_impl(e, x, groups, n_groups, t, z, guided, guidance_scale, eps_scratch, x_out, nullptr, workspace,
                              workspace_bytes, stream);
}

int32_t ditto_p_sample_ragged_multistep(ditto_engine_t* e, const float* x, const ditto_seq_group_t* groups, int64_t n_groups,
                                        const int64_t* t, const float* z, int32_t guided, float guidance_scale, float* eps_scratch,
                                        float* x_out, float* hist, void* workspace, int64_t workspace_bytes, void* stream) {
  DITTO_TRY(require_multistep(e, hist, "p_sample_ragged_multistep"));
  return p_sample_ragged_impl(e, x, groups, n_groups, t, z, guided, guidance_scale, eps_scratch, x_out, hist, workspace,
                              workspace_bytes, stream);
}

static int32_t p_sample_ragged_rng_impl(ditto_engine_t* e, const float* x, const ditto_seq_group_t* groups, int64_t n_groups, int64_t* t,
                                        uint64_t* rng, int32_t guided, float guidance_scale, float* eps_scratch, float* x_out,
                                        float* hist, void* workspace, int64_t workspace_bytes, int32_t advance, void* stream) {
  DITTO_REQUIRE(e && x && t && rng && eps_scratch && x_out && workspace, DITTO_E_BADARG, "p_sample_ragged_rng: null argument");
  DITTO_REQUIRE(e->finalized && e->have_schedule && !e->blocks_only, DITTO_E_STATE, "p_sample_ragged_rng: engine not finalized / schedule not loaded");
  std::vector<SeqGroup> gs;
  DITTO_TRY(parse_groups(e, groups, n_groups, true, gs));
  int64_t n_t = 0;
  for (const SeqGroup& g : gs) {
    DITTO_REQUIRE(g.n == (guided ? 2 : 1) * g.n_x, DITTO_E_BADARG, "p_sample_ragged_rng: n_seq must be n_x (unguided) or 2 n_x (guided)");
    n_t += g.n;
  }
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  DITTO_TRY(forward_impl(e, x, t, gs.data(), static_cast<int>(gs.size()), eps_scratch, workspace, workspace_bytes, st));
  const int64_t H = e->H;
  std::unique_lock<std::recursive_mutex> fork_lock(e->fork_mutex, std::defer_lock);
  if (gs.size() > 1 && e->n_side > 0) fork_lock.lock();
  Fork fork(e, st);
  DITTO_TRY(fork.begin(static_cast<int>(gs.size())));
  for (size_t gi = 0; gi < gs.size(); ++gi) {
    const SeqGroup& g = gs[gi];
    const int64_t per = g.T * H;
    const float* ec = eps_scratch + g.row0 * H;
    // element offset = position in the packed latent buffer: every element of the batch draws its own normal
    DITTO_TRY(launch_update_rng(e, ec, guided ? ec + g.n_x * per : nullptr, x + g.xrow0 * H, rng, t + g.seq0, g.n, guidance_scale,
                                x_out + g.xrow0 * H, hist ? hist + g.xrow0 * H : nullptr, g.n_x, per, g.xrow0 * H, false,
                                fork.stream(static_cast<int>(gi))));
  }
  DITTO_TRY(fork.end());
  if (advance) DITTO_TRY(launch_step_advance(reinterpret_cast<unsigned long long*>(rng), t, n_t, st));
  return 0;
}

int32_t ditto_p_sample_ragged_rng(ditto_engine_t* e, const float* x, const ditto_seq_group_t* groups, int64_t n_groups, int64_t* t,
                                  uint64_t* rng, int32_t guided, float guidance_scale, float* eps_scratch, float* x_out, void* workspace,
                                  int64_t workspace_bytes, int32_t advance, void* stream) {
  return p_sample_ragged_rng_impl(e, x, groups, n_groups, t, rng, guided, guidance_scale, eps_scratch, x_out, nullptr, workspace,
                                  workspace_bytes, advance, stream);
}

int32_t ditto_p_sample_ragged_multistep_rng(ditto_engine_t* e, const float* x, const ditto_seq_group_t* groups, int64_t n_groups,
                                            int64_t* t, uint64_t* rng, int32_t guided, float guidance_scale, float* eps_scratch,
                                            float* x_out, float* hist, void* workspace, int64_t workspace_bytes, int32_t advance,
                                            void* stream) {
  DITTO_TRY(require_multistep(e, hist, "p_sample_ragged_multistep_rng"));
  return p_sample_ragged_rng_impl(e, x, groups, n_groups, t, rng, guided, guidance_scale, eps_scratch, x_out, hist, workspace,
                                  workspace_bytes, advance, stream);
}

int32_t ditto_p_sample_ragged_known(ditto_engine_t* e, const float* x, const ditto_seq_group_t* groups, int64_t n_groups, int64_t* t,
                                    const float* z, uint64_t* rng, int32_t guided, float guidance_scale, float* eps_scratch, float* x_out,
                                    float* hist, const float* known, const uint8_t* known_mask, void* workspace, int64_t workspace_bytes,
                                    int32_t advance, void* stream) {
  DITTO_REQUIRE(e && x && t && eps_scratch && x_out && workspace, DITTO_E_BADARG, "p_sample_ragged_known: null argument");
  DITTO_REQUIRE(e->finalized && !e->blocks_only, DITTO_E_STATE, "p_sample_ragged_known: engine not finalized");
  DITTO_TRY(require_known(e, z, rng, hist, known, known_mask, advance, "p_sample_ragged_known"));
  std::vector<SeqGroup> gs;
  DITTO_TRY(parse_groups(e, groups, n_groups, true, gs));
  int64_t n_t = 0;
  for (const SeqGroup& g : gs) {
    DITTO_REQUIRE(g.n == (guided ? 2 : 1) * g.n_x, DITTO_E_BADARG, "p_sample_ragged_known: n_seq must be n_x (unguided) or 2 n_x (guided)");
    n_t += g.n;
  }
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  DITTO_TRY(forward_impl(e, x, t, gs.data(), static_cast<int>(gs.size()), eps_scratch, workspace, workspace_bytes, st));
  const int64_t H = e->H;
  std::unique_lock<std::recursive_mutex> fork_lock(e->fork_mutex, std::defer_lock);
  if (gs.size() > 1 && e->n_side > 0) fork_lock.lock();
  Fork fork(e, st);
  DITTO_TRY(fork.begin(static_cast<int>(gs.size())));
  for (size_t gi = 0; gi < gs.size(); ++gi) {
    const SeqGroup& g = gs[gi];
    const int64_t per = g.T * H;
    const float* ec = eps_scratch + g.row0 * H;
    // x, z, hist, known: packed rows from xrow0; the mask: one byte per packed row; noise offset = packed element position
    DITTO_TRY(launch_update_known(e, ec, guided ? ec + g.n_x * per : nullptr, x + g.xrow0 * H, z ? z + g.xrow0 * H : nullptr, rng,
                                  t + g.seq0, g.n, guidance_scale, x_out + g.xrow0 * H, hist ? hist + g.xrow0 * H : nullptr,
                                  known + g.xrow0 * H, known_mask + g.xrow0, g.n_x, g.T, g.xrow0 * H, false,
                                  fork.stream(static_cast<int>(gi))));
  }
  DITTO_TRY(fork.end());
  if (advance) DITTO_TRY(launch_step_advance(reinterpret_cast<unsigned long long*>(rng), t, n_t, st));
  return 0;
}

// ---- block-level operators (the reference's component signatures, src/components/DiT.py) -----------------------------
int32_t ditto_dit_block(ditto_engine_t* e, int32_t layer, const float* x, const void* ctx, int64_t n_seq, int64_t T, int64_t S, float* out,
                        void* workspace, int64_t workspace_bytes, void* stream) {
  DITTO_REQUIRE(e && x && ctx && out && workspace, DITTO_E_BADARG, "dit_block: null argument");
  DITTO_REQUIRE(e->finalized, DITTO_E_STATE, "dit_block: engine not finalized");
  DITTO_REQUIRE(layer >= 0 && layer < e->L, DITTO_E_BADARG, "dit_block: layer out of range");
  DITTO_REQUIRE(n_seq > 0 && T > 0 && S > 0 && T <= e->maxT, DITTO_E_BADARG, "dit_block: bad sizes");
  SeqGroup g;
  g.n = n_seq; g.n_x = n_seq; g.T = T; g.S = S; g.ctx = ctx;
  return forward_impl(e, x, nullptr, &g, 1, out, workspace, workspace_bytes, static_cast<cudaStream_t>(stream), layer);
}

// the three sections of DiT.forward on their own: LayerNorm -> section -> + residual
static int32_t dit_section(ditto_engine_t* e, int32_t layer, int stage, const char* what, const float* x, const void* ctx, int64_t n_seq,
                           int64_t T, int64_t S, float* out, void* workspace, int64_t workspace_bytes, void* stream) {
  DITTO_REQUIRE(e && x && ctx && out && workspace, DITTO_E_BADARG, std::string(what) + ": null argument");
  DITTO_REQUIRE(e->finalized, DITTO_E_STATE, std::string(what) + ": engine not finalized");
  DITTO_REQUIRE(layer >= 0 && layer < e->L, DITTO_E_BADARG, std::string(what) + ": layer out of range");
  DITTO_REQUIRE(n_seq > 0 && T > 0 && S > 0 && T <= e->maxT, DITTO_E_BADARG, std::string(what) + ": bad sizes");
  SeqGroup g;
  g.n = n_seq; g.n_x = n_seq; g.T = T; g.S = S; g.ctx = ctx;
  return forward_impl(e, x, nullptr, &g, 1, out, workspace, workspace_bytes, static_cast<cudaStream_t>(stream), layer, stage);
}
int32_t ditto_attn_self(ditto_engine_t* e, int32_t layer, const float* x, const void* ctx, int64_t n_seq, int64_t T, int64_t S, float* out,
                        void* workspace, int64_t workspace_bytes, void* stream) {
  return dit_section(e, layer, 1, "attn_self", x, ctx, n_seq, T, S, out, workspace, workspace_bytes, stream);
}
int32_t ditto_attn_cross(ditto_engine_t* e, int32_t layer, const float* x, const void* ctx, int64_t n_seq, int64_t T, int64_t S, float* out,
                         void* workspace, int64_t workspace_bytes, void* stream) {
  return dit_section(e, layer, 2, "attn_cross", x, ctx, n_seq, T, S, out, workspace, workspace_bytes, stream);
}
int32_t ditto_gated_mlp(ditto_engine_t* e, int32_t layer, const float* x, const void* ctx, int64_t n_seq, int64_t T, int64_t S, float* out,
                        void* workspace, int64_t workspace_bytes, void* stream) {
  return dit_section(e, layer, 3, "gated_mlp", x, ctx, n_seq, T, S, out, workspace, workspace_bytes, stream);
}

int64_t ditto_adaln_workspace_bytes(int64_t n_seq, int64_t H, int64_t time_dim, int64_t text_dim) {
  if (n_seq <= 0 || H <= 0 || time_dim <= 0 || text_dim <= 0) return -1;
  Arena a(nullptr);
  a.take<float>(n_seq * time_dim); a.take<float>(n_seq * 2 * H); a.take<float>(n_seq * text_dim); a.take<float>(n_seq * 2 * H);
  return static_cast<int64_t>(a.off + 256);
}

int32_t ditto_adaln(const float* x, const float* time_emb, const float* text_emb, const float* w_time, const float* b_time,
                    const float* w_text, const float* b_text, float* out, int64_t n_seq, int64_t T, int64_t S, int64_t H, int64_t time_dim,
                    int64_t text_dim, void* workspace, int64_t workspace_bytes, void* stream) {
  DITTO_REQUIRE(x && time_emb && text_emb && w_time && b_time && w_text && b_text && out && workspace, DITTO_E_BADARG, "adaln: null argument");
  DITTO_REQUIRE(n_seq > 0 && T > 0 && S > 0 && H > 0 && H % 4 == 0 && H <= 1024 && time_dim % 4 == 0 && text_dim > 0, DITTO_E_UNSUPPORTED,
                "adaln: need H % 4 == 0, H <= 1024, time_dim % 4 == 0");
  DITTO_REQUIRE(ditto_adaln_workspace_bytes(n_seq, H, time_dim, text_dim) <= workspace_bytes, DITTO_E_WORKSPACE, "adaln: workspace too small");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  Arena a(workspace);
  float* ts = a.take<float>(n_seq * time_dim);
  float* tm = a.take<float>(n_seq * 2 * H);
  float* pooled = a.take<float>(n_seq * text_dim);
  float* xm = a.take<float>(n_seq * 2 * H);
  // [time_scale | time_shift] = Linear(SiLU(time_emb))  (DiT.py:14-17,30);  [text_scale | text_shift] = Linear(SiLU(mean_S text))  (:27,31)
  DITTO_CUDA(cudaMemcpyAsync(ts, time_emb, sizeof(float) * n_seq * time_dim, cudaMemcpyDeviceToDevice, st));
  DITTO_TRY(launch_silu(ts, n_seq * time_dim, st));
  DITTO_TRY(sgemm_nt(ts, time_dim, w_time, time_dim, tm, 2 * H, b_time, nullptr, 0, 1.f, static_cast<int>(n_seq), static_cast<int>(2 * H),
                     static_cast<int>(time_dim), st));
  DITTO_TRY(launch_mean_silu(text_emb, pooled, n_seq, static_cast<int>(S), static_cast<int>(text_dim), st));
  DITTO_TRY(sgemm_nt(pooled, text_dim, w_text, text_dim, xm, 2 * H, b_text, nullptr, 0, 1.f, static_cast<int>(n_seq), static_cast<int>(2 * H),
                     static_cast<int>(text_dim), st));
  // LN_noaffine(x) (1 + ts + xs) + (tb + xb)  (DiT.py:34-39): the fused kernel with one table row per sequence and no LN1 stage
  return launch_adaln_ln(x, n_seq, tm, xm, nullptr, static_cast<int>(n_seq), nullptr, nullptr, out, nullptr, false, nullptr, n_seq,
                         static_cast<int>(T), static_cast<int>(H), st);
}

int32_t ditto_rope(const float* t, const float* pos, float* out, int64_t batch, int64_t T, int64_t heads, int64_t head_dim, void* stream) {
  DITTO_REQUIRE(t && pos && out, DITTO_E_BADARG, "rope: null argument");
  DITTO_REQUIRE(batch >= 0 && T > 0 && heads > 0 && head_dim > 0 && head_dim % 2 == 0, DITTO_E_BADARG, "rope: bad sizes (head_dim must be even)");
  return launch_rope_angles(t, pos, out, batch, static_cast<int>(T), static_cast<int>(heads), static_cast<int>(head_dim),
                            static_cast<cudaStream_t>(stream));
}

int32_t ditto_attn_self768(const void* qkv, int64_t ld, int64_t n_seq, int64_t T, float alpha, float* h, const float* gamma,
                           const float* beta, void* u_out, int32_t flags, void* stream) {
  DITTO_REQUIRE(qkv && h && n_seq > 0 && T > 0 && T < (1ll << 30), DITTO_E_BADARG, "attn_self768: bad argument");
  Flash768Params f;
  f.qkv = static_cast<const bf16*>(qkv); f.ld = ld; f.n_seq = n_seq; f.T = static_cast<int>(T); f.H = 768; f.alpha = alpha; f.h = h;
  f.gamma = gamma; f.beta = beta; f.u_out = static_cast<bf16*>(u_out); f.force_rescale = (flags & 1) != 0; f.dbg = flags >> 8; f.tag = PC_FLASH768;
  return launch_flash768(f, static_cast<cudaStream_t>(stream));
}

// ---- developer options: A/B switches of the kernels (tools/, tests/); the library never reads the environment ------
int32_t ditto_debug_option(const char* name, int32_t value) {
  DITTO_REQUIRE(name != nullptr, DITTO_E_BADARG, "debug_option: null name");
  struct Opt { const char* n; int* p; };
  const Opt opts[] = {
      {"no_pair", &g_opt.no_pair}, {"cluster_m", &g_opt.cluster_m}, {"cluster_n", &g_opt.cluster_n}, {"generic_epi", &g_opt.generic_epi},
      {"stages_1cta", &g_opt.stages_1cta}, {"stages_pair", &g_opt.stages_pair}, {"no_mcast", &g_opt.no_mcast}, {"xf_rows", &g_opt.xf_rows}, {"xf_prefetch", &g_opt.xf_prefetch},
      {"no_defer_ln", &g_opt.no_defer_ln}, {"no_fused_attn", &g_opt.no_fused_attn}, {"no_flash", &g_opt.no_flash},
      {"no_flash768", &g_opt.no_flash768}, {"no_fused_cross", &g_opt.no_fused_cross}, {"defer_ln2", &g_opt.defer_ln2},
      {"pv_transpose", &g_opt.pv_transpose}, {"rope_table", &g_opt.rope_table}, {"rope_generic", &g_opt.rope_generic},
      {"glu_generic", &g_opt.glu_generic}, {"no_rope_fast32", &g_opt.no_rope_fast32}, {"no_pv_perm4", &g_opt.no_pv_perm4},
      {"side_streams", &g_opt.side_streams}, {"no_fused_ln", &g_opt.no_fused_ln}, {"flash768_quad", &g_opt.flash768_quad},
      {"no_fc2_ln", &g_opt.no_fc2_ln}, {"no_cross_flash", &g_opt.no_cross_flash}, {"no_const_text", &g_opt.no_const_text}, {"dbg_nostore", &g_opt.dbg_nostore}};
  if (strcmp(name, "reset") == 0) { g_opt = DebugOptions(); return 0; }
  for (const Opt& o : opts)
    if (strcmp(name, o.n) == 0) { *o.p = value; return 0; }
  set_error(std::string("debug_option: unknown option '") + name + "'");
  return DITTO_E_BADARG;
}

// ---- single operators ---------------------------------------------------------------------------------
int32_t ditto_layernorm(const float* x, const float* gamma, const float* beta, void* y, int32_t out_bf16, int64_t rows, int64_t H,
                        void* stream) {
  DITTO_REQUIRE(x && y && rows >= 0 && H > 0, DITTO_E_BADARG, "layernorm: bad argument");
  return launch_layernorm(x, gamma, beta, y, out_bf16 != 0, rows, static_cast<int>(H), static_cast<cudaStream_t>(stream));
}

int32_t ditto_gemm_f32(const float* A, int64_t lda, int64_t strideA, const float* B, int64_t ldb, int64_t strideB, int32_t b_is_nk,
                       float* C, int64_t ldc, int64_t strideC, const float* bias, const float* resid, float alpha, int64_t M, int64_t N,
                       int64_t K, int64_t batch, void* stream) {
  DITTO_REQUIRE(A && B && C && batch >= 1, DITTO_E_BADARG, "gemm_f32: bad argument");
  SgemmParams p;
  p.A = A; p.lda = lda; p.sA_outer = strideA; p.B = B; p.ldb = ldb; p.sB_outer = strideB; p.b_is_nk = b_is_nk != 0;
  p.C = C; p.ldc = ldc; p.sC_outer = strideC; p.bias = bias; p.resid = resid; p.ldr = ldc; p.sR_outer = strideC; p.alpha = alpha;
  p.M = static_cast<int>(M); p.N = static_cast<int>(N); p.K = static_cast<int>(K); p.batch_outer = static_cast<int>(batch);
  return launch_sgemm(p, static_cast<cudaStream_t>(stream));
}

int32_t ditto_gemm_resid_ln_weight_row(int32_t packed_row) { return packed_row >= 0 ? gemm_resid_ln_weight_row(packed_row) : -1; }
int32_t ditto_gemm_resid_ln(const void* A, int64_t lda, const void* W, int64_t ldw, const float* bias, float* h, int64_t ldh,
                            const float* gamma, const float* beta, void* u, int64_t ldu, int64_t M, int64_t N, int64_t K, void* stream) {
  DITTO_REQUIRE(A && W && bias && h && M > 0 && M < (1ll << 31) && N > 0 && K > 0 && N < (1 << 20) && K < (1 << 24), DITTO_E_BADARG,
                "gemm_resid_ln: bad argument");
  GemmResidLnParams f;
  f.A = static_cast<const bf16*>(A); f.lda = lda; f.W = static_cast<const bf16*>(W); f.ldw = ldw; f.bias = bias;
  f.h = h; f.ldh = ldh; f.gamma = gamma; f.beta = beta; f.u = static_cast<bf16*>(u); f.ldu = ldu;
  f.M = static_cast<int>(M); f.N = static_cast<int>(N); f.K = static_cast<int>(K);
  return launch_gemm_resid_ln(f, static_cast<cudaStream_t>(stream));
}

int32_t ditto_gemm_bf16(const void* A, int64_t lda, const void* W, int64_t ldw, void* C, int64_t ldc, int32_t out_bf16,
                        const float* bias, const float* resid, int64_t ldr, float alpha, int64_t M, int64_t N, int64_t K, void* stream) {
  DITTO_REQUIRE(A && W && C, DITTO_E_BADARG, "gemm_bf16: null argument");
  TcGemmParams p;
  p.A.ptr = static_cast<const bf16*>(A); p.A.rows = M; p.A.cols = K; p.A.ld = lda;
  p.B.ptr = static_cast<const bf16*>(W); p.B.rows = N; p.B.cols = K; p.B.ld = ldw;
  p.M = static_cast<int>(M); p.N = static_cast<int>(N); p.K = static_cast<int>(K);
  p.alpha = alpha; p.bias = bias; p.out = C; p.out_bf16 = out_bf16 != 0; p.ldo = ldc; p.resid = resid; p.ldr = ldr;
  return launch_tc_gemm(p, static_cast<cudaStream_t>(stream));
}

int32_t ditto_cast_bf16(const float* x, void* y, int64_t n, void* stream) {
  DITTO_REQUIRE(x && y && n >= 0, DITTO_E_BADARG, "cast_bf16: bad argument");
  return launch_cast_bf16(x, static_cast<bf16*>(y), n, static_cast<cudaStream_t>(stream));
}

#pragma GCC visibility pop
}  // extern "C"
