// C ABI of libmudpt_b200.so (include/mudpt_b200.h): handle, frozen-weight conversion, tower
// forward / dgrad-only backward orchestration (to the prompts, and through the vision stem to the images).  All launches go to the caller's stream; no
// device synchronisation happens here (except the one-time read of logit_scale in set_weight).
#include "../../include/mudpt_b200.h"

#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "attention.h"
#include "augment.h"
#include "gemm.h"
#include "head.h"
#include "launch_count.h"
#include "prompt.h"
#include "peer.h"
#include "rowops.h"

namespace mudpt {
std::atomic<long long> g_launch_counter{0};
}

using namespace mudpt;
typedef __nv_bfloat16 bf16;

static thread_local std::string g_err;

namespace {

constexpr float kLnEps = 1e-5f;  // nn.LayerNorm default (clip/model.py:164)

struct Layer {
  // bf16 GEMM operands: forward uses the [out,in] weight as stored, dgrad the transposed copy
  bf16 *w_in = nullptr, *w_in_t = nullptr, *w_out = nullptr, *w_out_t = nullptr;
  bf16 *w_fc = nullptr, *w_fc_t = nullptr, *w_pr = nullptr, *w_pr_t = nullptr;
  float *b_in = nullptr, *b_out = nullptr, *b_fc = nullptr, *b_pr = nullptr;
  float *ln1_g = nullptr, *ln1_b = nullptr, *ln2_g = nullptr, *ln2_b = nullptr;
  // LayerNorm folded into the Linear that follows it (rowops.cu fold_layernorm): fp32 sources kept for re-folding,
  // folded bf16 weight (+ transposed), folded bias, column sums, interleaved (colsum, bias')
  float *w_in_f32 = nullptr, *w_fc_f32 = nullptr;
  bf16 *w_in_ln = nullptr, *w_in_t_ln = nullptr, *w_fc_ln = nullptr, *w_fc_t_ln = nullptr;
  float *b_in_ln = nullptr, *b_fc_ln = nullptr, *cs_in = nullptr, *cs_fc = nullptr;
  float2 *sb_in = nullptr, *sb_fc = nullptr;
  int have = 0;  // bit per tensor
};

// Device memory of one kind (tower input, training workspace, inference workspace): allocated together and released
// together when the tower outgrows it.
struct AllocGroup {
  std::vector<void*> ptrs;
  size_t bytes = 0;  // requested bytes (mudpt_workspace_bytes; each cudaMalloc adds 256 B of slack)
};

// The buffers one forward walk of a tower writes (tower_forward).  The training view gives every layer its own
// activations, which the backward reads; the inference view (Tower::inf) aliases the same few buffers in every layer.
struct FwdView {
  int S = 0, rows = 0;  // sequences and token rows of the walk (the row layout is the tower's)
  double attn_sq = 0;   // sum over sequences of length^2
  std::vector<float*> x_in, x_mid;  // [layers + 1], [layers]
  std::vector<bf16*> xb_in, xb_mid;  // fused LayerNorm: bf16 copies of x_in / x_mid ...
  std::vector<float2*> st_in, st_mid;  // ... and their per-64-column partial statistics
  std::vector<bf16*> qkv, o, h;  // h empty: c_fc writes QuickGELU(h) only (EPI_GELU_ONLY / EPI_LN_GELU_ONLY)
  std::vector<float*> lse;
  bf16 *a_buf = nullptr, *g_buf = nullptr;
  // pruned last block: S gathered rows
  float *pr_x = nullptr, *pr_xm = nullptr, *pr_xo = nullptr;
  bf16 *pr_o = nullptr, *pr_xmb = nullptr, *pr_h = nullptr, *pr_g = nullptr, *pr_a = nullptr;
  float2* pr_stm = nullptr;
  float* head_ws = nullptr;
  GemmWorkspace* gws = nullptr;
  bool fused = false, pruned = false;  // set by the walk: the formulation it ran
};

struct Tower {
  int d = 0, H = 0, layers = 0, n_ctx = 0, row0 = 0, depth = 0;
  bool causal = false;
  int L = 0;        // current tokens per sequence (ragged: the longest sequence)
  int S = 0;        // current sequences
  int rows = 0;     // token rows: S * L, or (ragged) the sum of the sequence lengths
  double attn_sq = 0;  // sum over sequences of length^2 (attention FLOP counts)
  size_t stem_per_seq = 0;  // vision: bf16 elements of one image's extracted patches (np * Kp); text: 0
  // Ragged text tower (mudpt_text_set_classes_ragged): sequence s occupies the packed rows [seq_off[s], seq_off[s + 1]),
  // tok_pos[row] = the row's position in its sequence; sel_rows / p0_rows hold absolute rows (row stride row_L() = 0).
  // The LayerNorms run stand-alone (the fused GEMM epilogues locate prompt rows with row % L).
  bool ragged = false;
  int *seq_off = nullptr, *tok_pos = nullptr;
  int* eot = nullptr;  // text: absolute EOT row of every class
  int row_L() const { return ragged ? 0 : L; }
  const int* packed_pos() const { return ragged ? tok_pos : nullptr; }  // (the arrays outlive a switch back to padded)
  const int* packed_off() const { return ragged ? seq_off : nullptr; }
  // tower input (x_in[0], xb_in[0], st_in[0], p0_rows; text: seq_off, tok_pos, eot): mudpt_text_set_classes* or the
  // vision stem writes it, the training walk reads it (and splices its layer-0 prompt rows into it), so does the backward
  AllocGroup in_mem;
  size_t in_rows = 0, in_S = 0;
  // training workspace (everything else above and below): allocated at the first mudpt_*_forward
  AllocGroup train_mem;
  size_t cap_rows = 0, cap_S = 0;
  std::vector<Layer> lw;
  bool fold_dirty = true;  // a tensor that enters the LayerNorm folding changed since the last fold
  // saved activations, per layer
  std::vector<float*> x_in, x_mid;
  std::vector<bf16*> qkv, o, h;
  std::vector<float*> lse;
  // fused LayerNorm: bf16 copies of the LN inputs (GEMM A operands) + their per-64-column partial statistics
  std::vector<bf16*> xb_in, xb_mid;
  std::vector<float2*> st_in, st_mid;
  float2* dots = nullptr;  // row dots for the fused LayerNorm backward [rows, dot_cap]
  int dot_cap = 0;
  // transients
  bf16 *a_buf = nullptr, *g_buf = nullptr, *dh_buf = nullptr, *do_buf = nullptr, *dqkv_buf = nullptr, *dx_bf16 = nullptr;
  float *dx = nullptr, *dsum = nullptr, *splice_ws = nullptr, *head_ws = nullptr;  // head_ws: feature_head_workspace_floats(S, d, e)
  bf16* patches = nullptr;  // vision stem: [S, np, Kp]
  // exact work skipping (SURVEY.md H5): after the last block's attention only one row per sequence is consumed
  // (CLS, clip/model.py:548; EOT, trainers/mudpt.py:154), so its out-proj / MLP run on S gathered rows
  const int* sel_rows = nullptr;  // consumed row per sequence (null: row 0)
  bf16 *pr_o = nullptr, *pr_xmb = nullptr, *pr_h = nullptr, *pr_g = nullptr, *pr_a = nullptr, *pr_dxb = nullptr, *pr_dh = nullptr,
       *pr_do = nullptr;
  float *pr_x = nullptr, *pr_xm = nullptr, *pr_xo = nullptr, *pr_dx = nullptr;
  float2 *pr_stm = nullptr, *pr_dots = nullptr;
  bool fwd_pruned = false;
  // ... and below block 0 only the spliced prompt rows carry a gradient anyone reads (everything else of the tower input
  // is frozen: patch / token embeddings, cls, positional embeddings), so block 0's d in-proj and LN1 backward run on
  // the S * n_ctx gathered prompt rows
  int* p0_rows = nullptr;  // absolute row of prompt token j of sequence s: s * L + row0 + j
  int p0_S = 0, p0_L = 0;  // shape p0_rows was built for
  bf16 *p0_dqkv = nullptr, *p0_a = nullptr, *p0_dxb = nullptr;
  float *p0_x = nullptr, *p0_dx = nullptr;
  GemmWorkspace gws;             // stream-K scratch of this tower's stream
  // image gradients (mudpt_vision_backward_images): what the stem backward cannot keep in the backward transients that are
  // free after block 0 -- allocated at the first such call, reported with the training workspace (DESIGN.md section 3)
  AllocGroup img_mem;
  size_t img_S = 0;
  float* img_dpatch = nullptr;   // [S * np, Kp] fp32 patch gradient, where it does not fit in g_buf
  float* img_dprompt = nullptr;  // [depth, n_ctx, d]: the splice backward's sink when no prompt gradient is asked for
  bool fwd_done = false;
  bool fwd_fused = false;  // the saved activations belong to the fused-LayerNorm formulation
  int first_splice = 0;  // 0: layer 0 splices prompts[0]; 1: layer-0 rows kept as given
  // forward-only walk (mudpt_*_infer): a workspace of its own, so that it touches nothing the backward reads
  struct Infer {
    AllocGroup mem;
    size_t rows = 0, S = 0;
    bool fused = false;  // holds the bf16 copies + statistics of the fused LayerNorm
    FwdView v;
    GemmWorkspace gws;
    bf16* patches = nullptr;
  } inf;
};

}  // namespace

// Optional per-kernel-class timing with CUDA events on the launch stream (bench.py's roofline leg).
enum ProfCat { PC_GEMM = 0, PC_ATTN_FWD, PC_ATTN_BWD, PC_LN_FWD, PC_LN_BWD, PC_SPLICE, PC_HEAD, PC_STEM,
               // the eight GEMMs of a block, forward and dgrad (PC_GEMM: everything else -- patch embedding, pruned tail)
               PC_GEMM_QKV, PC_GEMM_OUT, PC_GEMM_FC, PC_GEMM_PROJ, PC_GEMM_DPROJ, PC_GEMM_DFC, PC_GEMM_DOUT, PC_GEMM_DQKV, PC_COUNT };
struct ProfRec { int cat; cudaEvent_t e0, e1; double flops, bytes; };
struct Prof {
  bool on = false;
  std::vector<ProfRec> recs;
  std::vector<cudaEvent_t> pool;
  cudaEvent_t get() {
    if (!pool.empty()) { cudaEvent_t e = pool.back(); pool.pop_back(); return e; }
    cudaEvent_t e; cudaEventCreate(&e); return e;
  }
};

struct mudpt_handle {
  mudpt_config cfg;
  std::string err;
  Prof prof;
  Tower vis, txt;
  // vision stem / heads
  bf16* w_conv = nullptr;  // [dv, Kp] bf16 (Kp = 3*p*p padded to a multiple of 8)
  bf16* w_conv_t = nullptr;  // [Kp, dv] transposed copy: B operand of the patch dgrad (padding rows zero)
  int Kp = 0;
  float *cls = nullptr, *pos_v = nullptr, *ln_pre_g = nullptr, *ln_pre_b = nullptr, *ln_post_g = nullptr,
        *ln_post_b = nullptr, *proj_v = nullptr;
  float *pos_t = nullptr, *ln_final_g = nullptr, *ln_final_b = nullptr, *proj_t = nullptr;
  float logit_scale_exp = 0.f;
  int stem_have = 0;
  float* head_ws = nullptr;
  size_t head_ws_cap = 0;
  std::vector<void*> allocs;
  long long launches_at_create = 0;
  // options (mudpt_set_option): LayerNorm folded into the GEMMs (default) or the stand-alone LN kernels -- the
  // fallback for checkpoints whose residual stream has a row mean far above its spread (bf16(x) instead of
  // bf16(LN(x)) as the GEMM operand would lose the signal there)
  int ln_fused = -1;  // -1 = by tower size (see ln_fused_for), 0 = never, 1 = always
  // LayerNorm dgrad in the dgrad GEMMs' epilogues (EPI_LN_BWD) instead of the stand-alone kernel.  Off by default:
  // measured on B200 the row dots it needs cost more at their producers (GELU' epilogue +66 us, attention backward
  // +82 us per block at the cfg-2 shapes) than the fused epilogue saves (60 us): profiles/r02_ln_fusion_ab.txt
  bool ln_bwd_fused = false;
  bool ln_bwd_bf16x = true;  // env MUDPT_LN_BWD_BF16X
  // exact work skipping (SURVEY.md H5): the last block's out-proj / MLP on the CLS / EOT rows only
  bool prune = true;
  // Gradient of the residual stream kept in bf16 between the LayerNorm backward kernels (the dgrad GEMMs read that copy
  // as their A operand anyway); fp32 rows are written for the deep-prompt window only, which is all the splice backward
  // reads.  8 instead of 14 B per element on the HBM-bound LayerNorm backward; each of the 2 x layers updates rounds the
  // stream to bf16 (2^-9 relative): measured effect on the prompt gradients in profiles/r02_grad_stream_bf16.txt.
  // Not used when the dense input gradient is requested (CoCoOp's d_x0) or with ln_bwd_fused.  env MUDPT_GRAD_BF16
  bool grad_bf16 = true;
};

namespace {

int fail(mudpt_handle* h, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  if (h) h->err = buf;
  g_err = buf;
  return -1;
}

#define CK(h, expr)                                   \
  do {                                                \
    const char* _e = (expr);                          \
    if (_e) return fail((h), "%s (%s:%d)", _e, __FILE__, __LINE__); \
  } while (0)

#define CUDA_OK(h, expr)                                                                    \
  do {                                                                                      \
    cudaError_t _c = (expr);                                                                \
    if (_c != cudaSuccess) return fail((h), "%s: %s (%s:%d)", #expr, cudaGetErrorString(_c), __FILE__, __LINE__); \
  } while (0)

// CK with optional event bracketing: category, algorithmic FLOPs and bytes of the launch
#define CKP(h, st, cat, fl, by, expr)                                         \
  do {                                                                        \
    cudaEvent_t _e0 = nullptr, _e1 = nullptr;                                 \
    if ((h)->prof.on) { _e0 = (h)->prof.get(); _e1 = (h)->prof.get(); cudaEventRecord(_e0, (st)); } \
    const char* _e = (expr);                                                  \
    if (_e) return fail((h), "%s (%s:%d)", _e, __FILE__, __LINE__);           \
    if ((h)->prof.on) { cudaEventRecord(_e1, (st)); (h)->prof.recs.push_back(ProfRec{(cat), _e0, _e1, (double)(fl), (double)(by)}); } \
  } while (0)

template <typename T>
cudaError_t dev_alloc(mudpt_handle* h, T** p, size_t n, AllocGroup* group = nullptr) {
  void* q = nullptr;
  cudaError_t c = cudaMalloc(&q, n * sizeof(T) + 256);
  if (c != cudaSuccess) return c;
  if (group) {
    group->ptrs.push_back(q);
    group->bytes += n * sizeof(T);
  } else {
    h->allocs.push_back(q);
  }
  *p = reinterpret_cast<T*>(q);
  return cudaSuccess;
}

// (cudaFree waits for the device, so nothing in flight still uses the released buffers)
void release(AllocGroup& g) {
  for (void* p : g.ptrs) cudaFree(p);
  g.ptrs.clear();
  g.bytes = 0;
  gemm_clear_tensor_map_cache();
}

bool env_flag(const char* name, bool dflt) {
  const char* e = getenv(name);
  return e ? atoi(e) != 0 : dflt;
}

// Measured on B200 (profiles/r02_ln_fusion_ab.txt): folding the LayerNorm into the GEMMs saves its 4 B/element read
// but makes the four forward epilogues heavier (+2 B/element bf16 copy, statistics, rank-1 correction).  For the
// large HBM-bound tower (text, 77,000 rows) that is a gain; for ~6,000-row towers, whose 25-40 us GEMMs are
// launch / epilogue bound, the stand-alone LayerNorm kernels are faster: choose by row count unless told otherwise.
// (ragged towers: always the stand-alone kernels, which take the packed positions)
bool ln_fused_for(const mudpt_handle* h, const Tower& t, int rows) {
  return !t.ragged && (h->ln_fused == 1 || (h->ln_fused < 0 && rows >= 32768));
}

// Shape of the tower for S sequences of L tokens, or (off != null: host row offsets [S+1]) for S packed sequences of at
// most L tokens, and the memory of its input.  The workspaces follow at the first walk that needs them.  Each kind of
// memory grows to the largest shape seen; the outgrown buffers are released first (a CoCoOp-style caller whose B x C
// changes would otherwise pile up GBs until mudpt_destroy).
int ensure_input(mudpt_handle* h, Tower& t, int S, int L, const int* off = nullptr) {
  const size_t rows = off ? static_cast<size_t>(off[S]) : static_cast<size_t>(S) * L;
  t.S = S;
  t.L = L;
  t.rows = static_cast<int>(rows);
  t.ragged = off != nullptr;
  t.attn_sq = static_cast<double>(S) * L * L;
  if (off) {
    t.attn_sq = 0;
    for (int q = 0; q < S; ++q) t.attn_sq += static_cast<double>(off[q + 1] - off[q]) * (off[q + 1] - off[q]);
  }
  if (rows > t.in_rows || static_cast<size_t>(S) > t.in_S) {
    release(t.in_mem);
    t.in_rows = rows > t.in_rows ? rows : t.in_rows;
    t.in_S = static_cast<size_t>(S) > t.in_S ? S : t.in_S;
    const size_t R = t.in_rows, Sn = t.in_S, d = t.d;
    AllocGroup* g = &t.in_mem;
    CUDA_OK(h, dev_alloc(h, &t.x_in[0], R * d, g));
    CUDA_OK(h, dev_alloc(h, &t.xb_in[0], R * d, g));
    CUDA_OK(h, dev_alloc(h, &t.st_in[0], R * (d / 64), g));
    if (t.n_ctx > 0) CUDA_OK(h, dev_alloc(h, &t.p0_rows, Sn * t.n_ctx, g));
    if (t.causal) {  // text
      CUDA_OK(h, dev_alloc(h, &t.seq_off, Sn + 1, g));
      CUDA_OK(h, dev_alloc(h, &t.tok_pos, R, g));
      CUDA_OK(h, dev_alloc(h, &t.eot, Sn, g));
    }
    t.p0_S = 0;
    t.fwd_done = false;
  }
  const size_t R0 = static_cast<size_t>(S) * t.n_ctx;
  if (R0 > 0 && (off || t.p0_S != S || t.p0_L != L)) {
    std::vector<int> r(R0);
    for (int q = 0; q < S; ++q)
      for (int j = 0; j < t.n_ctx; ++j) r[static_cast<size_t>(q) * t.n_ctx + j] = (off ? off[q] : q * L) + t.row0 + j;
    CUDA_OK(h, cudaMemcpy(t.p0_rows, r.data(), R0 * sizeof(int), cudaMemcpyHostToDevice));  // (set-up: shapes change rarely)
    t.p0_S = S;
    t.p0_L = off ? -1 : L;  // (packed rows: rebuilt on the next set-up)
  }
  return 0;
}

// Training workspace for the tower's current shape: the saved activations of every layer (x_in[1..]), the forward and
// backward transients, the pruned blocks' rows, the feature head's, stream-K and splice scratch, the vision stem's patches
int ensure_train(mudpt_handle* h, Tower& t, cudaStream_t st) {
  if (static_cast<size_t>(t.rows) <= t.cap_rows && static_cast<size_t>(t.S) <= t.cap_S) return 0;
  release(t.train_mem);
  t.cap_rows = static_cast<size_t>(t.rows) > t.cap_rows ? t.rows : t.cap_rows;
  t.cap_S = static_cast<size_t>(t.S) > t.cap_S ? t.S : t.cap_S;
  const size_t rows = t.cap_rows, Ss = t.cap_S, d = t.d, parts = d / 64, R0 = Ss * t.n_ctx;
  AllocGroup* g = &t.train_mem;
  for (int i = 1; i <= t.layers; ++i) {
    CUDA_OK(h, dev_alloc(h, &t.x_in[i], rows * d, g));
    CUDA_OK(h, dev_alloc(h, &t.xb_in[i], rows * d, g));
    CUDA_OK(h, dev_alloc(h, &t.st_in[i], rows * parts, g));
  }
  for (int i = 0; i < t.layers; ++i) {
    CUDA_OK(h, dev_alloc(h, &t.x_mid[i], rows * d, g));
    CUDA_OK(h, dev_alloc(h, &t.xb_mid[i], rows * d, g));
    CUDA_OK(h, dev_alloc(h, &t.st_mid[i], rows * parts, g));
    CUDA_OK(h, dev_alloc(h, &t.qkv[i], rows * 3 * d, g));
    CUDA_OK(h, dev_alloc(h, &t.o[i], rows * d, g));
    CUDA_OK(h, dev_alloc(h, &t.h[i], rows * 4 * d, g));
    CUDA_OK(h, dev_alloc(h, &t.lse[i], rows * t.H, g));
  }
  const int dots_mlp = (4 * t.d + gemm_dots_span(4 * t.d) - 1) / gemm_dots_span(4 * t.d);
  t.dot_cap = dots_mlp > 3 * t.H ? dots_mlp : 3 * t.H;
  CUDA_OK(h, dev_alloc(h, &t.dots, rows * t.dot_cap, g));
  CUDA_OK(h, dev_alloc(h, &t.a_buf, rows * d, g));
  CUDA_OK(h, dev_alloc(h, &t.g_buf, rows * 4 * d, g));
  CUDA_OK(h, dev_alloc(h, &t.dh_buf, rows * 4 * d, g));
  CUDA_OK(h, dev_alloc(h, &t.do_buf, rows * d, g));
  CUDA_OK(h, dev_alloc(h, &t.dqkv_buf, rows * 3 * d, g));
  CUDA_OK(h, dev_alloc(h, &t.dx_bf16, rows * d, g));
  CUDA_OK(h, dev_alloc(h, &t.dx, rows * d, g));
  CUDA_OK(h, dev_alloc(h, &t.dsum, rows * t.H, g));
  CUDA_OK(h, dev_alloc(h, &t.pr_o, Ss * d, g));
  CUDA_OK(h, dev_alloc(h, &t.pr_xmb, Ss * d, g));
  CUDA_OK(h, dev_alloc(h, &t.pr_h, Ss * 4 * d, g));
  CUDA_OK(h, dev_alloc(h, &t.pr_g, Ss * 4 * d, g));
  CUDA_OK(h, dev_alloc(h, &t.pr_a, Ss * d, g));
  CUDA_OK(h, dev_alloc(h, &t.pr_dxb, Ss * d, g));
  CUDA_OK(h, dev_alloc(h, &t.pr_dh, Ss * 4 * d, g));
  CUDA_OK(h, dev_alloc(h, &t.pr_do, Ss * d, g));
  CUDA_OK(h, dev_alloc(h, &t.pr_x, Ss * d, g));
  CUDA_OK(h, dev_alloc(h, &t.pr_xm, Ss * d, g));
  CUDA_OK(h, dev_alloc(h, &t.pr_xo, Ss * d, g));
  CUDA_OK(h, dev_alloc(h, &t.pr_dx, Ss * d, g));
  CUDA_OK(h, dev_alloc(h, &t.pr_stm, Ss * parts, g));
  CUDA_OK(h, dev_alloc(h, &t.pr_dots, Ss * dots_mlp, g));
  if (R0 > 0) {
    CUDA_OK(h, dev_alloc(h, &t.p0_dqkv, R0 * 3 * d, g));
    CUDA_OK(h, dev_alloc(h, &t.p0_a, R0 * d, g));
    CUDA_OK(h, dev_alloc(h, &t.p0_dxb, R0 * d, g));
    CUDA_OK(h, dev_alloc(h, &t.p0_x, R0 * d, g));
    CUDA_OK(h, dev_alloc(h, &t.p0_dx, R0 * d, g));
  }
  // gathered CLS / EOT rows of the feature head + split-K partials
  CUDA_OK(h, dev_alloc(h, &t.head_ws, feature_head_workspace_floats(static_cast<int>(Ss), t.d, h->cfg.embed_dim), g));
  CUDA_OK(h, dev_alloc(h, &t.gws.partials, gemm_workspace_partial_bytes() / sizeof(float), g));
  CUDA_OK(h, dev_alloc(h, &t.gws.flags, gemm_workspace_flag_bytes() / sizeof(unsigned), g));
  CUDA_OK(h, cudaMemset(t.gws.flags, 0, gemm_workspace_flag_bytes()));
  const size_t nws = splice_bwd_workspace_floats(t.n_ctx > 0 ? t.n_ctx : 1, t.d);
  CUDA_OK(h, dev_alloc(h, &t.splice_ws, nws, g));
  CUDA_OK(h, cudaMemset(t.splice_ws, 0, nws * sizeof(float)));  // (the kernel's tickets start at zero and are left at zero)
  if (t.stem_per_seq) {
    CUDA_OK(h, dev_alloc(h, &t.patches, Ss * t.stem_per_seq, g));
    CUDA_OK(h, cudaMemsetAsync(t.patches, 0, Ss * t.stem_per_seq * sizeof(bf16), st));  // (the K padding stays zero)
  }
  t.fwd_done = false;
  return 0;
}

// Inference workspace for a walk over S sequences / `rows` token rows (DESIGN.md section 3): two fp32 residual buffers the
// layers use alternately (x_in, x_mid) with their bf16 copies and statistics when the LayerNorm is fused, one a_buf / qkv /
// o / g / lse shared by every layer, the pruned block's rows, the feature head's and stream-K scratch, the stem's patches.
// Nothing in it is read by a backward.
int ensure_infer(mudpt_handle* h, Tower& t, int S, int rows, bool fused, cudaStream_t st) {
  Tower::Infer& f = t.inf;
  if (!f.mem.ptrs.empty() && static_cast<size_t>(rows) <= f.rows && static_cast<size_t>(S) <= f.S && (f.fused || !fused)) return 0;
  release(f.mem);
  f.rows = static_cast<size_t>(rows) > f.rows ? rows : f.rows;
  f.S = static_cast<size_t>(S) > f.S ? S : f.S;
  f.fused = f.fused || fused;
  const size_t R = f.rows, Ss = f.S, d = t.d, parts = d / 64;
  AllocGroup* g = &f.mem;
  FwdView& v = f.v;
  float* x[2];
  bf16* xb[2] = {nullptr, nullptr};
  float2* xs[2] = {nullptr, nullptr};
  for (int k = 0; k < 2; ++k) {
    CUDA_OK(h, dev_alloc(h, &x[k], R * d, g));
    if (f.fused) {
      CUDA_OK(h, dev_alloc(h, &xb[k], R * d, g));
      CUDA_OK(h, dev_alloc(h, &xs[k], R * parts, g));
    }
  }
  bf16 *qkv, *o;
  float* lse;
  CUDA_OK(h, dev_alloc(h, &v.a_buf, R * d, g));
  CUDA_OK(h, dev_alloc(h, &qkv, R * 3 * d, g));
  CUDA_OK(h, dev_alloc(h, &o, R * d, g));
  CUDA_OK(h, dev_alloc(h, &v.g_buf, R * 4 * d, g));
  CUDA_OK(h, dev_alloc(h, &lse, R * t.H, g));
  v.x_in.assign(t.layers + 1, x[0]);
  v.x_mid.assign(t.layers, x[1]);
  v.xb_in.assign(t.layers + 1, xb[0]);
  v.xb_mid.assign(t.layers, xb[1]);
  v.st_in.assign(t.layers + 1, xs[0]);
  v.st_mid.assign(t.layers, xs[1]);
  v.qkv.assign(t.layers, qkv);
  v.o.assign(t.layers, o);
  v.h.clear();
  v.lse.assign(t.layers, lse);
  CUDA_OK(h, dev_alloc(h, &v.pr_x, Ss * d, g));
  CUDA_OK(h, dev_alloc(h, &v.pr_o, Ss * d, g));
  CUDA_OK(h, dev_alloc(h, &v.pr_xm, Ss * d, g));
  CUDA_OK(h, dev_alloc(h, &v.pr_xmb, Ss * d, g));
  CUDA_OK(h, dev_alloc(h, &v.pr_stm, Ss * parts, g));
  CUDA_OK(h, dev_alloc(h, &v.pr_g, Ss * 4 * d, g));
  CUDA_OK(h, dev_alloc(h, &v.pr_a, Ss * d, g));
  CUDA_OK(h, dev_alloc(h, &v.pr_xo, Ss * d, g));
  v.pr_h = nullptr;
  CUDA_OK(h, dev_alloc(h, &v.head_ws, feature_head_workspace_floats(static_cast<int>(Ss), t.d, h->cfg.embed_dim), g));
  CUDA_OK(h, dev_alloc(h, &f.gws.partials, gemm_workspace_partial_bytes() / sizeof(float), g));
  CUDA_OK(h, dev_alloc(h, &f.gws.flags, gemm_workspace_flag_bytes() / sizeof(unsigned), g));
  CUDA_OK(h, cudaMemset(f.gws.flags, 0, gemm_workspace_flag_bytes()));
  v.gws = &f.gws;
  if (t.stem_per_seq) {
    CUDA_OK(h, dev_alloc(h, &f.patches, Ss * t.stem_per_seq, g));
    CUDA_OK(h, cudaMemsetAsync(f.patches, 0, Ss * t.stem_per_seq * sizeof(bf16), st));
  }
  return 0;
}

// the training walk's view of the tower: every layer its own buffers
FwdView train_view(Tower& t) {
  FwdView v;
  v.S = t.S; v.rows = t.rows; v.attn_sq = t.attn_sq;
  v.x_in = t.x_in; v.x_mid = t.x_mid; v.xb_in = t.xb_in; v.xb_mid = t.xb_mid; v.st_in = t.st_in; v.st_mid = t.st_mid;
  v.qkv = t.qkv; v.o = t.o; v.h = t.h; v.lse = t.lse;
  v.a_buf = t.a_buf; v.g_buf = t.g_buf;
  v.pr_x = t.pr_x; v.pr_xm = t.pr_xm; v.pr_xo = t.pr_xo; v.pr_o = t.pr_o; v.pr_xmb = t.pr_xmb; v.pr_h = t.pr_h; v.pr_g = t.pr_g;
  v.pr_a = t.pr_a; v.pr_stm = t.pr_stm;
  v.head_ws = t.head_ws; v.gws = &t.gws;
  return v;
}

// ---------------------------------------------------------------------------- weights
int store_f32(mudpt_handle* h, float** dst, const float* src, int64_t numel, int64_t expect, const char* name,
              cudaStream_t st) {
  if (numel != expect) return fail(h, "weight %s: expected %lld elements, got %lld", name, (long long)expect, (long long)numel);
  if (!*dst) CUDA_OK(h, dev_alloc(h, dst, static_cast<size_t>(numel)));
  CUDA_OK(h, cudaMemcpyAsync(*dst, src, numel * sizeof(float), cudaMemcpyDeviceToDevice, st));
  return 0;
}
// [rows(out), cols(in)] fp32 -> bf16 as stored + bf16 transposed
int store_gemm_weight(mudpt_handle* h, bf16** w, bf16** wt, const float* src, int64_t numel, int rows, int cols,
                      const char* name, cudaStream_t st) {
  if (numel != static_cast<int64_t>(rows) * cols)
    return fail(h, "weight %s: expected %d x %d elements, got %lld", name, rows, cols, (long long)numel);
  if (!*w) CUDA_OK(h, dev_alloc(h, w, static_cast<size_t>(numel)));
  CK(h, cast_to_bf16(src, *w, static_cast<size_t>(numel), st));
  if (wt) {
    if (!*wt) CUDA_OK(h, dev_alloc(h, wt, static_cast<size_t>(numel)));
    CK(h, transpose_cast_bf16(src, *wt, rows, cols, st));
  }
  return 0;
}

enum LayerBits {
  LB_W_IN = 1 << 0, LB_B_IN = 1 << 1, LB_W_OUT = 1 << 2, LB_B_OUT = 1 << 3, LB_W_FC = 1 << 4, LB_B_FC = 1 << 5,
  LB_W_PR = 1 << 6, LB_B_PR = 1 << 7, LB_LN1_G = 1 << 8, LB_LN1_B = 1 << 9, LB_LN2_G = 1 << 10, LB_LN2_B = 1 << 11,
  LB_ALL = (1 << 12) - 1
};
enum StemBits {
  SB_CONV = 1 << 0, SB_CLS = 1 << 1, SB_POS_V = 1 << 2, SB_LNPRE_G = 1 << 3, SB_LNPRE_B = 1 << 4, SB_LNPOST_G = 1 << 5,
  SB_LNPOST_B = 1 << 6, SB_PROJ_V = 1 << 7, SB_POS_T = 1 << 8, SB_LNF_G = 1 << 9, SB_LNF_B = 1 << 10, SB_PROJ_T = 1 << 11,
  SB_SCALE = 1 << 12, SB_ALL = (1 << 13) - 1
};

int set_block_weight(mudpt_handle* h, Tower& t, int layer, const char* sub, const float* data, int64_t numel,
                     const char* full, cudaStream_t st) {
  if (layer < 0 || layer >= t.layers) return fail(h, "weight %s: layer out of range", full);
  Layer& l = t.lw[layer];
  const int d = t.d;
  int rc = 0;
  if (!strcmp(sub, "attn.in_proj_weight")) {
    rc = store_gemm_weight(h, &l.w_in, &l.w_in_t, data, numel, 3 * d, d, full, st);
    if (!rc) rc = store_f32(h, &l.w_in_f32, data, numel, static_cast<int64_t>(3) * d * d, full, st);
    l.have |= LB_W_IN;
  }
  else if (!strcmp(sub, "attn.in_proj_bias")) { rc = store_f32(h, &l.b_in, data, numel, 3 * d, full, st); l.have |= LB_B_IN; }
  else if (!strcmp(sub, "attn.out_proj.weight")) { rc = store_gemm_weight(h, &l.w_out, &l.w_out_t, data, numel, d, d, full, st); l.have |= LB_W_OUT; }
  else if (!strcmp(sub, "attn.out_proj.bias")) { rc = store_f32(h, &l.b_out, data, numel, d, full, st); l.have |= LB_B_OUT; }
  else if (!strcmp(sub, "mlp.c_fc.weight")) {
    rc = store_gemm_weight(h, &l.w_fc, &l.w_fc_t, data, numel, 4 * d, d, full, st);
    if (!rc) rc = store_f32(h, &l.w_fc_f32, data, numel, static_cast<int64_t>(4) * d * d, full, st);
    l.have |= LB_W_FC;
  }
  else if (!strcmp(sub, "mlp.c_fc.bias")) { rc = store_f32(h, &l.b_fc, data, numel, 4 * d, full, st); l.have |= LB_B_FC; }
  else if (!strcmp(sub, "mlp.c_proj.weight")) { rc = store_gemm_weight(h, &l.w_pr, &l.w_pr_t, data, numel, d, 4 * d, full, st); l.have |= LB_W_PR; }
  else if (!strcmp(sub, "mlp.c_proj.bias")) { rc = store_f32(h, &l.b_pr, data, numel, d, full, st); l.have |= LB_B_PR; }
  else if (!strcmp(sub, "ln_1.weight")) { rc = store_f32(h, &l.ln1_g, data, numel, d, full, st); l.have |= LB_LN1_G; }
  else if (!strcmp(sub, "ln_1.bias")) { rc = store_f32(h, &l.ln1_b, data, numel, d, full, st); l.have |= LB_LN1_B; }
  else if (!strcmp(sub, "ln_2.weight")) { rc = store_f32(h, &l.ln2_g, data, numel, d, full, st); l.have |= LB_LN2_G; }
  else if (!strcmp(sub, "ln_2.bias")) { rc = store_f32(h, &l.ln2_b, data, numel, d, full, st); l.have |= LB_LN2_B; }
  else return 1;
  t.fold_dirty = true;
  return rc;
}

// LayerNorm -> Linear folding of every block (once per weight load)
int ensure_folded(mudpt_handle* h, Tower& t, cudaStream_t st) {
  if (!t.fold_dirty) return 0;
  const int d = t.d;
  for (Layer& l : t.lw) {
    if (!l.w_in_ln) {
      CUDA_OK(h, dev_alloc(h, &l.w_in_ln, static_cast<size_t>(3) * d * d));
      CUDA_OK(h, dev_alloc(h, &l.w_in_t_ln, static_cast<size_t>(3) * d * d));
      CUDA_OK(h, dev_alloc(h, &l.w_fc_ln, static_cast<size_t>(4) * d * d));
      CUDA_OK(h, dev_alloc(h, &l.w_fc_t_ln, static_cast<size_t>(4) * d * d));
      CUDA_OK(h, dev_alloc(h, &l.b_in_ln, static_cast<size_t>(3) * d));
      CUDA_OK(h, dev_alloc(h, &l.b_fc_ln, static_cast<size_t>(4) * d));
      CUDA_OK(h, dev_alloc(h, &l.cs_in, static_cast<size_t>(3) * d));
      CUDA_OK(h, dev_alloc(h, &l.cs_fc, static_cast<size_t>(4) * d));
      CUDA_OK(h, dev_alloc(h, &l.sb_in, static_cast<size_t>(3) * d));
      CUDA_OK(h, dev_alloc(h, &l.sb_fc, static_cast<size_t>(4) * d));
    }
    CK(h, fold_layernorm(l.w_in_f32, l.ln1_g, l.ln1_b, l.b_in, l.w_in_ln, l.w_in_t_ln, l.b_in_ln, l.cs_in, l.sb_in, 3 * d, d, st));
    CK(h, fold_layernorm(l.w_fc_f32, l.ln2_g, l.ln2_b, l.b_fc, l.w_fc_ln, l.w_fc_t_ln, l.b_fc_ln, l.cs_fc, l.sb_fc, 4 * d, d, st));
  }
  t.fold_dirty = false;
  return 0;
}

// ---------------------------------------------------------------------------- tower passes
// Per block (clip/model.py:275-301): [splice] ; x += attn(ln_1(x)) ; x += c_proj(QuickGELU(c_fc(ln_2(x)))).
//
// Fused formulation (default): no LayerNorm kernel and no splice kernel inside the layer loop.  The residual GEMMs
// (out-proj, c_proj) write the new residual row as fp32 + bf16 + partial statistics (and the NEXT block's spliced
// prompt rows in place of the computed ones); the QKV / c_fc GEMMs read the bf16 row as their A operand and apply
// the normalisation in their epilogue (EPI_LN_*: gamma folded into the weight, mean as a rank-1 correction).
// Precondition of the fused path: v.x_in[0], v.xb_in[0], v.st_in[0] hold the tower input (layer-0 splice excepted).
// The walk writes the buffers of `v` only (and, with a layer-0 splice, the prompt rows of v.x_in[0]); with v.h empty the
// c_fc GEMMs write QuickGELU(h) alone (no backward will need h): the same values as the training walk, bit for bit.
int tower_forward(mudpt_handle* h, Tower& t, FwdView& v, const float* prompts, int first_splice_layer, cudaStream_t st) {
  const int M = v.rows, d = t.d;
  const double Md = static_cast<double>(M), dd = d;
  const double attn_fl = 4.0 * t.H * v.attn_sq * 64.0;  // QK^T + PV, dense count
  const bool fused = ln_fused_for(h, t, M);
  const bool pruned = h->prune;
  const bool keep_h = !v.h.empty();
  const double fc_out = keep_h ? 2.0 : 1.0;  // bf16 outputs of c_fc
  const int parts = d / 64;
  auto spliced = [&](int i) { return i < t.depth && i >= first_splice_layer && t.n_ctx > 0 && i < t.layers; };
  if (fused && ensure_folded(h, t, st)) return -1;
  for (int i = 0; i < t.layers; ++i) {
    const Layer& w = t.lw[i];
    // the stand-alone LayerNorm does the block's splice in the same pass; the fused form splices in the previous block's
    // residual epilogue (layer 0: a kernel of its own, with the statistics of the spliced rows)
    if (spliced(i) && fused && i == 0) {
      const float* pr = prompts + static_cast<size_t>(i) * t.n_ctx * d;
      CKP(h, st, PC_SPLICE, 0, 2.0 * v.S * t.n_ctx * dd * 4, splice_fwd_stats(v.x_in[i], v.xb_in[i], v.st_in[i], pr, v.S, t.L, t.row0, t.n_ctx, d, st));
    }
    // x + attn(ln_1(x))   (clip/model.py:299)
    GemmEpilogue e1;
    e1.out0 = v.qkv[i]; e1.ldc = 3 * d;
    if (fused) {
      e1.mode = EPI_LN_BF16; e1.bias = w.b_in_ln; e1.colsum = w.cs_in; e1.ln_stats = v.st_in[i]; e1.ln_parts = parts; e1.ln_width = d; e1.ln_eps = kLnEps;
      CKP(h, st, PC_GEMM_QKV, 2.0 * Md * 3 * dd * dd, 2 * (Md * dd + 3 * dd * dd + Md * 3 * dd),
          gemm_bf16_tn(v.xb_in[i], d, w.w_in_ln, d, e1, M, 3 * d, d, st, v.gws));
    } else {
      CKP(h, st, PC_LN_FWD, 0, Md * dd * 6,
          layernorm_fwd_splice(v.x_in[i], spliced(i) ? prompts + static_cast<size_t>(i) * t.n_ctx * d : nullptr, t.L, t.row0,
                               spliced(i) ? t.n_ctx : 0, w.ln1_g, w.ln1_b, v.a_buf, true, M, d, kLnEps, st, t.packed_pos()));
      e1.mode = EPI_BF16; e1.bias = w.b_in;
      CKP(h, st, PC_GEMM_QKV, 2.0 * Md * 3 * dd * dd, 2 * (Md * dd + 3 * dd * dd + Md * 3 * dd),
          gemm_bf16_tn(v.a_buf, d, w.w_in, d, e1, M, 3 * d, d, st, v.gws));
    }
    CKP(h, st, PC_ATTN_FWD, attn_fl, Md * dd * 2 * 4,
        t.ragged ? attention_varlen_fwd(v.qkv[i], v.o[i], v.lse[i], t.seq_off, v.S, t.L, t.H, d, st)
                 : attention_fwd(v.qkv[i], v.o[i], v.lse[i], v.S, t.L, t.H, d, t.causal, st));
    if (pruned && i == t.layers - 1) {
      // the block's output is consumed on one row per sequence: out-proj and the MLP on S gathered rows
      const int S = v.S;
      const double Sd = S;
      CKP(h, st, PC_SPLICE, 0, Sd * dd * 12, gather_rows(v.x_in[i], v.o[i], t.sel_rows, S, t.row_L(), v.pr_x, v.pr_o, d, st));
      GemmEpilogue p2;
      p2.out0 = v.pr_xm; p2.bias = w.b_out; p2.resid = v.pr_x; p2.ldc = d;
      if (fused) { p2.mode = EPI_RESID_STATS; p2.out2 = v.pr_xmb; p2.stats_out = v.pr_stm; }
      else p2.mode = EPI_RESID_F32;
      CKP(h, st, PC_GEMM, 2.0 * Sd * dd * dd, 2 * (Sd * dd + dd * dd) + 10 * Sd * dd, gemm_bf16_tn(v.pr_o, d, w.w_out, d, p2, S, d, d, st, v.gws));
      GemmEpilogue p3;
      p3.ldc = 4 * d;
      if (keep_h) { p3.out0 = v.pr_h; p3.out1 = v.pr_g; }
      else p3.out0 = v.pr_g;
      if (fused) {
        p3.mode = keep_h ? EPI_LN_GELU : EPI_LN_GELU_ONLY; p3.bias = w.b_fc_ln; p3.colsum = w.cs_fc; p3.ln_stats = v.pr_stm; p3.ln_parts = parts;
        p3.ln_width = d; p3.ln_eps = kLnEps;
        CKP(h, st, PC_GEMM, 2.0 * Sd * 4 * dd * dd, 2 * (Sd * dd + 4 * dd * dd + fc_out * Sd * 4 * dd), gemm_bf16_tn(v.pr_xmb, d, w.w_fc_ln, d, p3, S, 4 * d, d, st, v.gws));
      } else {
        CKP(h, st, PC_LN_FWD, 0, Sd * dd * 6, layernorm_fwd(v.pr_xm, w.ln2_g, w.ln2_b, v.pr_a, true, S, d, kLnEps, st));
        p3.mode = keep_h ? EPI_GELU : EPI_GELU_ONLY; p3.bias = w.b_fc;
        CKP(h, st, PC_GEMM, 2.0 * Sd * 4 * dd * dd, 2 * (Sd * dd + 4 * dd * dd + fc_out * Sd * 4 * dd), gemm_bf16_tn(v.pr_a, d, w.w_fc, d, p3, S, 4 * d, d, st, v.gws));
      }
      GemmEpilogue p4;
      p4.mode = EPI_RESID_F32; p4.out0 = v.pr_xo; p4.bias = w.b_pr; p4.resid = v.pr_xm; p4.ldc = d;
      CKP(h, st, PC_GEMM, 2.0 * Sd * 4 * dd * dd, 2 * (Sd * 4 * dd + 4 * dd * dd) + 8 * Sd * dd, gemm_bf16_tn(v.pr_g, 4 * d, w.w_pr, 4 * d, p4, S, d, 4 * d, st, v.gws));
      break;
    }
    GemmEpilogue e2;
    e2.out0 = v.x_mid[i]; e2.bias = w.b_out; e2.resid = v.x_in[i]; e2.ldc = d;
    if (fused) { e2.mode = EPI_RESID_STATS; e2.out2 = v.xb_mid[i]; e2.stats_out = v.st_mid[i]; }
    else e2.mode = EPI_RESID_F32;
    CKP(h, st, PC_GEMM_OUT, 2.0 * Md * dd * dd, 2 * (Md * dd + dd * dd) + (fused ? 10 : 8) * Md * dd,
        gemm_bf16_tn(v.o[i], d, w.w_out, d, e2, M, d, d, st, v.gws));
    // x + c_proj(QuickGELU(c_fc(ln_2(x))))   (clip/model.py:300)
    GemmEpilogue e3;
    e3.ldc = 4 * d;
    if (keep_h) { e3.out0 = v.h[i]; e3.out1 = v.g_buf; }
    else e3.out0 = v.g_buf;
    if (fused) {
      e3.mode = keep_h ? EPI_LN_GELU : EPI_LN_GELU_ONLY; e3.bias = w.b_fc_ln; e3.colsum = w.cs_fc; e3.ln_stats = v.st_mid[i]; e3.ln_parts = parts;
      e3.ln_width = d; e3.ln_eps = kLnEps;
      CKP(h, st, PC_GEMM_FC, 2.0 * Md * 4 * dd * dd, 2 * (Md * dd + 4 * dd * dd + fc_out * Md * 4 * dd),
          gemm_bf16_tn(v.xb_mid[i], d, w.w_fc_ln, d, e3, M, 4 * d, d, st, v.gws));
    } else {
      CKP(h, st, PC_LN_FWD, 0, Md * dd * 6, layernorm_fwd(v.x_mid[i], w.ln2_g, w.ln2_b, v.a_buf, true, M, d, kLnEps, st));
      e3.mode = keep_h ? EPI_GELU : EPI_GELU_ONLY; e3.bias = w.b_fc;
      CKP(h, st, PC_GEMM_FC, 2.0 * Md * 4 * dd * dd, 2 * (Md * dd + 4 * dd * dd + fc_out * Md * 4 * dd),
          gemm_bf16_tn(v.a_buf, d, w.w_fc, d, e3, M, 4 * d, d, st, v.gws));
    }
    GemmEpilogue e4;
    e4.out0 = v.x_in[i + 1]; e4.bias = w.b_pr; e4.resid = v.x_mid[i]; e4.ldc = d;
    if (fused) {
      e4.mode = EPI_RESID_STATS; e4.out2 = v.xb_in[i + 1]; e4.stats_out = v.st_in[i + 1];
      if (spliced(i + 1)) {  // the next block's prompt rows replace the computed ones (they get no gradient: splice_bwd)
        e4.splice_prompt = prompts + static_cast<size_t>(i + 1) * t.n_ctx * d;
        e4.splice_row0 = t.row0; e4.splice_n = t.n_ctx; e4.splice_L = t.L;
      }
    } else {
      e4.mode = EPI_RESID_F32;
    }
    CKP(h, st, PC_GEMM_PROJ, 2.0 * Md * 4 * dd * dd, 2 * (Md * 4 * dd + 4 * dd * dd) + (fused ? 10 : 8) * Md * dd,
        gemm_bf16_tn(v.g_buf, 4 * d, w.w_pr, 4 * d, e4, M, d, 4 * d, st, v.gws));
  }
  v.fused = fused;
  v.pruned = pruned;
  return 0;
}

// x (and the row stride) the feature head reads its one row per sequence from, after a walk over `v`
const float* tower_head_input(const Tower& t, const FwdView& v, const int** rows, int* L) {
  if (v.pruned) { *rows = nullptr; *L = 1; return v.pr_xo; }
  *rows = t.sel_rows; *L = t.row_L();
  return v.x_in[t.layers];
}

// the training walk: saves the activations for the backward
int tower_forward_train(mudpt_handle* h, Tower& t, const float* prompts, int first_splice_layer, cudaStream_t st, FwdView& v) {
  v = train_view(t);
  if (tower_forward(h, t, v, prompts, first_splice_layer, st)) return -1;
  t.fwd_done = true;
  t.fwd_fused = v.fused;
  t.fwd_pruned = v.pruned;
  return 0;
}

// Precondition: t.dx / t.dx_bf16 hold the gradient w.r.t. the tower output x_in[layers].
//
// Fused formulation: the LayerNorm dgrad  dx += rstd (g - mean(g) - xhat mean(g xhat)),  g = dy gamma, runs in the
// epilogue of the dgrad GEMM that produces g (through the gamma-folded weight).  Its two row means do not need g:
//   mean(g) = (1/d) dout . colsum,   mean(g xhat) = (1/d) dout . (y - b')      (dout = the GEMM's A operand, y = the
// saved output of the forward LN-GEMM), so the PRODUCER of dout (GELU' epilogue, attention backward) emits them.
int tower_backward(mudpt_handle* h, Tower& t, float* d_prompts, int first_splice_layer, cudaStream_t st, bool need_dx0 = false) {
  const int M = t.rows, d = t.d;
  const double Md = static_cast<double>(M), dd = d;
  const double attn_fl = 2.5 * 4.0 * t.H * t.attn_sq * 64.0;  // SURVEY.md 8d: 2.5x forward
  const bool fused = t.fwd_fused && h->ln_bwd_fused;  // (the fused forward also keeps the fp32 LN inputs the kernel needs)
  // stand-alone LayerNorm backward after a fused forward: the bf16 row + its exact statistics instead of the fp32 row
  // (14 instead of 16 B/element on an HBM-bound kernel; xhat from bf16(x) -- the operand precision of every GEMM here)
  const bool xstats = t.fwd_fused && !fused && h->ln_bwd_bf16x;
  const int parts = d / 64;
  const int dots_mlp = (4 * d + gemm_dots_span(4 * d) - 1) / gemm_dots_span(4 * d);
  // bf16 gradient stream (see mudpt_handle::grad_bf16): the stand-alone LayerNorm backward reads the residual gradient
  // from t.dx_bf16 and writes it back there; t.dx (fp32) gets the rows of the deep-prompt window only.
  const bool gb = h->grad_bf16 && !fused && !need_dx0;
  const double ln_bwd_bytes = (gb ? 6.0 : 12.0) + (xstats ? 2.0 : 4.0);  // dy 2, x, residual in, gradient out (+ its bf16 copy)
  bool f32_whole = true;  // t.dx holds the whole stream in fp32 (head_backward / the pruned last block write both copies)
  auto ln_bwd_main = [&](const void* xrow, const float2* stats, const float* gamma, bool has_resid, bool whole_f32_out) -> const char* {
    if (!gb)
      return layernorm_bwd(t.a_buf, true, xrow, stats, gamma, has_resid ? t.dx : nullptr, t.dx, t.dx_bf16, M, d, kLnEps, st);
    const bool rb = has_resid && !f32_whole;
    const void* resid = !has_resid ? nullptr : (rb ? static_cast<const void*>(t.dx_bf16) : static_cast<const void*>(t.dx));
    const char* e = layernorm_bwd_stream(t.a_buf, true, xrow, stats, gamma, resid, rb, t.dx, t.dx_bf16, M, d, kLnEps, t.L, t.row0,
                                         whole_f32_out ? -1 : t.n_ctx, st, t.packed_pos());
    f32_whole = whole_f32_out;
    return e;
  };
  for (int i = t.layers - 1; i >= 0; --i) {
    const Layer& w = t.lw[i];
    const bool tail_pruned = t.fwd_pruned && i == t.layers - 1;
    if (tail_pruned) {
      // Precondition here: t.pr_dx / t.pr_dxb hold the gradient of the S consumed rows of the block output.
      const int S = t.S;
      const double Sd = S;
      GemmEpilogue p1;
      p1.out0 = t.pr_dh; p1.aux = t.pr_h; p1.ldc = 4 * d;
      if (fused) { p1.mode = EPI_GELU_BWD_DOTS; p1.sb = w.sb_fc; p1.dots_out = t.pr_dots; }
      else p1.mode = EPI_GELU_BWD;
      CKP(h, st, PC_GEMM, 2.0 * Sd * 4 * dd * dd, 2 * (Sd * dd + 4 * dd * dd + 2 * Sd * 4 * dd), gemm_bf16_tn(t.pr_dxb, d, w.w_pr_t, d, p1, S, 4 * d, d, st, &t.gws));
      GemmEpilogue p2;
      p2.ldc = d;
      if (fused) {
        p2.mode = EPI_LN_BWD; p2.out0 = t.pr_dx; p2.resid = t.pr_dx; p2.out2 = t.pr_dxb; p2.x2 = t.pr_xmb;
        p2.ln_stats = t.pr_stm; p2.ln_parts = parts; p2.ln_width = d; p2.ln_eps = kLnEps; p2.dots = t.pr_dots; p2.dot_parts = dots_mlp;
        CKP(h, st, PC_GEMM, 2.0 * Sd * 4 * dd * dd, 2 * (Sd * 4 * dd + 4 * dd * dd) + 12 * Sd * dd, gemm_bf16_tn(t.pr_dh, 4 * d, w.w_fc_t_ln, 4 * d, p2, S, d, 4 * d, st, &t.gws));
      } else {
        p2.mode = EPI_BF16; p2.out0 = t.pr_a;
        CKP(h, st, PC_GEMM, 2.0 * Sd * 4 * dd * dd, 2 * (Sd * 4 * dd + 4 * dd * dd) + 2 * Sd * dd, gemm_bf16_tn(t.pr_dh, 4 * d, w.w_fc_t, 4 * d, p2, S, d, 4 * d, st, &t.gws));
        CKP(h, st, PC_LN_BWD, 0, Sd * dd * 16, layernorm_bwd(t.pr_a, true, t.pr_xm, nullptr, w.ln2_g, t.pr_dx, t.pr_dx, t.pr_dxb, S, d, kLnEps, st));
      }
      GemmEpilogue p3;
      p3.mode = EPI_BF16; p3.out0 = t.pr_do; p3.ldc = d;
      CKP(h, st, PC_GEMM, 2.0 * Sd * dd * dd, 2 * (2 * Sd * dd + dd * dd), gemm_bf16_tn(t.pr_dxb, d, w.w_out_t, d, p3, S, d, d, st, &t.gws));
      // dO of the whole block: zero but for the S consumed rows
      CUDA_OK(h, cudaMemsetAsync(t.do_buf, 0, static_cast<size_t>(M) * d * sizeof(bf16), st));
      CKP(h, st, PC_SPLICE, 0, Sd * dd * 4, scatter_rows_bf16(t.pr_do, t.sel_rows, S, t.row_L(), t.do_buf, d, st));
    } else {
    // MLP branch: dg = dx W_pr ; dh = dg * GELU'(h) ; dm = dh W_fc ; dx += LN2_bwd(dm)
    GemmEpilogue e1;
    e1.out0 = t.dh_buf; e1.aux = t.h[i]; e1.ldc = 4 * d;
    if (fused) { e1.mode = EPI_GELU_BWD_DOTS; e1.sb = w.sb_fc; e1.dots_out = t.dots; }
    else e1.mode = EPI_GELU_BWD;
    CKP(h, st, PC_GEMM_DPROJ, 2.0 * Md * 4 * dd * dd, 2 * (Md * dd + 4 * dd * dd + 2 * Md * 4 * dd),
        gemm_bf16_tn(t.dx_bf16, d, w.w_pr_t, d, e1, M, 4 * d, d, st, &t.gws));
    GemmEpilogue e2;
    e2.ldc = d;
    if (fused) {
      e2.mode = EPI_LN_BWD; e2.out0 = t.dx; e2.resid = t.dx; e2.out2 = t.dx_bf16; e2.x2 = t.xb_mid[i];
      e2.ln_stats = t.st_mid[i]; e2.ln_parts = parts; e2.ln_width = d; e2.ln_eps = kLnEps; e2.dots = t.dots; e2.dot_parts = dots_mlp;
      CKP(h, st, PC_GEMM_DFC, 2.0 * Md * 4 * dd * dd, 2 * (Md * 4 * dd + 4 * dd * dd) + 12 * Md * dd,
          gemm_bf16_tn(t.dh_buf, 4 * d, w.w_fc_t_ln, 4 * d, e2, M, d, 4 * d, st, &t.gws));
    } else {
      e2.mode = EPI_BF16; e2.out0 = t.a_buf;  // a_buf: forward transient, free during the backward
      CKP(h, st, PC_GEMM_DFC, 2.0 * Md * 4 * dd * dd, 2 * (Md * 4 * dd + 4 * dd * dd) + 2 * Md * dd,
          gemm_bf16_tn(t.dh_buf, 4 * d, w.w_fc_t, 4 * d, e2, M, d, 4 * d, st, &t.gws));
      CKP(h, st, PC_LN_BWD, 0, Md * dd * ln_bwd_bytes,
          ln_bwd_main(xstats ? static_cast<const void*>(t.xb_mid[i]) : t.x_mid[i], xstats ? t.st_mid[i] : nullptr, w.ln2_g, true, false));
    }
    // attention branch: dO = dx W_out ; (dQ,dK,dV) ; da = dQKV W_in ; dx += LN1_bwd(da)
    GemmEpilogue e3;
    e3.mode = EPI_BF16; e3.out0 = t.do_buf; e3.ldc = d;
    CKP(h, st, PC_GEMM_DOUT, 2.0 * Md * dd * dd, 2 * (2 * Md * dd + dd * dd), gemm_bf16_tn(t.dx_bf16, d, w.w_out_t, d, e3, M, d, d, st, &t.gws));
    }
    CKP(h, st, PC_ATTN_BWD, attn_fl, Md * dd * 2 * 8,
        t.ragged ? attention_varlen_bwd(t.qkv[i], t.do_buf, t.lse[i], t.dqkv_buf, t.seq_off, t.S, t.L, t.H, d, st)
                 : attention_bwd(t.qkv[i], t.o[i], t.do_buf, t.lse[i], t.dsum, t.dqkv_buf, t.S, t.L, t.H, d, t.causal, st,
                                 fused ? w.sb_in : nullptr, fused ? t.dots : nullptr));
    // exact work skipping below block 0: only the prompt rows of its input gradient are ever read (by the splice backward)
    const bool head_pruned = i == 0 && h->prune && !fused && !tail_pruned && !need_dx0 && first_splice_layer == 0 && t.depth > 0 &&
                             t.n_ctx > 0 && t.S * t.n_ctx < M;
    if (head_pruned) {
      const int R = t.S * t.n_ctx;
      const double Rd = R;
      CKP(h, st, PC_SPLICE, 0, Rd * dd * 12, gather_rows(nullptr, t.dqkv_buf, t.p0_rows, R, 0, nullptr, t.p0_dqkv, 3 * d, st));
      GemmEpilogue q4;
      q4.mode = EPI_BF16; q4.out0 = t.p0_a; q4.ldc = d;
      CKP(h, st, PC_GEMM, 2.0 * Rd * 3 * dd * dd, 2 * (Rd * 3 * dd + 3 * dd * dd) + 2 * Rd * dd,
          gemm_bf16_tn(t.p0_dqkv, 3 * d, w.w_in_t, 3 * d, q4, R, d, 3 * d, st, &t.gws));
      CKP(h, st, PC_SPLICE, 0, Rd * dd * 8, gather_rows(t.x_in[0], nullptr, t.p0_rows, R, 0, t.p0_x, nullptr, d, st));
      CKP(h, st, PC_SPLICE, 0, Rd * dd * 8, gather_rows(t.dx, nullptr, t.p0_rows, R, 0, t.p0_dx, nullptr, d, st));
      CKP(h, st, PC_LN_BWD, 0, Rd * dd * 16, layernorm_bwd(t.p0_a, true, t.p0_x, nullptr, w.ln1_g, t.p0_dx, t.p0_dx, t.p0_dxb, R, d, kLnEps, st));
      CKP(h, st, PC_SPLICE, 0, Rd * dd * 8, scatter_rows(t.p0_dx, t.p0_rows, R, 0, t.dx, nullptr, d, false, st));
      CKP(h, st, PC_SPLICE, 0, t.S * t.n_ctx * dd * 4, splice_bwd(t.dx, t.dx_bf16, d_prompts, t.splice_ws, t.S, t.L, t.row0, t.n_ctx, d, false, st, t.packed_off()));
      continue;
    }
    GemmEpilogue e4;
    e4.ldc = d;
    if (fused) {
      e4.mode = EPI_LN_BWD; e4.out0 = t.dx; e4.resid = tail_pruned ? nullptr : t.dx; e4.out2 = t.dx_bf16; e4.x2 = t.xb_in[i];
      e4.ln_stats = t.st_in[i]; e4.ln_parts = parts; e4.ln_width = d; e4.ln_eps = kLnEps; e4.dots = t.dots; e4.dot_parts = 3 * t.H;
      CKP(h, st, PC_GEMM_DQKV, 2.0 * Md * 3 * dd * dd, 2 * (Md * 3 * dd + 3 * dd * dd) + 12 * Md * dd,
          gemm_bf16_tn(t.dqkv_buf, 3 * d, w.w_in_t_ln, 3 * d, e4, M, d, 3 * d, st, &t.gws));
    } else {
      e4.mode = EPI_BF16; e4.out0 = t.a_buf;
      CKP(h, st, PC_GEMM_DQKV, 2.0 * Md * 3 * dd * dd, 2 * (Md * 3 * dd + 3 * dd * dd) + 2 * Md * dd,
          gemm_bf16_tn(t.dqkv_buf, 3 * d, w.w_in_t, 3 * d, e4, M, d, 3 * d, st, &t.gws));
      // (the pruned last block adds its S consumed rows into the fp32 stream right below: every fp32 row is written there)
      CKP(h, st, PC_LN_BWD, 0, Md * dd * (tail_pruned ? 8.0 + (xstats ? 2.0 : 4.0) : ln_bwd_bytes),
          ln_bwd_main(xstats ? static_cast<const void*>(t.xb_in[i]) : t.x_in[i], xstats ? t.st_in[i] : nullptr, w.ln1_g, !tail_pruned,
                      tail_pruned));
    }
    if (tail_pruned)  // the residual path of the S consumed rows (everything else of it is zero)
      CKP(h, st, PC_SPLICE, 0, t.S * dd * 14, scatter_rows(t.pr_dx, t.sel_rows, t.S, t.row_L(), t.dx, t.dx_bf16, d, true, st));
    // splice backward: the inserted prompt rows collect the batch-summed gradient; the rows
    // they overwrote get none (clip/model.py:281-297, SURVEY.md 3.3)
    if (i < t.depth && i >= first_splice_layer && t.n_ctx > 0)
      CKP(h, st, PC_SPLICE, 0, t.S * t.n_ctx * dd * 4,
          splice_bwd(t.dx, t.dx_bf16, d_prompts + static_cast<size_t>(i) * t.n_ctx * d, t.splice_ws, t.S, t.L, t.row0, t.n_ctx, d, i > 0, st,
                     t.packed_off()));
  }
  return 0;
}

// Gradient of the feature head into the tower output: the S consumed rows only (pruned: a dense [S, d] buffer;
// otherwise scattered into the zeroed full gradient).
int head_backward(mudpt_handle* h, Tower& t, const float* d_f, const float* gamma, const float* proj, cudaStream_t st) {
  const int e = h->cfg.embed_dim;
  if (t.fwd_pruned) {
    CK(h, feature_head_bwd(d_f, t.pr_xo, nullptr, gamma, proj, t.pr_dx, t.pr_dxb, t.head_ws, t.S, 1, t.d, e, kLnEps, st));
    return 0;
  }
  const size_t n = static_cast<size_t>(t.rows) * t.d;
  CUDA_OK(h, cudaMemsetAsync(t.dx, 0, n * sizeof(float), st));
  CUDA_OK(h, cudaMemsetAsync(t.dx_bf16, 0, n * sizeof(bf16), st));
  CK(h, feature_head_bwd(d_f, t.x_in[t.layers], t.sel_rows, gamma, proj, t.dx, t.dx_bf16, t.head_ws, t.S, t.row_L(), t.d, e, kLnEps, st));
  return 0;
}

bool tower_complete(const Tower& t) {
  for (const Layer& l : t.lw)
    if (l.have != LB_ALL) return false;
  return true;
}

}  // namespace

// =============================================================================== C ABI
extern "C" {

int mudpt_abi_version(void) { return MUDPT_ABI_VERSION; }
const char* mudpt_global_last_error(void) { return g_err.c_str(); }
const char* mudpt_last_error(mudpt_handle* h) { return h ? h->err.c_str() : g_err.c_str(); }

int mudpt_create(const mudpt_config* cfg, mudpt_handle** out) {
  if (!cfg || !out) return fail(nullptr, "mudpt_create: null argument");
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0)
    return fail(nullptr, "mudpt_create: no CUDA device (there is no CPU fallback)");
  if (cfg->device < 0 || cfg->device >= ndev) return fail(nullptr, "mudpt_create: bad device ordinal %d", cfg->device);
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, cfg->device) != cudaSuccess) return fail(nullptr, "cudaGetDeviceProperties failed");
  if (prop.major != 10) return fail(nullptr, "mudpt_create: device is sm_%d%d; this library is built for sm_100a only", prop.major, prop.minor);
  if (cfg->vision_width % 64 || cfg->transformer_width % 64 || cfg->transformer_width != cfg->transformer_heads * 64)
    return fail(nullptr, "mudpt_create: tower widths must be heads * 64");
  if (cfg->image_resolution % cfg->vision_patch_size) return fail(nullptr, "mudpt_create: resolution %% patch != 0");
  if (cfg->prompt_depth < 1 || cfg->n_ctx < 0) return fail(nullptr, "mudpt_create: PROMPT_DEPTH should be > 0");
  if (cfg->embed_dim != cfg->transformer_width)
    return fail(nullptr, "mudpt_create: embed_dim must equal transformer_width (clip/model.py:519, trainers/mudpt.py:175)");
  cudaSetDevice(cfg->device);
  mudpt_handle* h = new mudpt_handle();
  h->cfg = *cfg;
  const int np = (cfg->image_resolution / cfg->vision_patch_size) * (cfg->image_resolution / cfg->vision_patch_size);
  Tower& v = h->vis;
  v.d = cfg->vision_width; v.H = cfg->vision_width / 64; v.layers = cfg->vision_layers; v.n_ctx = cfg->n_ctx;
  v.L = np + 1 + cfg->n_ctx; v.row0 = np + 1; v.depth = cfg->prompt_depth; v.causal = false;
  v.lw.resize(v.layers);
  Tower& t = h->txt;
  t.d = cfg->transformer_width; t.H = cfg->transformer_heads; t.layers = cfg->transformer_layers; t.n_ctx = cfg->n_ctx;
  t.L = cfg->context_length; t.row0 = 1; t.depth = cfg->prompt_depth; t.causal = true;
  t.lw.resize(t.layers);
  h->Kp = (3 * cfg->vision_patch_size * cfg->vision_patch_size + 7) & ~7;
  v.stem_per_seq = static_cast<size_t>(np) * h->Kp;
  for (Tower* w : {&v, &t}) {
    w->x_in.assign(w->layers + 1, nullptr);
    w->xb_in.assign(w->layers + 1, nullptr);
    w->st_in.assign(w->layers + 1, nullptr);
    w->x_mid.assign(w->layers, nullptr);
    w->xb_mid.assign(w->layers, nullptr);
    w->st_mid.assign(w->layers, nullptr);
    w->qkv.assign(w->layers, nullptr);
    w->o.assign(w->layers, nullptr);
    w->h.assign(w->layers, nullptr);
    w->lse.assign(w->layers, nullptr);
  }
  h->launches_at_create = g_launch_counter.load();
  h->ln_fused = getenv("MUDPT_LN_FUSED") ? (atoi(getenv("MUDPT_LN_FUSED")) != 0 ? 1 : 0) : -1;
  h->ln_bwd_fused = env_flag("MUDPT_LN_BWD_FUSED", false);
  h->ln_bwd_bf16x = env_flag("MUDPT_LN_BWD_BF16X", true);
  h->prune = env_flag("MUDPT_PRUNE", true);
  h->grad_bf16 = env_flag("MUDPT_GRAD_BF16", true);
  *out = h;
  return 0;
}

void mudpt_destroy(mudpt_handle* h) {
  if (!h) return;
  cudaSetDevice(h->cfg.device);
  for (void* p : h->allocs) cudaFree(p);
  for (Tower* t : {&h->vis, &h->txt})
    for (AllocGroup* g : {&t->in_mem, &t->train_mem, &t->inf.mem, &t->img_mem})
      for (void* p : g->ptrs) cudaFree(p);
  for (ProfRec& r : h->prof.recs) { cudaEventDestroy(r.e0); cudaEventDestroy(r.e1); }
  for (cudaEvent_t e : h->prof.pool) cudaEventDestroy(e);
  gemm_clear_tensor_map_cache();
  delete h;
}

int mudpt_set_option(mudpt_handle* h, const char* name, int32_t value) {
  if (!h || !name) return fail(h, "mudpt_set_option: null argument");
  if (!strcmp(name, "ln_fused")) h->ln_fused = value < 0 ? -1 : (value != 0 ? 1 : 0);
  else if (!strcmp(name, "ln_bwd_fused")) h->ln_bwd_fused = value != 0;
  else if (!strcmp(name, "prune")) h->prune = value != 0;
  else if (!strcmp(name, "grad_stream_bf16")) h->grad_bf16 = value != 0;
  else return fail(h, "mudpt_set_option: unknown option %s", name);
  h->vis.fwd_done = h->txt.fwd_done = false;  // saved activations belong to the previous formulation
  return 0;
}

int mudpt_set_weight(mudpt_handle* h, const char* name, const float* data, int64_t numel, void* stream) {
  if (!h || !name || !data) return fail(h, "mudpt_set_weight: null argument");
  cudaSetDevice(h->cfg.device);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const mudpt_config& c = h->cfg;
  const int dv = c.vision_width, dt = c.transformer_width, e = c.embed_dim;
  const int np = (c.image_resolution / c.vision_patch_size) * (c.image_resolution / c.vision_patch_size);
  int layer = -1, off = 0;
  if (sscanf(name, "visual.transformer.resblocks.%d.%n", &layer, &off) == 1 && off > 0)
    return set_block_weight(h, h->vis, layer, name + off, data, numel, name, st);
  if (sscanf(name, "transformer.resblocks.%d.%n", &layer, &off) == 1 && off > 0)
    return set_block_weight(h, h->txt, layer, name + off, data, numel, name, st);
  int rc = 1;
  if (!strcmp(name, "visual.conv1.weight")) {
    const int k = 3 * c.vision_patch_size * c.vision_patch_size;
    if (numel != static_cast<int64_t>(dv) * k) return fail(h, "weight %s: bad size", name);
    if (!h->w_conv) CUDA_OK(h, dev_alloc(h, &h->w_conv, static_cast<size_t>(dv) * h->Kp));
    CUDA_OK(h, cudaMemsetAsync(h->w_conv, 0, static_cast<size_t>(dv) * h->Kp * sizeof(bf16), st));
    if (h->Kp == k) {
      CK(h, cast_to_bf16(data, h->w_conv, static_cast<size_t>(numel), st));
    } else {  // padded rows (ViT-L/14: 588 -> 592)
      for (int r = 0; r < dv; ++r) CK(h, cast_to_bf16(data + static_cast<size_t>(r) * k, h->w_conv + static_cast<size_t>(r) * h->Kp, k, st));
    }
    // [k, dv] transposed + (Kp - k) zero rows
    if (!h->w_conv_t) CUDA_OK(h, dev_alloc(h, &h->w_conv_t, static_cast<size_t>(h->Kp) * dv));
    if (h->Kp != k)
      CUDA_OK(h, cudaMemsetAsync(h->w_conv_t + static_cast<size_t>(k) * dv, 0, static_cast<size_t>(h->Kp - k) * dv * sizeof(bf16), st));
    CK(h, transpose_cast_bf16(data, h->w_conv_t, dv, k, st));
    h->stem_have |= SB_CONV; rc = 0;
  } else if (!strcmp(name, "visual.class_embedding")) { rc = store_f32(h, &h->cls, data, numel, dv, name, st); h->stem_have |= SB_CLS; }
  else if (!strcmp(name, "visual.positional_embedding")) { rc = store_f32(h, &h->pos_v, data, numel, static_cast<int64_t>(np + 1) * dv, name, st); h->stem_have |= SB_POS_V; }
  else if (!strcmp(name, "visual.ln_pre.weight")) { rc = store_f32(h, &h->ln_pre_g, data, numel, dv, name, st); h->stem_have |= SB_LNPRE_G; }
  else if (!strcmp(name, "visual.ln_pre.bias")) { rc = store_f32(h, &h->ln_pre_b, data, numel, dv, name, st); h->stem_have |= SB_LNPRE_B; }
  else if (!strcmp(name, "visual.ln_post.weight")) { rc = store_f32(h, &h->ln_post_g, data, numel, dv, name, st); h->stem_have |= SB_LNPOST_G; }
  else if (!strcmp(name, "visual.ln_post.bias")) { rc = store_f32(h, &h->ln_post_b, data, numel, dv, name, st); h->stem_have |= SB_LNPOST_B; }
  else if (!strcmp(name, "visual.proj")) { rc = store_f32(h, &h->proj_v, data, numel, static_cast<int64_t>(dv) * e, name, st); h->stem_have |= SB_PROJ_V; }
  else if (!strcmp(name, "positional_embedding")) { rc = store_f32(h, &h->pos_t, data, numel, static_cast<int64_t>(c.context_length) * dt, name, st); h->stem_have |= SB_POS_T; }
  else if (!strcmp(name, "ln_final.weight")) { rc = store_f32(h, &h->ln_final_g, data, numel, dt, name, st); h->stem_have |= SB_LNF_G; }
  else if (!strcmp(name, "ln_final.bias")) { rc = store_f32(h, &h->ln_final_b, data, numel, dt, name, st); h->stem_have |= SB_LNF_B; }
  else if (!strcmp(name, "text_projection")) { rc = store_f32(h, &h->proj_t, data, numel, static_cast<int64_t>(dt) * e, name, st); h->stem_have |= SB_PROJ_T; }
  else if (!strcmp(name, "logit_scale")) {
    if (numel != 1) return fail(h, "weight logit_scale: expected 1 element");
    float v = 0.f;
    CUDA_OK(h, cudaMemcpyAsync(&v, data, sizeof(float), cudaMemcpyDeviceToHost, st));
    CUDA_OK(h, cudaStreamSynchronize(st));
    h->logit_scale_exp = expf(v);  // logit_scale.exp(), trainers/mudpt.py:181 (frozen)
    h->stem_have |= SB_SCALE; rc = 0;
  }
  return rc;
}

int mudpt_weights_complete(mudpt_handle* h) {
  if (!h) return fail(h, "null handle");
  if (h->stem_have != SB_ALL) return fail(h, "stem/head weights missing (mask 0x%x of 0x%x)", h->stem_have, SB_ALL);
  if (!tower_complete(h->vis)) return fail(h, "vision tower weights incomplete");
  if (!tower_complete(h->txt)) return fail(h, "text tower weights incomplete");
  return 0;
}

// conv1 as a GEMM over extracted patches, scattered to token rows 1..np with +pos (clip/model.py:527-531), the CLS rows,
// then ln_pre in place (:541) -- the prompt rows are overwritten by the layer-0 splice with prompts[0] = ln_pre(visual_ctx +
// shared_ctx), which is identical for every image -- and, for the fused LayerNorm, the bf16 copy + statistics of x0
static int vision_stem(mudpt_handle* h, const float* images, int B, bf16* patches, float* x0, bf16* xb0, float2* st0, cudaStream_t st) {
  const mudpt_config& c = h->cfg;
  const Tower& t = h->vis;
  const int np = t.row0 - 1;
  CK(h, im2col_bf16(images, patches, B, c.image_resolution, c.vision_patch_size, h->Kp, st));
  GemmEpilogue ep;
  ep.mode = EPI_PATCH; ep.out0 = x0; ep.resid = h->pos_v; ep.ldc = t.d; ep.patch_np = np; ep.patch_L = t.L;
  CK(h, gemm_bf16_tn(patches, h->Kp, h->w_conv, h->Kp, ep, B * np, t.d, h->Kp, st));
  CK(h, write_cls_rows(x0, h->cls, h->pos_v, B, t.L, t.d, st));
  CK(h, layernorm_fwd(x0, h->ln_pre_g, h->ln_pre_b, x0, false, B * t.L, t.d, kLnEps, st));
  if (ln_fused_for(h, t, B * t.L)) CK(h, rowstats(x0, xb0, st0, B * t.L, t.d, st));
  return 0;
}

int mudpt_vision_forward(mudpt_handle* h, const float* images, int32_t B, const float* prompts, float* f_img, void* stream) {
  if (!h || !images || !f_img || (!prompts && h->cfg.n_ctx > 0)) return fail(h, "mudpt_vision_forward: null argument");
  if (B <= 0) return fail(h, "mudpt_vision_forward: empty batch");
  if (mudpt_weights_complete(h)) return -1;
  cudaSetDevice(h->cfg.device);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  Tower& t = h->vis;
  if (ensure_input(h, t, B, t.row0 + t.n_ctx) || ensure_train(h, t, st)) return -1;
  if (vision_stem(h, images, B, t.patches, t.x_in[0], t.xb_in[0], t.st_in[0], st)) return -1;
  t.sel_rows = nullptr;  // CLS row (clip/model.py:548)
  FwdView v;
  if (tower_forward_train(h, t, prompts, 0, st, v)) return -1;
  const int* rows; int Lh;
  const float* xh = tower_head_input(t, v, &rows, &Lh);
  CK(h, feature_head_fwd(xh, rows, h->ln_post_g, h->ln_post_b, h->proj_v, f_img, v.head_ws, B, Lh, t.d, h->cfg.embed_dim, kLnEps, st));
  return 0;
}

int mudpt_vision_infer(mudpt_handle* h, const float* images, int32_t B, const float* prompts, float* f_img, void* stream) {
  if (!h || !images || !f_img || (!prompts && h->cfg.n_ctx > 0)) return fail(h, "mudpt_vision_infer: null argument");
  if (B <= 0) return fail(h, "mudpt_vision_infer: empty batch");
  if (mudpt_weights_complete(h)) return -1;
  cudaSetDevice(h->cfg.device);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  Tower& t = h->vis;
  const int M = B * t.L;
  if (ensure_infer(h, t, B, M, ln_fused_for(h, t, M), st)) return -1;
  FwdView& v = t.inf.v;
  v.S = B; v.rows = M; v.attn_sq = static_cast<double>(B) * t.L * t.L;
  if (vision_stem(h, images, B, t.inf.patches, v.x_in[0], v.xb_in[0], v.st_in[0], st)) return -1;
  if (tower_forward(h, t, v, prompts, 0, st)) return -1;
  const int* rows; int Lh;
  const float* xh = tower_head_input(t, v, &rows, &Lh);
  CK(h, feature_head_fwd(xh, rows, h->ln_post_g, h->ln_post_b, h->proj_v, f_img, v.head_ws, B, Lh, t.d, h->cfg.embed_dim, kLnEps, st));
  return 0;
}

int mudpt_vision_backward(mudpt_handle* h, const float* d_f_img, float* d_prompts, void* stream) {
  if (!h || !d_f_img || !d_prompts) return fail(h, "mudpt_vision_backward: null argument");
  Tower& t = h->vis;
  if (!t.fwd_done) return fail(h, "mudpt_vision_backward: no forward pass to differentiate");
  cudaSetDevice(h->cfg.device);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (head_backward(h, t, d_f_img, h->ln_post_g, h->proj_v, st)) return -1;
  return tower_backward(h, t, d_prompts, 0, st);
}

// The fp32 patch gradient [S * np, Kp] goes to g_buf (the forward's QuickGELU transient, which no backward reads) where it
// fits: per image L * 4d bf16 against np * Kp fp32 -- ViT-B/16 and ViT-L/14 yes, ViT-B/32 (Kp = 4d) no.
static bool dpatch_in_g_buf(const mudpt_handle* h) {
  const Tower& t = h->vis;
  return static_cast<size_t>(t.row0 - 1) * h->Kp * sizeof(float) <= static_cast<size_t>(t.L) * 4 * t.d * sizeof(bf16);
}

// Image-gradient memory beyond the training workspace (Tower::img_mem), for the tower's current batch
static int ensure_image_grad(mudpt_handle* h, Tower& t) {
  if (static_cast<size_t>(t.S) <= t.img_S) return 0;  // (img_S = 0 until the first call)
  release(t.img_mem);
  t.img_S = t.S;
  t.img_dpatch = t.img_dprompt = nullptr;
  AllocGroup* g = &t.img_mem;
  if (!dpatch_in_g_buf(h)) CUDA_OK(h, dev_alloc(h, &t.img_dpatch, t.img_S * (t.row0 - 1) * h->Kp, g));
  if (t.n_ctx > 0) CUDA_OK(h, dev_alloc(h, &t.img_dprompt, static_cast<size_t>(t.depth) * t.n_ctx * t.d, g));
  return 0;
}

// Backward of the stem (vision_stem) into the images, on the patch rows b * L + 1 + p: x = conv1(img) + pos, y = ln_pre(x).
// Precondition: t.dx holds dL/dy for every row in fp32 (tower_backward with need_dx0).  The CLS rows (class_embedding is
// frozen) and the prompt rows (their ln_pre belongs to the prompt algebra; their gradient went to d_prompts[0]) are dropped.
//   1. x again from the kept bf16 patches with the forward's own patch GEMM: bitwise the rows ln_pre normalised
//   2. ln_pre dgrad over the row map b * np + p <- b * L + 1 + p, bf16 compact rows
//   3. patch dgrad d_patches [S * np, Kp] = dy_ln . W_conv (the transposed bf16 copy), fp32, returned in *dpatch
// The output stage (col2im for the image gradient, or the PGD update) reads *dpatch.
// Scratch: x in dh_buf, dy_ln in a_buf, d_patches in g_buf or img_dpatch -- transients no one reads after block 0.
static int stem_backward(mudpt_handle* h, cudaStream_t st, const float** dpatch_out) {
  Tower& t = h->vis;
  const int B = t.S, np = t.row0 - 1, d = t.d, Kp = h->Kp, M = B * np;
  const double Md = M, dd = d, Kd = Kp;
  float* x = reinterpret_cast<float*>(t.dh_buf);
  GemmEpilogue ep;
  ep.mode = EPI_PATCH; ep.out0 = x; ep.resid = h->pos_v; ep.ldc = d; ep.patch_np = np; ep.patch_L = t.L;
  CKP(h, st, PC_STEM, 2.0 * Md * dd * Kd, 2 * (Md * Kd + dd * Kd) + 8 * Md * dd, gemm_bf16_tn(t.patches, Kp, h->w_conv, Kp, ep, M, d, Kp, st));
  CKP(h, st, PC_LN_BWD, 0, Md * dd * 10, layernorm_bwd_rows(t.dx, x, h->ln_pre_g, t.a_buf, M, d, kLnEps, np, t.L, 1, st));
  float* dpatch = dpatch_in_g_buf(h) ? reinterpret_cast<float*>(t.g_buf) : t.img_dpatch;
  GemmEpilogue e2;
  e2.mode = EPI_F32; e2.out0 = dpatch; e2.ldc = Kp;
  CKP(h, st, PC_GEMM, 2.0 * Md * Kd * dd, 2 * (Md * dd + Kd * dd) + 4 * Md * Kd, gemm_bf16_tn(t.a_buf, d, h->w_conv_t, d, e2, M, Kp, d, st, &t.gws));
  *dpatch_out = dpatch;
  return 0;
}

// The vision backward of the last forward down to the patch gradient: head, dense tower backward, stem backward
static int image_backward(mudpt_handle* h, const float* d_f_img, float* d_prompts, cudaStream_t st, const float** dpatch) {
  Tower& t = h->vis;
  if (ensure_image_grad(h, t)) return -1;
  if (head_backward(h, t, d_f_img, h->ln_post_g, h->proj_v, st)) return -1;
  // without d_prompts the splice backward still runs (layers > 0 zero the rows their prompts overwrote) into a sink
  if (tower_backward(h, t, d_prompts ? d_prompts : t.img_dprompt, 0, st, /*need_dx0=*/true)) return -1;
  return stem_backward(h, st, dpatch);
}

int mudpt_vision_backward_images(mudpt_handle* h, const float* d_f_img, float* d_prompts, float* d_images, void* stream) {
  if (!h || !d_f_img || !d_images) return fail(h, "mudpt_vision_backward_images: null argument");
  Tower& t = h->vis;
  if (!t.fwd_done) return fail(h, "mudpt_vision_backward_images: no forward pass to differentiate");
  cudaSetDevice(h->cfg.device);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const mudpt_config& c = h->cfg;
  const float* dpatch;
  if (image_backward(h, d_f_img, d_prompts, st, &dpatch)) return -1;
  CKP(h, st, PC_STEM, 0, 8.0 * t.S * 3 * c.image_resolution * c.image_resolution,
      col2im_f32(dpatch, d_images, t.S, c.image_resolution, c.vision_patch_size, h->Kp, st));
  return 0;
}

static PgdParams pgd_params(const float* mean_host, const float* std_host, float eps, float alpha) {
  PgdParams p;
  for (int c = 0; c < 3; ++c) { p.mean[c] = mean_host[c]; p.std[c] = std_host[c]; }
  p.eps = eps; p.alpha = alpha;
  return p;
}

int mudpt_vision_pgd_step(mudpt_handle* h, const float* d_f_img, float* x_adv, const float* x_clean, float* x_norm,
                          const float* mean_host, const float* std_host, float eps, float alpha, void* stream) {
  if (!h || !d_f_img || !x_adv || !x_clean || !x_norm || !mean_host || !std_host)
    return fail(h, "mudpt_vision_pgd_step: null argument");
  Tower& t = h->vis;
  if (!t.fwd_done) return fail(h, "mudpt_vision_pgd_step: no forward pass to differentiate");
  const PgdParams prm = pgd_params(mean_host, std_host, eps, alpha);
  if (const char* e = pgd_linf_check(prm)) return fail(h, "mudpt_vision_pgd_step: %s", e);
  cudaSetDevice(h->cfg.device);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const mudpt_config& c = h->cfg;
  const float* dpatch;
  if (image_backward(h, d_f_img, nullptr, st, &dpatch)) return -1;
  CKP(h, st, PC_STEM, 0, 20.0 * t.S * 3 * c.image_resolution * c.image_resolution,
      pgd_linf_f32(dpatch, x_adv, x_clean, x_norm, t.S, c.image_resolution, c.vision_patch_size, h->Kp, prm, st));
  return 0;
}

int mudpt_text_set_classes(mudpt_handle* h, const float* embeddings, int32_t C, int32_t src_len, int32_t seq_len,
                           const int32_t* eot_host, void* stream) {
  if (!h || !embeddings || !eot_host) return fail(h, "mudpt_text_set_classes: null argument");
  const mudpt_config& c = h->cfg;
  if (C <= 0 || seq_len <= 0 || seq_len > src_len || src_len > c.context_length)
    return fail(h, "mudpt_text_set_classes: bad lengths (C=%d src_len=%d seq_len=%d)", C, src_len, seq_len);
  if (seq_len < 1 + c.n_ctx) return fail(h, "mudpt_text_set_classes: seq_len shorter than SOT + n_ctx");
  for (int i = 0; i < C; ++i)
    if (eot_host[i] < 0 || eot_host[i] >= seq_len) return fail(h, "mudpt_text_set_classes: eot[%d]=%d outside seq_len %d", i, eot_host[i], seq_len);
  if (!(h->stem_have & SB_POS_T)) return fail(h, "mudpt_text_set_classes: positional_embedding not set");
  cudaSetDevice(c.device);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  Tower& t = h->txt;
  if (ensure_input(h, t, C, seq_len)) return -1;
  CUDA_OK(h, cudaMemcpyAsync(t.eot, eot_host, C * sizeof(int), cudaMemcpyHostToDevice, st));
  CUDA_OK(h, cudaStreamSynchronize(st));  // eot_host may be freed by the caller after return
  CK(h, add_positional(t.x_in[0], embeddings, h->pos_t, C, seq_len, src_len, t.d, st));
  CK(h, rowstats(t.x_in[0], t.xb_in[0], t.st_in[0], C * seq_len, t.d, st));  // (the prompt rows are rewritten every step)
  t.fwd_done = false;
  return 0;
}

int mudpt_text_set_classes_ragged(mudpt_handle* h, const float* embeddings, int32_t C, int32_t src_len, const int32_t* len_host,
                                  const int32_t* eot_host, void* stream) {
  if (!h || !embeddings || !len_host || !eot_host) return fail(h, "mudpt_text_set_classes_ragged: null argument");
  const mudpt_config& c = h->cfg;
  if (C <= 0 || src_len <= 0 || src_len > c.context_length)
    return fail(h, "mudpt_text_set_classes_ragged: bad lengths (C=%d src_len=%d)", C, src_len);
  const int max_ok = src_len < attention_varlen_max_len() ? src_len : attention_varlen_max_len();
  int max_len = 0;
  for (int i = 0; i < C; ++i) {
    if (len_host[i] < 1 + c.n_ctx || len_host[i] > max_ok)
      return fail(h, "mudpt_text_set_classes_ragged: len[%d]=%d outside [%d, %d] (SOT + n_ctx .. src_len, at most %d)", i, len_host[i],
                  1 + c.n_ctx, max_ok, attention_varlen_max_len());
    if (eot_host[i] < 0 || eot_host[i] >= len_host[i])
      return fail(h, "mudpt_text_set_classes_ragged: eot[%d]=%d outside len %d", i, eot_host[i], len_host[i]);
    max_len = len_host[i] > max_len ? len_host[i] : max_len;
  }
  if (!(h->stem_have & SB_POS_T)) return fail(h, "mudpt_text_set_classes_ragged: positional_embedding not set");
  cudaSetDevice(c.device);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  Tower& t = h->txt;
  std::vector<int> off(C + 1, 0), sel(C);
  for (int i = 0; i < C; ++i) {
    off[i + 1] = off[i] + len_host[i];
    sel[i] = off[i] + eot_host[i];  // absolute EOT row
  }
  const int M = off[C];
  std::vector<int> pos(M);
  for (int i = 0; i < C; ++i)
    for (int j = 0; j < len_host[i]; ++j) pos[off[i] + j] = j;
  if (ensure_input(h, t, C, max_len, off.data())) return -1;
  CUDA_OK(h, cudaMemcpyAsync(t.eot, sel.data(), C * sizeof(int), cudaMemcpyHostToDevice, st));
  CUDA_OK(h, cudaMemcpyAsync(t.seq_off, off.data(), (C + 1) * sizeof(int), cudaMemcpyHostToDevice, st));
  CUDA_OK(h, cudaMemcpyAsync(t.tok_pos, pos.data(), M * sizeof(int), cudaMemcpyHostToDevice, st));
  CUDA_OK(h, cudaStreamSynchronize(st));  // (the host vectors go out of scope)
  CK(h, add_positional(t.x_in[0], embeddings, h->pos_t, C, max_len, src_len, t.d, st, t.seq_off));
  t.fwd_done = false;
  return 0;
}

int mudpt_text_forward(mudpt_handle* h, const float* prompts, int32_t splice_layer0, float* f_txt, void* stream) {
  if (!h || !f_txt || (!prompts && h->cfg.n_ctx > 0)) return fail(h, "mudpt_text_forward: null argument");
  if (mudpt_weights_complete(h)) return -1;
  Tower& t = h->txt;
  if (t.in_rows == 0 || t.S <= 0) return fail(h, "mudpt_text_forward: call mudpt_text_set_classes first");
  cudaSetDevice(h->cfg.device);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (ensure_train(h, t, st)) return -1;
  t.sel_rows = t.eot;  // EOT row (trainers/mudpt.py:154)
  FwdView v;
  if (tower_forward_train(h, t, prompts, splice_layer0 ? 0 : 1, st, v)) return -1;
  const int* rows; int Lh;
  const float* xh = tower_head_input(t, v, &rows, &Lh);
  CK(h, feature_head_fwd(xh, rows, h->ln_final_g, h->ln_final_b, h->proj_t, f_txt, v.head_ws, t.S, Lh, t.d, h->cfg.embed_dim, kLnEps, st));
  t.first_splice = splice_layer0 ? 0 : 1;  // the backward must mirror the forward's splice set
  return 0;
}

int mudpt_text_infer(mudpt_handle* h, const float* prompts, int32_t splice_layer0, float* f_txt, void* stream) {
  if (!h || !f_txt || (!prompts && h->cfg.n_ctx > 0)) return fail(h, "mudpt_text_infer: null argument");
  if (mudpt_weights_complete(h)) return -1;
  Tower& t = h->txt;
  if (t.in_rows == 0 || t.S <= 0) return fail(h, "mudpt_text_infer: call mudpt_text_set_classes first");
  cudaSetDevice(h->cfg.device);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const bool fused = ln_fused_for(h, t, t.rows);
  if (ensure_infer(h, t, t.S, t.rows, fused, st)) return -1;
  FwdView& v = t.inf.v;
  v.S = t.S; v.rows = t.rows; v.attn_sq = t.attn_sq;
  // The walk splices the layer-0 prompt rows into its input in place.  The class set's input belongs to the training walk
  // (its backward reads those rows again), so with a layer-0 splice this walk starts from a copy in its own residual buffer.
  if (splice_layer0 && t.n_ctx > 0 && t.layers > 0) {
    const size_t n = static_cast<size_t>(t.rows) * t.d;
    v.x_in[0] = v.x_in[t.layers];
    v.xb_in[0] = v.xb_in[t.layers];
    v.st_in[0] = v.st_in[t.layers];
    CUDA_OK(h, cudaMemcpyAsync(v.x_in[0], t.x_in[0], n * sizeof(float), cudaMemcpyDeviceToDevice, st));
    if (fused) {
      CUDA_OK(h, cudaMemcpyAsync(v.xb_in[0], t.xb_in[0], n * sizeof(bf16), cudaMemcpyDeviceToDevice, st));
      CUDA_OK(h, cudaMemcpyAsync(v.st_in[0], t.st_in[0], n / 64 * sizeof(float2), cudaMemcpyDeviceToDevice, st));
    }
  } else {  // read only
    v.x_in[0] = t.x_in[0];
    v.xb_in[0] = t.xb_in[0];
    v.st_in[0] = t.st_in[0];
  }
  t.sel_rows = t.eot;
  if (tower_forward(h, t, v, prompts, splice_layer0 ? 0 : 1, st)) return -1;
  const int* rows; int Lh;
  const float* xh = tower_head_input(t, v, &rows, &Lh);
  CK(h, feature_head_fwd(xh, rows, h->ln_final_g, h->ln_final_b, h->proj_t, f_txt, v.head_ws, t.S, Lh, t.d, h->cfg.embed_dim, kLnEps, st));
  return 0;
}

int mudpt_workspace_bytes(mudpt_handle* h, int32_t tower, int32_t kind, int64_t* bytes) {
  if (!h || !bytes) return fail(h, "mudpt_workspace_bytes: null argument");
  if (tower != MUDPT_TOWER_VISION && tower != MUDPT_TOWER_TEXT) return fail(h, "mudpt_workspace_bytes: bad tower %d", tower);
  Tower& t = tower == MUDPT_TOWER_VISION ? h->vis : h->txt;
  const AllocGroup* g = kind == 0 ? &t.train_mem : kind == 1 ? &t.inf.mem : kind == 2 ? &t.in_mem : nullptr;
  if (!g) return fail(h, "mudpt_workspace_bytes: kind must be 0 (training workspace), 1 (inference workspace) or 2 (tower input)");
  *bytes = static_cast<int64_t>(g->bytes + (kind == 0 ? t.img_mem.bytes : 0));  // (image gradients: with the training workspace)
  return 0;
}

int mudpt_text_backward(mudpt_handle* h, const float* d_f_txt, float* d_prompts, float* d_x0, void* stream) {
  if (!h || !d_f_txt || (!d_prompts && h->cfg.n_ctx > 0)) return fail(h, "mudpt_text_backward: null argument");
  Tower& t = h->txt;
  if (!t.fwd_done) return fail(h, "mudpt_text_backward: no forward pass to differentiate");
  cudaSetDevice(h->cfg.device);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const size_t n = static_cast<size_t>(t.rows) * t.d;
  if (head_backward(h, t, d_f_txt, h->ln_final_g, h->proj_t, st)) return -1;
  if (tower_backward(h, t, d_prompts, t.first_splice, st, d_x0 != nullptr)) return -1;
  if (d_x0 && t.ragged) CK(h, unpack_rows(t.dx, t.seq_off, t.S, t.L, t.d, d_x0, st));
  else if (d_x0) CUDA_OK(h, cudaMemcpyAsync(d_x0, t.dx, n * sizeof(float), cudaMemcpyDeviceToDevice, st));
  return 0;
}

int mudpt_logits_head(mudpt_handle* h, const float* f_img, const float* f_txt, const int64_t* labels, int32_t B,
                      int32_t C, float inv_global_batch, float* logits, float* loss, float* d_f_img, float* d_f_txt,
                      void* stream) {
  if (!h || !f_img || !f_txt || !logits) return fail(h, "mudpt_logits_head: null argument");
  if (labels && !loss) return fail(h, "mudpt_logits_head: loss output required with labels");
  if (!(h->stem_have & SB_SCALE)) return fail(h, "mudpt_logits_head: logit_scale not set");
  cudaSetDevice(h->cfg.device);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const size_t need = logits_head_workspace_floats(B, C, h->cfg.embed_dim);
  if (need > h->head_ws_cap) {
    CUDA_OK(h, dev_alloc(h, &h->head_ws, need));
    h->head_ws_cap = need;
  }
  CK(h, logits_head(f_img, f_txt, reinterpret_cast<const long long*>(labels), h->logit_scale_exp, B, C, h->cfg.embed_dim,
                    inv_global_batch, h->head_ws, logits, loss, d_f_img, d_f_txt, st));
  return 0;
}

int mudpt_logits_backward(mudpt_handle* h, const float* f_img, const float* f_txt, const float* dlogits, int32_t B,
                          int32_t C, float* d_f_img, float* d_f_txt, void* stream) {
  if (!h || !f_img || !f_txt || !dlogits || !d_f_img || !d_f_txt) return fail(h, "mudpt_logits_backward: null argument");
  cudaSetDevice(h->cfg.device);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const size_t need = logits_head_workspace_floats(B, C, h->cfg.embed_dim);
  if (need > h->head_ws_cap) {
    CUDA_OK(h, dev_alloc(h, &h->head_ws, need));
    h->head_ws_cap = need;
  }
  CK(h, logits_head_bwd(f_img, f_txt, dlogits, h->logit_scale_exp, B, C, h->cfg.embed_dim, h->head_ws, d_f_img, d_f_txt, st));
  return 0;
}

// ---------------------------------------------------------------------------- unit pieces
#define CKG(expr)                                       \
  do {                                                  \
    const char* _e = (expr);                            \
    if (_e) return fail(nullptr, "%s", _e);             \
  } while (0)

int mudpt_layernorm_forward(const float* x, const float* gamma, const float* beta, void* out, int32_t out_bf16,
                            int32_t rows, int32_t width, void* stream) {
  CKG(layernorm_fwd(x, gamma, beta, out, out_bf16 != 0, rows, width, kLnEps, static_cast<cudaStream_t>(stream)));
  return 0;
}
int mudpt_layernorm_backward(const float* dy, const float* x, const float* gamma, const float* resid, float* dx,
                             uint16_t* dx_bf16, int32_t rows, int32_t width, void* stream) {
  CKG(layernorm_bwd(dy, false, x, nullptr, gamma, resid, dx, reinterpret_cast<bf16*>(dx_bf16), rows, width, kLnEps, static_cast<cudaStream_t>(stream)));
  return 0;
}
int mudpt_layernorm_backward_stream(const uint16_t* dy, const void* x, const float* x_stats, const float* gamma, const void* resid,
                                    int32_t resid_bf16, float* dx, uint16_t* dx_bf16, int32_t rows, int32_t width, int32_t win_L,
                                    int32_t win_row0, int32_t win_n, void* stream) {
  CKG(layernorm_bwd_stream(dy, true, x, reinterpret_cast<const float2*>(x_stats), gamma, resid, resid_bf16 != 0, dx,
                           reinterpret_cast<bf16*>(dx_bf16), rows, width, kLnEps, win_L, win_row0, win_n, static_cast<cudaStream_t>(stream)));
  return 0;
}
int mudpt_splice_forward(float* x, const float* prompt, int32_t S, int32_t L, int32_t row0, int32_t n, int32_t width, void* stream) {
  CKG(splice_fwd(x, prompt, S, L, row0, n, width, static_cast<cudaStream_t>(stream)));
  return 0;
}
int mudpt_splice_backward(float* dx, uint16_t* dx_bf16, float* d_prompt, int32_t S, int32_t L, int32_t row0, int32_t n,
                          int32_t width, int32_t zero_rows, void* stream) {
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  float* ws = nullptr;  // unit entry point: stream-ordered scratch (the towers own a persistent one)
  if (cudaMallocAsync(reinterpret_cast<void**>(&ws), splice_bwd_workspace_floats(n, width) * sizeof(float), st) != cudaSuccess)
    return fail(nullptr, "mudpt_splice_backward: scratch allocation failed");
  cudaMemsetAsync(ws, 0, splice_bwd_workspace_floats(n, width) * sizeof(float), st);
  const char* e = splice_bwd(dx, reinterpret_cast<bf16*>(dx_bf16), d_prompt, ws, S, L, row0, n, width, zero_rows != 0, st);
  cudaFreeAsync(ws, st);
  if (e) return fail(nullptr, "%s", e);
  return 0;
}
int mudpt_attention_forward(const uint16_t* qkv, uint16_t* o, float* lse2, int32_t S, int32_t L, int32_t H, int32_t causal, void* stream) {
  CKG(attention_fwd(reinterpret_cast<const bf16*>(qkv), reinterpret_cast<bf16*>(o), lse2, S, L, H, H * 64, causal != 0, static_cast<cudaStream_t>(stream)));
  return 0;
}
int mudpt_attention_backward(const uint16_t* qkv, const uint16_t* o, const uint16_t* d_o, const float* lse2, float* dsum,
                             uint16_t* dqkv, int32_t S, int32_t L, int32_t H, int32_t causal, void* stream) {
  CKG(attention_bwd(reinterpret_cast<const bf16*>(qkv), reinterpret_cast<const bf16*>(o), reinterpret_cast<const bf16*>(d_o),
                    lse2, dsum, reinterpret_cast<bf16*>(dqkv), S, L, H, H * 64, causal != 0, static_cast<cudaStream_t>(stream)));
  return 0;
}
int mudpt_attention_varlen_forward(const uint16_t* qkv, uint16_t* o, float* lse2, const int32_t* seq_off, int32_t S, int32_t max_len,
                                   int32_t H, void* stream) {
  CKG(attention_varlen_fwd(reinterpret_cast<const bf16*>(qkv), reinterpret_cast<bf16*>(o), lse2, seq_off, S, max_len, H, H * 64,
                           static_cast<cudaStream_t>(stream)));
  return 0;
}
int mudpt_attention_varlen_backward(const uint16_t* qkv, const uint16_t* d_o, const float* lse2, uint16_t* dqkv, const int32_t* seq_off,
                                    int32_t S, int32_t max_len, int32_t H, void* stream) {
  CKG(attention_varlen_bwd(reinterpret_cast<const bf16*>(qkv), reinterpret_cast<const bf16*>(d_o), lse2, reinterpret_cast<bf16*>(dqkv),
                           seq_off, S, max_len, H, H * 64, static_cast<cudaStream_t>(stream)));
  return 0;
}
// stream-K scratch of the handle-less GEMM entry points (tests, one stream at a time)
static GemmWorkspace* unit_workspace() {
  static GemmWorkspace ws;
  if (!ws.partials) {
    void *p = nullptr, *f = nullptr;
    if (cudaMalloc(&p, gemm_workspace_partial_bytes()) != cudaSuccess || cudaMalloc(&f, gemm_workspace_flag_bytes()) != cudaSuccess)
      return nullptr;
    cudaMemset(f, 0, gemm_workspace_flag_bytes());
    ws.partials = static_cast<float*>(p);
    ws.flags = static_cast<unsigned*>(f);
  }
  return &ws;
}

int mudpt_gemm_fused(const uint16_t* A, const uint16_t* B, int32_t M, int32_t N, int32_t K, const mudpt_gemm_epilogue* e,
                     void* stream) {
  if (!A || !B || !e) return fail(nullptr, "mudpt_gemm_fused: null argument");
  GemmEpilogue ep;
  ep.mode = e->mode; ep.ldc = e->ldc; ep.out0 = e->out0; ep.out1 = e->out1; ep.out2 = e->out2; ep.bias = e->bias;
  ep.resid = e->resid; ep.aux = e->aux; ep.ln_stats = reinterpret_cast<const float2*>(e->ln_stats); ep.ln_parts = e->ln_parts;
  ep.ln_width = e->ln_width; ep.ln_eps = e->ln_eps; ep.dot_parts = e->dot_parts; ep.colsum = e->colsum;
  ep.stats_out = reinterpret_cast<float2*>(e->stats_out); ep.splice_prompt = e->splice_prompt; ep.splice_row0 = e->splice_row0;
  ep.splice_n = e->splice_n; ep.splice_L = e->splice_L > 0 ? e->splice_L : 1; ep.x2 = e->x2;
  ep.dots = reinterpret_cast<const float2*>(e->dots); ep.sb = reinterpret_cast<const float2*>(e->sb);
  ep.dots_out = reinterpret_cast<float2*>(e->dots_out);
  gemm_set_stream_k(e->stream_k);
  const char* err = gemm_bf16_tn(reinterpret_cast<const bf16*>(A), K, reinterpret_cast<const bf16*>(B), K, ep, M, N, K,
                                 static_cast<cudaStream_t>(stream), e->stream_k != 0 ? unit_workspace() : nullptr);
  gemm_set_stream_k(-2);  // back to the process default
  if (err) return fail(nullptr, "%s", err);
  return 0;
}
int32_t mudpt_gemm_dots_span(int32_t N) { return gemm_dots_span(N); }
int mudpt_rowstats(const float* x, uint16_t* xb, float* stats, int32_t rows, int32_t width, void* stream) {
  CKG(rowstats(x, reinterpret_cast<bf16*>(xb), reinterpret_cast<float2*>(stats), rows, width, static_cast<cudaStream_t>(stream)));
  return 0;
}
int mudpt_fold_layernorm(const float* W, const float* gamma, const float* beta, const float* bias, uint16_t* Wl,
                         uint16_t* Wlt, float* bias_l, float* colsum, float* sb, int32_t N, int32_t K, void* stream) {
  CKG(fold_layernorm(W, gamma, beta, bias, reinterpret_cast<bf16*>(Wl), reinterpret_cast<bf16*>(Wlt), bias_l, colsum,
                     reinterpret_cast<float2*>(sb), N, K, static_cast<cudaStream_t>(stream)));
  return 0;
}
int mudpt_attention_backward_dots(const uint16_t* qkv, const uint16_t* o, const uint16_t* d_o, const float* lse2,
                                  float* dsum, uint16_t* dqkv, int32_t S, int32_t L, int32_t H, int32_t causal,
                                  const float* ln_sb, float* ln_dots, void* stream) {
  CKG(attention_bwd(reinterpret_cast<const bf16*>(qkv), reinterpret_cast<const bf16*>(o), reinterpret_cast<const bf16*>(d_o),
                    lse2, dsum, reinterpret_cast<bf16*>(dqkv), S, L, H, H * 64, causal != 0, static_cast<cudaStream_t>(stream),
                    reinterpret_cast<const float2*>(ln_sb), reinterpret_cast<float2*>(ln_dots)));
  return 0;
}
int mudpt_gemm_bf16(const uint16_t* A, const uint16_t* B, int32_t M, int32_t N, int32_t K, int32_t mode, void* out0,
                    void* out1, const float* bias, const float* resid, const void* aux, int32_t ldc, int32_t patch_np,
                    int32_t patch_L, void* stream) {
  GemmEpilogue ep;
  ep.mode = mode; ep.out0 = out0; ep.out1 = out1; ep.bias = bias; ep.resid = resid; ep.aux = aux; ep.ldc = ldc;
  ep.patch_np = patch_np > 0 ? patch_np : 1; ep.patch_L = patch_L > 0 ? patch_L : 1;
  CKG(gemm_bf16_tn(reinterpret_cast<const bf16*>(A), K, reinterpret_cast<const bf16*>(B), K, ep, M, N, K, static_cast<cudaStream_t>(stream),
                   unit_workspace()));
  return 0;
}
int mudpt_set_attention_tc(int32_t mode) {
  attention_tc_set_mode(mode);
  return 0;
}
int mudpt_im2col(const float* images, uint16_t* patches, int32_t B, int32_t R, int32_t patch, int32_t ld, void* stream) {
  CKG(im2col_bf16(images, reinterpret_cast<bf16*>(patches), B, R, patch, ld, static_cast<cudaStream_t>(stream)));
  return 0;
}
int mudpt_col2im(const float* patches, float* images, int32_t B, int32_t R, int32_t patch, int32_t ld, void* stream) {
  CKG(col2im_f32(patches, images, B, R, patch, ld, static_cast<cudaStream_t>(stream)));
  return 0;
}
int mudpt_pgd_linf_update(const float* dpatch, int32_t ld, float* x_adv, const float* x_clean, float* x_norm, int32_t B,
                          int32_t R, int32_t patch, const float* mean_host, const float* std_host, float eps, float alpha,
                          void* stream) {
  if (!dpatch || !x_adv || !x_clean || !x_norm || !mean_host || !std_host) return fail(nullptr, "mudpt_pgd_linf_update: null argument");
  CKG(pgd_linf_f32(dpatch, x_adv, x_clean, x_norm, B, R, patch, ld, pgd_params(mean_host, std_host, eps, alpha),
                   static_cast<cudaStream_t>(stream)));
  return 0;
}
int mudpt_peer_all_gather_rows(const void* peers_dev, int32_t world, int32_t n_total, int32_t width, float* out, void* stream) {
  if (!peers_dev || !out) return fail(nullptr, "mudpt_peer_all_gather_rows: null argument");
  CKG(peer_gather_rows(reinterpret_cast<const float* const*>(peers_dev), world, n_total, width, out, static_cast<cudaStream_t>(stream)));
  return 0;
}
int mudpt_peer_reduce_scatter_rows(const void* peers_dev, int32_t world, int32_t rank, int32_t n_total, int32_t width, float* out,
                                   void* stream) {
  if (!peers_dev || !out) return fail(nullptr, "mudpt_peer_reduce_scatter_rows: null argument");
  CKG(peer_reduce_scatter_rows(reinterpret_cast<const float* const*>(peers_dev), world, rank, n_total, width, out,
                               static_cast<cudaStream_t>(stream)));
  return 0;
}
int mudpt_cast_bf16(const float* in, uint16_t* out, int64_t numel, void* stream) {
  CKG(cast_to_bf16(in, reinterpret_cast<bf16*>(out), static_cast<size_t>(numel), static_cast<cudaStream_t>(stream)));
  return 0;
}

static PromptArgs to_prompt_args(const mudpt_prompt_args* p) {
  PromptArgs a;
  a.n = p->n; a.depth = p->depth; a.dt = p->dt; a.dv = p->dv; a.eps = p->eps;
  a.ctx = p->ctx; a.deep = p->deep; a.We = p->We; a.be = p->be; a.Wd = p->Wd; a.bd = p->bd; a.vctx = p->vctx; a.vdeep = p->vdeep;
  a.Wv = p->Wv; a.bv = p->bv; a.ln_g = p->ln_g; a.ln_b = p->ln_b; a.pos = p->pos; a.P_v = p->P_v; a.P_t = p->P_t; a.ln_in = p->ln_in;
  a.dP_v = p->dP_v; a.dP_t = p->dP_t; a.u = p->u; a.d_ctx = p->d_ctx; a.d_deep = p->d_deep; a.d_We = p->d_We; a.d_be = p->d_be;
  a.d_Wd = p->d_Wd; a.d_bd = p->d_bd; a.d_vctx = p->d_vctx; a.d_vdeep = p->d_vdeep; a.d_Wv = p->d_Wv; a.d_bv = p->d_bv;
  return a;
}
int mudpt_prompt_forward(const mudpt_prompt_args* args, void* stream) {
  if (!args) return fail(nullptr, "mudpt_prompt_forward: null argument");
  CKG(prompt_forward(to_prompt_args(args), static_cast<cudaStream_t>(stream)));
  return 0;
}
int mudpt_prompt_backward(const mudpt_prompt_args* args, void* stream) {
  if (!args) return fail(nullptr, "mudpt_prompt_backward: null argument");
  CKG(prompt_backward(to_prompt_args(args), static_cast<cudaStream_t>(stream)));
  return 0;
}

int mudpt_sgd_step(void* const* params, const void* const* grads, void* const* bufs, const int64_t* numel, int32_t n,
                   float lr, float momentum, float dampening, float weight_decay, int32_t nesterov, int32_t first_step,
                   void* stream) {
  if (!params || !grads || !numel || (momentum != 0.f && !bufs)) return fail(nullptr, "mudpt_sgd_step: null argument");
  CKG(sgd_step(params, grads, bufs, reinterpret_cast<const long long*>(numel), n, lr, momentum, dampening, weight_decay,
               nesterov != 0, first_step != 0, static_cast<cudaStream_t>(stream)));
  return 0;
}

int64_t mudpt_augment_workspace_bytes(const mudpt_image_desc* descs_host, int32_t n, int32_t out_h, int32_t out_w) {
  const char* e = nullptr;
  const long long b = augment_workspace_bytes(descs_host, n, out_h, out_w, &e);
  if (e) return fail(nullptr, "%s", e);
  return b;
}
int mudpt_augment_images(const mudpt_image_desc* descs, const mudpt_image_desc* descs_host, int32_t n, int32_t out_h,
                         int32_t out_w, const float* mean_host, const float* std_host, void* workspace,
                         int64_t workspace_bytes, float* out, void* stream) {
  CKG(augment_images(descs, descs_host, n, out_h, out_w, mean_host, std_host, workspace, workspace_bytes, out,
                     static_cast<cudaStream_t>(stream)));
  return 0;
}

int mudpt_debug_buffer(mudpt_handle* h, int32_t tower, const char* name, int32_t layer, void** ptr, int64_t* numel) {
  if (!h || !name || !ptr || !numel) return fail(h, "mudpt_debug_buffer: null argument");
  Tower& t = tower == MUDPT_TOWER_VISION ? h->vis : h->txt;
  if (t.cap_rows == 0) return fail(h, "mudpt_debug_buffer: tower has no workspace yet");
  const int64_t rows = t.rows;
  if (!strcmp(name, "dx")) { *ptr = t.dx; *numel = rows * t.d; return 0; }
  if (!strcmp(name, "x_in")) {
    if (layer < 0 || layer > t.layers) return fail(h, "mudpt_debug_buffer: layer out of range");
    *ptr = t.x_in[layer]; *numel = rows * t.d; return 0;
  }
  if (layer < 0 || layer >= t.layers) return fail(h, "mudpt_debug_buffer: layer out of range");
  if (!strcmp(name, "x_mid")) { *ptr = t.x_mid[layer]; *numel = rows * t.d; return 0; }
  if (!strcmp(name, "qkv")) { *ptr = t.qkv[layer]; *numel = rows * 3 * t.d; return 0; }
  if (!strcmp(name, "o")) { *ptr = t.o[layer]; *numel = rows * t.d; return 0; }
  if (!strcmp(name, "h")) { *ptr = t.h[layer]; *numel = rows * 4 * t.d; return 0; }
  if (!strcmp(name, "lse")) { *ptr = t.lse[layer]; *numel = rows * t.H; return 0; }
  return fail(h, "mudpt_debug_buffer: unknown buffer %s", name);
}

int mudpt_profile_begin(mudpt_handle* h) {
  if (!h) return fail(h, "null handle");
  for (ProfRec& r : h->prof.recs) { h->prof.pool.push_back(r.e0); h->prof.pool.push_back(r.e1); }
  h->prof.recs.clear();
  h->prof.on = true;
  return 0;
}

// out[cat*4 + {0,1,2,3}] = {total ms, launches, algorithmic FLOPs, algorithmic bytes}; cat order:
// gemm (other), attn_fwd, attn_bwd, ln_fwd, ln_bwd, splice, head, stem, gemm_qkv, gemm_out, gemm_fc, gemm_proj,
// gemm_dproj, gemm_dfc, gemm_dout, gemm_dqkv.  Blocks until the recorded work is done.
// With peaks (TFLOP/s, GB/s) > 0 a fifth value per class: the sum over its launches of the time the launch would take at
// the bound that applies to it, max(FLOPs / peak, algorithmic bytes / hbm) -- per launch, so a class that mixes
// tensor-bound and HBM-bound launches is measured against the right one each time.
static int profile_collect(mudpt_handle* h, double* out_host, int stride, double peak_tflops, double hbm_gbs) {
  h->prof.on = false;
  for (int i = 0; i < PC_COUNT * stride; ++i) out_host[i] = 0.0;
  for (ProfRec& r : h->prof.recs) {
    CUDA_OK(h, cudaEventSynchronize(r.e1));
    float ms = 0.f;
    CUDA_OK(h, cudaEventElapsedTime(&ms, r.e0, r.e1));
    out_host[r.cat * stride + 0] += ms;
    out_host[r.cat * stride + 1] += 1.0;
    out_host[r.cat * stride + 2] += r.flops;
    out_host[r.cat * stride + 3] += r.bytes;
    if (stride > 4 && peak_tflops > 0 && hbm_gbs > 0) {
      const double t_fl = r.flops / (peak_tflops * 1e12), t_by = r.bytes / (hbm_gbs * 1e9);
      out_host[r.cat * stride + 4] += 1e3 * (t_fl > t_by ? t_fl : t_by);
    }
    h->prof.pool.push_back(r.e0);
    h->prof.pool.push_back(r.e1);
  }
  h->prof.recs.clear();
  return 0;
}

int mudpt_profile_end(mudpt_handle* h, double* out_host, int32_t n_out) {
  if (!h || !out_host) return fail(h, "mudpt_profile_end: null argument");
  if (n_out < PC_COUNT * 4) return fail(h, "mudpt_profile_end: output too small");
  return profile_collect(h, out_host, 4, 0.0, 0.0);
}

int mudpt_profile_end_bound(mudpt_handle* h, double* out_host, int32_t n_out, double peak_tflops, double hbm_gbs) {
  if (!h || !out_host) return fail(h, "mudpt_profile_end_bound: null argument");
  if (n_out < PC_COUNT * 5) return fail(h, "mudpt_profile_end_bound: output too small");
  return profile_collect(h, out_host, 5, peak_tflops, hbm_gbs);
}

int64_t mudpt_launch_count(mudpt_handle* h) { return h ? g_launch_counter.load() - h->launches_at_create : 0; }

#ifdef MUDPT_BRINGUP
int mudpt_bringup_simt_gemm(int on) { gemm_set_bringup_simt(on != 0); return 0; }
#endif

}  // extern "C"
