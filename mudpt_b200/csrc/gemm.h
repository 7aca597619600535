// Internal interface of the tcgen05 GEMM (see gemm.cu).
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stddef.h>

namespace mudpt {

enum GemmEpilogueMode {
  EPI_BF16 = 0,       // out0(bf16) = acc (+ bias)                          QKV in-proj; dgrad of out-proj
  EPI_F32 = 1,        // out0(f32)  = acc (+ bias)
  EPI_RESID_F32 = 2,  // out0(f32)  = acc + bias + resid(f32)               out-proj / c_proj + residual
  EPI_GELU = 3,       // out0(bf16) = h = acc + bias; out1(bf16) = QuickGELU(h)   c_fc
  EPI_GELU_BWD = 4,   // out0(bf16) = acc * QuickGELU'(aux(bf16))           dgrad of c_proj
  EPI_PATCH = 5,      // out0(f32)[img*L + 1 + p] = acc + resid[1 + p]       conv1 patch embedding
  // ---- LayerNorm folded into the GEMMs (clip/model.py:164-170, 299-300).  The LN input row x is kept as a bf16
  // copy (the A operand) plus per-row partial statistics; gamma is folded into the weight (W' = W diag(gamma)),
  // beta into the bias (b' = b + W beta), and the mean enters as a rank-1 correction with colsum[c] = sum_k W'[c,k]:
  //     LN(x) W^T + b  =  rstd * (x W'^T - mean * colsum) + b'
  EPI_LN_BF16 = 7,      // out0(bf16) = rstd*(acc - mean*colsum) + bias                       LN1 + QKV in-proj
  EPI_LN_GELU = 8,      // out0(bf16) = h = (same); out1(bf16) = QuickGELU(h)                 LN2 + c_fc
  EPI_RESID_STATS = 9,  // out0(f32) = x = acc + bias + resid; out2(bf16) = x; stats_out = per-row partial (sum, M2) of x
                        // per 64 columns; rows (r % splice_L) in [splice_row0, +splice_n) take splice_prompt instead
                        // (the deep-prompt splice of the NEXT block, clip/model.py:281-297, bit-exact copy)
  EPI_LN_BWD = 10,      // LN dgrad fused into the dgrad GEMM through the folded weight (acc = dy*gamma = g):
                        //   out0(f32) = resid + rstd*(g - c1 - xhat*c2), out2(bf16) = same,  xhat = (x2 - mean)*rstd,
                        //   c1 = mean_k(g), c2 = mean_k(g*xhat) computed by the PRODUCER of the GEMM's A operand from
                        //   c1 = (1/d) sum_c dout_c colsum_c,  c2 = (1/d) sum_c dout_c (y_c - b'_c)   (y = saved LN-GEMM output)
  EPI_GELU_BWD_DOTS = 11,  // EPI_GELU_BWD + dots_out[row][col/span] = partial (sum dh*colsum, sum dh*(h - b')) for the above
  // ---- forward-only c_fc (no backward will read the pre-activation h): one bf16 output, bitwise out1 of modes 3 / 8
  EPI_GELU_ONLY = 12,     // out0(bf16) = QuickGELU(acc + bias)
  EPI_LN_GELU_ONLY = 13,  // out0(bf16) = QuickGELU(rstd*(acc - mean*colsum) + bias)
};

struct GemmEpilogue {
  int mode = EPI_BF16;
  void* out0 = nullptr;
  void* out1 = nullptr;
  const float* bias = nullptr;   // [N] or null
  const float* resid = nullptr;  // EPI_RESID_*: [M, ldc] f32; EPI_LN_BWD: residual gradient; EPI_PATCH: positional embedding [np+1, ldc]
  const void* aux = nullptr;     // EPI_GELU_BWD*: h [M, ldc] bf16
  int ldc = 0;                   // leading dimension (elements) of out0/out1/out2/resid/aux/x2
  int patch_np = 1;              // EPI_PATCH: patches per image
  int patch_L = 1;               // EPI_PATCH: tokens per image (np + 1 + n_ctx)
  // ---- fused LayerNorm
  const float2* ln_stats = nullptr;  // [M, ln_parts] partial (sum, M2) of the LN input row, one per 64 columns
  int ln_parts = 0;
  int ln_width = 0;                  // width of the LN input row
  float ln_eps = 1e-5f;
  const float* colsum = nullptr;     // EPI_LN_BF16 / EPI_LN_GELU: [N]
  void* out2 = nullptr;              // EPI_RESID_STATS / EPI_LN_BWD: bf16 copy of out0
  float2* stats_out = nullptr;       // EPI_RESID_STATS: [M, N/64]
  const float* splice_prompt = nullptr;  // EPI_RESID_STATS: [splice_n, N] fp32 or null
  int splice_row0 = 0, splice_n = 0, splice_L = 1;
  const void* x2 = nullptr;          // EPI_LN_BWD: bf16 copy of the LN input x [M, ldc]
  const float2* dots = nullptr;      // EPI_LN_BWD: [M, dot_parts] partial (sum dout*colsum, sum dout*(y - b'))
  int dot_parts = 0;
  const float2* sb = nullptr;        // EPI_GELU_BWD_DOTS: [N] (colsum_c, b'_c) of the LN-GEMM whose output is aux
  float2* dots_out = nullptr;        // EPI_GELU_BWD_DOTS: [M, N / gemm_dots_span(N)]
};

// Stream-K scratch of one stream: fp32 partial accumulator tiles that travel through L2 between CTAs of the same
// launch + their ready flags.  Launches that share a workspace must be stream-ordered.
struct GemmWorkspace {
  float* partials = nullptr;
  unsigned* flags = nullptr;  // zero-initialised once; every launch leaves them zero
};
size_t gemm_workspace_partial_bytes();
size_t gemm_workspace_flag_bytes();

// columns covered by one partial of EPI_GELU_BWD_DOTS for an N-column output
int gemm_dots_span(int N);

// C = A[M,K] * B[N,K]^T with the fused epilogue. Returns nullptr on success, else a static
// error string. Asynchronous on `stream`.  ws == nullptr: whole-tile scheduling only (no stream-K).
const char* gemm_bf16_tn(const __nv_bfloat16* A, int lda, const __nv_bfloat16* B, int ldb, const GemmEpilogue& ep,
                         int M, int N, int K, cudaStream_t stream, const GemmWorkspace* ws = nullptr);
// cached 3D TMA descriptor (bf16, 64-column boxes of box1 rows, 128B swizzle) for the attention kernels
const char* tensor_map_3d_bf16(const void* ptr, int d0, int d1, int d2, long long stride1, long long stride2, int box1,
                               CUtensorMap* out);
void gemm_clear_tensor_map_cache();
// 0 = whole tiles only, 1 = always cut, -1 = cost model, -2 = back to the process default (env MUDPT_GEMM_SK)
void gemm_set_stream_k(int mode);
#ifdef MUDPT_BRINGUP
void gemm_set_bringup_simt(bool on);
#endif

}  // namespace mudpt
