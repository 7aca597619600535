// Internal interface of the row kernels (see rowops.cu). All return nullptr on success.
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stddef.h>

namespace mudpt {
const char* layernorm_fwd(const float* x, const float* gamma, const float* beta, void* out, bool out_bf16, int M, int d,
                          float eps, cudaStream_t stream);
// LayerNorm with the deep-prompt splice of the block done in the same pass: rows (row % L) in [row0, row0 + n) are first
// overwritten with prompt[row % L - row0] (verbatim).  tok_pos != null (packed variable-length sequences, [M] device
// int32): tok_pos[row] is the position of the row in its sequence and takes the place of row % L (L is then unused).
const char* layernorm_fwd_splice(float* x, const float* prompt, int L, int row0, int n, const float* gamma, const float* beta,
                                 void* out, bool out_bf16, int M, int d, float eps, cudaStream_t stream, const int* tok_pos = nullptr);
// x: fp32 rows, or (stats != nullptr) their bf16 copy + per-64-column partial statistics (fused-LayerNorm towers)
const char* layernorm_bwd(const void* dy, bool dy_bf16, const void* x, const float2* stats, const float* gamma, const float* resid,
                          float* dx, __nv_bfloat16* dx_bf16, int M, int d, float eps, cudaStream_t stream);
// The same with the gradient stream kept in bf16: resid is the fp32 stream or (resid_bf16) its bf16 copy, which may alias
// dx_bf16; dx (fp32) may be null; win_n >= 0 writes fp32 rows only where (row % win_L) is in [win_row0, win_row0 + win_n)
// (the deep-prompt rows the splice backward sums), win_n < 0 writes every row.  win_pos != null: the position of row r is
// win_pos[r] (packed variable-length sequences) instead of r % win_L.
const char* layernorm_bwd_stream(const void* dy, bool dy_bf16, const void* x, const float2* stats, const float* gamma,
                                 const void* resid, bool resid_bf16, float* dx, __nv_bfloat16* dx_bf16, int M, int d, float eps,
                                 int win_L, int win_row0, int win_n, cudaStream_t stream, const int* win_pos = nullptr);
// LayerNorm dgrad of `per` rows out of every sequence of L rows, compacted: out[r] (bf16) from dy / x (fp32) at row
// (r / per) * L + row0 + r % per, r < M; no residual (the vision stem's ln_pre on the patch rows)
const char* layernorm_bwd_rows(const float* dy, const float* x, const float* gamma, __nv_bfloat16* out, int M, int d, float eps,
                               int per, int L, int row0, cudaStream_t stream);
const char* splice_fwd(float* x, const float* prompt, int S, int L, int row0, int n, int d, cudaStream_t stream);
size_t splice_bwd_workspace_floats(int n, int d);  // must be zero-initialised once (it ends with the kernel's tickets)
// seq_off != null: packed variable-length sequences ([S+1] device int32), sequence s's prompt rows start at seq_off[s] + row0
const char* splice_bwd(float* dx, __nv_bfloat16* dx_bf16, float* dprompt, float* workspace, int S, int L, int row0, int n,
                       int d, bool zero_rows, cudaStream_t stream, const int* seq_off = nullptr);
// fused-LayerNorm plumbing (see rowops.cu): bf16 copy + per-64-column partial statistics of fp32 rows
const char* rowstats(const float* x, __nv_bfloat16* xb, float2* stats, int M, int d, cudaStream_t stream);
const char* splice_fwd_stats(float* x, __nv_bfloat16* xb, float2* stats, const float* prompt, int S, int L, int row0, int n,
                             int d, cudaStream_t stream);
const char* fold_layernorm(const float* W, const float* gamma, const float* beta, const float* bias, __nv_bfloat16* Wl,
                           __nv_bfloat16* Wlt, float* bias_l, float* colsum, float2* sb, int N, int K, cudaStream_t stream);
// rows / row stride L of the three below: row s * L + rows[s] (L = 0: rows[] are absolute row indices)
const char* scatter_rows(const float* src, const int* rows, int S, int L, float* x, __nv_bfloat16* xb, int d, bool accumulate,
                         cudaStream_t stream);
const char* scatter_rows_bf16(const __nv_bfloat16* src, const int* rows, int S, int L, __nv_bfloat16* x, int d, cudaStream_t stream);
const char* gather_rows(const float* src_f, const __nv_bfloat16* src_b, const int* rows, int S, int L, float* dst_f,
                        __nv_bfloat16* dst_b, int d, cudaStream_t stream);
const char* im2col_bf16(const float* img, __nv_bfloat16* out, int B, int R, int p, int ldo, cudaStream_t stream);
// inverse of im2col_bf16's index map, fp32 (patch rows of row stride ldi >= 3*p*p -> [B, 3, R, R], every element written once)
const char* col2im_f32(const float* cols, float* img, int B, int R, int p, int ldi, cudaStream_t stream);
// One l-inf PGD step in pixel space (include/mudpt_b200.h, mudpt_pgd_linf_update): the patch gradient cols (col2im_f32's
// layout, dL/d x_norm) -> x_adv [B, 3, R, R] in place and x_norm = (x_adv - mean) / std, IEEE fp32
struct PgdParams { float mean[3], std[3], eps, alpha; };
const char* pgd_linf_check(const PgdParams& prm);  // nullptr, or why the parameters are rejected
const char* pgd_linf_f32(const float* cols, float* x_adv, const float* x_clean, float* x_norm, int B, int R, int p, int ldi,
                         const PgdParams& prm, cudaStream_t stream);
const char* write_cls_rows(float* x, const float* cls, const float* pos, int S, int L, int d, cudaStream_t stream);
// seq_off != null: packed variable-length output rows (L = the longest sequence)
const char* add_positional(float* x0, const float* emb, const float* pos, int S, int L, int Lsrc, int d, cudaStream_t stream,
                           const int* seq_off = nullptr);
// packed variable-length rows [seq_off[S], d] -> [S, L, d], zero past each sequence's length
const char* unpack_rows(const float* x, const int* seq_off, int S, int L, int d, float* out, cudaStream_t stream);
const char* cast_to_bf16(const float* in, __nv_bfloat16* out, size_t n, cudaStream_t stream);
const char* transpose_cast_bf16(const float* in, __nv_bfloat16* out, int rows, int cols, cudaStream_t stream);
}  // namespace mudpt
