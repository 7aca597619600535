// Internal interface of the attention kernels (see attention.cu).
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>

namespace mudpt {
// qkv [S*L, 3d] bf16 (row = sequence*L + token; head h owns columns [64h, 64h+64) of each third),
// o [S*L, d] bf16, lse2 [S, H, L] fp32 = log2-domain log-sum-exp of the scaled scores.
const char* attention_fwd(const __nv_bfloat16* qkv, __nv_bfloat16* o, float* lse2, int S, int L, int H, int d,
                          bool causal, cudaStream_t stream);
// dsum [S, H, L] fp32 scratch (rowsum(dO*O)), dqkv [S*L, 3d] bf16 out.
// ln_dots != null (fused LayerNorm backward of the in-proj, gemm.h EPI_LN_BWD): also ln_dots[row, which*H + h] =
// (sum_c g_c colsum_c, sum_c g_c (y_c - b'_c)) over the 64 columns of head h of dq / dk / dv (which = 0 / 1 / 2),
// with ln_sb [3d] = (colsum, b') of the LN-folded in-proj and y = the saved qkv.
const char* attention_bwd(const __nv_bfloat16* qkv, const __nv_bfloat16* o, const __nv_bfloat16* d_o, const float* lse2,
                          float* dsum, __nv_bfloat16* dqkv, int S, int L, int H, int d, bool causal, cudaStream_t stream,
                          const float2* ln_sb = nullptr, float2* ln_dots = nullptr);
// Causal attention over packed variable-length sequences (the ragged text tower): sequence s occupies rows [seq_off[s], seq_off[s+1]) of qkv / o /
// dqkv (seq_off: device int32 [S+1], lengths 1..attention_varlen_max_len(), max_len = the longest), lse2 [seq_off[S] * H]
// holds sequence s's [H, len_s] block at seq_off[s] * H.  Warp-MMA kernels only (the tcgen05 tensor maps assume one L).
int attention_varlen_max_len();
const char* attention_varlen_fwd(const __nv_bfloat16* qkv, __nv_bfloat16* o, float* lse2, const int* seq_off, int S, int max_len,
                                 int H, int d, cudaStream_t stream);
const char* attention_varlen_bwd(const __nv_bfloat16* qkv, const __nv_bfloat16* d_o, const float* lse2, __nv_bfloat16* dqkv,
                                 const int* seq_off, int S, int max_len, int H, int d, cudaStream_t stream,
                                 const float2* ln_sb = nullptr, float2* ln_dots = nullptr);
// tcgen05 / TMEM path (attention_tc.cu); attention_fwd dispatches to it when eligible.
// mode: 0 = never, 1 = default (forward: non-causal sequences of 129..256 tokens; backward: 65..80 and 129..256 tokens),
//       2 = every length the kernels support
void attention_tc_set_mode(int mode);
bool attention_tc_fwd_eligible(int L, bool causal);
bool attention_tc_bwd_eligible(int L, bool causal);
const char* attention_tc_bwd(const __nv_bfloat16* qkv, const __nv_bfloat16* o, const __nv_bfloat16* d_o, const float* lse2,
                             float* dsum, __nv_bfloat16* dqkv, int S, int L, int H, int d, bool causal, cudaStream_t stream);
const char* attention_tc_fwd(const __nv_bfloat16* qkv, __nv_bfloat16* o, float* lse2, int S, int L, int H, int d, bool causal,
                             cudaStream_t stream);
}  // namespace mudpt
