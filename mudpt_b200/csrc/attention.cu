// Flash-style multi-head self-attention, forward and dgrad, for the short fixed sequences of
// the CLIP towers: vision L = 197 + n_ctx (no mask), text L <= 77 (causal mask,
// clip/model.py:810-816), head width 64.  Replaces the scaled_dot_product_attention call
// inside nn.MultiheadAttention (clip/model.py:271-273) and its autograd backward.
//
// Whole K/V (resp. Q/dO) of one (sequence, head) fits in shared memory, so each CTA owns a
// block of 16*nwarps rows and every warp is the sole owner of 16 of them: no atomics and no
// cross-warp reductions anywhere.
//   forward : S = QK^T, online softmax, O = PV, LSE (log2 domain) saved
//   dQ pass : rows = queries.  P recomputed from LSE, dP = dO V^T, dS = P*(dP - D), dQ = dS K
//   dKV pass: rows = keys.     P^T, dV = P^T dO, dP^T = V dO^T, dS^T, dK = dS^T Q
// With L <= ~260 and head width 64 the kernel is bound by its Q/K/V/O traffic, not by MMA
// rate (SURVEY.md appendix C: ~100 FLOP/B vision, ~38 text), so the products run on warp-level
// mma.sync (HMMA) tiles fed by ldmatrix from XOR-swizzled shared memory.  The backward passes
// work on 32-column chunks and re-read their A fragments from shared memory instead of pinning
// them in registers: that keeps them under ~128 registers so 4 CTAs fit per SM.
#include "attention.h"

#include <cstdlib>
#include <type_traits>

#include "common.cuh"
#include "launch_count.h"

namespace mudpt {

static constexpr int DH = 64;         // head width (all CLIP ViT towers)
static constexpr int ROW_BYTES = 128; // 64 bf16

__device__ __forceinline__ uint32_t swz(int row, int chunk) {
  return static_cast<uint32_t>(row * ROW_BYTES + ((chunk ^ (row & 7)) << 4));
}

// Load `nrows` rows x 64 bf16 columns into a swizzled smem tile; global row = row_begin + r,
// rows >= row_limit are zero-filled.
__device__ __forceinline__ void load_tile(uint32_t tile, const bf16* g, int ld, int row_begin, int row_limit, int nrows) {
  const int c = threadIdx.x & 7, r0 = threadIdx.x >> 3, rstep = blockDim.x >> 3;
  if ((rstep & 7) == 0) {
    // CTAs of >= 64 threads: a thread's rows are 8k apart, so its swizzled 16 B slot is loop-invariant
    // and both addresses advance by constants (the load loop was ~15 % of all issued instructions)
    uint32_t dst = tile + static_cast<uint32_t>(r0 * ROW_BYTES + ((c ^ (r0 & 7)) << 4));
    const bf16* src = g + static_cast<size_t>(row_begin + r0) * ld + c * 8;
    const size_t sstep = static_cast<size_t>(rstep) * ld;
    for (int r = r0; r < nrows; r += rstep) {
      const bool ok = row_begin + r < row_limit;
      cp_async16(dst, ok ? src : g, ok);
      dst += rstep * ROW_BYTES;
      src += sstep;
    }
  } else {
    for (int r = r0; r < nrows; r += rstep) {
      const int gr = row_begin + r;
      const bool ok = gr < row_limit;
      cp_async16(tile + swz(r, c), g + static_cast<size_t>(ok ? gr : 0) * ld + c * 8, ok);
    }
  }
}

__device__ __forceinline__ void load_a_frag(uint32_t (&a)[4], uint32_t tile, int row0, int ks, int lane) {
  ldsm_x4(tile + swz(row0 + (lane & 15), ks * 2 + (lane >> 4)), a[0], a[1], a[2], a[3]);
}

// acc(16 x 16*NG) = A(16 rows of tileA at row0, 64 dh) * T[c0 .. c0+16*NG)^T -- contraction over the
// head dimension.  Only 16-column groups g in [g_lo, g_hi) are computed, the rest stay 0.
// k-step outermost: consecutive MMAs hit different accumulators (no back-to-back dependency).
template <int NG>
__device__ __forceinline__ void mma_rows_x_cols(float (&acc)[2 * NG][4], uint32_t tileA, int row0, uint32_t tile, int c0,
                                                int g_lo, int g_hi, int lane) {
#pragma unroll
  for (int ks = 0; ks < 4; ++ks) {
    uint32_t a[4];
    load_a_frag(a, tileA, row0, ks, lane);
#pragma unroll
    for (int g = 0; g < NG; ++g) {
      if (g >= g_lo && g < g_hi) {
        uint32_t b0, b1, b2, b3;
        ldsm_x4(tile + swz(c0 + g * 16 + (lane & 7) + ((lane >> 4) << 3), ks * 2 + ((lane >> 3) & 1)), b0, b1, b2, b3);
        mma16816(acc[2 * g], a, b0, b1);
        mma16816(acc[2 * g + 1], a, b2, b3);
      }
    }
  }
}

// out(16 x 64dh) += P(16 x 16*NG) * T[c0 .. c0+16*NG)  -- contraction over the tile rows; P comes
// straight from accumulator registers (converted to bf16 A fragments).
template <int NG>
__device__ __forceinline__ void mma_p_x_tile(float (&out)[8][4], const float (&p)[2 * NG][4], uint32_t tile, int c0,
                                             int g_lo, int g_hi, int lane) {
#pragma unroll
  for (int g = 0; g < NG; ++g) {
    if (g >= g_lo && g < g_hi) {
      uint32_t a[4];
      a[0] = pack_bf16(p[2 * g][0], p[2 * g][1]);
      a[1] = pack_bf16(p[2 * g][2], p[2 * g][3]);
      a[2] = pack_bf16(p[2 * g + 1][0], p[2 * g + 1][1]);
      a[3] = pack_bf16(p[2 * g + 1][2], p[2 * g + 1][3]);
#pragma unroll
      for (int dp = 0; dp < 4; ++dp) {
        uint32_t b0, b1, b2, b3;
        ldsm_x4_t(tile + swz(c0 + g * 16 + (lane & 7) + (((lane >> 3) & 1) << 3), dp * 2 + (lane >> 4)), b0, b1, b2, b3);
        mma16816(out[2 * dp], a, b0, b1);
        mma16816(out[2 * dp + 1], a, b2, b3);
      }
    }
  }
}

// Optional by-product of the backward stores (fused LayerNorm backward, gemm.h EPI_LN_BWD): the row dots of the
// stored gradient slice with the column sums of the LN-folded in-proj weight and with (y - b'), y = the saved
// forward value of the same slice (q, k or v).  One partial per (row, slice): dots[row * parts + part].
struct RowDots {
  const float2* sb = nullptr;  // (colsum, b') of the slice's 64 columns
  const bf16* y = nullptr;     // forward values, same indexing as the gradient slice
  float2* out = nullptr;       // null: no dots
  int parts = 0, part = 0;
};

// Write a warp's 16 x 64 fp32 accumulator (scaled) as bf16 to global rows, staged through the
// warp's own (no longer needed) 16 smem rows so the global stores are 16 B and coalesced.
__device__ __forceinline__ void store_rows_bf16(const float (&acc)[8][4], float scale0, float scale1, uint8_t* smem_gen,
                                                uint32_t tile_off, int row0, bf16* g, int ld, int grow0, int row_limit,
                                                int lane, const RowDots dots = RowDots()) {
  __syncwarp();
#pragma unroll
  for (int nt = 0; nt < 8; ++nt) {
    const int r_lo = row0 + (lane >> 2), r_hi = r_lo + 8;
    const int within = (lane & 3) * 4;  // byte offset of this thread's column pair inside the 16 B chunk nt
    *reinterpret_cast<uint32_t*>(smem_gen + tile_off + swz(r_lo, nt) + within) = pack_bf16(acc[nt][0] * scale0, acc[nt][1] * scale0);
    *reinterpret_cast<uint32_t*>(smem_gen + tile_off + swz(r_hi, nt) + within) = pack_bf16(acc[nt][2] * scale1, acc[nt][3] * scale1);
  }
  __syncwarp();
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int idx = i * 32 + lane;
    const int r = idx >> 3, c = idx & 7;
    const int gr = grow0 + r;
    const bool valid = gr < row_limit;
    uint4 v = *reinterpret_cast<const uint4*>(smem_gen + tile_off + swz(row0 + r, c));
    if (valid) *reinterpret_cast<uint4*>(g + static_cast<size_t>(gr) * ld + c * 8) = v;
    if (dots.out != nullptr) {  // (warp-uniform) 8 lanes share a row: the rounded values that the dgrad GEMM will read
      float d1 = 0.f, d2 = 0.f;
      if (valid) {
        const uint4 y = *reinterpret_cast<const uint4*>(dots.y + static_cast<size_t>(gr) * ld + c * 8);
        const uint32_t vw[4] = {v.x, v.y, v.z, v.w}, yw[4] = {y.x, y.y, y.z, y.w};
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const float4 sb2 = __ldg(reinterpret_cast<const float4*>(dots.sb + c * 8 + 2 * q));  // (cs, b', cs, b') of 2 columns
          const float2 gv = unpack_bf16(vw[q]), yv = unpack_bf16(yw[q]);
          d1 += gv.x * sb2.x + gv.y * sb2.z;
          d2 += gv.x * (yv.x - sb2.y) + gv.y * (yv.y - sb2.w);
        }
      }
#pragma unroll
      for (int o = 4; o > 0; o >>= 1) {
        d1 += __shfl_xor_sync(0xffffffffu, d1, o);
        d2 += __shfl_xor_sync(0xffffffffu, d2, o);
      }
      if (valid && c == 0) dots.out[static_cast<size_t>(gr) * dots.parts + dots.part] = make_float2(d1, d2);
    }
  }
}

template <int N>
__device__ __forceinline__ void zero_acc(float (&a)[N][4]) {
#pragma unroll
  for (int i = 0; i < N; ++i) a[i][0] = a[i][1] = a[i][2] = a[i][3] = 0.f;
}

// One 64-key chunk of the online-softmax forward for a warp's 16 query rows.
// FULL: all four 16-key groups are visible to every row (no guards, no mask).
template <bool CAUSAL, bool FULL>
__device__ __forceinline__ void fwd_chunk(float (&oacc)[8][4], float (&m_run)[2], float (&l_run)[2], uint32_t sQ, uint32_t sK,
                                          uint32_t sV, int row0, int c0, int g_hi, int L, const int (&qrow)[2],
                                          float scale_log2e, int lane) {
  float sacc[8][4];
  zero_acc(sacc);
  mma_rows_x_cols<4>(sacc, sQ, row0, sK, c0, 0, FULL ? 4 : g_hi, lane);
  float mx[2] = {-INFINITY, -INFINITY};
#pragma unroll
  for (int nt = 0; nt < 8; ++nt) {
    if (FULL || nt < 2 * g_hi) {
      if constexpr (!FULL) {
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const int col = c0 + nt * 8 + (lane & 3) * 2 + (e & 1);
          const bool ok = col < L && (!CAUSAL || col <= qrow[e >> 1]);
          sacc[nt][e] = ok ? sacc[nt][e] : -INFINITY;
        }
      }
      mx[0] = fmaxf(mx[0], fmaxf(sacc[nt][0], sacc[nt][1]));
      mx[1] = fmaxf(mx[1], fmaxf(sacc[nt][2], sacc[nt][3]));
    }
  }
  f32x2 alpha2[2], nm2[2];
#pragma unroll
  for (int r = 0; r < 2; ++r) {
    mx[r] = fmaxf(mx[r], __shfl_xor_sync(0xffffffffu, mx[r], 1));
    mx[r] = fmaxf(mx[r], __shfl_xor_sync(0xffffffffu, mx[r], 2));
    const float m_new = fmaxf(m_run[r], mx[r] * scale_log2e);  // running max of the scaled scores (log2 domain)
    const float m_use = (m_new == -INFINITY) ? 0.f : m_new;
    const float alpha = exp2f(m_run[r] - m_use);  // m_run = -inf -> 0
    m_run[r] = m_new;
    l_run[r] *= alpha;
    alpha2[r] = f2_pack(alpha, alpha);
    nm2[r] = f2_pack(-m_use, -m_use);
  }
  const f32x2 sc2 = f2_pack(scale_log2e, scale_log2e);
  f32x2 ls[2] = {f2_pack(0.f, 0.f), f2_pack(0.f, 0.f)};
#pragma unroll
  for (int nt = 0; nt < 8; ++nt) {
    if (FULL || nt < 2 * g_hi) {
#pragma unroll
      for (int r = 0; r < 2; ++r) {
        float a, b;
        f2_unpack(f2_fma(f2_pack(sacc[nt][2 * r], sacc[nt][2 * r + 1]), sc2, nm2[r]), a, b);
        a = exp2f(a);
        b = exp2f(b);
        sacc[nt][2 * r] = a;
        sacc[nt][2 * r + 1] = b;
        ls[r] = f2_add(ls[r], f2_pack(a, b));
      }
    }
#pragma unroll
    for (int r = 0; r < 2; ++r) {
      float a, b;
      f2_unpack(f2_mul(f2_pack(oacc[nt][2 * r], oacc[nt][2 * r + 1]), alpha2[r]), a, b);
      oacc[nt][2 * r] = a;
      oacc[nt][2 * r + 1] = b;
    }
  }
#pragma unroll
  for (int r = 0; r < 2; ++r) {
    float a, b;
    f2_unpack(ls[r], a, b);
    l_run[r] += a + b;
  }
  mma_p_x_tile<4>(oacc, sacc, sV, c0, 0, FULL ? 4 : g_hi, lane);
}

// ---------------------------------------------------------------------------------------
// forward
// ---------------------------------------------------------------------------------------
template <bool CAUSAL>
__global__ void __launch_bounds__(256) attn_fwd_kernel(const bf16* __restrict__ qkv, bf16* __restrict__ o,
                                                       float* __restrict__ lse2, int L, int H, int d, float scale_log2e) {
  extern __shared__ __align__(128) uint8_t smem[];
  const int nwarps = blockDim.x >> 5, BQ = nwarps * 16;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int sh = blockIdx.y, s = sh / H, h = sh - s * H;
  const int q0 = blockIdx.x * BQ;
  const int kv_len = CAUSAL ? min(L, q0 + BQ) : L;
  const int kv_rows = (kv_len + 15) & ~15;
  const int Lp = (L + 15) & ~15;
  const uint32_t sQ = smem_u32(smem), sK = sQ + BQ * ROW_BYTES, sV = sK + Lp * ROW_BYTES;
  const int ld = 3 * d;
  const bf16* base = qkv + static_cast<size_t>(s) * L * ld + h * DH;
  pdl_wait();
  pdl_trigger();
  load_tile(sQ, base, ld, q0, L, BQ);
  load_tile(sK, base + d, ld, 0, L, kv_rows);
  load_tile(sV, base + 2 * d, ld, 0, L, kv_rows);
  cp_async_commit();
  cp_async_wait_all();
  __syncthreads();

  const int row0 = warp * 16;
  if (q0 + row0 >= L) return;  // whole warp out of range (no further block-wide syncs below)
  float oacc[8][4];
  zero_acc(oacc);
  float m_run[2] = {-INFINITY, -INFINITY}, l_run[2] = {0.f, 0.f};
  const int qrow[2] = {q0 + row0 + (lane >> 2), q0 + row0 + (lane >> 2) + 8};
  const int kv_warp = CAUSAL ? min(kv_len, q0 + row0 + 16) : kv_len;  // keys this warp can see

  for (int c0 = 0; c0 < kv_warp; c0 += 64) {
    const int g_hi = min(4, (kv_warp - c0 + 15) >> 4);
    // the kernel is instruction-bound (ncu: 3 % of the issued instructions are MMAs): chunks that lie
    // entirely inside the valid / causal region take a straight-line path without per-group guards or
    // mask arithmetic (3 of the 4 chunks of a 199-token vision sequence)
    const bool need_mask = (c0 + 64 > L) || (CAUSAL && c0 + 63 > q0 + row0);
    if (g_hi == 4 && !need_mask) fwd_chunk<CAUSAL, true>(oacc, m_run, l_run, sQ, sK, sV, row0, c0, 4, L, qrow, scale_log2e, lane);
    else fwd_chunk<CAUSAL, false>(oacc, m_run, l_run, sQ, sK, sV, row0, c0, g_hi, L, qrow, scale_log2e, lane);
  }
  float inv[2];
#pragma unroll
  for (int r = 0; r < 2; ++r) {
    l_run[r] += __shfl_xor_sync(0xffffffffu, l_run[r], 1);
    l_run[r] += __shfl_xor_sync(0xffffffffu, l_run[r], 2);
    inv[r] = l_run[r] > 0.f ? 1.f / l_run[r] : 0.f;
    if ((lane & 3) == 0 && qrow[r] < L)
      lse2[(static_cast<size_t>(s) * H + h) * L + qrow[r]] = m_run[r] + log2f(l_run[r]);
  }
  store_rows_bf16(oacc, inv[0], inv[1], smem, 0, row0, o + static_cast<size_t>(s) * L * d + h * DH, d, q0 + row0, L, lane);
}

// ---------------------------------------------------------------------------------------
// backward, dQ pass (rows = queries).  Also produces D = rowsum(dO * O) for the dKV pass.
// ---------------------------------------------------------------------------------------
template <bool CAUSAL>
__global__ void __launch_bounds__(256, 2) attn_bwd_dq_kernel(const bf16* __restrict__ qkv, const bf16* __restrict__ o,
                                                             const bf16* __restrict__ d_o, const float* __restrict__ lse2,
                                                             float* __restrict__ dsum, bf16* __restrict__ dqkv, int L,
                                                             int H, int d, float scale, float scale_log2e,
                                                             const float2* __restrict__ ln_sb, float2* __restrict__ ln_dots) {
  extern __shared__ __align__(128) uint8_t smem[];
  const int nwarps = blockDim.x >> 5, BQ = nwarps * 16;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int sh = blockIdx.y, s = sh / H, h = sh - s * H;
  const int q0 = blockIdx.x * BQ;
  const int kv_len = CAUSAL ? min(L, q0 + BQ) : L;
  const int kv_rows = (kv_len + 15) & ~15;
  const int Lp = (L + 15) & ~15;
  const uint32_t sQ = smem_u32(smem), sdO = sQ + BQ * ROW_BYTES, sO = sdO + BQ * ROW_BYTES;
  const uint32_t sK = sO + BQ * ROW_BYTES, sV = sK + Lp * ROW_BYTES;
  const int ld = 3 * d;
  const size_t seq_row = static_cast<size_t>(s) * L;
  const bf16* base = qkv + seq_row * ld + h * DH;
  pdl_wait();
  pdl_trigger();
  load_tile(sQ, base, ld, q0, L, BQ);
  load_tile(sdO, d_o + seq_row * d + h * DH, d, q0, L, BQ);
  load_tile(sO, o + seq_row * d + h * DH, d, q0, L, BQ);
  load_tile(sK, base + d, ld, 0, L, kv_rows);
  load_tile(sV, base + 2 * d, ld, 0, L, kv_rows);
  cp_async_commit();
  cp_async_wait_all();
  __syncthreads();

  const int row0 = warp * 16;
  if (q0 + row0 >= L) return;
  // D_i = sum_j dO_ij O_ij for the warp's 16 rows: lane -> (row = lane/2, half = lane%2)
  float dpart = 0.f;
  {
    const int r = row0 + (lane >> 1);
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      const int chunk = (lane & 1) * 4 + c;
      uint4 a = *reinterpret_cast<const uint4*>(smem + (sdO - sQ) + swz(r, chunk));
      uint4 b = *reinterpret_cast<const uint4*>(smem + (sO - sQ) + swz(r, chunk));
      const uint32_t* pa = reinterpret_cast<const uint32_t*>(&a);
      const uint32_t* pb = reinterpret_cast<const uint32_t*>(&b);
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        float2 x = unpack_bf16(pa[i]), y = unpack_bf16(pb[i]);
        dpart += x.x * y.x + x.y * y.y;
      }
    }
    dpart += __shfl_xor_sync(0xffffffffu, dpart, 1);
  }
  const int qrow[2] = {q0 + row0 + (lane >> 2), q0 + row0 + (lane >> 2) + 8};
  float Dr[2], lse[2];
  Dr[0] = __shfl_sync(0xffffffffu, dpart, (lane >> 2) * 2);
  Dr[1] = __shfl_sync(0xffffffffu, dpart, ((lane >> 2) + 8) * 2);
  const size_t stat_base = (static_cast<size_t>(s) * H + h) * L;
  if ((lane & 1) == 0) {
    const int r = q0 + row0 + (lane >> 1);
    if (r < L) dsum[stat_base + r] = dpart;
  }
#pragma unroll
  for (int r = 0; r < 2; ++r) lse[r] = qrow[r] < L ? lse2[stat_base + qrow[r]] : 0.f;

  float dq[8][4];
  zero_acc(dq);
  const int kv_warp = CAUSAL ? min(kv_len, q0 + row0 + 16) : kv_len;
  const f32x2 c2 = f2_pack(scale_log2e, scale_log2e);
  const f32x2 nl2[2] = {f2_pack(-lse[0], -lse[0]), f2_pack(-lse[1], -lse[1])};
  const f32x2 nD2[2] = {f2_pack(-Dr[0], -Dr[0]), f2_pack(-Dr[1], -Dr[1])};
  // one 32-key chunk; FULL: both 16-key groups visible to every row (no guards / mask)
  auto chunk = [&](auto full_tag, int c0, int g_hi) {
    constexpr bool FULL = decltype(full_tag)::value;
    float sacc[4][4], dp[4][4];
    zero_acc(sacc);
    zero_acc(dp);
    mma_rows_x_cols<2>(sacc, sQ, row0, sK, c0, 0, FULL ? 2 : g_hi, lane);
    mma_rows_x_cols<2>(dp, sdO, row0, sV, c0, 0, FULL ? 2 : g_hi, lane);
    // rows >= L of the last tile carry lse = 0 and finite garbage: they are never stored, so only the
    // column mask matters
#pragma unroll
    for (int nt = 0; nt < 4; ++nt) {
      if (FULL || nt < 2 * g_hi) {
#pragma unroll
        for (int r = 0; r < 2; ++r) {
          float a, b;
          f2_unpack(f2_fma(f2_pack(sacc[nt][2 * r], sacc[nt][2 * r + 1]), c2, nl2[r]), a, b);
          a = exp2f(a);
          b = exp2f(b);
          if constexpr (!FULL) {
            const int col = c0 + nt * 8 + (lane & 3) * 2;
            const int lim = CAUSAL ? min(L - 1, qrow[r]) : L - 1;
            a = col <= lim ? a : 0.f;
            b = col + 1 <= lim ? b : 0.f;
          }
          f2_unpack(f2_mul(f2_pack(a, b), f2_add(f2_pack(dp[nt][2 * r], dp[nt][2 * r + 1]), nD2[r])), sacc[nt][2 * r],
                    sacc[nt][2 * r + 1]);  // dS (unscaled)
        }
      }
    }
    mma_p_x_tile<2>(dq, sacc, sK, c0, 0, FULL ? 2 : g_hi, lane);
  };
  for (int c0 = 0; c0 < kv_warp; c0 += 32) {
    const int g_hi = min(2, (kv_warp - c0 + 15) >> 4);
    const bool need_mask = (c0 + 32 > L) || (CAUSAL && c0 + 31 > q0 + row0);
    if (g_hi == 2 && !need_mask) chunk(std::true_type{}, c0, 2);
    else chunk(std::false_type{}, c0, g_hi);
  }
  RowDots rd;
  if (ln_dots != nullptr) { rd.sb = ln_sb + h * DH; rd.y = base; rd.out = ln_dots + seq_row * 3 * H; rd.parts = 3 * H; rd.part = h; }
  store_rows_bf16(dq, scale, scale, smem, 0, row0, dqkv + seq_row * ld + h * DH, ld, q0 + row0, L, lane, rd);
}

// ---------------------------------------------------------------------------------------
// backward, dK/dV pass (rows = keys)
// ---------------------------------------------------------------------------------------
template <bool CAUSAL>
__global__ void __launch_bounds__(256, 2) attn_bwd_dkv_kernel(const bf16* __restrict__ qkv, const bf16* __restrict__ d_o,
                                                              const float* __restrict__ lse2, const float* __restrict__ dsum,
                                                              bf16* __restrict__ dqkv, int L, int H, int d, float scale,
                                                              float scale_log2e, const float2* __restrict__ ln_sb,
                                                              float2* __restrict__ ln_dots) {
  extern __shared__ __align__(128) uint8_t smem[];
  const int nwarps = blockDim.x >> 5, BKV = nwarps * 16;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int sh = blockIdx.y, s = sh / H, h = sh - s * H;
  const int k0 = blockIdx.x * BKV;
  const int Lp = (L + 15) & ~15;
  const uint32_t sK = smem_u32(smem), sV = sK + BKV * ROW_BYTES, sQ = sV + BKV * ROW_BYTES, sdO = sQ + Lp * ROW_BYTES;
  float* sLse = reinterpret_cast<float*>(smem + (2 * BKV + 2 * Lp) * ROW_BYTES);
  float* sD = sLse + Lp;
  const int ld = 3 * d;
  const size_t seq_row = static_cast<size_t>(s) * L;
  const bf16* base = qkv + seq_row * ld + h * DH;
  const int q_blk = CAUSAL ? (k0 & ~15) : 0;  // queries below the block's first key never see it
  pdl_wait();
  pdl_trigger();
  load_tile(sK, base + d, ld, k0, L, BKV);
  load_tile(sV, base + 2 * d, ld, k0, L, BKV);
  load_tile(sQ + q_blk * ROW_BYTES, base, ld, q_blk, L, Lp - q_blk);
  load_tile(sdO + q_blk * ROW_BYTES, d_o + seq_row * d + h * DH, d, q_blk, L, Lp - q_blk);
  cp_async_commit();
  const size_t stat_base = (static_cast<size_t>(s) * H + h) * L;
  for (int i = threadIdx.x; i < Lp; i += blockDim.x) {
    sLse[i] = i < L ? lse2[stat_base + i] : 0.f;
    sD[i] = i < L ? dsum[stat_base + i] : 0.f;
  }
  cp_async_wait_all();
  __syncthreads();

  const int row0 = warp * 16;
  if (k0 + row0 >= L) return;
  float dk[8][4], dv[8][4];
  zero_acc(dk);
  zero_acc(dv);
  const int krow[2] = {k0 + row0 + (lane >> 2), k0 + row0 + (lane >> 2) + 8};
  const int q_first = CAUSAL ? (k0 + row0) : 0;  // first query that can see any of this warp's keys
  const f32x2 c2 = f2_pack(scale_log2e, scale_log2e);
  // one chunk of 32 queries (columns); FULL: both 16-query groups see all of this warp's keys
  auto chunk = [&](auto full_tag, int c0, int g_lo, int g_hi) {
    constexpr bool FULL = decltype(full_tag)::value;
    float st[4][4], dpt[4][4];
    zero_acc(st);
    zero_acc(dpt);
    mma_rows_x_cols<2>(st, sK, row0, sQ, c0, FULL ? 0 : g_lo, FULL ? 2 : g_hi, lane);
    mma_rows_x_cols<2>(dpt, sV, row0, sdO, c0, FULL ? 0 : g_lo, FULL ? 2 : g_hi, lane);
    // key rows >= L only pollute their own (never stored) dK/dV rows; the query (column) mask is
    // needed only where the chunk crosses L or the causal diagonal of this warp's 16 keys
#pragma unroll
    for (int nt = 0; nt < 4; ++nt) {
      if (FULL || (nt >= 2 * g_lo && nt < 2 * g_hi)) {
        const int qi = c0 + nt * 8 + (lane & 3) * 2;  // query index (column), < Lp here
        const float2 l2 = *reinterpret_cast<const float2*>(sLse + qi);
        const float2 d2 = *reinterpret_cast<const float2*>(sD + qi);
        const f32x2 nl = f2_pack(-l2.x, -l2.y), nd = f2_pack(-d2.x, -d2.y);
#pragma unroll
        for (int r = 0; r < 2; ++r) {
          float a, b;
          f2_unpack(f2_fma(f2_pack(st[nt][2 * r], st[nt][2 * r + 1]), c2, nl), a, b);
          a = exp2f(a);
          b = exp2f(b);
          if constexpr (!FULL) {
            a = (qi < L && (!CAUSAL || krow[r] <= qi)) ? a : 0.f;
            b = (qi + 1 < L && (!CAUSAL || krow[r] <= qi + 1)) ? b : 0.f;
          }
          st[nt][2 * r] = a;  // P^T
          st[nt][2 * r + 1] = b;
          f2_unpack(f2_mul(f2_pack(a, b), f2_add(f2_pack(dpt[nt][2 * r], dpt[nt][2 * r + 1]), nd)), dpt[nt][2 * r],
                    dpt[nt][2 * r + 1]);  // dS^T (unscaled), in place
        }
      }
    }
    mma_p_x_tile<2>(dv, st, sdO, c0, FULL ? 0 : g_lo, FULL ? 2 : g_hi, lane);
    mma_p_x_tile<2>(dk, dpt, sQ, c0, FULL ? 0 : g_lo, FULL ? 2 : g_hi, lane);
  };
  for (int c0 = q_first & ~31; c0 < L; c0 += 32) {
    const int g_lo = max(0, (q_first - c0) >> 4);
    const int g_hi = min(2, (L - c0 + 15) >> 4);
    const bool need_mask = (c0 + 32 > L) || (CAUSAL && c0 < k0 + row0 + 15);
    if (g_lo == 0 && g_hi == 2 && !need_mask) chunk(std::true_type{}, c0, 0, 2);
    else chunk(std::false_type{}, c0, g_lo, g_hi);
  }
  bf16* out = dqkv + seq_row * ld + h * DH;
  RowDots rk, rv;
  if (ln_dots != nullptr) {
    rk.sb = ln_sb + d + h * DH; rk.y = base + d; rk.out = ln_dots + seq_row * 3 * H; rk.parts = 3 * H; rk.part = H + h;
    rv = rk; rv.sb = ln_sb + 2 * d + h * DH; rv.y = base + 2 * d; rv.part = 2 * H + h;
  }
  store_rows_bf16(dk, scale, scale, smem, 0, row0, out + d, ld, k0 + row0, L, lane, rk);
  store_rows_bf16(dv, 1.f, 1.f, smem, BKV * ROW_BYTES, row0, out + 2 * d, ld, k0 + row0, L, lane, rv);
}

// =======================================================================================
// Short sequences (L <= 128: the text tower, 77 tokens or fewer after EOT truncation).
//
// One CTA per (sequence, head), one warp per 16-row tile, Q / K / V (and dO, O) loaded ONCE.
// The whole score row block of a warp (16 x 16*T, T = visible 16-key groups) lives in registers,
// so the softmax is a single pass (no running max / rescale) and the code is straight-line per T
// (dispatch on T: no per-group guards -- the generic kernels above spend ~2/3 of their issue
// slots on those).  The backward is ONE kernel: phase 1 (rows = queries) computes S, P, dP, dS
// once (D = rowsum(P dP): O is not loaded), dQ = dS K, and parks P / dS as bf16 in shared memory (over the dead K / V tiles);
// phase 2 (rows = keys) reads them transposed with ldmatrix.trans: dV = P^T dO, dK = dS^T Q.
// 5 MMA products instead of 7, one exp per score instead of two, a third of the tile loads.
// =======================================================================================
static constexpr int SHORT_MAX_TILES = 8;

__device__ __forceinline__ uint32_t ps_stride(int Lp) { return static_cast<uint32_t>(2 * Lp + 16); }  // bytes; odd multiple of 16: conflict-free ldmatrix

template <bool CAUSAL, int T>
__device__ __forceinline__ void short_fwd_body(uint8_t* smem, uint32_t sQ, uint32_t sK, uint32_t sV, int t, int L, int lane,
                                               float scale_log2e, bf16* o_base, int d, float* lse_base) {
  const int row0 = t * 16;
  uint32_t qa[4][4];
#pragma unroll
  for (int ks = 0; ks < 4; ++ks) load_a_frag(qa[ks], sQ, row0, ks, lane);
  float s[2 * T][4];
  zero_acc(s);
#pragma unroll
  for (int ks = 0; ks < 4; ++ks) {
#pragma unroll
    for (int g = 0; g < T; ++g) {
      uint32_t b0, b1, b2, b3;
      ldsm_x4(sK + swz(g * 16 + (lane & 7) + ((lane >> 4) << 3), ks * 2 + ((lane >> 3) & 1)), b0, b1, b2, b3);
      mma16816(s[2 * g], qa[ks], b0, b1);
      mma16816(s[2 * g + 1], qa[ks], b2, b3);
    }
  }
  const int qr = row0 + (lane >> 2);
  // only the last visible group can hold invisible keys (the causal diagonal / columns >= L)
#pragma unroll
  for (int nt = 2 * T - 2; nt < 2 * T; ++nt) {
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const int col = nt * 8 + (lane & 3) * 2 + (e & 1);
      const bool ok = col < L && (!CAUSAL || col <= qr + 8 * (e >> 1));
      s[nt][e] = ok ? s[nt][e] : -INFINITY;
    }
  }
  float m[2] = {-INFINITY, -INFINITY};
#pragma unroll
  for (int nt = 0; nt < 2 * T; ++nt) {
    m[0] = fmaxf(m[0], fmaxf(s[nt][0], s[nt][1]));
    m[1] = fmaxf(m[1], fmaxf(s[nt][2], s[nt][3]));
  }
  f32x2 nm[2];
#pragma unroll
  for (int r = 0; r < 2; ++r) {
    m[r] = fmaxf(m[r], __shfl_xor_sync(0xffffffffu, m[r], 1));
    m[r] = fmaxf(m[r], __shfl_xor_sync(0xffffffffu, m[r], 2));
    m[r] = (m[r] == -INFINITY) ? 0.f : m[r] * scale_log2e;  // scaled max (log2 domain)
    nm[r] = f2_pack(-m[r], -m[r]);
  }
  const f32x2 sc = f2_pack(scale_log2e, scale_log2e);
  f32x2 lsum[2] = {f2_pack(0.f, 0.f), f2_pack(0.f, 0.f)};
  uint32_t pk[2 * T][2];  // P as bf16 A fragments
#pragma unroll
  for (int nt = 0; nt < 2 * T; ++nt) {
#pragma unroll
    for (int r = 0; r < 2; ++r) {
      float a, b;
      f2_unpack(f2_fma(f2_pack(s[nt][2 * r], s[nt][2 * r + 1]), sc, nm[r]), a, b);
      a = exp2f(a);
      b = exp2f(b);
      lsum[r] = f2_add(lsum[r], f2_pack(a, b));
      pk[nt][r] = pack_bf16(a, b);
    }
  }
  float oacc[8][4];
  zero_acc(oacc);
#pragma unroll
  for (int g = 0; g < T; ++g) {
    const uint32_t a[4] = {pk[2 * g][0], pk[2 * g][1], pk[2 * g + 1][0], pk[2 * g + 1][1]};
#pragma unroll
    for (int dp = 0; dp < 4; ++dp) {
      uint32_t b0, b1, b2, b3;
      ldsm_x4_t(sV + swz(g * 16 + (lane & 7) + (((lane >> 3) & 1) << 3), dp * 2 + (lane >> 4)), b0, b1, b2, b3);
      mma16816(oacc[2 * dp], a, b0, b1);
      mma16816(oacc[2 * dp + 1], a, b2, b3);
    }
  }
  float inv[2];
#pragma unroll
  for (int r = 0; r < 2; ++r) {
    float a, b;
    f2_unpack(lsum[r], a, b);
    float l = a + b;
    l += __shfl_xor_sync(0xffffffffu, l, 1);
    l += __shfl_xor_sync(0xffffffffu, l, 2);
    inv[r] = l > 0.f ? 1.f / l : 0.f;
    const int row = qr + 8 * r;
    if ((lane & 3) == 0 && row < L) lse_base[row] = m[r] + log2f(l);
  }
  store_rows_bf16(oacc, inv[0], inv[1], smem, 0, row0, o_base, d, row0, L, lane);
}

// MAXT = most 16-row tiles (warps) this instantiation handles: sizes the register budget, so that the
// 77-token text tower (5 tiles) does not pay for 128-token sequences (8 tiles).
constexpr int short_min_ctas(int maxt, bool bwd) { return maxt <= 2 ? 8 : maxt <= 5 ? (bwd ? 3 : 5) : (bwd ? 1 : 2); }

// One (sequence, head) problem: the sequence occupies rows [seq_row, seq_row + L) of qkv / o, its lse2 row block starts at
// lse_base.  The CTA may have more warps than the sequence has 16-row tiles (variable-length launches are sized by the
// longest sequence): those warps help with the loads and leave after the only block-wide barrier.
template <bool CAUSAL, int MAXT>
__device__ __forceinline__ void short_fwd_cta(uint8_t* smem, const bf16* qkv, bf16* o, float* lse_base, size_t seq_row, int L, int h,
                                              int d, float scale_log2e) {
  const int nw = blockDim.x >> 5, Lp = nw * 16;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t sQ = smem_u32(smem), sK = sQ + Lp * ROW_BYTES, sV = sK + Lp * ROW_BYTES;
  const int ld = 3 * d;
  const bf16* base = qkv + seq_row * ld + h * DH;
  load_tile(sQ, base, ld, 0, L, Lp);
  load_tile(sK, base + d, ld, 0, L, Lp);
  load_tile(sV, base + 2 * d, ld, 0, L, Lp);
  cp_async_commit();
  cp_async_wait_all();
  __syncthreads();
  const int nt = (L + 15) >> 4;
  if (warp >= nt) return;
  bf16* ob = o + seq_row * d + h * DH;
  const int T = CAUSAL ? warp + 1 : nt;
#define MUDPT_FWD_CASE(k) \
  case k: if constexpr (MAXT >= k) short_fwd_body<CAUSAL, k>(smem, sQ, sK, sV, warp, L, lane, scale_log2e, ob, d, lse_base); break;
  switch (T) {
    MUDPT_FWD_CASE(1) MUDPT_FWD_CASE(2) MUDPT_FWD_CASE(3) MUDPT_FWD_CASE(4)
    MUDPT_FWD_CASE(5) MUDPT_FWD_CASE(6) MUDPT_FWD_CASE(7) MUDPT_FWD_CASE(8)
    default: break;
  }
#undef MUDPT_FWD_CASE
}

template <bool CAUSAL, int MAXT>
__global__ void __launch_bounds__(MAXT * 32, short_min_ctas(MAXT, false)) attn_short_fwd_kernel(const bf16* __restrict__ qkv, bf16* __restrict__ o,
                                                                              float* __restrict__ lse2, int L, int H, int d,
                                                                              float scale_log2e) {
  extern __shared__ __align__(128) uint8_t smem[];
  const int sh = blockIdx.x, s = sh / H, h = sh - s * H;
  pdl_wait();
  pdl_trigger();
  short_fwd_cta<CAUSAL, MAXT>(smem, qkv, o, lse2 + (static_cast<size_t>(s) * H + h) * L, static_cast<size_t>(s) * L, L, h, d, scale_log2e);
}

// Packed variable-length causal sequences (the ragged text tower): sequence s occupies rows [seq_off[s], seq_off[s + 1]); its
// lse2 block is [H, len_s] at seq_off[s] * H (with equal lengths: the layout and the results of attn_short_fwd_kernel).
// 3 instead of 5 resident CTAs for the 3-5 tile forward: its 16 x 80 score block, P fragments, Q fragments and output
// accumulator need ~110 registers, and 5 (4) CTAs cap it at 80 (96), where it spills.
constexpr int varlen_min_ctas(int maxt, bool bwd) { return maxt <= 2 ? 8 : maxt <= 5 ? 3 : (bwd ? 1 : 2); }

template <int MAXT>
__global__ void __launch_bounds__(MAXT * 32, varlen_min_ctas(MAXT, false)) attn_varlen_fwd_kernel(const bf16* __restrict__ qkv, bf16* __restrict__ o,
                                                                               float* __restrict__ lse2, const int* __restrict__ seq_off,
                                                                               int H, int d, float scale_log2e) {
  extern __shared__ __align__(128) uint8_t smem[];
  const int sh = blockIdx.x, s = sh / H, h = sh - s * H;
  pdl_wait();
  pdl_trigger();
  const int r0 = seq_off[s], L = seq_off[s + 1] - r0;
  short_fwd_cta<true, MAXT>(smem, qkv, o, lse2 + static_cast<size_t>(r0) * H + static_cast<size_t>(h) * L, r0, L, h, d, scale_log2e);
}

// Phase 1 of the fused backward for query tile t: returns dQ in `dq`, P / dS (bf16, accumulator
// fragment layout) in pp / ds.
template <bool CAUSAL, int T, int MAXT>
__device__ __forceinline__ void short_bwd_phase1(uint32_t sQ, uint32_t sdO, uint32_t sK, uint32_t sV, int t, int L, int lane,
                                                 float scale_log2e, float lse0, float lse1, float (&dq)[8][4],
                                                 uint32_t (&pp)[2 * MAXT][2], uint32_t (&ds)[2 * MAXT][2]) {
  const int row0 = t * 16;
  float sc[2 * T][4], dp[2 * T][4];
  zero_acc(sc);
  zero_acc(dp);
#pragma unroll
  for (int ks = 0; ks < 4; ++ks) {
    uint32_t qa[4], da[4];
    load_a_frag(qa, sQ, row0, ks, lane);
    load_a_frag(da, sdO, row0, ks, lane);
#pragma unroll
    for (int g = 0; g < T; ++g) {
      const uint32_t off = swz(g * 16 + (lane & 7) + ((lane >> 4) << 3), ks * 2 + ((lane >> 3) & 1));
      uint32_t b0, b1, b2, b3;
      ldsm_x4(sK + off, b0, b1, b2, b3);
      mma16816(sc[2 * g], qa, b0, b1);
      mma16816(sc[2 * g + 1], qa, b2, b3);
      ldsm_x4(sV + off, b0, b1, b2, b3);
      mma16816(dp[2 * g], da, b0, b1);
      mma16816(dp[2 * g + 1], da, b2, b3);
    }
  }
  const int qr = row0 + (lane >> 2);
  const f32x2 c2 = f2_pack(scale_log2e, scale_log2e);
  const f32x2 nl[2] = {f2_pack(-lse0, -lse0), f2_pack(-lse1, -lse1)};
  // P in place of the scores; D_i = sum_j P_ij dP_ij (== sum_k dO_ik O_ik, without loading O: the whole row
  // block is in registers here)
  f32x2 dsum2[2] = {f2_pack(0.f, 0.f), f2_pack(0.f, 0.f)};
#pragma unroll
  for (int nt = 0; nt < 2 * T; ++nt) {
#pragma unroll
    for (int r = 0; r < 2; ++r) {
      float a, b;
      f2_unpack(f2_fma(f2_pack(sc[nt][2 * r], sc[nt][2 * r + 1]), c2, nl[r]), a, b);
      a = exp2f(a);
      b = exp2f(b);
      if (nt >= 2 * T - 2) {  // only the last visible group can hold invisible keys
        const int col = nt * 8 + (lane & 3) * 2;
        const int lim = CAUSAL ? min(L - 1, qr + 8 * r) : L - 1;
        a = col <= lim ? a : 0.f;
        b = col + 1 <= lim ? b : 0.f;
      }
      sc[nt][2 * r] = a;
      sc[nt][2 * r + 1] = b;
      dsum2[r] = f2_fma(f2_pack(a, b), f2_pack(dp[nt][2 * r], dp[nt][2 * r + 1]), dsum2[r]);
    }
  }
  f32x2 nD[2];
#pragma unroll
  for (int r = 0; r < 2; ++r) {
    float a, b;
    f2_unpack(dsum2[r], a, b);
    float D = a + b;
    D += __shfl_xor_sync(0xffffffffu, D, 1);
    D += __shfl_xor_sync(0xffffffffu, D, 2);
    nD[r] = f2_pack(-D, -D);
  }
#pragma unroll
  for (int nt = 0; nt < 2 * T; ++nt) {
#pragma unroll
    for (int r = 0; r < 2; ++r) {
      const f32x2 p2 = f2_pack(sc[nt][2 * r], sc[nt][2 * r + 1]);
      float x, y;
      f2_unpack(f2_mul(p2, f2_add(f2_pack(dp[nt][2 * r], dp[nt][2 * r + 1]), nD[r])), x, y);  // dS (unscaled)
      pp[nt][r] = pack_bf16(sc[nt][2 * r], sc[nt][2 * r + 1]);
      ds[nt][r] = pack_bf16(x, y);
    }
  }
  zero_acc(dq);
#pragma unroll
  for (int g = 0; g < T; ++g) {
    const uint32_t a[4] = {ds[2 * g][0], ds[2 * g][1], ds[2 * g + 1][0], ds[2 * g + 1][1]};
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      uint32_t b0, b1, b2, b3;
      ldsm_x4_t(sK + swz(g * 16 + (lane & 7) + (((lane >> 3) & 1) << 3), q * 2 + (lane >> 4)), b0, b1, b2, b3);
      mma16816(dq[2 * q], a, b0, b1);
      mma16816(dq[2 * q + 1], a, b2, b3);
    }
  }
}

// One (sequence, head) problem of the fused backward (rows [seq_row, seq_row + L), lse2 row block at lse_base).  Warps
// past the sequence's last 16-row tile (variable-length launches) do no work but reach both block-wide barriers.
template <bool CAUSAL, int MAXT>
__device__ __forceinline__ void short_bwd_cta(uint8_t* smem, const bf16* qkv, const bf16* d_o, const float* lse_base, bf16* dqkv,
                                              size_t seq_row, int L, int h, int H, int d, float scale, float scale_log2e,
                                              const float2* ln_sb, float2* ln_dots) {
  const int nw = blockDim.x >> 5, Lp = nw * 16;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // [Q | dO | K | V | pad]; after phase 1 the K / V / pad region is reused for P and dS
  const uint32_t tile_bytes = Lp * ROW_BYTES;
  const uint32_t sQ = smem_u32(smem), sdO = sQ + tile_bytes, sK = sdO + tile_bytes, sV = sK + tile_bytes;
  const int ld = 3 * d;
  const bf16* base = qkv + seq_row * ld + h * DH;
  load_tile(sQ, base, ld, 0, L, Lp);
  load_tile(sdO, d_o + seq_row * d + h * DH, d, 0, L, Lp);
  load_tile(sK, base + d, ld, 0, L, Lp);
  load_tile(sV, base + 2 * d, ld, 0, L, Lp);
  cp_async_commit();
  const int row0 = warp * 16;
  const int qr = row0 + (lane >> 2);
  // rows >= L: lse = 0 with zero Q / dO rows gives finite p, dP = 0, hence D = 0 and dS = 0: no contribution to dK / dV
  const float lse0 = qr < L ? lse_base[qr] : 0.f;
  const float lse1 = qr + 8 < L ? lse_base[qr + 8] : 0.f;
  cp_async_wait_all();
  __syncthreads();

  float dq[8][4];
  uint32_t pp[2 * MAXT][2], ds[2 * MAXT][2];
  const int ntiles = (L + 15) >> 4;  // live tiles; warps past them take part in the barriers only
  const bool live = warp < ntiles;
  const int T = !live ? 0 : CAUSAL ? warp + 1 : ntiles;
#define MUDPT_BWD_CASE(k) \
  case k: if constexpr (MAXT >= k) short_bwd_phase1<CAUSAL, k, MAXT>(sQ, sdO, sK, sV, warp, L, lane, scale_log2e, lse0, lse1, dq, pp, ds); break;
  switch (T) {
    MUDPT_BWD_CASE(1) MUDPT_BWD_CASE(2) MUDPT_BWD_CASE(3) MUDPT_BWD_CASE(4)
    MUDPT_BWD_CASE(5) MUDPT_BWD_CASE(6) MUDPT_BWD_CASE(7) MUDPT_BWD_CASE(8)
    default: break;
  }
#undef MUDPT_BWD_CASE
  __syncthreads();  // every warp is done with K / V / O: the region becomes P | dS
  const uint32_t stride = ps_stride(Lp);
  uint8_t* gP = smem + 2 * tile_bytes;
  uint8_t* gS = gP + Lp * stride;
  if (live) {
    // accumulator fragment layout: rows (lane/4, +8), column pair 2*(lane%4) of each 8-column tile
    const uint32_t r_lo = static_cast<uint32_t>(row0 + (lane >> 2)) * stride + (lane & 3) * 4;
    const uint32_t r_hi = r_lo + 8 * stride;
#pragma unroll
    for (int nt = 0; nt < 2 * MAXT; ++nt) {
      if (nt < 2 * T) {
        *reinterpret_cast<uint32_t*>(gP + r_lo + nt * 16) = pp[nt][0];
        *reinterpret_cast<uint32_t*>(gP + r_hi + nt * 16) = pp[nt][1];
        *reinterpret_cast<uint32_t*>(gS + r_lo + nt * 16) = ds[nt][0];
        *reinterpret_cast<uint32_t*>(gS + r_hi + nt * 16) = ds[nt][1];
      }
    }
  }
  __syncthreads();

  // phase 2: rows = this warp's 16 keys; query groups g that can see them
  float dk[8][4], dv[8][4];
  zero_acc(dk);
  zero_acc(dv);
  const uint32_t aP = smem_u32(gP), aS = smem_u32(gS);
  for (int g = CAUSAL ? warp : 0; live && g < ntiles; ++g) {
    // A = (P^T)[keys row0.., queries 16g..]: 8x8 blocks of P (rows = queries) read transposed.
    // a0..a3 = blocks (queries 0-7, keys 0-7), (q 0-7, keys 8-15), (q 8-15, keys 0-7), (q 8-15, keys 8-15):
    // lanes 8i..8i+7 address the 8 query rows of block i
    const uint32_t off = static_cast<uint32_t>(g * 16 + (lane & 7) + ((lane >> 4) << 3)) * stride +
                         static_cast<uint32_t>(row0 + (((lane >> 3) & 1) << 3)) * 2;
    uint32_t pa[4], sa[4];
    ldsm_x4_t(aP + off, pa[0], pa[1], pa[2], pa[3]);
    ldsm_x4_t(aS + off, sa[0], sa[1], sa[2], sa[3]);
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const uint32_t boff = swz(g * 16 + (lane & 7) + (((lane >> 3) & 1) << 3), q * 2 + (lane >> 4));
      uint32_t b0, b1, b2, b3;
      ldsm_x4_t(sdO + boff, b0, b1, b2, b3);
      mma16816(dv[2 * q], pa, b0, b1);
      mma16816(dv[2 * q + 1], pa, b2, b3);
      ldsm_x4_t(sQ + boff, b0, b1, b2, b3);
      mma16816(dk[2 * q], sa, b0, b1);
      mma16816(dk[2 * q + 1], sa, b2, b3);
    }
  }
  __syncthreads();  // all reads of Q / dO / P / dS are done: the Q and dO tiles become store staging
  bf16* out = dqkv + seq_row * ld + h * DH;
  if (live) {
    RowDots rq, rk, rv;
    if (ln_dots != nullptr) {
      rq.sb = ln_sb + h * DH; rq.y = base; rq.out = ln_dots + seq_row * 3 * H; rq.parts = 3 * H; rq.part = h;
      rk = rq; rk.sb = ln_sb + d + h * DH; rk.y = base + d; rk.part = H + h;
      rv = rq; rv.sb = ln_sb + 2 * d + h * DH; rv.y = base + 2 * d; rv.part = 2 * H + h;
    }
    store_rows_bf16(dq, scale, scale, smem, 0, row0, out, ld, row0, L, lane, rq);
    store_rows_bf16(dk, scale, scale, smem, tile_bytes, row0, out + d, ld, row0, L, lane, rk);
    __syncwarp();
    store_rows_bf16(dv, 1.f, 1.f, smem, 0, row0, out + 2 * d, ld, row0, L, lane, rv);
  }
}

template <bool CAUSAL, int MAXT>
__global__ void __launch_bounds__(MAXT * 32, short_min_ctas(MAXT, true)) attn_short_bwd_kernel(const bf16* __restrict__ qkv, const bf16* __restrict__ o,
                                                                              const bf16* __restrict__ d_o,
                                                                              const float* __restrict__ lse2,
                                                                              bf16* __restrict__ dqkv, int L, int H, int d,
                                                                              float scale, float scale_log2e,
                                                                              const float2* __restrict__ ln_sb,
                                                                              float2* __restrict__ ln_dots) {
  extern __shared__ __align__(128) uint8_t smem[];
  const int sh = blockIdx.x, s = sh / H, h = sh - s * H;
  pdl_wait();
  pdl_trigger();
  short_bwd_cta<CAUSAL, MAXT>(smem, qkv, d_o, lse2 + (static_cast<size_t>(s) * H + h) * L, dqkv, static_cast<size_t>(s) * L, L, h, H, d,
                              scale, scale_log2e, ln_sb, ln_dots);
}

// Backward of attn_varlen_fwd_kernel (same packed layout).
template <int MAXT>
__global__ void __launch_bounds__(MAXT * 32, varlen_min_ctas(MAXT, true)) attn_varlen_bwd_kernel(const bf16* __restrict__ qkv,
                                                                               const bf16* __restrict__ d_o,
                                                                               const float* __restrict__ lse2,
                                                                               bf16* __restrict__ dqkv, const int* __restrict__ seq_off,
                                                                               int H, int d, float scale, float scale_log2e,
                                                                               const float2* __restrict__ ln_sb,
                                                                               float2* __restrict__ ln_dots) {
  extern __shared__ __align__(128) uint8_t smem[];
  const int sh = blockIdx.x, s = sh / H, h = sh - s * H;
  pdl_wait();
  pdl_trigger();
  const int r0 = seq_off[s], L = seq_off[s + 1] - r0;
  short_bwd_cta<true, MAXT>(smem, qkv, d_o, lse2 + static_cast<size_t>(r0) * H + static_cast<size_t>(h) * L, dqkv, r0, L, h, H, d,
                              scale, scale_log2e, ln_sb, ln_dots);
}

static size_t short_bwd_smem(int Lp) {
  const size_t tiles = 4u * Lp * ROW_BYTES;                       // Q dO K V
  const size_t need = 2u * Lp * ROW_BYTES + 2u * Lp * (2 * Lp + 16);  // Q dO P dS
  return tiles > need ? tiles : need;
}

// ---------------------------------------------------------------------------------------
// host launchers
// ---------------------------------------------------------------------------------------
// Warps (16-row tiles) per CTA.  The problems are tiny, so what matters is how many independent
// load->compute->store chains an SM has in flight: short sequences (text) use 2-warp CTAs, which
// doubles the resident CTAs per SM; long ones (vision) are limited by the K/V tile in shared memory
// anyway and keep 4 warps per CTA to amortise it.  MUDPT_ATTN_WARPS overrides (tuning aid).
static int pick_warps(int L) {
  const int tiles = (L + 15) / 16;
  static int forced = -1;
  if (forced < 0) {
    const char* e = getenv("MUDPT_ATTN_WARPS");
    forced = e ? atoi(e) : 0;
  }
  if (forced > 0) return forced > 8 ? 8 : (tiles >= forced ? forced : tiles);
  // as few CTAs per (sequence, head) as 8-warp CTAs allow, rows spread evenly: 199 tokens = 13 tiles ->
  // 2 CTAs of 7 warps (each K/V tile is then loaded twice instead of four times)
  const int ctas = (tiles + 7) / 8;
  return (tiles + ctas - 1) / ctas;
}

// L <= 128: the single-pass kernels (MUDPT_ATTN_SHORT=0 forces the generic ones; tuning / A-B aid)
static bool use_short(int L) {
  static int en = -1;
  if (en < 0) {
    const char* e = getenv("MUDPT_ATTN_SHORT");
    en = e ? (atoi(e) != 0) : 1;
  }
  return en && L <= 16 * SHORT_MAX_TILES;
}

template <typename K>
static const char* set_smem(K kern, size_t bytes) {
  if (bytes > 227 * 1024) return "attention: sequence too long for the shared-memory resident kernel";
  if (bytes > 48 * 1024 &&
      cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(bytes)) != cudaSuccess)
    return "attention: cudaFuncSetAttribute failed";
  return nullptr;
}

const char* attention_fwd(const bf16* qkv, bf16* o, float* lse2, int S, int L, int H, int d, bool causal,
                          cudaStream_t stream) {
  if (S <= 0 || L <= 0) return nullptr;
  if (d != H * DH) return "attention: head width must be 64";
  if (attention_tc_fwd_eligible(L, causal)) return attention_tc_fwd(qkv, o, lse2, S, L, H, d, causal, stream);
  const float sl2 = 0.125f * 1.4426950408889634f;
  if (use_short(L)) {
    const int tiles = (L + 15) / 16;
    const size_t sm = 3u * tiles * 16 * ROW_BYTES;
    const char* es = nullptr;
#define MUDPT_LAUNCH_FWD(C, MT)                                                                        \
  do {                                                                                                 \
    if ((es = set_smem(attn_short_fwd_kernel<C, MT>, sm))) return es;                                  \
    launch_pdl(attn_short_fwd_kernel<C, MT>, dim3(S * H), dim3(tiles * 32), sm, stream, qkv, o, lse2, L, H, d, sl2); \
  } while (0)
    if (causal) { if (tiles <= 2) MUDPT_LAUNCH_FWD(true, 2); else if (tiles <= 5) MUDPT_LAUNCH_FWD(true, 5); else MUDPT_LAUNCH_FWD(true, 8); }
    else { if (tiles <= 2) MUDPT_LAUNCH_FWD(false, 2); else if (tiles <= 5) MUDPT_LAUNCH_FWD(false, 5); else MUDPT_LAUNCH_FWD(false, 8); }
#undef MUDPT_LAUNCH_FWD
    count_launch(1);
    return launch_status("attention fwd (short) launch failed");
  }
  const int nw = pick_warps(L), BQ = nw * 16, Lp = (L + 15) & ~15;
  const size_t smem = static_cast<size_t>(BQ + 2 * Lp) * ROW_BYTES;
  dim3 grid((L + BQ - 1) / BQ, S * H);
  const char* e;
  if (causal) {
    if ((e = set_smem(attn_fwd_kernel<true>, smem))) return e;
    launch_pdl(attn_fwd_kernel<true>, grid, dim3(nw * 32), smem, stream, qkv, o, lse2, L, H, d, sl2);
  } else {
    if ((e = set_smem(attn_fwd_kernel<false>, smem))) return e;
    launch_pdl(attn_fwd_kernel<false>, grid, dim3(nw * 32), smem, stream, qkv, o, lse2, L, H, d, sl2);
  }
  count_launch(1);
  return launch_status("attention fwd launch failed");
}

// Varlen launches (causal): one CTA per (sequence, head), sized by the longest sequence (16-row tiles, <= SHORT_MAX_TILES).
int attention_varlen_max_len() { return 16 * SHORT_MAX_TILES; }

const char* attention_varlen_fwd(const bf16* qkv, bf16* o, float* lse2, const int* seq_off, int S, int max_len, int H, int d,
                                 cudaStream_t stream) {
  if (S <= 0) return nullptr;
  if (d != H * DH) return "attention: head width must be 64";
  if (max_len <= 0 || max_len > 16 * SHORT_MAX_TILES) return "attention (varlen): sequences must have 1..128 tokens";
  const float sl2 = 0.125f * 1.4426950408889634f;
  const int tiles = (max_len + 15) / 16;
  const size_t sm = 3u * tiles * 16 * ROW_BYTES;
  const char* es = nullptr;
#define MUDPT_LAUNCH_VFWD(MT)                                                                                     \
  do {                                                                                                            \
    if ((es = set_smem(attn_varlen_fwd_kernel<MT>, sm))) return es;                                               \
    launch_pdl(attn_varlen_fwd_kernel<MT>, dim3(S * H), dim3(tiles * 32), sm, stream, qkv, o, lse2, seq_off, H, d, sl2); \
  } while (0)
  if (tiles <= 2) MUDPT_LAUNCH_VFWD(2); else if (tiles <= 5) MUDPT_LAUNCH_VFWD(5); else MUDPT_LAUNCH_VFWD(8);
#undef MUDPT_LAUNCH_VFWD
  count_launch(1);
  return launch_status("attention fwd (varlen) launch failed");
}

const char* attention_varlen_bwd(const bf16* qkv, const bf16* d_o, const float* lse2, bf16* dqkv, const int* seq_off, int S, int max_len,
                                 int H, int d, cudaStream_t stream, const float2* ln_sb, float2* ln_dots) {
  if (S <= 0) return nullptr;
  if (d != H * DH) return "attention: head width must be 64";
  if (max_len <= 0 || max_len > 16 * SHORT_MAX_TILES) return "attention (varlen): sequences must have 1..128 tokens";
  const int tiles = (max_len + 15) / 16;
  const size_t sm = short_bwd_smem(tiles * 16);
  const char* es = nullptr;
  const float sc = 0.125f, sl2s = 0.125f * 1.4426950408889634f;
#define MUDPT_LAUNCH_VBWD(MT)                                                                                      \
  do {                                                                                                             \
    if ((es = set_smem(attn_varlen_bwd_kernel<MT>, sm))) return es;                                                \
    launch_pdl(attn_varlen_bwd_kernel<MT>, dim3(S * H), dim3(tiles * 32), sm, stream, qkv, d_o, lse2, dqkv, seq_off, H, d, sc, sl2s, \
               ln_sb, ln_dots);                                                                                    \
  } while (0)
  if (tiles <= 2) MUDPT_LAUNCH_VBWD(2); else if (tiles <= 5) MUDPT_LAUNCH_VBWD(5); else MUDPT_LAUNCH_VBWD(8);
#undef MUDPT_LAUNCH_VBWD
  count_launch(1);
  return launch_status("attention bwd (varlen) launch failed");
}

const char* attention_bwd(const bf16* qkv, const bf16* o, const bf16* d_o, const float* lse2, float* dsum, bf16* dqkv,
                          int S, int L, int H, int d, bool causal, cudaStream_t stream, const float2* ln_sb, float2* ln_dots) {
  if (S <= 0 || L <= 0) return nullptr;
  if (d != H * DH) return "attention: head width must be 64";
  if (ln_dots == nullptr && attention_tc_bwd_eligible(L, causal))  // (the row-dot by-product exists in the warp-MMA kernels only)
    return attention_tc_bwd(qkv, o, d_o, lse2, dsum, dqkv, S, L, H, d, causal, stream);
  if (use_short(L)) {
    const int tiles = (L + 15) / 16;
    const size_t sm = short_bwd_smem(tiles * 16);
    const char* es = nullptr;
    const float sc = 0.125f, sl2s = 0.125f * 1.4426950408889634f;
#define MUDPT_LAUNCH_BWD(C, MT)                                                                                  \
  do {                                                                                                           \
    if ((es = set_smem(attn_short_bwd_kernel<C, MT>, sm))) return es;                                            \
    launch_pdl(attn_short_bwd_kernel<C, MT>, dim3(S * H), dim3(tiles * 32), sm, stream, qkv, o, d_o, lse2, dqkv, L, H, d, sc, sl2s, ln_sb, ln_dots); \
  } while (0)
    if (causal) { if (tiles <= 2) MUDPT_LAUNCH_BWD(true, 2); else if (tiles <= 5) MUDPT_LAUNCH_BWD(true, 5); else MUDPT_LAUNCH_BWD(true, 8); }
    else { if (tiles <= 2) MUDPT_LAUNCH_BWD(false, 2); else if (tiles <= 5) MUDPT_LAUNCH_BWD(false, 5); else MUDPT_LAUNCH_BWD(false, 8); }
#undef MUDPT_LAUNCH_BWD
    count_launch(1);
    return launch_status("attention bwd (short) launch failed");
  }
  const int nw = pick_warps(L), BQ = nw * 16, Lp = (L + 15) & ~15;
  const size_t smem_q = static_cast<size_t>(3 * BQ + 2 * Lp) * ROW_BYTES;
  const size_t smem_kv = static_cast<size_t>(2 * BQ + 2 * Lp) * ROW_BYTES + 2 * Lp * sizeof(float);
  const float scale = 0.125f, sl2 = 0.125f * 1.4426950408889634f;
  dim3 grid((L + BQ - 1) / BQ, S * H);
  const char* e;
  if (causal) {
    if ((e = set_smem(attn_bwd_dq_kernel<true>, smem_q))) return e;
    if ((e = set_smem(attn_bwd_dkv_kernel<true>, smem_kv))) return e;
    launch_pdl(attn_bwd_dq_kernel<true>, grid, dim3(nw * 32), smem_q, stream, qkv, o, d_o, lse2, dsum, dqkv, L, H, d, scale, sl2, ln_sb, ln_dots);
    launch_pdl(attn_bwd_dkv_kernel<true>, grid, dim3(nw * 32), smem_kv, stream, qkv, d_o, lse2, dsum, dqkv, L, H, d, scale, sl2, ln_sb, ln_dots);
  } else {
    if ((e = set_smem(attn_bwd_dq_kernel<false>, smem_q))) return e;
    if ((e = set_smem(attn_bwd_dkv_kernel<false>, smem_kv))) return e;
    launch_pdl(attn_bwd_dq_kernel<false>, grid, dim3(nw * 32), smem_q, stream, qkv, o, d_o, lse2, dsum, dqkv, L, H, d, scale, sl2, ln_sb, ln_dots);
    launch_pdl(attn_bwd_dkv_kernel<false>, grid, dim3(nw * 32), smem_kv, stream, qkv, d_o, lse2, dsum, dqkv, L, H, d, scale, sl2, ln_sb, ln_dots);
  }
  count_launch(2);
  return launch_status("attention bwd launch failed");
}

}  // namespace mudpt
