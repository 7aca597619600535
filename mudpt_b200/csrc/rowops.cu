// HBM-bound row kernels of the MuDPT towers: LayerNorm forward / dgrad-only backward,
// the deep-prompt splice (indexed row overwrite, bit-exact) and its backward (sum over
// sequences + zeroing), patch extraction (im2col + bf16 cast) and weight re-layout.
//
//   LayerNorm ......... clip/model.py:164-170 (fp32 statistics, eps 1e-5, biased variance)
//   splice ............ clip/model.py:281-297 (text rows 1..n, vision last n rows)
//   patch extraction .. clip/model.py:527-529 (conv1 with stride == kernel == patch)
#include "rowops.h"

#include <cmath>
#include <cstdint>
#include <cstdlib>

#include "common.cuh"
#include "launch_count.h"

namespace mudpt {

static constexpr int LN_MAXV = 8;  // float4 per lane -> width <= 1024

// ------------------------------------------------------------------ LayerNorm forward
// One warp per row, NV float4 per lane (NV = ceil(width / 128), compile-time so that narrow towers
// do not pay registers for wide ones). OUT_BF16: normalized row as bf16 (GEMM A operand); else fp32
// (may alias x).
template <int NV, bool OUT_BF16>
// sp_prompt != nullptr: the deep-prompt splice of the block is done here too -- rows whose position (row % sp_L, or sp_pos[row]
// for packed variable-length sequences) is in [sp_row0, sp_row0 + sp_n) take their values from sp_prompt (copied verbatim into x: bit-exact, clip/model.py:281-297) before being normalised.
// (x is read through the read-only path; x_w is the same buffer, written for spliced rows only -- rows that are never read)
__global__ void __launch_bounds__(256) ln_fwd_kernel(const float* __restrict__ x, float* __restrict__ x_w,
                                                     const float* __restrict__ gamma, const float* __restrict__ beta,
                                                     void* __restrict__ out, int M, int d, float eps,
                                                     const float* __restrict__ sp_prompt, int sp_L, int sp_row0, int sp_n,
                                                     const int* __restrict__ sp_pos) {
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  pdl_wait();
  pdl_trigger();
  if (row >= M) return;
  float* xr = x_w + static_cast<size_t>(row) * d;
  const float* src = x + static_cast<size_t>(row) * d;
  bool spliced = false;
  if (sp_prompt != nullptr) {
    const int pos = (sp_pos != nullptr ? sp_pos[row] : row % sp_L) - sp_row0;
    if (pos >= 0 && pos < sp_n) {
      src = sp_prompt + static_cast<size_t>(pos) * d;
      spliced = true;
    }
  }
  float4 v[NV];
  float sum = 0.f;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const int c = (i * 32 + lane) * 4;
    if (c < d) {
      v[i] = *reinterpret_cast<const float4*>(src + c);
      sum += (v[i].x + v[i].y) + (v[i].z + v[i].w);
    }
  }
  if (spliced) {  // (warp-uniform; after every load of the row has been issued)
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      const int c = (i * 32 + lane) * 4;
      if (c < d) *reinterpret_cast<float4*>(xr + c) = v[i];
    }
  }
  const float mean = warp_sum(sum) / d;
  float sq = 0.f;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const int c = (i * 32 + lane) * 4;
    if (c < d) {
      const float a = v[i].x - mean, b = v[i].y - mean, e = v[i].z - mean, f = v[i].w - mean;
      sq += (a * a + b * b) + (e * e + f * f);
    }
  }
  const float rstd = rsqrtf(warp_sum(sq) / d + eps);
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const int c = (i * 32 + lane) * 4;
    if (c < d) {
      const float4 g = *reinterpret_cast<const float4*>(gamma + c);
      const float4 b = *reinterpret_cast<const float4*>(beta + c);
      float4 y;
      y.x = (v[i].x - mean) * rstd * g.x + b.x;
      y.y = (v[i].y - mean) * rstd * g.y + b.y;
      y.z = (v[i].z - mean) * rstd * g.z + b.z;
      y.w = (v[i].w - mean) * rstd * g.w + b.w;
      if constexpr (OUT_BF16) {
        uint2 u;
        u.x = pack_bf16(y.x, y.y);
        u.y = pack_bf16(y.z, y.w);
        *reinterpret_cast<uint2*>(reinterpret_cast<bf16*>(out) + static_cast<size_t>(row) * d + c) = u;
      } else {
        *reinterpret_cast<float4*>(reinterpret_cast<float*>(out) + static_cast<size_t>(row) * d + c) = y;
      }
    }
  }
}

static int pick_nv(int d) {
  const int nv = (d + 127) / 128;
  return nv <= 1 ? 1 : nv <= 2 ? 2 : nv <= 4 ? 4 : nv <= 6 ? 6 : 8;
}

// rows (= warps) per CTA of the LayerNorm kernels: experiment hook MUDPT_LN_WARPS (1..8)
static int ln_warps() {
  static const int w = getenv("MUDPT_LN_WARPS") ? atoi(getenv("MUDPT_LN_WARPS")) : 8;
  return w < 1 ? 1 : (w > 8 ? 8 : w);
}

template <int NV>
static void launch_ln_fwd(float* x, const float* gamma, const float* beta, void* out, bool out_bf16, int M, int d, float eps,
                          const float* sp_prompt, int sp_L, int sp_row0, int sp_n, const int* sp_pos, cudaStream_t stream) {
  const int wpc = ln_warps();
  const int grid = (M + wpc - 1) / wpc;
  if (out_bf16)
    launch_pdl(ln_fwd_kernel<NV, true>, dim3(grid), dim3(32 * wpc), 0, stream, x, x, gamma, beta, out, M, d, eps, sp_prompt, sp_L, sp_row0, sp_n, sp_pos);
  else
    launch_pdl(ln_fwd_kernel<NV, false>, dim3(grid), dim3(32 * wpc), 0, stream, x, x, gamma, beta, out, M, d, eps, sp_prompt, sp_L, sp_row0, sp_n, sp_pos);
}

// (defined with the pipeline kernels below) true when the shared-memory pipeline took the launch; *err is set if it failed
static bool ln_fwd_pipe_try(float* x, const float* gamma, const float* beta, bf16* out, int M, int d, float eps, const float* sp_prompt,
                            int sp_L, int sp_row0, int sp_n, const int* sp_pos, cudaStream_t stream, const char** err);

static const char* ln_fwd_dispatch(float* x, const float* gamma, const float* beta, void* out, bool out_bf16, int M, int d, float eps,
                                   const float* sp_prompt, int sp_L, int sp_row0, int sp_n, const int* sp_pos, cudaStream_t stream) {
  if (M <= 0) return nullptr;
  if (d % 4 != 0 || d > LN_MAXV * 128) return "layernorm: width must be a multiple of 4 and <= 1024";
  if (out_bf16) {
    const char* e = nullptr;
    if (ln_fwd_pipe_try(x, gamma, beta, reinterpret_cast<bf16*>(out), M, d, eps, sp_prompt, sp_L, sp_row0, sp_n, sp_pos, stream, &e)) {
      if (e) return e;
      count_launch(1);
      return launch_status("layernorm fwd (pipeline) launch failed");
    }
  }
  switch (pick_nv(d)) {
    case 1: launch_ln_fwd<1>(x, gamma, beta, out, out_bf16, M, d, eps, sp_prompt, sp_L, sp_row0, sp_n, sp_pos, stream); break;
    case 2: launch_ln_fwd<2>(x, gamma, beta, out, out_bf16, M, d, eps, sp_prompt, sp_L, sp_row0, sp_n, sp_pos, stream); break;
    case 4: launch_ln_fwd<4>(x, gamma, beta, out, out_bf16, M, d, eps, sp_prompt, sp_L, sp_row0, sp_n, sp_pos, stream); break;
    case 6: launch_ln_fwd<6>(x, gamma, beta, out, out_bf16, M, d, eps, sp_prompt, sp_L, sp_row0, sp_n, sp_pos, stream); break;
    default: launch_ln_fwd<8>(x, gamma, beta, out, out_bf16, M, d, eps, sp_prompt, sp_L, sp_row0, sp_n, sp_pos, stream); break;
  }
  count_launch(1);
  return launch_status("layernorm fwd launch failed");
}

const char* layernorm_fwd(const float* x, const float* gamma, const float* beta, void* out, bool out_bf16, int M, int d,
                          float eps, cudaStream_t stream) {
  // (x is only written for spliced rows: none here)
  return ln_fwd_dispatch(const_cast<float*>(x), gamma, beta, out, out_bf16, M, d, eps, nullptr, 1, 0, 0, nullptr, stream);
}

const char* layernorm_fwd_splice(float* x, const float* prompt, int L, int row0, int n, const float* gamma, const float* beta,
                                 void* out, bool out_bf16, int M, int d, float eps, cudaStream_t stream, const int* tok_pos) {
  if (n <= 0 || prompt == nullptr) return ln_fwd_dispatch(x, gamma, beta, out, out_bf16, M, d, eps, nullptr, 1, 0, 0, nullptr, stream);
  if (tok_pos != nullptr) {
    if (row0 < 0) return "layernorm + splice: bad geometry";
    return ln_fwd_dispatch(x, gamma, beta, out, out_bf16, M, d, eps, prompt, 1, row0, n, tok_pos, stream);
  }
  if (L <= 0 || row0 < 0 || row0 + n > L || M % L != 0) return "layernorm + splice: bad geometry";
  return ln_fwd_dispatch(x, gamma, beta, out, out_bf16, M, d, eps, prompt, L, row0, n, nullptr, stream);
}

// Registers holding the residual-gradient piece of a lane: fp32 (float4) or the packed bf16 form (uint2)
template <bool BF16> struct ResidRegs;
template <> struct ResidRegs<false> {
  typedef float4 type;
  __device__ __forceinline__ static float4 zero() { return make_float4(0.f, 0.f, 0.f, 0.f); }
  __device__ __forceinline__ static float4 f32(const float4& r) { return r; }
};
template <> struct ResidRegs<true> {
  typedef uint2 type;
  __device__ __forceinline__ static uint2 zero() { return make_uint2(0u, 0u); }
  __device__ __forceinline__ static float4 f32(const uint2& r) {
    const float2 a = unpack_bf16(r.x), b = unpack_bf16(r.y);
    return make_float4(a.x, a.y, b.x, b.y);
  }
};

// ------------------------------------------------------------------ LayerNorm backward (dgrad only)
// dx = resid + rstd * (g - mean(g) - xhat * mean(g * xhat)),  g = dy * gamma.
// gamma/beta are frozen (trainers/mudpt.py:205-212): no dgamma/dbeta. Statistics are
// recomputed from the saved fp32 input row. dx may alias resid. Also emits the bf16 copy of dx
// that feeds the next dgrad GEMM.  DY_BF16: dy comes from a bf16 GEMM epilogue.
// X_STATS: the row comes as its bf16 copy + per-64-column partial statistics (the form the fused-LayerNorm forward
// keeps, rowops.cu "fused-LayerNorm plumbing"): 2 B instead of 4 B per element read, exact fp32 mean / rstd.
// RESID_BF16: the residual gradient is read from the bf16 copy of the stream (it may alias dx_bf16: every lane reads its
// own elements before it writes them).  win_n >= 0 restricts the fp32 output to the rows of the deep-prompt window,
// (row % win_L, or win_pos[row] for packed variable-length sequences) in [win_row0, win_row0 + win_n) -- the only fp32 rows anyone reads when the gradient stream is kept in
// bf16 (the splice backward sums them); win_n < 0: every row.  8 instead of 14 B per element on an HBM-bound kernel.
template <int NV, bool DY_BF16, bool X_STATS, bool RESID_BF16>
__global__ void __launch_bounds__(256, NV == 4 ? 4 : 1) ln_bwd_kernel(const void* __restrict__ dy, const void* __restrict__ xv,
                                                     const float2* __restrict__ stats, const float* __restrict__ gamma,
                                                     const void* resid, float* dx, bf16* dx_bf16, int M, int d,
                                                     float eps, int win_L, int win_row0, int win_n,
                                                     const int* __restrict__ win_pos) {
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  pdl_wait();
  pdl_trigger();
  if (row >= M) return;
  const size_t off = static_cast<size_t>(row) * d;
  const float* x = reinterpret_cast<const float*>(xv);
  bool write_f32 = dx != nullptr;  // (warp-uniform)
  if (win_n >= 0) {
    const int pos = (win_pos != nullptr ? win_pos[row] : row % win_L) - win_row0;
    write_f32 = write_f32 && pos >= 0 && pos < win_n;
  }
  float4 v[NV], g[NV];
  typename ResidRegs<RESID_BF16>::type rs[NV];
  float sum = 0.f;
  // issue every load of the row up front (x, dy, residual gradient): 3 streams in flight per lane.  The residual must be
  // in registers before the first store: dx may alias it, so a load placed after a store of the row is ordered behind it
  // and every 16-byte piece pays its own memory round trip (measured on the single-wave launches of 6-10 thousand rows)
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const int c = (i * 32 + lane) * 4;
    rs[i] = ResidRegs<RESID_BF16>::zero();
    if (c < d) {
      if (resid != nullptr) {
        if constexpr (RESID_BF16) rs[i] = *reinterpret_cast<const uint2*>(reinterpret_cast<const bf16*>(resid) + off + c);
        else rs[i] = *reinterpret_cast<const float4*>(reinterpret_cast<const float*>(resid) + off + c);
      }
      if constexpr (X_STATS) {
        const uint2 u = *reinterpret_cast<const uint2*>(reinterpret_cast<const bf16*>(xv) + off + c);
        const float2 a = unpack_bf16(u.x), b = unpack_bf16(u.y);
        v[i] = make_float4(a.x, a.y, b.x, b.y);
      } else {
        v[i] = *reinterpret_cast<const float4*>(x + off + c);
      }
      if constexpr (DY_BF16) {
        const uint2 u = *reinterpret_cast<const uint2*>(reinterpret_cast<const bf16*>(dy) + off + c);
        const float2 a = unpack_bf16(u.x), b = unpack_bf16(u.y);
        g[i] = make_float4(a.x, a.y, b.x, b.y);
      } else {
        g[i] = *reinterpret_cast<const float4*>(reinterpret_cast<const float*>(dy) + off + c);
      }
      sum += (v[i].x + v[i].y) + (v[i].z + v[i].w);
    }
  }
  float mean, rstd;
  if constexpr (X_STATS) {
    // lane p holds the partial of columns [64 p, 64 p + 64): exact pairwise combination (no cancellation)
    const int parts = (d + 63) >> 6;
    float2 st = make_float2(0.f, 0.f);
    float np = 0.f;
    if (lane < parts) {
      st = stats[static_cast<size_t>(row) * parts + lane];
      const int rem = d - lane * 64;
      np = static_cast<float>(rem < 64 ? rem : 64);
    }
    mean = warp_sum(st.x) / d;
    const float dm = np > 0.f ? st.x / np - mean : 0.f;
    rstd = rsqrtf(warp_sum(st.y + np * dm * dm) / d + eps);
#pragma unroll
    for (int i = 0; i < NV; ++i) { v[i].x -= mean; v[i].y -= mean; v[i].z -= mean; v[i].w -= mean; }
  } else {
    mean = warp_sum(sum) / d;
    float sq = 0.f;
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      const int c = (i * 32 + lane) * 4;
      if (c < d) {
        v[i].x -= mean; v[i].y -= mean; v[i].z -= mean; v[i].w -= mean;
        sq += (v[i].x * v[i].x + v[i].y * v[i].y) + (v[i].z * v[i].z + v[i].w * v[i].w);
      }
    }
    rstd = rsqrtf(warp_sum(sq) / d + eps);
  }
  float s1 = 0.f, s2 = 0.f;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const int c = (i * 32 + lane) * 4;
    if (c < d) {
      const float4 gm = *reinterpret_cast<const float4*>(gamma + c);
      v[i].x *= rstd; v[i].y *= rstd; v[i].z *= rstd; v[i].w *= rstd;  // xhat
      g[i].x *= gm.x; g[i].y *= gm.y; g[i].z *= gm.z; g[i].w *= gm.w;
      s1 += (g[i].x + g[i].y) + (g[i].z + g[i].w);
      s2 += (g[i].x * v[i].x + g[i].y * v[i].y) + (g[i].z * v[i].z + g[i].w * v[i].w);
    }
  }
  s1 = warp_sum(s1) / d;
  s2 = warp_sum(s2) / d;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const int c = (i * 32 + lane) * 4;
    if (c < d) {
      const float4 r = ResidRegs<RESID_BF16>::f32(rs[i]);
      float4 o;
      o.x = r.x + rstd * (g[i].x - s1 - v[i].x * s2);
      o.y = r.y + rstd * (g[i].y - s1 - v[i].y * s2);
      o.z = r.z + rstd * (g[i].z - s1 - v[i].z * s2);
      o.w = r.w + rstd * (g[i].w - s1 - v[i].w * s2);
      if (write_f32) *reinterpret_cast<float4*>(dx + off + c) = o;
      if (dx_bf16 != nullptr) {
        uint2 u;
        u.x = pack_bf16(o.x, o.y);
        u.y = pack_bf16(o.z, o.w);
        *reinterpret_cast<uint2*>(dx_bf16 + off + c) = u;
      }
    }
  }
}

template <int NV, bool RB>
static void launch_ln_bwd(const void* dy, bool dy_bf16, const void* x, const float2* stats, const float* gamma, const void* resid,
                          float* dx, bf16* dx_bf16, int M, int d, float eps, int win_L, int win_row0, int win_n,
                          const int* win_pos, cudaStream_t stream) {
  const int wpc = ln_warps();
  const int grid = (M + wpc - 1) / wpc;
  const dim3 blk(32 * wpc);
  if (stats != nullptr) {  // (bf16 dy only: the dgrad GEMM's output)
    launch_pdl(ln_bwd_kernel<NV, true, true, RB>, dim3(grid), blk, 0, stream, dy, x, stats, gamma, resid, dx, dx_bf16, M, d, eps,
               win_L, win_row0, win_n, win_pos);
  } else if (dy_bf16) {
    launch_pdl(ln_bwd_kernel<NV, true, false, RB>, dim3(grid), blk, 0, stream, dy, x, stats, gamma, resid, dx, dx_bf16, M, d, eps,
               win_L, win_row0, win_n, win_pos);
  } else {
    launch_pdl(ln_bwd_kernel<NV, false, false, RB>, dim3(grid), blk, 0, stream, dy, x, stats, gamma, resid, dx, dx_bf16, M, d, eps,
               win_L, win_row0, win_n, win_pos);
  }
}

template <bool RB>
static void dispatch_ln_bwd(const void* dy, bool dy_bf16, const void* x, const float2* stats, const float* gamma, const void* resid,
                            float* dx, bf16* dx_bf16, int M, int d, float eps, int win_L, int win_row0, int win_n,
                            const int* win_pos, cudaStream_t stream) {
  switch (pick_nv(d)) {
    case 1: launch_ln_bwd<1, RB>(dy, dy_bf16, x, stats, gamma, resid, dx, dx_bf16, M, d, eps, win_L, win_row0, win_n, win_pos, stream); break;
    case 2: launch_ln_bwd<2, RB>(dy, dy_bf16, x, stats, gamma, resid, dx, dx_bf16, M, d, eps, win_L, win_row0, win_n, win_pos, stream); break;
    case 4: launch_ln_bwd<4, RB>(dy, dy_bf16, x, stats, gamma, resid, dx, dx_bf16, M, d, eps, win_L, win_row0, win_n, win_pos, stream); break;
    case 6: launch_ln_bwd<6, RB>(dy, dy_bf16, x, stats, gamma, resid, dx, dx_bf16, M, d, eps, win_L, win_row0, win_n, win_pos, stream); break;
    default: launch_ln_bwd<8, RB>(dy, dy_bf16, x, stats, gamma, resid, dx, dx_bf16, M, d, eps, win_L, win_row0, win_n, win_pos, stream); break;
  }
}

// ------------------------------------------------------------------ LayerNorm backward over a row map
// out[r] = bf16(rstd (g - mean(g) - xhat mean(g xhat))), g = dy[src] * gamma, for the compact rows r < M, where the source
// row is src = (r / per) * L + row0 + r % per: one block of `per` rows out of every sequence of L rows.  fp32 dy and x,
// statistics recomputed from x, no residual.  The vision stem's ln_pre backward on the patch rows of every image (the
// output is the A operand of the patch dgrad GEMM); the same arithmetic as ln_bwd_kernel.
template <int NV>
__global__ void __launch_bounds__(256) ln_bwd_rows_kernel(const float* __restrict__ dy, const float* __restrict__ x,
                                                          const float* __restrict__ gamma, bf16* __restrict__ out, int M, int d,
                                                          float eps, int per, int L, int row0) {
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  pdl_wait();
  pdl_trigger();
  if (row >= M) return;
  const int seq = row / per;
  const size_t src = (static_cast<size_t>(seq) * L + row0 + (row - seq * per)) * d;
  float4 v[NV], g[NV];
  float sum = 0.f;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const int c = (i * 32 + lane) * 4;
    if (c < d) {
      v[i] = *reinterpret_cast<const float4*>(x + src + c);
      g[i] = *reinterpret_cast<const float4*>(dy + src + c);
      sum += (v[i].x + v[i].y) + (v[i].z + v[i].w);
    }
  }
  const float mean = warp_sum(sum) / d;
  float sq = 0.f;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const int c = (i * 32 + lane) * 4;
    if (c < d) {
      v[i].x -= mean; v[i].y -= mean; v[i].z -= mean; v[i].w -= mean;
      sq += (v[i].x * v[i].x + v[i].y * v[i].y) + (v[i].z * v[i].z + v[i].w * v[i].w);
    }
  }
  const float rstd = rsqrtf(warp_sum(sq) / d + eps);
  float s1 = 0.f, s2 = 0.f;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const int c = (i * 32 + lane) * 4;
    if (c < d) {
      const float4 gm = *reinterpret_cast<const float4*>(gamma + c);
      v[i].x *= rstd; v[i].y *= rstd; v[i].z *= rstd; v[i].w *= rstd;  // xhat
      g[i].x *= gm.x; g[i].y *= gm.y; g[i].z *= gm.z; g[i].w *= gm.w;
      s1 += (g[i].x + g[i].y) + (g[i].z + g[i].w);
      s2 += (g[i].x * v[i].x + g[i].y * v[i].y) + (g[i].z * v[i].z + g[i].w * v[i].w);
    }
  }
  s1 = warp_sum(s1) / d;
  s2 = warp_sum(s2) / d;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const int c = (i * 32 + lane) * 4;
    if (c < d) {
      float4 o;
      o.x = rstd * (g[i].x - s1 - v[i].x * s2);
      o.y = rstd * (g[i].y - s1 - v[i].y * s2);
      o.z = rstd * (g[i].z - s1 - v[i].z * s2);
      o.w = rstd * (g[i].w - s1 - v[i].w * s2);
      uint2 u;
      u.x = pack_bf16(o.x, o.y);
      u.y = pack_bf16(o.z, o.w);
      *reinterpret_cast<uint2*>(out + static_cast<size_t>(row) * d + c) = u;
    }
  }
}

template <int NV>
static void launch_ln_bwd_rows(const float* dy, const float* x, const float* gamma, bf16* out, int M, int d, float eps, int per,
                               int L, int row0, cudaStream_t stream) {
  const int wpc = ln_warps();
  launch_pdl(ln_bwd_rows_kernel<NV>, dim3((M + wpc - 1) / wpc), dim3(32 * wpc), 0, stream, dy, x, gamma, out, M, d, eps, per, L, row0);
}

const char* layernorm_bwd_rows(const float* dy, const float* x, const float* gamma, bf16* out, int M, int d, float eps, int per,
                               int L, int row0, cudaStream_t stream) {
  if (M <= 0) return nullptr;
  if (d % 4 != 0 || d > LN_MAXV * 128) return "layernorm: width must be a multiple of 4 and <= 1024";
  if (per <= 0 || row0 < 0 || row0 + per > L) return "layernorm bwd (row map): bad geometry";
  switch (pick_nv(d)) {
    case 1: launch_ln_bwd_rows<1>(dy, x, gamma, out, M, d, eps, per, L, row0, stream); break;
    case 2: launch_ln_bwd_rows<2>(dy, x, gamma, out, M, d, eps, per, L, row0, stream); break;
    case 4: launch_ln_bwd_rows<4>(dy, x, gamma, out, M, d, eps, per, L, row0, stream); break;
    case 6: launch_ln_bwd_rows<6>(dy, x, gamma, out, M, d, eps, per, L, row0, stream); break;
    default: launch_ln_bwd_rows<8>(dy, x, gamma, out, M, d, eps, per, L, row0, stream); break;
  }
  count_launch(1);
  return launch_status("layernorm bwd (row map) launch failed");
}

// ------------------------------------------------------------------ LayerNorm backward, shared-memory pipeline
// The register kernel above has one row per warp in flight: measured on the bf16 gradient stream it moves 3.5 TB/s where
// 6.5 are available (ncu: every warp waits a full DRAM round trip per row, 45 % of the warp slots, no byte in flight while
// a row is being reduced).  Here the loads are taken off the warps: a persistent CTA walks blocks of 8 consecutive
// rows; ONE thread issues the block's rows -- contiguous in memory, so one 1-D bulk copy (cp.async.bulk, the TMA engine)
// per operand: dy, x, residual gradient, statistics -- into a ring of `stages` shared-memory slots that complete on
// mbarriers, `stages - 1` blocks ahead of the math; the 8 warps take a row each from the slot into registers, the slot is
// refilled at once (the bytes in flight per SM no longer depend on occupancy), and the row is reduced and stored from
// registers.  The residual gradient may alias the bf16 output: a row is read (bulk copy completed) before the same CTA
// writes it, and no other CTA touches it.
__device__ __forceinline__ void bulk_load_1d(void* smem_dst, const void* gsrc, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(smem_dst)),
               "l"(gsrc), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void warp_sum2(float& a, float& b) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    a += __shfl_xor_sync(0xffffffffu, a, o);
    b += __shfl_xor_sync(0xffffffffu, b, o);
  }
}
__device__ __forceinline__ void unpack8_bf16(const uint4& u, float (&f)[8]) {
  const float2 a = unpack_bf16(u.x), b = unpack_bf16(u.y), c = unpack_bf16(u.z), e = unpack_bf16(u.w);
  f[0] = a.x; f[1] = a.y; f[2] = b.x; f[3] = b.y; f[4] = c.x; f[5] = c.y; f[6] = e.x; f[7] = e.y;
}

struct LnPipeArgs {
  const bf16* dy;
  const void* x;        // bf16 rows (X_STATS) or fp32 rows
  const float2* stats;  // X_STATS: [M, d / 64] partial (sum, M2)
  const float* gamma;
  const void* resid;    // RESID 1: bf16 rows (may alias dx_bf16), 2: fp32 rows
  float* dx;            // fp32 output (window rows only when win_n >= 0) or null
  bf16* dx_bf16;        // bf16 output or null
  int M, d;
  float eps;
  int win_L, win_row0, win_n;
  const int* win_pos;   // or null: the window position of a row is row % win_L
  int stages;
  unsigned stage_bytes;
};

static constexpr int kPipeBarBytes = 128;
__host__ __device__ constexpr unsigned align128(unsigned v) { return (v + 127u) & ~127u; }

// d = NP * 256 exactly: lane l owns the 8 columns [(i * 32 + l) * 8, +8) of piece i < NP, no width predicates (other widths
// take the register kernel).  RESID: 0 none, 1 bf16, 2 fp32.  One row per warp and block (two rows per warp -- 16 KB bulk
// copies, half the barriers -- measured no faster and need twice the ring).  Addresses, ring slot / phase and the position in
// the deep-prompt window advance incrementally: the first version spent 40 % of its 480 instructions per row on 64-bit index
// arithmetic, width predicates and divisions (ncu source page), and the kernel is issue-bound once the loads are off the warps.
template <int NP, bool X_STATS, int RESID>
__global__ void __launch_bounds__(256) ln_bwd_pipe_kernel(const LnPipeArgs a) {
  extern __shared__ __align__(128) uint8_t ln_pipe_smem[];
  constexpr int ROWS = 8;  // one row per warp
  constexpr unsigned d = NP * 256u;
  constexpr unsigned XB = X_STATS ? 2u : 4u;
  constexpr unsigned RB = RESID == 1 ? 2u : (RESID == 2 ? 4u : 0u);
  constexpr unsigned parts = d >> 6;
  constexpr unsigned dy_off = 0, x_off = ROWS * d * 2u, r_off = x_off + ROWS * d * XB, st_off = r_off + ROWS * d * RB;
  const unsigned warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  uint64_t* full = reinterpret_cast<uint64_t*>(ln_pipe_smem);
  float* gam = reinterpret_cast<float*>(ln_pipe_smem + kPipeBarBytes);
  uint8_t* stage0 = ln_pipe_smem + kPipeBarBytes + align128(d * 4u);
  const int nblk = (a.M + ROWS - 1) / ROWS;
  const int stages = a.stages;
  if (threadIdx.x == 0) {
    for (int s = 0; s < stages; ++s) mbar_init(&full[s], 1);
    fence_mbar_init();
  }
  __syncthreads();
  pdl_wait();
  auto issue = [&](int blk, int s) {  // one thread: the rows of block `blk` into slot `s`
    const int r0 = blk * ROWS;
    const unsigned nr = static_cast<unsigned>(a.M - r0 < ROWS ? a.M - r0 : ROWS);
    uint8_t* st = stage0 + static_cast<size_t>(s) * a.stage_bytes;
    mbar_expect_tx(&full[s], nr * d * (2u + XB + RB) + (X_STATS ? nr * parts * 8u : 0u));
    bulk_load_1d(st + dy_off, a.dy + static_cast<size_t>(r0) * d, nr * d * 2u, &full[s]);
    bulk_load_1d(st + x_off, reinterpret_cast<const uint8_t*>(a.x) + static_cast<size_t>(r0) * d * XB, nr * d * XB, &full[s]);
    if constexpr (RESID != 0)
      bulk_load_1d(st + r_off, reinterpret_cast<const uint8_t*>(a.resid) + static_cast<size_t>(r0) * d * RB, nr * d * RB, &full[s]);
    if constexpr (X_STATS) bulk_load_1d(st + st_off, a.stats + static_cast<size_t>(r0) * parts, nr * parts * 8u, &full[s]);
  };
  if (threadIdx.x == 0) {
    for (int s = 0; s < stages; ++s) {
      const int blk = blockIdx.x + s * gridDim.x;
      if (blk < nblk) issue(blk, s);
    }
  }
  for (unsigned c = threadIdx.x * 4; c < d; c += 256 * 4) *reinterpret_cast<float4*>(gam + c) = *reinterpret_cast<const float4*>(a.gamma + c);
  pdl_trigger();
  __syncthreads();  // gamma staged
  constexpr float inv_d = 1.f / static_cast<float>(d);
  // this warp's row inside a slot, this lane's 8 columns inside a piece
  const unsigned o_dy = dy_off + warp * d * 2u + lane * 16u;
  const unsigned o_x = x_off + warp * d * XB + lane * 8u * XB;
  const unsigned o_r = r_off + warp * d * RB + lane * 8u * RB;
  const unsigned o_st = st_off + (warp * parts + lane) * 8u;
  const float* gl = gam + lane * 8u;
  const float np = lane < parts ? 64.f : 0.f;  // (d is a multiple of 64: every partial statistic covers 64 columns)
  const bool windowed = a.win_n >= 0;
  const int row_step = ROWS * static_cast<int>(gridDim.x);
  int row = static_cast<int>(blockIdx.x) * ROWS + static_cast<int>(warp);
  int pos = 0, pos_step = 0;  // row % win_L, advanced without a division per row
  if (windowed) {
    pos = row % a.win_L;
    pos_step = row_step % a.win_L;
  }
  int s = 0;
  uint32_t phase = 0;
  const uint8_t* st = stage0;
  for (int blk = blockIdx.x; blk < nblk; blk += gridDim.x) {
    mbar_wait(&full[s], phase);
    // ---- the row: shared memory -> registers
    float gg[NP][8], xc[NP][8];
    uint4 rq[RESID == 1 ? NP : 1];
    float4 rf[RESID == 2 ? NP : 1][2];
    float2 stp = make_float2(0.f, 0.f);
#pragma unroll
    for (int i = 0; i < NP; ++i) {
      unpack8_bf16(*reinterpret_cast<const uint4*>(st + o_dy + i * 512u), gg[i]);
      if constexpr (X_STATS) {
        unpack8_bf16(*reinterpret_cast<const uint4*>(st + o_x + i * 512u), xc[i]);
      } else {
        const float4 u0 = *reinterpret_cast<const float4*>(st + o_x + i * 1024u);
        const float4 u1 = *reinterpret_cast<const float4*>(st + o_x + i * 1024u + 16u);
        xc[i][0] = u0.x; xc[i][1] = u0.y; xc[i][2] = u0.z; xc[i][3] = u0.w;
        xc[i][4] = u1.x; xc[i][5] = u1.y; xc[i][6] = u1.z; xc[i][7] = u1.w;
      }
      if constexpr (RESID == 1) rq[i] = *reinterpret_cast<const uint4*>(st + o_r + i * 512u);
      if constexpr (RESID == 2) {
        rf[i][0] = *reinterpret_cast<const float4*>(st + o_r + i * 1024u);
        rf[i][1] = *reinterpret_cast<const float4*>(st + o_r + i * 1024u + 16u);
      }
    }
    if constexpr (X_STATS) {
      if (lane < parts) stp = *reinterpret_cast<const float2*>(st + o_st);
    }
    __syncthreads();  // every warp holds its row: the slot is free
    if (threadIdx.x == 0) {
      const int nb = blk + stages * static_cast<int>(gridDim.x);
      fence_proxy_async_smem();  // the warps' reads of the slot (ordered by the barrier) before the async-proxy refill
      if (nb < nblk) issue(nb, s);
    }
    if (++s == stages) { s = 0; phase ^= 1u; st = stage0; } else { st += a.stage_bytes; }
    if (row < a.M) {  // (warp-uniform)
      // ---- g = dy * gamma, s1 = mean(g); mean of x
      float s1 = 0.f, sx = 0.f;
#pragma unroll
      for (int i = 0; i < NP; ++i) {
        const float4 g0 = *reinterpret_cast<const float4*>(gl + i * 256), g1 = *reinterpret_cast<const float4*>(gl + i * 256 + 4);
        gg[i][0] *= g0.x; gg[i][1] *= g0.y; gg[i][2] *= g0.z; gg[i][3] *= g0.w;
        gg[i][4] *= g1.x; gg[i][5] *= g1.y; gg[i][6] *= g1.z; gg[i][7] *= g1.w;
        s1 += ((gg[i][0] + gg[i][1]) + (gg[i][2] + gg[i][3])) + ((gg[i][4] + gg[i][5]) + (gg[i][6] + gg[i][7]));
        if constexpr (!X_STATS)
          sx += ((xc[i][0] + xc[i][1]) + (xc[i][2] + xc[i][3])) + ((xc[i][4] + xc[i][5]) + (xc[i][6] + xc[i][7]));
      }
      if constexpr (X_STATS) sx = stp.x;
      warp_sum2(s1, sx);
      s1 *= inv_d;
      const float mean = sx * inv_d;
      // ---- centred row, its second moment (exact: partial M2 + shift, or recomputed) and C = sum g (x - mean)
      float m2 = 0.f, cc = 0.f;
#pragma unroll
      for (int i = 0; i < NP; ++i) {
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          xc[i][j] -= mean;
          cc = fmaf(gg[i][j], xc[i][j], cc);
          if constexpr (!X_STATS) m2 = fmaf(xc[i][j], xc[i][j], m2);
        }
      }
      if constexpr (X_STATS) {
        const float dm = np > 0.f ? stp.x * (1.f / 64.f) - mean : 0.f;
        m2 = stp.y + np * dm * dm;
      }
      warp_sum2(m2, cc);
      const float rstd = rsqrtf(m2 * inv_d + a.eps);
      const float k2 = -(rstd * rstd * rstd * (cc * inv_d));  // -rstd^2 * s2 with s2 = mean(g * xhat) = rstd * mean(g (x - mean))
      const float c0 = -rstd * s1;
      // ---- dx = resid + rstd * (g - s1 - xhat * s2) = (resid - rstd * s1) + rstd * g - (x - mean) * rstd^3 * mean(g (x - mean))
      const int wp = a.win_pos != nullptr ? a.win_pos[row] : pos;
      const bool write_f32 = a.dx != nullptr && (!windowed || (wp >= a.win_row0 && wp < a.win_row0 + a.win_n));
      const size_t off = static_cast<size_t>(row) * d + lane * 8u;
#pragma unroll
      for (int i = 0; i < NP; ++i) {
        float r[8];
        if constexpr (RESID == 1) {
          unpack8_bf16(rq[i], r);
        } else if constexpr (RESID == 2) {
          r[0] = rf[i][0].x; r[1] = rf[i][0].y; r[2] = rf[i][0].z; r[3] = rf[i][0].w;
          r[4] = rf[i][1].x; r[5] = rf[i][1].y; r[6] = rf[i][1].z; r[7] = rf[i][1].w;
        } else {
#pragma unroll
          for (int j = 0; j < 8; ++j) r[j] = 0.f;
        }
        float o[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) o[j] = fmaf(k2, xc[i][j], fmaf(rstd, gg[i][j], r[j] + c0));
        if (write_f32) {
          *reinterpret_cast<float4*>(a.dx + off + i * 256) = make_float4(o[0], o[1], o[2], o[3]);
          *reinterpret_cast<float4*>(a.dx + off + i * 256 + 4) = make_float4(o[4], o[5], o[6], o[7]);
        }
        if (a.dx_bf16 != nullptr) {
          uint4 u;
          u.x = pack_bf16(o[0], o[1]); u.y = pack_bf16(o[2], o[3]); u.z = pack_bf16(o[4], o[5]); u.w = pack_bf16(o[6], o[7]);
          *reinterpret_cast<uint4*>(a.dx_bf16 + off + i * 256) = u;
        }
      }
    }
    row += row_step;
    if (windowed) {
      pos += pos_step;
      if (pos >= a.win_L) pos -= a.win_L;
    }
  }
}

// LayerNorm forward (bf16 output, optional deep-prompt splice) on the same pipeline (clip/model.py:299-300).  An experiment that
// did not pay at the shapes where the forward LayerNorm is a stand-alone kernel (see ln_fwd_pipe_mode()): kept behind
// MUDPT_LN_FWD_PIPE=1 for towers whose forward LayerNorm is not folded into the GEMMs at tens of thousands of rows.
struct LnFwdPipeArgs {
  const float* x;   // fp32 rows (read by the bulk copies)
  float* x_w;       // the same buffer: spliced rows are written back (rows no bulk copy of another CTA reads)
  const float* gamma;
  const float* beta;
  bf16* out;
  int M;
  float eps;
  const float* sp_prompt;  // or null
  int sp_L, sp_row0, sp_n;
  const int* sp_pos;       // or null: the position of a row is row % sp_L
  int stages;
  unsigned stage_bytes;
};

template <int NP>
__global__ void __launch_bounds__(256) ln_fwd_pipe_kernel(const LnFwdPipeArgs a) {
  extern __shared__ __align__(128) uint8_t ln_pipe_smem[];
  constexpr int ROWS = 8;
  constexpr unsigned d = NP * 256u;
  const unsigned warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  uint64_t* full = reinterpret_cast<uint64_t*>(ln_pipe_smem);
  float* gam = reinterpret_cast<float*>(ln_pipe_smem + kPipeBarBytes);
  float* bet = gam + d;
  uint8_t* stage0 = ln_pipe_smem + kPipeBarBytes + align128(d * 8u);
  const int nblk = (a.M + ROWS - 1) / ROWS;
  const int stages = a.stages;
  if (threadIdx.x == 0) {
    for (int s = 0; s < stages; ++s) mbar_init(&full[s], 1);
    fence_mbar_init();
  }
  __syncthreads();
  pdl_wait();
  auto issue = [&](int blk, int s) {
    const int r0 = blk * ROWS;
    const unsigned nr = static_cast<unsigned>(a.M - r0 < ROWS ? a.M - r0 : ROWS);
    mbar_expect_tx(&full[s], nr * d * 4u);
    bulk_load_1d(stage0 + static_cast<size_t>(s) * a.stage_bytes, a.x + static_cast<size_t>(r0) * d, nr * d * 4u, &full[s]);
  };
  if (threadIdx.x == 0) {
    for (int s = 0; s < stages; ++s) {
      const int blk = blockIdx.x + s * gridDim.x;
      if (blk < nblk) issue(blk, s);
    }
  }
  for (unsigned c = threadIdx.x * 4; c < d; c += 256 * 4) {
    *reinterpret_cast<float4*>(gam + c) = *reinterpret_cast<const float4*>(a.gamma + c);
    *reinterpret_cast<float4*>(bet + c) = *reinterpret_cast<const float4*>(a.beta + c);
  }
  pdl_trigger();
  __syncthreads();
  constexpr float inv_d = 1.f / static_cast<float>(d);
  const unsigned o_x = warp * d * 4u + lane * 32u;
  const float* gl = gam + lane * 8u;
  const float* bl = bet + lane * 8u;
  const bool splicing = a.sp_prompt != nullptr;
  const int row_step = ROWS * static_cast<int>(gridDim.x);
  int row = static_cast<int>(blockIdx.x) * ROWS + static_cast<int>(warp);
  int pos = 0, pos_step = 0;
  if (splicing) {
    pos = row % a.sp_L;
    pos_step = row_step % a.sp_L;
  }
  int s = 0;
  uint32_t phase = 0;
  const uint8_t* st = stage0;
  for (int blk = blockIdx.x; blk < nblk; blk += gridDim.x) {
    mbar_wait(&full[s], phase);
    float xv[NP][8];
#pragma unroll
    for (int i = 0; i < NP; ++i) {
      const float4 u0 = *reinterpret_cast<const float4*>(st + o_x + i * 1024u);
      const float4 u1 = *reinterpret_cast<const float4*>(st + o_x + i * 1024u + 16u);
      xv[i][0] = u0.x; xv[i][1] = u0.y; xv[i][2] = u0.z; xv[i][3] = u0.w;
      xv[i][4] = u1.x; xv[i][5] = u1.y; xv[i][6] = u1.z; xv[i][7] = u1.w;
    }
    __syncthreads();  // every warp holds its row: the slot is free
    if (threadIdx.x == 0) {
      const int nb = blk + stages * static_cast<int>(gridDim.x);
      fence_proxy_async_smem();
      if (nb < nblk) issue(nb, s);
    }
    if (++s == stages) { s = 0; phase ^= 1u; st = stage0; } else { st += a.stage_bytes; }
    if (row < a.M) {  // (warp-uniform)
      const size_t off = static_cast<size_t>(row) * d + lane * 8u;
      const int sp = a.sp_pos != nullptr ? a.sp_pos[row] : pos;
      if (splicing && sp >= a.sp_row0 && sp < a.sp_row0 + a.sp_n) {
        // the deep-prompt splice of the block (clip/model.py:281-297): the row takes the prompt's values, copied verbatim
        // into the residual stream (bit-exact), and is normalised like any other
        const float* src = a.sp_prompt + static_cast<size_t>(sp - a.sp_row0) * d + lane * 8u;
#pragma unroll
        for (int i = 0; i < NP; ++i) {
          const float4 u0 = *reinterpret_cast<const float4*>(src + i * 256), u1 = *reinterpret_cast<const float4*>(src + i * 256 + 4);
          xv[i][0] = u0.x; xv[i][1] = u0.y; xv[i][2] = u0.z; xv[i][3] = u0.w;
          xv[i][4] = u1.x; xv[i][5] = u1.y; xv[i][6] = u1.z; xv[i][7] = u1.w;
          *reinterpret_cast<float4*>(a.x_w + off + i * 256) = u0;
          *reinterpret_cast<float4*>(a.x_w + off + i * 256 + 4) = u1;
        }
      }
      float sum = 0.f;
#pragma unroll
      for (int i = 0; i < NP; ++i)
        sum += ((xv[i][0] + xv[i][1]) + (xv[i][2] + xv[i][3])) + ((xv[i][4] + xv[i][5]) + (xv[i][6] + xv[i][7]));
      const float mean = warp_sum(sum) * inv_d;
      float sq = 0.f;
#pragma unroll
      for (int i = 0; i < NP; ++i) {
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          xv[i][j] -= mean;
          sq = fmaf(xv[i][j], xv[i][j], sq);
        }
      }
      const float rstd = rsqrtf(warp_sum(sq) * inv_d + a.eps);
#pragma unroll
      for (int i = 0; i < NP; ++i) {
        const float4 g0 = *reinterpret_cast<const float4*>(gl + i * 256), g1 = *reinterpret_cast<const float4*>(gl + i * 256 + 4);
        const float4 b0 = *reinterpret_cast<const float4*>(bl + i * 256), b1 = *reinterpret_cast<const float4*>(bl + i * 256 + 4);
        uint4 u;
        u.x = pack_bf16(fmaf(xv[i][0] * rstd, g0.x, b0.x), fmaf(xv[i][1] * rstd, g0.y, b0.y));
        u.y = pack_bf16(fmaf(xv[i][2] * rstd, g0.z, b0.z), fmaf(xv[i][3] * rstd, g0.w, b0.w));
        u.z = pack_bf16(fmaf(xv[i][4] * rstd, g1.x, b1.x), fmaf(xv[i][5] * rstd, g1.y, b1.y));
        u.w = pack_bf16(fmaf(xv[i][6] * rstd, g1.z, b1.z), fmaf(xv[i][7] * rstd, g1.w, b1.w));
        *reinterpret_cast<uint4*>(a.out + off + i * 256) = u;
      }
    }
    row += row_step;
    if (splicing) {
      pos += pos_step;
      if (pos >= a.sp_L) pos -= a.sp_L;
    }
  }
}

static int ln_pipe_env(const char* name, int dflt) {
  const char* e = getenv(name);
  return e ? atoi(e) : dflt;
}

static const char kLnPipeNoFit[] = "layernorm bwd (pipeline): row too wide for the shared-memory ring";

template <int NP, bool X_STATS, int RESID>
static const char* launch_ln_pipe(LnPipeArgs a, cudaStream_t stream) {
  constexpr int ROWS = 8;
  auto kern = ln_bwd_pipe_kernel<NP, X_STATS, RESID>;
  static int sms = 0;
  static bool attr_done = false;
  if (!attr_done) {
    if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024 - 1024) != cudaSuccess)
      return "layernorm bwd (pipeline): cudaFuncSetAttribute failed";
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    if (sms <= 0) sms = 148;
    attr_done = true;
  }
  const unsigned row_bytes = static_cast<unsigned>(a.d) * (2u + (X_STATS ? 2u : 4u) + (RESID == 1 ? 2u : RESID == 2 ? 4u : 0u)) +
                             (X_STATS ? static_cast<unsigned>(a.d >> 6) * 8u : 0u);
  a.stage_bytes = align128(ROWS * row_bytes);
  const unsigned fixed = kPipeBarBytes + align128(a.d * 4u);
  // As many CTAs per SM as fit with at least 2 slots each, at most 3 (registers), at most 4 slots.  Measured on the text
  // tower (77,000 x 512, 315 MB): 3 CTAs x 2 slots 52 us (0.92 of HBM), 2 x 4 slots 61 us, 1 x 4 slots 94 us, register kernel
  // 87 us -- the warps' row math is what has to be covered, not the depth of the ring (profiles/r02_ln_bwd_pipe.txt)
  static const int want_ctas = ln_pipe_env("MUDPT_LN_PIPE_CTAS", 3);
  static const int want_stages = ln_pipe_env("MUDPT_LN_PIPE_STAGES", 4);
  // registers bound the co-resident CTAs too (the persistent grid must not be larger than what runs at once: a CTA that
  // waits for a free SM starts its share when the others are done)
  static int reg_ctas = 0;
  if (reg_ctas == 0) {
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&reg_ctas, kern, 256, 0) != cudaSuccess || reg_ctas < 1) reg_ctas = 1;
  }
  int ctas = want_ctas < 1 ? 1 : (want_ctas < reg_ctas ? want_ctas : reg_ctas);
  int stages = 0;
  for (; ctas >= 1; --ctas) {
    const unsigned budget = (227u * 1024u - 1024u * ctas) / ctas;  // 1 KB per CTA is reserved by the driver
    stages = budget > fixed ? static_cast<int>((budget - fixed) / a.stage_bytes) : 0;
    if (stages >= 2) break;
  }
  if (ctas < 1 || stages < 2) return kLnPipeNoFit;  // (the caller falls back to the register kernel)
  if (stages > want_stages) stages = want_stages < 2 ? 2 : want_stages;
  if (stages > 8) stages = 8;
  a.stages = stages;
  const int nblk = (a.M + ROWS - 1) / ROWS;
  const int grid = nblk < ctas * sms ? nblk : ctas * sms;
  launch_pdl(kern, dim3(grid), dim3(256), fixed + static_cast<size_t>(stages) * a.stage_bytes, stream, a);
  return nullptr;
}

template <bool X_STATS, int RESID>
static const char* dispatch_ln_pipe_np(const LnPipeArgs& a, cudaStream_t stream) {
  switch ((a.d + 255) / 256) {
    case 1: return launch_ln_pipe<1, X_STATS, RESID>(a, stream);
    case 2: return launch_ln_pipe<2, X_STATS, RESID>(a, stream);
    case 3: return launch_ln_pipe<3, X_STATS, RESID>(a, stream);
    default: return launch_ln_pipe<4, X_STATS, RESID>(a, stream);
  }
}

static const char* dispatch_ln_pipe(const LnPipeArgs& a, bool x_stats, int resid, cudaStream_t stream) {
  if (x_stats) {
    return resid == 0 ? dispatch_ln_pipe_np<true, 0>(a, stream)
                      : resid == 1 ? dispatch_ln_pipe_np<true, 1>(a, stream) : dispatch_ln_pipe_np<true, 2>(a, stream);
  }
  return resid == 0 ? dispatch_ln_pipe_np<false, 0>(a, stream)
                    : resid == 1 ? dispatch_ln_pipe_np<false, 1>(a, stream) : dispatch_ln_pipe_np<false, 2>(a, stream);
}

// MUDPT_LN_BWD_PIPE: 0 = register kernel only, 1 (default) = shared-memory pipeline where it applies
static int ln_bwd_pipe_mode() {
  static const int m = ln_pipe_env("MUDPT_LN_BWD_PIPE", 1);
  return m;
}

// MUDPT_LN_FWD_PIPE: 1 = the pipeline for bf16-output LayerNorm forward of 512 / 768 / 1024-wide rows, 0 (default) = register
// kernel.  Measured (profiles/r02_ln_bwd_pipe.txt): at the 6-10 thousand rows of the stand-alone forward LayerNorms the
// pipeline is SLOWER (12.5 against 10.9 us per launch; N = 1 vision tower 13.3 against 12.0): with one operand and 2.7 rounds
// of row blocks its prologue (barriers, gamma / beta staging, the first bulk copy) is not amortised.  Parity-tested, off.
static int ln_fwd_pipe_mode() {
  static const int m = ln_pipe_env("MUDPT_LN_FWD_PIPE", 0);
  return m;
}

template <int NP>
static const char* launch_ln_fwd_pipe(LnFwdPipeArgs a, cudaStream_t stream) {
  constexpr int ROWS = 8;
  constexpr unsigned d = NP * 256u;
  auto kern = ln_fwd_pipe_kernel<NP>;
  static int sms = 0, reg_ctas = 0;
  static bool attr_done = false;
  if (!attr_done) {
    if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024 - 1024) != cudaSuccess)
      return "layernorm fwd (pipeline): cudaFuncSetAttribute failed";
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    if (sms <= 0) sms = 148;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&reg_ctas, kern, 256, 0) != cudaSuccess || reg_ctas < 1) reg_ctas = 1;
    attr_done = true;
  }
  a.stage_bytes = ROWS * d * 4u;
  const unsigned fixed = kPipeBarBytes + align128(d * 8u);
  static const int want_ctas = ln_pipe_env("MUDPT_LN_PIPE_CTAS", 3);
  static const int want_stages = ln_pipe_env("MUDPT_LN_PIPE_STAGES", 4);
  int ctas = want_ctas < 1 ? 1 : (want_ctas < reg_ctas ? want_ctas : reg_ctas);
  int stages = 0;
  for (; ctas >= 1; --ctas) {
    const unsigned budget = (227u * 1024u - 1024u * ctas) / ctas;
    stages = budget > fixed ? static_cast<int>((budget - fixed) / a.stage_bytes) : 0;
    if (stages >= 2) break;
  }
  if (ctas < 1 || stages < 2) return kLnPipeNoFit;
  if (stages > want_stages) stages = want_stages < 2 ? 2 : want_stages;
  if (stages > 8) stages = 8;
  a.stages = stages;
  const int nblk = (a.M + ROWS - 1) / ROWS;
  const int grid = nblk < ctas * sms ? nblk : ctas * sms;
  launch_pdl(kern, dim3(grid), dim3(256), fixed + static_cast<size_t>(stages) * a.stage_bytes, stream, a);
  return nullptr;
}

static bool ln_fwd_pipe_try(float* x, const float* gamma, const float* beta, bf16* out, int M, int d, float eps, const float* sp_prompt,
                            int sp_L, int sp_row0, int sp_n, const int* sp_pos, cudaStream_t stream, const char** err) {
  *err = nullptr;
  if (ln_fwd_pipe_mode() <= 0 || d % 256 != 0 || d > 1024 || M < 64) return false;
  LnFwdPipeArgs a;
  a.x = x; a.x_w = x; a.gamma = gamma; a.beta = beta; a.out = out; a.M = M; a.eps = eps;
  a.sp_prompt = sp_prompt; a.sp_L = sp_L > 0 ? sp_L : 1; a.sp_row0 = sp_row0; a.sp_n = sp_n; a.sp_pos = sp_pos; a.stages = 0; a.stage_bytes = 0;
  const char* e = d == 256 ? launch_ln_fwd_pipe<1>(a, stream)
                           : d == 512 ? launch_ln_fwd_pipe<2>(a, stream) : d == 768 ? launch_ln_fwd_pipe<3>(a, stream) : launch_ln_fwd_pipe<4>(a, stream);
  if (e == kLnPipeNoFit) return false;
  *err = e;
  return true;
}

// x: fp32 rows, or (stats != nullptr) their bf16 copy with the per-64-column partial statistics.
// resid: fp32 rows, or (resid_bf16) the bf16 copy of the gradient stream; dx (fp32) and dx_bf16 may each be null (not both);
// win_n >= 0: fp32 rows are written inside the deep-prompt window only (see the kernel).
const char* layernorm_bwd_stream(const void* dy, bool dy_bf16, const void* x, const float2* stats, const float* gamma,
                                 const void* resid, bool resid_bf16, float* dx, bf16* dx_bf16, int M, int d, float eps,
                                 int win_L, int win_row0, int win_n, cudaStream_t stream, const int* win_pos) {
  if (M <= 0) return nullptr;
  if (d % 4 != 0 || d > LN_MAXV * 128) return "layernorm: width must be a multiple of 4 and <= 1024";
  if (stats != nullptr && (!dy_bf16 || d % 64 != 0)) return "layernorm: the bf16-input form needs bf16 dy and width % 64 == 0";
  if (dx == nullptr && dx_bf16 == nullptr) return "layernorm bwd: no output";
  if (win_pos != nullptr) win_L = 1;  // (positions come from win_pos)
  if (win_n > 0 && win_pos == nullptr && (win_L <= 0 || win_row0 < 0 || win_row0 + win_n > win_L)) return "layernorm bwd: bad window";
  if (win_n >= 0 && win_L <= 0) win_L = 1;
  // bf16 dy, width a multiple of 256 (one 8-column piece per lane and 256 columns: 512 / 768 / 1024, the widths of the CLIP towers)
  if (ln_bwd_pipe_mode() > 0 && dy_bf16 && d % 256 == 0 && M >= 64) {
    LnPipeArgs a;
    a.dy = reinterpret_cast<const bf16*>(dy); a.x = x; a.stats = stats; a.gamma = gamma; a.resid = resid; a.dx = dx; a.dx_bf16 = dx_bf16;
    a.M = M; a.d = d; a.eps = eps; a.win_L = win_L; a.win_row0 = win_row0; a.win_n = win_n; a.win_pos = win_pos; a.stages = 0; a.stage_bytes = 0;
    const int rk = resid == nullptr ? 0 : (resid_bf16 ? 1 : 2);
    const char* e = dispatch_ln_pipe(a, stats != nullptr, rk, stream);
    if (e == nullptr) {
      count_launch(1);
      return launch_status("layernorm bwd (pipeline) launch failed");
    }
    if (e != kLnPipeNoFit) return e;
  }
  if (resid_bf16 && resid != nullptr)
    dispatch_ln_bwd<true>(dy, dy_bf16, x, stats, gamma, resid, dx, dx_bf16, M, d, eps, win_L, win_row0, win_n, win_pos, stream);
  else
    dispatch_ln_bwd<false>(dy, dy_bf16, x, stats, gamma, resid, dx, dx_bf16, M, d, eps, win_L, win_row0, win_n, win_pos, stream);
  count_launch(1);
  return launch_status("layernorm bwd launch failed");
}

const char* layernorm_bwd(const void* dy, bool dy_bf16, const void* x, const float2* stats, const float* gamma, const float* resid,
                          float* dx, bf16* dx_bf16, int M, int d, float eps, cudaStream_t stream) {
  if (dx == nullptr) return "layernorm bwd: no fp32 output";
  return layernorm_bwd_stream(dy, dy_bf16, x, stats, gamma, resid, false, dx, dx_bf16, M, d, eps, 1, 0, -1, stream);
}

// ------------------------------------------------------------------ deep-prompt splice
// x[s, row0 + r, :] = prompt[r, :] for every sequence s: the values are copied verbatim.
__global__ void splice_fwd_kernel(float* __restrict__ x, const float* __restrict__ prompt, int L, int row0, int n, int d) {
  const int s = blockIdx.x, r = blockIdx.y;
  pdl_wait();
  pdl_trigger();
  float4* dst = reinterpret_cast<float4*>(x + (static_cast<size_t>(s) * L + row0 + r) * d);
  const float4* src = reinterpret_cast<const float4*>(prompt + static_cast<size_t>(r) * d);
  for (int c = threadIdx.x; c < d / 4; c += blockDim.x) dst[c] = src[c];
}

const char* splice_fwd(float* x, const float* prompt, int S, int L, int row0, int n, int d, cudaStream_t stream) {
  if (S <= 0 || n <= 0) return nullptr;
  if (d % 4 != 0 || row0 < 0 || row0 + n > L) return "splice: bad geometry";
  launch_pdl(splice_fwd_kernel, dim3(S, n), dim3(128), 0, stream, x, prompt, L, row0, n, d);
  count_launch(1);
  return launch_status("splice fwd launch failed");
}

// dprompt[r, :] = sum_s dx[s, row0 + r, :] (packed variable-length sequences: row seq_off[s] + row0 + r); optionally the rows of dx (fp32 and bf16 copy) are
// then zeroed (the overwritten activations receive no gradient, SURVEY.md 3.3).
// Deterministic two-stage reduction: stage 1 sums a fixed slice of the sequences per block
// (fixed partition over 8 warps, fixed-order smem reduction) into partial[slice][r][:],
// stage 2 adds the slices in order.
static constexpr int SPLICE_MAX_SLICES = 64;

__global__ void __launch_bounds__(256) splice_bwd_partial_kernel(float* __restrict__ dx, bf16* __restrict__ dx_bf16,
                                                                 float* __restrict__ partial, int S, int L, int row0,
                                                                 int n, int d, int per_slice, int zero_rows,
                                                                 const int* __restrict__ seq_off) {
  __shared__ float4 part[8][32];
  const int r = blockIdx.x, slice = blockIdx.z;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int c = (blockIdx.y * 32 + lane) * 4;
  const int s_end = min(S, (slice + 1) * per_slice);
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
  pdl_wait();
  pdl_trigger();
  if (c < d) {
    for (int s = slice * per_slice + warp; s < s_end; s += 8) {
      const size_t off = ((seq_off != nullptr ? static_cast<size_t>(seq_off[s]) : static_cast<size_t>(s) * L) + row0 + r) * d + c;
      const float4 v = *reinterpret_cast<const float4*>(dx + off);
      acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
      if (zero_rows) {
        *reinterpret_cast<float4*>(dx + off) = make_float4(0.f, 0.f, 0.f, 0.f);
        if (dx_bf16 != nullptr) *reinterpret_cast<uint2*>(dx_bf16 + off) = make_uint2(0u, 0u);
      }
    }
  }
  part[warp][lane] = acc;
  __syncthreads();
  if (warp == 0 && c < d) {
    float4 t = part[0][lane];
#pragma unroll
    for (int w = 1; w < 8; ++w) {
      t.x += part[w][lane].x; t.y += part[w][lane].y; t.z += part[w][lane].z; t.w += part[w][lane].w;
    }
    *reinterpret_cast<float4*>(partial + (static_cast<size_t>(slice) * n + r) * d + c) = t;
  }
}

// The same two stages in ONE launch: every block writes its slice's partial, then the LAST block to finish (atomic ticket)
// adds the slices in slice order -- the result does not depend on which block that is, so it stays deterministic.
__global__ void __launch_bounds__(256) splice_bwd_fused_kernel(float* __restrict__ dx, bf16* __restrict__ dx_bf16,
                                                               float* __restrict__ partial, float* __restrict__ dprompt,
                                                               unsigned* __restrict__ ticket, int S, int L, int row0, int n, int d,
                                                               int per_slice, int zero_rows, const int* __restrict__ seq_off) {
  __shared__ float4 part[8][32];
  __shared__ unsigned s_last;
  const int r = blockIdx.x, slice = blockIdx.z, nslices = gridDim.z;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int c = (blockIdx.y * 32 + lane) * 4;
  const int s_end = min(S, (slice + 1) * per_slice);
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
  pdl_wait();
  pdl_trigger();
  if (c < d) {
    for (int s = slice * per_slice + warp; s < s_end; s += 8) {
      const size_t off = ((seq_off != nullptr ? static_cast<size_t>(seq_off[s]) : static_cast<size_t>(s) * L) + row0 + r) * d + c;
      const float4 v = *reinterpret_cast<const float4*>(dx + off);
      acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
      if (zero_rows) {
        *reinterpret_cast<float4*>(dx + off) = make_float4(0.f, 0.f, 0.f, 0.f);
        if (dx_bf16 != nullptr) *reinterpret_cast<uint2*>(dx_bf16 + off) = make_uint2(0u, 0u);
      }
    }
  }
  part[warp][lane] = acc;
  __syncthreads();
  if (warp == 0 && c < d) {
    float4 t = part[0][lane];
#pragma unroll
    for (int w = 1; w < 8; ++w) {
      t.x += part[w][lane].x; t.y += part[w][lane].y; t.z += part[w][lane].z; t.w += part[w][lane].w;
    }
    *reinterpret_cast<float4*>(partial + (static_cast<size_t>(slice) * n + r) * d + c) = t;
  }
  // ticket per (prompt row, column block): the last of its nslices blocks reduces them
  __threadfence();
  __syncthreads();
  unsigned* tk = ticket + blockIdx.x * gridDim.y + blockIdx.y;
  if (threadIdx.x == 0) s_last = atomicAdd(tk, 1u) == static_cast<unsigned>(nslices - 1) ? 1u : 0u;
  __syncthreads();
  if (s_last == 0u) return;
  __threadfence();
  if (warp == 0 && c < d) {
    float4 t = __ldcg(reinterpret_cast<const float4*>(partial + static_cast<size_t>(r) * d + c));
    for (int sl = 1; sl < nslices; ++sl) {
      const float4 v = __ldcg(reinterpret_cast<const float4*>(partial + (static_cast<size_t>(sl) * n + r) * d + c));
      t.x += v.x; t.y += v.y; t.z += v.z; t.w += v.w;
    }
    *reinterpret_cast<float4*>(dprompt + static_cast<size_t>(r) * d + c) = t;
  }
  if (threadIdx.x == 0) *tk = 0u;  // leave the ticket clear for the next launch
}

__global__ void splice_bwd_final_kernel(const float* __restrict__ partial, float* __restrict__ dprompt, int nslices, int nd) {
  const int i = (blockIdx.x * blockDim.x + threadIdx.x) * 4;
  pdl_wait();
  pdl_trigger();
  if (i >= nd) return;
  float4 t = *reinterpret_cast<const float4*>(partial + i);
  for (int sl = 1; sl < nslices; ++sl) {
    const float4 v = *reinterpret_cast<const float4*>(partial + static_cast<size_t>(sl) * nd + i);
    t.x += v.x; t.y += v.y; t.z += v.z; t.w += v.w;
  }
  *reinterpret_cast<float4*>(dprompt + i) = t;
}

// partials [SPLICE_MAX_SLICES][n][d] + (as the tail of the same allocation) one ticket per (row, 128-column block), zeroed once
static size_t splice_ticket_slots(int n, int d) { return static_cast<size_t>(n) * ((d + 127) / 128); }
size_t splice_bwd_workspace_floats(int n, int d) { return static_cast<size_t>(SPLICE_MAX_SLICES) * n * d + splice_ticket_slots(n, d); }

const char* splice_bwd(float* dx, bf16* dx_bf16, float* dprompt, float* workspace, int S, int L, int row0, int n, int d,
                       bool zero_rows, cudaStream_t stream, const int* seq_off) {
  if (n <= 0) return nullptr;
  if (d % 4 != 0 || row0 < 0 || (seq_off == nullptr && row0 + n > L)) return "splice: bad geometry";
  int nslices = (S + 15) / 16;  // >= 16 sequences per block
  if (nslices > SPLICE_MAX_SLICES) nslices = SPLICE_MAX_SLICES;
  if (nslices < 1) nslices = 1;
  const int per_slice = (S + nslices - 1) / nslices;
  // the tickets live behind the partials and must be zero before the first launch (the owner of the workspace zeroes it once)
  unsigned* ticket = reinterpret_cast<unsigned*>(workspace + static_cast<size_t>(SPLICE_MAX_SLICES) * n * d);
  launch_pdl(splice_bwd_fused_kernel, dim3(n, (d + 127) / 128, nslices), dim3(256), 0, stream, dx, dx_bf16, workspace, dprompt, ticket,
             S, L, row0, n, d, per_slice, zero_rows ? 1 : 0, seq_off);
  count_launch(1);
  return launch_status("splice bwd launch failed");
}

// ------------------------------------------------------------------ fused-LayerNorm plumbing
// With LayerNorm folded into the GEMMs (gemm.h, EPI_LN_*), an LN input row lives as fp32 (residual stream),
// a bf16 copy (the GEMM's A operand) and partial statistics (sum, M2 about the partial's own mean) per 64
// columns.  The GEMM epilogues produce all three for the rows they write; these kernels do it for rows that do
// not come out of a GEMM: the tower inputs and the layer-0 prompt rows.
//
// 16 lanes own one 64-column span (one float4 each): v = the lane's 4 values -> (sum, M2) of the span in all 16 lanes
__device__ __forceinline__ float2 span_stats(const float4& v) {
  float s = (v.x + v.y) + (v.z + v.w);
#pragma unroll
  for (int o = 8; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  const float m = s * (1.f / 64.f);
  const float a = v.x - m, b = v.y - m, c = v.z - m, e = v.w - m;
  float q = (a * a + b * b) + (c * c + e * e);
#pragma unroll
  for (int o = 8; o > 0; o >>= 1) q += __shfl_xor_sync(0xffffffffu, q, o);
  return make_float2(s, q);
}

// xb[row, :] = bf16(x[row, :]), stats[row, p] = (sum, M2) of columns [64p, 64p + 64).  One warp per row.
__global__ void __launch_bounds__(256) rowstats_kernel(const float* __restrict__ x, bf16* __restrict__ xb,
                                                       float2* __restrict__ stats, int M, int d) {
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  pdl_wait();
  pdl_trigger();
  if (row >= M) return;
  const int parts = d >> 6;
  for (int p0 = 0; p0 < parts; p0 += 2) {  // (warp-uniform trip count; a trailing odd span leaves lanes 16..31 idle)
    const int p = p0 + (lane >> 4);
    const bool ok = p < parts;
    const size_t off = static_cast<size_t>(row) * d + (ok ? p : p0) * 64 + (lane & 15) * 4;
    const float4 v = *reinterpret_cast<const float4*>(x + off);
    const float2 st = span_stats(v);
    if (ok) {
      uint2 u;
      u.x = pack_bf16(v.x, v.y);
      u.y = pack_bf16(v.z, v.w);
      *reinterpret_cast<uint2*>(xb + off) = u;
      if ((lane & 15) == 0) stats[static_cast<size_t>(row) * parts + p] = st;
    }
  }
}

const char* rowstats(const float* x, bf16* xb, float2* stats, int M, int d, cudaStream_t stream) {
  if (M <= 0) return nullptr;
  if (d % 64 != 0) return "rowstats: width must be a multiple of 64";
  launch_pdl(rowstats_kernel, dim3((M + 7) / 8), dim3(256), 0, stream, x, xb, stats, M, d);
  count_launch(1);
  return launch_status("rowstats launch failed");
}

// Splice with the bf16 copy and the statistics of the spliced rows (values copied verbatim into x: bit-exact).
__global__ void __launch_bounds__(128) splice_fwd_stats_kernel(float* __restrict__ x, bf16* __restrict__ xb,
                                                               float2* __restrict__ stats, const float* __restrict__ prompt,
                                                               int L, int row0, int d) {
  const int s = blockIdx.x, r = blockIdx.y;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  pdl_wait();
  pdl_trigger();
  const int parts = d >> 6;
  const size_t row = static_cast<size_t>(s) * L + row0 + r;
  for (int p0 = 2 * warp; p0 < parts; p0 += 8) {
    const int p = p0 + (lane >> 4);
    const bool ok = p < parts;
    const int c = (ok ? p : p0) * 64 + (lane & 15) * 4;
    const float4 v = *reinterpret_cast<const float4*>(prompt + static_cast<size_t>(r) * d + c);
    const float2 st = span_stats(v);
    if (ok) {
      *reinterpret_cast<float4*>(x + row * d + c) = v;
      uint2 u;
      u.x = pack_bf16(v.x, v.y);
      u.y = pack_bf16(v.z, v.w);
      *reinterpret_cast<uint2*>(xb + row * d + c) = u;
      if ((lane & 15) == 0) stats[row * parts + p] = st;
    }
  }
}

const char* splice_fwd_stats(float* x, bf16* xb, float2* stats, const float* prompt, int S, int L, int row0, int n, int d,
                             cudaStream_t stream) {
  if (S <= 0 || n <= 0) return nullptr;
  if (d % 64 != 0 || row0 < 0 || row0 + n > L) return "splice: bad geometry";
  launch_pdl(splice_fwd_stats_kernel, dim3(S, n), dim3(128), 0, stream, x, xb, stats, prompt, L, row0, d);
  count_launch(1);
  return launch_status("splice fwd (stats) launch failed");
}

// LayerNorm folded into the following Linear (weights frozen, done once at weight-load time):
//   W'[n,k] = bf16(W[n,k] * gamma[k])  (+ the K-major transposed copy for the dgrad GEMM)
//   colsum[n] = sum_k W'[n,k] (of the ROUNDED weight: it must cancel what the tensor cores compute for a constant row)
//   bias'[n] = bias[n] + sum_k W[n,k] * beta[k],   sb[n] = (colsum[n], bias'[n])
// One warp per output row n.
__global__ void __launch_bounds__(256) fold_ln_kernel(const float* __restrict__ W, const float* __restrict__ gamma,
                                                      const float* __restrict__ beta, const float* __restrict__ bias,
                                                      bf16* __restrict__ Wl, bf16* __restrict__ Wlt, float* __restrict__ bias_l,
                                                      float* __restrict__ colsum, float2* __restrict__ sb, int N, int K) {
  const int n = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (n >= N) return;
  float cs = 0.f, bd = 0.f;
  for (int k = lane; k < K; k += 32) {
    const float w = W[static_cast<size_t>(n) * K + k];
    const bf16 wl = __float2bfloat16(w * gamma[k]);
    Wl[static_cast<size_t>(n) * K + k] = wl;
    Wlt[static_cast<size_t>(k) * N + n] = wl;
    cs += __bfloat162float(wl);
    bd += w * beta[k];
  }
  cs = warp_sum(cs);
  bd = warp_sum(bd);
  if (lane == 0) {
    const float b = bias[n] + bd;
    bias_l[n] = b;
    colsum[n] = cs;
    sb[n] = make_float2(cs, b);
  }
}

const char* fold_layernorm(const float* W, const float* gamma, const float* beta, const float* bias, bf16* Wl, bf16* Wlt,
                           float* bias_l, float* colsum, float2* sb, int N, int K, cudaStream_t stream) {
  if (N <= 0 || K <= 0) return nullptr;
  fold_ln_kernel<<<(N + 7) / 8, 256, 0, stream>>>(W, gamma, beta, bias, Wl, Wlt, bias_l, colsum, sb, N, K);
  count_launch(1);
  return launch_status("fold_layernorm launch failed");
}

// x[rows[i], :] (+)= src[i, :] for S rows (fp32 + optional bf16 copy of the result): scatters the S live rows of a
// pruned pass back into a full [M, d] buffer.
__global__ void scatter_rows_kernel(const float* __restrict__ src, const int* __restrict__ rows, int L, float* __restrict__ x,
                                    bf16* __restrict__ xb, int d, int accumulate) {
  const int s = blockIdx.x;
  pdl_wait();
  pdl_trigger();
  const size_t row = static_cast<size_t>(s) * L + (rows ? rows[s] : 0);
  for (int c = threadIdx.x * 4; c < d; c += blockDim.x * 4) {
    float4 v = *reinterpret_cast<const float4*>(src + static_cast<size_t>(s) * d + c);
    if (accumulate) {
      const float4 o = *reinterpret_cast<const float4*>(x + row * d + c);
      v.x += o.x; v.y += o.y; v.z += o.z; v.w += o.w;
    }
    *reinterpret_cast<float4*>(x + row * d + c) = v;
    if (xb != nullptr) {
      uint2 u;
      u.x = pack_bf16(v.x, v.y);
      u.y = pack_bf16(v.z, v.w);
      *reinterpret_cast<uint2*>(xb + row * d + c) = u;
    }
  }
}
const char* scatter_rows(const float* src, const int* rows, int S, int L, float* x, bf16* xb, int d, bool accumulate,
                         cudaStream_t stream) {
  if (S <= 0) return nullptr;
  if (d % 4 != 0) return "scatter_rows: width must be a multiple of 4";
  launch_pdl(scatter_rows_kernel, dim3(S), dim3(128), 0, stream, src, rows, L, x, xb, d, accumulate ? 1 : 0);
  count_launch(1);
  return launch_status("scatter_rows launch failed");
}

__global__ void scatter_rows_bf16_kernel(const bf16* __restrict__ src, const int* __restrict__ rows, int L, bf16* __restrict__ x, int d) {
  const int s = blockIdx.x;
  pdl_wait();
  pdl_trigger();
  const size_t row = static_cast<size_t>(s) * L + (rows ? rows[s] : 0);
  for (int c = threadIdx.x * 8; c < d; c += blockDim.x * 8)
    *reinterpret_cast<uint4*>(x + row * d + c) = *reinterpret_cast<const uint4*>(src + static_cast<size_t>(s) * d + c);
}
const char* scatter_rows_bf16(const bf16* src, const int* rows, int S, int L, bf16* x, int d, cudaStream_t stream) {
  if (S <= 0) return nullptr;
  if (d % 8 != 0) return "scatter_rows_bf16: width must be a multiple of 8";
  launch_pdl(scatter_rows_bf16_kernel, dim3(S), dim3(128), 0, stream, src, rows, L, x, d);
  count_launch(1);
  return launch_status("scatter_rows_bf16 launch failed");
}

// dst[i, :] = src[s*L + rows[s], :] for S rows, fp32 and/or bf16 sources (either may be null): gathers the CLS / EOT
// rows the last block still needs after attention.
__global__ void gather_rows_kernel(const float* __restrict__ src_f, const bf16* __restrict__ src_b, const int* __restrict__ rows,
                                   int L, float* __restrict__ dst_f, bf16* __restrict__ dst_b, int d) {
  const int s = blockIdx.x;
  pdl_wait();
  pdl_trigger();
  const size_t row = static_cast<size_t>(s) * L + (rows ? rows[s] : 0);
  for (int c = threadIdx.x * 4; c < d; c += blockDim.x * 4) {
    if (src_f != nullptr) *reinterpret_cast<float4*>(dst_f + static_cast<size_t>(s) * d + c) = *reinterpret_cast<const float4*>(src_f + row * d + c);
    if (src_b != nullptr) *reinterpret_cast<uint2*>(dst_b + static_cast<size_t>(s) * d + c) = *reinterpret_cast<const uint2*>(src_b + row * d + c);
  }
}
const char* gather_rows(const float* src_f, const bf16* src_b, const int* rows, int S, int L, float* dst_f, bf16* dst_b, int d,
                        cudaStream_t stream) {
  if (S <= 0) return nullptr;
  if (d % 4 != 0) return "gather_rows: width must be a multiple of 4";
  launch_pdl(gather_rows_kernel, dim3(S), dim3(128), 0, stream, src_f, src_b, rows, L, dst_f, dst_b, d);
  count_launch(1);
  return launch_status("gather_rows launch failed");
}

// ------------------------------------------------------------------ patch extraction
// patches[(b*gh + py)*gw + px, (c*p + iy)*p + ix] = image[b, c, py*p + iy, px*p + ix]  (bf16),
// row stride ldo >= 3*p*p (padding columns, if any, are zeroed once at allocation).
__global__ void im2col_kernel(const float* __restrict__ img, bf16* __restrict__ out, int R, int p, int ldo, size_t total2) {
  const size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= total2) return;
  const int gw = R / p;
  const int kdim = 3 * p * p;
  const size_t e = i * 2;  // 2 consecutive ix (p is even)
  const int col = static_cast<int>(e % kdim);
  const size_t row = e / kdim;
  const int ix = col % p, iy = (col / p) % p, c = col / (p * p);
  const int px = static_cast<int>(row % gw), py = static_cast<int>((row / gw) % gw);
  const int b = static_cast<int>(row / (static_cast<size_t>(gw) * gw));
  const float2 v = *reinterpret_cast<const float2*>(img + ((static_cast<size_t>(b) * 3 + c) * R + py * p + iy) * R + px * p + ix);
  *reinterpret_cast<uint32_t*>(out + row * ldo + col) = pack_bf16(v.x, v.y);
}

const char* im2col_bf16(const float* img, bf16* out, int B, int R, int p, int ldo, cudaStream_t stream) {
  if (B <= 0) return nullptr;
  if (R % p != 0 || p % 2 != 0 || ldo < 3 * p * p || ldo % 2 != 0) return "im2col: bad geometry";
  const size_t total2 = static_cast<size_t>(B) * 3 * R * R / 2;
  im2col_kernel<<<static_cast<unsigned>((total2 + 255) / 256), 256, 0, stream>>>(img, out, R, p, ldo, total2);
  count_launch(1);
  return launch_status("im2col launch failed");
}

// The inverse index map of im2col_kernel, fp32: image[b, c, py*p + iy, px*p + ix] = patches[(b*gh + py)*gw + px, (c*p + iy)*p + ix].
// Stride equals the kernel size, so this is a permutation: every image element is written exactly once, nothing is
// accumulated, and the padding columns >= 3*p*p of the rows are never read.  Threads walk the image (coalesced writes),
// two consecutive ix per thread (p is even, so both lie in one patch).
__global__ void col2im_kernel(const float* __restrict__ cols, float* __restrict__ img, int R, int p, int ldi, size_t total2) {
  const size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  pdl_wait();
  pdl_trigger();
  if (i >= total2) return;
  const size_t e = i * 2;
  const int x = static_cast<int>(e % R);
  const size_t r2 = e / R;
  const int y = static_cast<int>(r2 % R);
  const size_t bc = r2 / R;
  const int c = static_cast<int>(bc % 3);
  const size_t b = bc / 3;
  const int gw = R / p;
  const int px = x / p, ix = x - px * p, py = y / p, iy = y - py * p;
  const size_t row = (b * gw + py) * gw + px;
  const int col = (c * p + iy) * p + ix;
  *reinterpret_cast<float2*>(img + e) = *reinterpret_cast<const float2*>(cols + row * ldi + col);
}

const char* col2im_f32(const float* cols, float* img, int B, int R, int p, int ldi, cudaStream_t stream) {
  if (B <= 0) return nullptr;
  if (R % p != 0 || p % 2 != 0 || ldi < 3 * p * p || ldi % 2 != 0) return "col2im: bad geometry";
  const size_t total2 = static_cast<size_t>(B) * 3 * R * R / 2;
  launch_pdl(col2im_kernel, dim3(static_cast<unsigned>((total2 + 255) / 256)), dim3(256), 0, stream, cols, img, R, p, ldi, total2);
  count_launch(1);
  return launch_status("col2im launch failed");
}

// ------------------------------------------------------------------ l-inf PGD update
// IEEE fp32 arithmetic in inline PTX: the library builds with --use_fast_math, under which __fdiv_rn / __fadd_rn /
// __fsub_rn and fminf / fmaxf compile to their .ftz forms and would flush subnormal gradients and pixels to zero.
// PyTorch's element-wise kernels do not flush, and the update must be bitwise theirs.
__device__ __forceinline__ float add_ieee(float a, float b) { float r; asm("add.rn.f32 %0, %1, %2;" : "=f"(r) : "f"(a), "f"(b)); return r; }
__device__ __forceinline__ float sub_ieee(float a, float b) { float r; asm("sub.rn.f32 %0, %1, %2;" : "=f"(r) : "f"(a), "f"(b)); return r; }
__device__ __forceinline__ float div_ieee(float a, float b) { float r; asm("div.rn.f32 %0, %1, %2;" : "=f"(r) : "f"(a), "f"(b)); return r; }
__device__ __forceinline__ float max_ieee(float a, float b) { float r; asm("max.f32 %0, %1, %2;" : "=f"(r) : "f"(a), "f"(b)); return r; }
__device__ __forceinline__ float min_ieee(float a, float b) { float r; asm("min.f32 %0, %1, %2;" : "=f"(r) : "f"(a), "f"(b)); return r; }

// One pixel, op for op the PyTorch loop x = (x + alpha * (g / std).sign()).clamp(x0 - eps, x0 + eps).clamp(0, 1),
// xn = (x - mean) / std, where g / std is the autograd of the normalisation.  The sign is read from the bits of the
// quotient (torch.sign: 0 for +-0 and NaN); alpha * sign is exact, so the step is +0 or alpha with the quotient's sign bit.
__device__ __forceinline__ float pgd_pixel(float g, float x, float x0, float mean, float std, float eps, float alpha, float* xn) {
  const uint32_t q = __float_as_uint(div_ieee(g, std));
  const uint32_t mag = q & 0x7fffffffu;
  const float step = (mag == 0u || mag > 0x7f800000u) ? 0.f : __uint_as_float(__float_as_uint(alpha) | (q & 0x80000000u));
  float v = add_ieee(x, step);
  v = min_ieee(max_ieee(v, sub_ieee(x0, eps)), add_ieee(x0, eps));
  v = min_ieee(max_ieee(v, 0.f), 1.f);
  *xn = div_ieee(sub_ieee(v, mean), std);
  return v;
}

// The patch gradient is read through col2im_kernel's index map (never written as an image; padding columns not read);
// x_adv is updated in place and x_norm rewritten, two consecutive pixels per thread.
__global__ void pgd_linf_kernel(const float* __restrict__ cols, float* __restrict__ x_adv, const float* __restrict__ x_clean,
                                float* __restrict__ x_norm, int R, int p, int ldi, size_t total2, PgdParams prm) {
  const size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  pdl_wait();
  pdl_trigger();
  if (i >= total2) return;
  const size_t e = i * 2;
  const int x = static_cast<int>(e % R);
  const size_t r2 = e / R;
  const int y = static_cast<int>(r2 % R);
  const size_t bc = r2 / R;
  const int c = static_cast<int>(bc % 3);
  const size_t b = bc / 3;
  const int gw = R / p;
  const int px = x / p, ix = x - px * p, py = y / p, iy = y - py * p;
  const size_t row = (b * gw + py) * gw + px;
  const int col = (c * p + iy) * p + ix;
  const float2 g = *reinterpret_cast<const float2*>(cols + row * ldi + col);
  const float2 xa = *reinterpret_cast<const float2*>(x_adv + e);
  const float2 x0 = *reinterpret_cast<const float2*>(x_clean + e);
  const float m = prm.mean[c], s = prm.std[c];
  float2 o, n;
  o.x = pgd_pixel(g.x, xa.x, x0.x, m, s, prm.eps, prm.alpha, &n.x);
  o.y = pgd_pixel(g.y, xa.y, x0.y, m, s, prm.eps, prm.alpha, &n.y);
  *reinterpret_cast<float2*>(x_adv + e) = o;
  *reinterpret_cast<float2*>(x_norm + e) = n;
}

const char* pgd_linf_check(const PgdParams& prm) {
  if (!(std::isfinite(prm.eps) && prm.eps >= 0.f)) return "pgd: eps must be finite and >= 0";
  if (!(std::isfinite(prm.alpha) && prm.alpha > 0.f)) return "pgd: alpha must be finite and > 0";
  for (int c = 0; c < 3; ++c) {
    if (!(std::isfinite(prm.std[c]) && prm.std[c] > 0.f)) return "pgd: std must be finite and > 0";
    if (!std::isfinite(prm.mean[c])) return "pgd: mean must be finite";
  }
  return nullptr;
}

const char* pgd_linf_f32(const float* cols, float* x_adv, const float* x_clean, float* x_norm, int B, int R, int p, int ldi,
                         const PgdParams& prm, cudaStream_t stream) {
  if (const char* e = pgd_linf_check(prm)) return e;
  if (B <= 0) return nullptr;
  if (R % p != 0 || p % 2 != 0 || ldi < 3 * p * p || ldi % 2 != 0) return "pgd: bad geometry";
  for (const void* q : {static_cast<const void*>(cols), static_cast<const void*>(x_adv), static_cast<const void*>(x_clean),
                        static_cast<const void*>(x_norm)})
    if (reinterpret_cast<uintptr_t>(q) % 8 != 0) return "pgd: pointers must be 8-byte aligned";
  const size_t total2 = static_cast<size_t>(B) * 3 * R * R / 2;
  launch_pdl(pgd_linf_kernel, dim3(static_cast<unsigned>((total2 + 255) / 256)), dim3(256), 0, stream, cols, x_adv, x_clean,
             x_norm, R, p, ldi, total2, prm);
  count_launch(1);
  return launch_status("pgd launch failed");
}

// ------------------------------------------------------------------ small helpers
// out[s, 0, :] = cls[:] + pos[0, :]  (class token row of every image)
__global__ void cls_rows_kernel(float* __restrict__ x, const float* __restrict__ cls, const float* __restrict__ pos, int L, int d) {
  float* dst = x + static_cast<size_t>(blockIdx.x) * L * d;
  for (int c = threadIdx.x; c < d; c += blockDim.x) dst[c] = cls[c] + pos[c];
}
const char* write_cls_rows(float* x, const float* cls, const float* pos, int S, int L, int d, cudaStream_t stream) {
  if (S <= 0) return nullptr;
  cls_rows_kernel<<<S, 256, 0, stream>>>(x, cls, pos, L, d);
  count_launch(1);
  return launch_status("cls rows launch failed");
}

// x0[c, l, :] = emb[c, l, :] + pos[l, :] for l < L (L <= Lsrc): text-tower input, built once
// per class set (trainers/mudpt.py:143); the ctx rows are overwritten by the splice each step.
// seq_off != null: packed variable-length sequences, row seq_off[c] + l for l < seq_off[c+1] - seq_off[c] (L = the longest).
__global__ void add_pos_kernel(float* __restrict__ x0, const float* __restrict__ emb, const float* __restrict__ pos,
                               int L, int Lsrc, int d, const int* __restrict__ seq_off) {
  const int c = blockIdx.x, l = blockIdx.y;
  if (seq_off != nullptr && l >= seq_off[c + 1] - seq_off[c]) return;
  const float* src = emb + (static_cast<size_t>(c) * Lsrc + l) * d;
  float* dst = x0 + ((seq_off != nullptr ? static_cast<size_t>(seq_off[c]) : static_cast<size_t>(c) * L) + l) * d;
  for (int i = threadIdx.x; i < d; i += blockDim.x) dst[i] = src[i] + pos[static_cast<size_t>(l) * d + i];
}
const char* add_positional(float* x0, const float* emb, const float* pos, int S, int L, int Lsrc, int d, cudaStream_t stream,
                           const int* seq_off) {
  if (S <= 0) return nullptr;
  add_pos_kernel<<<dim3(S, L), 128, 0, stream>>>(x0, emb, pos, L, Lsrc, d, seq_off);
  count_launch(1);
  return launch_status("add_pos launch failed");
}

// out[s, l, :] = x[seq_off[s] + l, :] for l < len_s, 0 for len_s <= l < L: packed variable-length rows to the padded
// [S, L, d] layout (the dense input gradient of a ragged text tower; zero past each length is exact under the causal mask)
__global__ void unpack_rows_kernel(const float* __restrict__ x, const int* __restrict__ seq_off, int L, int d, float* __restrict__ out) {
  const int s = blockIdx.x, l = blockIdx.y;
  pdl_wait();
  pdl_trigger();
  const int r0 = seq_off[s], len = seq_off[s + 1] - r0;
  float4* dst = reinterpret_cast<float4*>(out + (static_cast<size_t>(s) * L + l) * d);
  const float4* src = reinterpret_cast<const float4*>(x + static_cast<size_t>(r0 + l) * d);
  for (int c = threadIdx.x; c < d / 4; c += blockDim.x) dst[c] = l < len ? src[c] : make_float4(0.f, 0.f, 0.f, 0.f);
}
const char* unpack_rows(const float* x, const int* seq_off, int S, int L, int d, float* out, cudaStream_t stream) {
  if (S <= 0 || L <= 0) return nullptr;
  if (d % 4 != 0) return "unpack_rows: width must be a multiple of 4";
  launch_pdl(unpack_rows_kernel, dim3(S, L), dim3(128), 0, stream, x, seq_off, L, d, out);
  count_launch(1);
  return launch_status("unpack_rows launch failed");
}

__global__ void cast_bf16_kernel(const float* __restrict__ in, bf16* __restrict__ out, size_t n) {
  const size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i < n) out[i] = __float2bfloat16(in[i]);
}
const char* cast_to_bf16(const float* in, bf16* out, size_t n, cudaStream_t stream) {
  if (n == 0) return nullptr;
  cast_bf16_kernel<<<static_cast<unsigned>((n + 255) / 256), 256, 0, stream>>>(in, out, n);
  count_launch(1);
  return launch_status("cast launch failed");
}

// out[c, r] = bf16(in[r, c])  (in: [rows, cols] fp32) -- the K-major copy used by dgrad GEMMs
__global__ void transpose_cast_kernel(const float* __restrict__ in, bf16* __restrict__ out, int rows, int cols) {
  __shared__ float tile[32][33];
  const int c0 = blockIdx.x * 32, r0 = blockIdx.y * 32;
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int r = r0 + i, c = c0 + threadIdx.x;
    tile[i][threadIdx.x] = (r < rows && c < cols) ? in[static_cast<size_t>(r) * cols + c] : 0.f;
  }
  __syncthreads();
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int c = c0 + i, r = r0 + threadIdx.x;
    if (c < cols && r < rows) out[static_cast<size_t>(c) * rows + r] = __float2bfloat16(tile[threadIdx.x][i]);
  }
}
const char* transpose_cast_bf16(const float* in, bf16* out, int rows, int cols, cudaStream_t stream) {
  if (rows <= 0 || cols <= 0) return nullptr;
  transpose_cast_kernel<<<dim3((cols + 31) / 32, (rows + 31) / 32), dim3(32, 8), 0, stream>>>(in, out, rows, cols);
  count_launch(1);
  return launch_status("transpose launch failed");
}

}  // namespace mudpt
