// tcgen05 / TMEM / TMA GEMM for the frozen-weight linear layers of the MuDPT towers.
//
//   C[M,N] = A[M,K] (bf16, row-major) x B[N,K]^T (bf16, row-major, i.e. nn.Linear's [out,in])
//
// Both operands are K-major, so forward GEMMs use the weight as stored and the dgrad GEMMs
// use a pre-transposed copy made once at weight-load time (weights are frozen,
// trainers/mudpt.py:205-212, so there is no wgrad and the transpose is free).
//
// Replaces the `addmm`/`mm` call sites of clip/model.py:273 (in-proj), :299 (out-proj),
// :300 (c_fc, c_proj), :527 (conv1 as a GEMM), their autograd dgrads, and -- through the EPI_LN_* /
// EPI_RESID_STATS epilogues -- the LayerNorms in front of them (:164-170) and the deep-prompt splice (:281-297).
//
// Structure (one persistent CTA per SM, 320 threads; CTA pairs in cta_group::2 mode):
//   warp 0      TMA producer   : cp.async.bulk.tensor 2D tiles (128B swizzle) into a smem ring
//   warp 1      MMA issuer     : one elected lane issues tcgen05.mma (128|256 x BN x 16), fp32
//                                accumulators in TMEM, double-buffered (2 x BN columns)
//   warps 2..9  epilogue       : tcgen05.ld the accumulator, apply the fused epilogue
//                                (bias / QuickGELU / residual / GELU' / LayerNorm forms / patch-embed scatter),
//                                hand 32 x 32 boxes to the TMA (UTMASTG; residual / saved
//                                pre-activation boxes arrive by UTMALDG one box ahead)
// The epilogue of tile i overlaps the MMAs of tile i+1 through the second TMEM buffer.  The kernel
// is launched with programmatic stream serialization: its prologue (barriers, TMEM allocation,
// descriptor prefetch) overlaps the tail of the previous kernel (pdl_wait() in common.cuh).
//
// Work decomposition (grouped stream-K).  Whole tiles are dealt round-robin to the units (CTAs or CTA pairs); when
// the tile count leaves a remainder of R tiles, the LAST g units give up their tile of the last full wave and share
// those g tiles plus the R remainder tiles as ONE contiguous range of k-blocks each (75 pair tiles on 74 pairs with
// g = 8: 67 units do one tile, 8 units do 9/8 of a tile -- 1.125 tile-times instead of 2).  A unit walks its range
// from the high end down, so the part of a tile that ends at the tile's last k-block comes last in its range: that
// unit ("finisher") runs the epilogue, after adding the fp32 partial accumulators that the lower-numbered
// unit(s) holding the rest of the tile wrote to an L2-resident scratch slot at the START of their ranges (one slot per
// CTA, one ready flag per epilogue warp: warp w of the finisher reads exactly what warp w of the contributor wrote,
// so the hand-over is warp to warp).  A finisher only ever waits for lower-numbered units, which the hardware
// dispatches first: no deadlock when another stream's kernel holds part of the machine.  g trades the imbalance
// R/g against the L2 traffic of g hand-overs (measured: all 74 pairs handing over 256 KB each costs ~9 us, more than
// a whole K = 768 tile), see plan_sk().
#include "gemm.h"

#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <mutex>
#include <unordered_map>

#include "common.cuh"
#include "launch_count.h"

namespace mudpt {

static constexpr int BM = 128;
static constexpr int BK = 64;  // 64 bf16 = 128 B = one swizzle row
static constexpr int kStatSpan = 64;  // columns per partial LayerNorm statistic (EPI_RESID_STATS -> EPI_LN_*)
// Epilogue warps per CTA (TMA warp + MMA warp + these).  The GELU' epilogue (dgrad of c_proj) has the longest
// per-element dependency chain (unpack, 6 packed fp32 ops, tanh, pack) and was latency-bound on 2 warps per
// scheduler (ncu: issue slots 39 % busy, stall_wait dominant): it runs 16 warps at <= 112 registers, with a
// single accumulator register set (4 warps per scheduler hide the TMEM load instead of a second set).
template <int MODE> struct GeluBwd { static constexpr bool value = (MODE == EPI_GELU_BWD || MODE == EPI_GELU_BWD_DOTS); };
template <int MODE> struct EpiWarps { static constexpr int value = GeluBwd<MODE>::value ? 16 : 8; };
template <int MODE> struct GemmThreads { static constexpr int value = 64 + 32 * EpiWarps<MODE>::value; };

// TWO = CTA pair (cta_group::2): the pair computes a 256 x BN tile, each CTA holds 128 rows of A
// and BN/2 rows of B per stage, so the B half that an SM reads from its shared memory feeds both
// tensor cores: 1/3 less operand traffic through shared memory per FLOP than two independent
// 128 x BN tiles (the 1-CTA mainloop is bound by exactly that traffic).
// Epilogue flavour per mode.  "Row" epilogues keep the TMEM layout (thread = accumulator row, 32
// consecutive columns in registers), do the fused math on packed fp32 pairs and hand 32 x 32
// boxes to the TMA (store; also the loads of residual / saved pre-activation / LN input) through 2 KB
// 64B-swizzled (bf16) or 4 KB 128B-swizzled (fp32) staging boxes.  Only the patch-embedding scatter keeps the
// transposing epilogue below.
template <int MODE> struct RowEpi { static constexpr bool value = (MODE != EPI_PATCH); };
template <int MODE> struct LnFwd { static constexpr bool value = (MODE == EPI_LN_BF16 || MODE == EPI_LN_GELU || MODE == EPI_LN_GELU_ONLY); };
// two bf16 outputs (h and QuickGELU(h))
template <int MODE> struct GeluFwd { static constexpr bool value = (MODE == EPI_GELU || MODE == EPI_LN_GELU); };
// one bf16 output: the fused value, or its QuickGELU (GeluOnly)
template <int MODE> struct GeluOnly { static constexpr bool value = (MODE == EPI_GELU_ONLY || MODE == EPI_LN_GELU_ONLY); };
template <int MODE> struct Bf16Fwd { static constexpr bool value = (MODE == EPI_BF16 || MODE == EPI_LN_BF16 || GeluOnly<MODE>::value); };
// fp32 output box with an optional second (bf16) box: residual + statistics, LayerNorm backward
template <int MODE> struct DualEpi { static constexpr bool value = (MODE == EPI_RESID_STATS || MODE == EPI_LN_BWD); };
template <int MODE> struct F32Epi { static constexpr bool value = (MODE == EPI_F32 || MODE == EPI_RESID_F32 || DualEpi<MODE>::value); };
// an fp32 box (residual / residual gradient) is TMA-loaded one box ahead and rewritten in place
template <int MODE> struct ResidEpi { static constexpr bool value = (MODE == EPI_RESID_F32 || DualEpi<MODE>::value); };
template <int MODE> struct PrefetchEpi { static constexpr bool value = (ResidEpi<MODE>::value || GeluBwd<MODE>::value); };
static constexpr int kUnitBytes = 32 * 64;  // 32 rows x 32 bf16, SWIZZLE_64B
static constexpr int kMaxSmem = 227 * 1024;

template <int BN, int MODE, bool TWO>
struct GemmCfg {
  static constexpr int kBRows = TWO ? BN / 2 : BN;
  static constexpr int kABytes = BM * BK * 2;
  static constexpr int kBBytes = kBRows * BK * 2;
  static constexpr int kStageBytes = kABytes + kBBytes;
  static constexpr int kTxBytes = TWO ? 2 * kStageBytes : kStageBytes;  // credited to the leader's barrier
  // staging per epilogue warp: one 4 KB transpose buffer (patch embedding), or TMA boxes: 2 bf16 units (4 for the
  // two-output c_fc), 2 fp32 boxes (= 4 units), or 2 fp32 boxes + 2 bf16 units for the dual-output modes
  static constexpr int kUnitsPerWarp = DualEpi<MODE>::value ? 6 : (GeluFwd<MODE>::value || F32Epi<MODE>::value) ? 4 : 2;
  static constexpr int kWarpStaging = RowEpi<MODE>::value ? kUnitsPerWarp * kUnitBytes : 32 * 32 * 4;
  static constexpr int kStagingBytes = EpiWarps<MODE>::value * kWarpStaging;
  static constexpr int kBarBytes = 512;
  static constexpr int kFit = (kMaxSmem - kStagingBytes - 1024 - kBarBytes) / kStageBytes;
  static constexpr int kStages = kFit < 6 ? kFit : 6;
  static_assert(kStages >= 2, "operand ring too shallow");
  static constexpr int kSmemBytes = kStages * kStageBytes + kStagingBytes + 1024 /*align slack*/ + kBarBytes;
  static constexpr int kTmemCols = 2 * BN;
};

// ---------------------------------------------------------------------------------------
// Work decomposition shared by the three warp roles
// ---------------------------------------------------------------------------------------
struct SkArgs {
  int dp_tiles;   // tiles [0, dp_tiles) are dealt whole, round-robin over all units
  int sk_tiles;   // tiles [dp_tiles, dp_tiles + sk_tiles) are cut into sk_units contiguous k-block ranges ...
  int sk_units;   // ... owned by the units [sk_first, sk_first + sk_units)
  int sk_first;
  float* partials;  // one slot of 128 x BN floats per CTA
  unsigned* flags;  // [CTA][16]
};

struct Seg {
  int tile, kb0, kb1;  // k-blocks [kb0, kb1) of `tile`
  bool finish;         // holds the tile's last k-block: runs the epilogue
  int n_contrib;       // finisher: partials to add, written by units unit-1 ... unit-n_contrib
};

// Only the two cursors are state; everything else is re-derived from kernel parameters (uniform registers /
// constant bank) on each step -- three roles hold an iterator each and the 16-warp epilogues have 96 registers.
struct SegIter {
  int dp_next, q;
  __device__ __forceinline__ static int cut(int v, const SkArgs& a, int num_kb) {  // lower end of the range of SK unit v
    return static_cast<int>(static_cast<long long>(v) * (a.sk_tiles * num_kb) / a.sk_units);
  }
  __device__ __forceinline__ void init(int unit, int num_kb, const SkArgs& a) {
    dp_next = unit;
    const int v = unit - a.sk_first;
    q = (a.sk_tiles > 0 && v >= 0 && v < a.sk_units) ? cut(v + 1, a, num_kb) : 0;
  }
  __device__ __forceinline__ bool next(Seg& s, int unit, int stride, int num_kb, const SkArgs& a) {
    if (dp_next < a.dp_tiles) {
      s.tile = dp_next; s.kb0 = 0; s.kb1 = num_kb; s.finish = true; s.n_contrib = 0;
      dp_next += stride;
      return true;
    }
    if (q > 0) {  // the unit's stream-K range, walked from the high end down (q == 0: none, or done)
      const int v = unit - a.sk_first;
      const int q_lo = cut(v, a, num_kb);
      const int ts = (q - 1) / num_kb, t0 = ts * num_kb;
      const int lo = q_lo > t0 ? q_lo : t0;
      s.tile = a.dp_tiles + ts; s.kb0 = lo - t0; s.kb1 = q - t0; s.finish = (s.kb1 == num_kb); s.n_contrib = 0;
      if (s.finish && s.kb0 > 0) {  // the rest of the tile is held by the units just below
        int w = v;
        do { --w; ++s.n_contrib; } while (cut(w, a, num_kb) > t0);
      }
      q = lo > q_lo ? lo : 0;  // (lo == q_lo: range exhausted)
      return true;
    }
    return false;
  }
};

__device__ __forceinline__ void flag_release(unsigned* f) {
  asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(f), "r"(1u) : "memory");
}
__device__ __forceinline__ unsigned flag_acquire(const unsigned* f) {
  unsigned v;
  asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(f) : "memory");
  return v;
}

// ---------------------------------------------------------------------------------------
// Fused epilogue on 4 consecutive columns of one row (transposing epilogue of the patch embedding
// and the bring-up SIMT kernel).
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ uint2 pack4_bf16(const float4& v) {
  uint2 u;
  u.x = pack_bf16(v.x, v.y);
  u.y = pack_bf16(v.z, v.w);
  return u;
}

// Extra per-element operand of the epilogue (residual / saved pre-activation / positional embedding),
// fetched ahead of time so that its DRAM latency overlaps the TMEM drain instead of serialising
// against the stores (out0 and the operand may alias as far as the compiler knows).
template <int MODE> struct EpiExtra { typedef float4 type; };
template <> struct EpiExtra<EPI_GELU_BWD> { typedef uint2 type; };  // 4 packed bf16: half the registers

// `row`/`col` must be in range (the caller clamps them): the load is unconditional so that the
// compiler can keep all prefetches of a chunk in flight (a predicated load + select forces a wait
// on every single load).
template <int MODE>
__device__ __forceinline__ typename EpiExtra<MODE>::type epilogue_prefetch(const GemmEpilogue& ep, int row, int col) {
  if constexpr (MODE == EPI_RESID_F32) {
    return __ldg(reinterpret_cast<const float4*>(ep.resid + static_cast<size_t>(row) * ep.ldc + col));
  } else if constexpr (MODE == EPI_GELU_BWD) {
    return __ldg(reinterpret_cast<const uint2*>(reinterpret_cast<const bf16*>(ep.aux) + static_cast<size_t>(row) * ep.ldc + col));
  } else if constexpr (MODE == EPI_PATCH) {
    const int p = row % ep.patch_np;
    return __ldg(reinterpret_cast<const float4*>(ep.resid + static_cast<size_t>(1 + p) * ep.ldc + col));
  } else {
    return make_float4(0.f, 0.f, 0.f, 0.f);
  }
}

template <int MODE>
__device__ __forceinline__ void epilogue4(const GemmEpilogue& ep, int row, int col, float4 v,
                                          const typename EpiExtra<MODE>::type& ex) {
  // row < M and col + 4 <= N are guaranteed by the caller (N % 8 == 0); bias already added.
  const size_t off = static_cast<size_t>(row) * ep.ldc + col;
  if constexpr (MODE == EPI_BF16) {
    *reinterpret_cast<uint2*>(reinterpret_cast<bf16*>(ep.out0) + off) = pack4_bf16(v);
  } else if constexpr (MODE == EPI_F32) {
    *reinterpret_cast<float4*>(reinterpret_cast<float*>(ep.out0) + off) = v;
  } else if constexpr (MODE == EPI_RESID_F32) {
    v.x += ex.x; v.y += ex.y; v.z += ex.z; v.w += ex.w;
    *reinterpret_cast<float4*>(reinterpret_cast<float*>(ep.out0) + off) = v;
  } else if constexpr (MODE == EPI_GELU) {
    // out0 = pre-activation h (kept for the backward GELU'), out1 = QuickGELU(h)
    if (ep.out0 != nullptr) *reinterpret_cast<uint2*>(reinterpret_cast<bf16*>(ep.out0) + off) = pack4_bf16(v);
    const float4 g = make_float4(quick_gelu(v.x), quick_gelu(v.y), quick_gelu(v.z), quick_gelu(v.w));
    *reinterpret_cast<uint2*>(reinterpret_cast<bf16*>(ep.out1) + off) = pack4_bf16(g);
  } else if constexpr (MODE == EPI_GELU_BWD) {
    // out0 = acc * QuickGELU'(h), h = saved bf16 pre-activation (prefetched, packed, in ex)
    const float2 h0 = unpack_bf16(ex.x), h1 = unpack_bf16(ex.y);
    v.x *= quick_gelu_grad(h0.x); v.y *= quick_gelu_grad(h0.y);
    v.z *= quick_gelu_grad(h1.x); v.w *= quick_gelu_grad(h1.y);
    *reinterpret_cast<uint2*>(reinterpret_cast<bf16*>(ep.out0) + off) = pack4_bf16(v);
  } else if constexpr (MODE == EPI_PATCH) {
    // patch-embedding scatter (clip/model.py:527-531): GEMM row r = image*np + p goes to token
    // row image*L + 1 + p of the residual stream, plus positional_embedding[1 + p] (in ex).
    const int img = row / ep.patch_np;
    const int p = row - img * ep.patch_np;
    v.x += ex.x; v.y += ex.y; v.z += ex.z; v.w += ex.w;
    const size_t o = (static_cast<size_t>(img) * ep.patch_L + 1 + p) * ep.ldc + col;
    *reinterpret_cast<float4*>(reinterpret_cast<float*>(ep.out0) + o) = v;
  }
}


// ---------------------------------------------------------------------------------------
// Row-layout epilogue, one call per epilogue warp.
//   quad = warp % 4 selects the 32 TMEM lanes (accumulator rows) the warp may read, half selects
//   which contiguous part of the tile's BN columns it drains, in boxes of 32 columns:
//     tcgen05.ld 32x32b.x32 (thread = row)  ->  fused math on packed fp32 pairs
//     ->  bf16: 4 x STS.128 into a 2 KB unit (64B swizzle), fp32: 8 x STS.128 into a 4 KB box (128B swizzle)
//     ->  TMA store.
//   The next box's accumulator columns are in flight (second register set) during the math.
//   Modes with an extra per-element operand TMA-load its box into the staging one box ahead
//   (also across tiles) and rewrite it in place.
//   TMA clips stores / zero-fills loads at the M and N tails, so there are no per-element predicates.
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t unit_slot(int lane, int j) {  // byte offset of 16 B chunk j of row `lane`
  return static_cast<uint32_t>(lane * 64 + ((j ^ ((lane >> 1) & 3)) << 4));
}

// v * QuickGELU'(h), QuickGELU'(h) = s (1 + 1.702 h (1 - s)), s = sigmoid(1.702 h); with a = 0.851 h, t = tanh(a):
//   QuickGELU'(h) = 0.5 (1 + t + a (1 - t^2)) = 0.5 + 0.5 p,  p = t + (-a)(t^2 - 1)
// one MUFU and six packed fp32 ops per pair
__device__ __forceinline__ f32x2 mul_quick_gelu_grad2(f32x2 v, f32x2 h) {
  const f32x2 a = f2_mul(h, f2_pack(0.851f, 0.851f));
  const f32x2 na = f2_mul(h, f2_pack(-0.851f, -0.851f));
  float a0, a1;
  f2_unpack(a, a0, a1);
  const f32x2 t = f2_pack(tanh_approx(a0), tanh_approx(a1));
  const f32x2 w = f2_fma(t, t, f2_pack(-1.f, -1.f));  // t^2 - 1
  const f32x2 p = f2_fma(na, w, t);
  const f32x2 vh = f2_mul(v, f2_pack(0.5f, 0.5f));
  return f2_fma(vh, p, vh);
}
// QuickGELU(v) = v sigmoid(1.702 v) = 0.5 v + 0.5 v tanh(0.851 v)
__device__ __forceinline__ f32x2 quick_gelu2(f32x2 v) {
  const f32x2 u = f2_mul(v, f2_pack(0.851f, 0.851f));
  float u0, u1;
  f2_unpack(u, u0, u1);
  const f32x2 t = f2_pack(tanh_approx(u0), tanh_approx(u1));
  const f32x2 hv = f2_mul(v, f2_pack(0.5f, 0.5f));
  return f2_fma(hv, t, hv);
}
__device__ __forceinline__ uint32_t pack_bf16_2(f32x2 v) {
  float lo, hi;
  f2_unpack(v, lo, hi);
  return pack_bf16(lo, hi);
}
__device__ __forceinline__ float f2_hsum(f32x2 v) {
  float lo, hi;
  f2_unpack(v, lo, hi);
  return lo + hi;
}

// Row statistics from the per-64-column partials (sum, M2 about the partial's own mean) written by
// EPI_RESID_STATS / the row kernels: Chan's pairwise update, so a large row mean costs no precision.
__device__ __forceinline__ void row_mean_rstd(const float2* __restrict__ st, int parts, int width, float eps, float& mean,
                                              float& rstd) {
  float n = 0.f, mu = 0.f, m2 = 0.f;
  for (int p = 0; p < parts; ++p) {
    const float2 v = __ldg(st + p);
    const int rem = width - p * kStatSpan;
    const float np = static_cast<float>(rem < kStatSpan ? rem : kStatSpan);
    const float nn = n + np;
    const float delta = v.x / np - mu;
    mu += delta * (np / nn);
    m2 += v.y + delta * delta * (n * np / nn);
    n = nn;
  }
  mean = mu;
  rstd = rsqrtf(m2 / static_cast<float>(width) + eps);
}

struct EpiMaps {
  const CUtensorMap *o0, *o1, *ex, *x2, *o2;
};

template <int BN, int MODE, bool TWO>
__device__ __forceinline__ void epilogue_rows(const EpiMaps mp, const GemmEpilogue& ep, const SkArgs& sk, const int M, const int N,
                                              const int num_n, const int num_kb, const int unit, const int unit_stride,
                                              const uint32_t rank, const uint32_t tmem_base, uint8_t* units, uint64_t* ex_bar,
                                              uint64_t* tmem_full_bar, uint64_t* tmem_empty_bar, const int warp,
                                              const int lane) {
  constexpr int TM = TWO ? 2 * BM : BM;
  constexpr int EW = EpiWarps<MODE>::value;
  constexpr int kParts = EW / 4;        // warps per TMEM lane quadrant
  constexpr int kCols = BN / kParts;    // columns per warp
  constexpr int kBoxes = kCols / 32;    // boxes per warp and tile
  constexpr int kBoxFloats = 32 * 32;
  const int we = warp - 2;
  const int quad = warp & 3, half = we >> 2;  // half = which column part of the tile
  auto box_origin = [&](int tile, int& row, int& col0) {
    const int m_blk = tile / num_n, n_blk = tile - m_blk * num_n;
    row = m_blk * TM + static_cast<int>(rank) * BM + quad * 32;
    col0 = n_blk * BN + half * kCols;
  };
  auto boxes_of = [&](int tile) {  // valid boxes of this warp in `tile` (warp-uniform)
    int row, col0;
    box_origin(tile, row, col0);
    if (row >= M || col0 >= N) return 0;
    const int nb = (N - col0 + 31) >> 5;
    return nb < kBoxes ? nb : kBoxes;
  };
  const bool has_resid = ep.resid != nullptr;
  // Modes with a TMA-loaded operand box: lane 0 walks one box ahead of the warp (over the tiles this unit
  // FINISHES, in order) and issues the loads
  SegIter pit;
  Seg psg;
  bool pf_valid = false;
  int pf_b = -1, pf_nb = 0;
  auto pf_advance = [&]() {
    bool ok;
    do { ok = pit.next(psg, unit, unit_stride, num_kb, sk); } while (ok && !psg.finish);
    pf_valid = ok;
    pf_nb = ok ? boxes_of(psg.tile) : 0;
  };
  auto prefetch_next = [&](const uint32_t pf_k) {  // pf_k = index of the box being requested (one ahead of the warp)
    for (;;) {
      ++pf_b;
      while (pf_valid && pf_b >= pf_nb) { pf_advance(); pf_b = 0; }
      if (!pf_valid) return;
      int row, col0;
      box_origin(psg.tile, row, col0);
      uint64_t* bar = &ex_bar[pf_k & 1];
      if constexpr (MODE == EPI_LN_BWD) {
        // residual gradient (fp32 box, optional) + LN input x (bf16 box): one barrier
        mbar_expect_tx(bar, kUnitBytes + (has_resid ? 2 * kUnitBytes : 0));
        if (has_resid) tma_load_2d(units + (pf_k & 1) * 2 * kUnitBytes, mp.ex, bar, col0 + pf_b * 32, row);
        tma_load_2d(units + 4 * kUnitBytes + (pf_k & 1) * kUnitBytes, mp.x2, bar, col0 + pf_b * 32, row);
      } else if constexpr (ResidEpi<MODE>::value) {  // fp32 residual: one 32 x 32 fp32 box (128 B rows, 4 KB = two units)
        mbar_expect_tx(bar, 2 * kUnitBytes);
        tma_load_2d(units + (pf_k & 1) * 2 * kUnitBytes, mp.ex, bar, col0 + pf_b * 32, row);
      } else {
        mbar_expect_tx(bar, kUnitBytes);
        tma_load_2d(units + (pf_k & 1) * kUnitBytes, mp.ex, bar, col0 + pf_b * 32, row);
      }
      return;
    }
  };
  if constexpr (PrefetchEpi<MODE>::value) {
    if (lane == 0) {
      pit.init(unit, num_kb, sk);
      pf_advance();
      prefetch_next(0u);
    }
  }

  uint32_t k = 0;  // boxes processed so far by this warp
  const bool has_bias = ep.bias != nullptr;
  // per-row state of the tile being finished (thread = accumulator row)
  int trow = 0;                               // this thread's global row
  float ln_a = 1.f, ln_b = 0.f;               // LayerNorm forward: rstd, -rstd * mean
  float bw_a1 = 0.f, bw_a0 = 0.f;             // LayerNorm backward: out = resid + ln_a * acc + bw_a1 * x + bw_a0
  int prow = -1;                              // EPI_RESID_STATS: spliced prompt row, or -1
  float g_sum = 0.f, g_m2 = 0.f, g_mean = 0.f;  // EPI_RESID_STATS: first box of the current 64-column granule
  f32x2 dot1 = f2_pack(0.f, 0.f), dot2 = f2_pack(0.f, 0.f);  // EPI_GELU_BWD_DOTS
  auto row_setup = [&](int row) {
    trow = row + lane;
    const int rc = trow < M ? trow : M - 1;
    if constexpr (LnFwd<MODE>::value || MODE == EPI_LN_BWD) {
      float mean, rstd;
      row_mean_rstd(ep.ln_stats + static_cast<size_t>(rc) * ep.ln_parts, ep.ln_parts, ep.ln_width, ep.ln_eps, mean, rstd);
      ln_a = rstd;
      ln_b = -rstd * mean;
      if constexpr (MODE == EPI_LN_BWD) {
        float c1 = 0.f, c2 = 0.f;
        const float2* dp = ep.dots + static_cast<size_t>(rc) * ep.dot_parts;
        for (int p = 0; p < ep.dot_parts; ++p) {
          const float2 v = __ldg(dp + p);
          c1 += v.x;
          c2 += v.y;
        }
        const float inv = 1.f / static_cast<float>(ep.ln_width);
        c1 *= inv;
        c2 *= inv;
        bw_a1 = -rstd * rstd * c2;
        bw_a0 = rstd * (rstd * c2 * mean - c1);
      }
    }
    if constexpr (MODE == EPI_RESID_STATS) {
      prow = -1;
      if (ep.splice_n > 0 && trow < M) {
        const int pos = trow % ep.splice_L - ep.splice_row0;
        if (pos >= 0 && pos < ep.splice_n) prow = pos;
      }
    }
  };
  // one box: r = 32 accumulator columns of this thread's row
  auto process = [&](uint32_t (&r)[32], int row, int col) {
    if constexpr (Bf16Fwd<MODE>::value || GeluFwd<MODE>::value) {
      constexpr bool LN = LnFwd<MODE>::value;
      float4 bv[8], sv[LN ? 8 : 1];
      if ((has_bias || LN) && col + 32 <= N) {  // the common case: no per-load guards
        const float4* bp = reinterpret_cast<const float4*>(ep.bias + col);
#pragma unroll
        for (int i = 0; i < 8; ++i) bv[i] = __ldg(bp + i);
        if constexpr (LN) {
          const float4* sp = reinterpret_cast<const float4*>(ep.colsum + col);
#pragma unroll
          for (int i = 0; i < 8; ++i) sv[i] = __ldg(sp + i);
        }
      } else {
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          bv[i] = make_float4(0.f, 0.f, 0.f, 0.f);
          if ((has_bias || LN) && col + 4 * i < N) bv[i] = __ldg(reinterpret_cast<const float4*>(ep.bias + col) + i);
          if constexpr (LN) {
            sv[i] = make_float4(0.f, 0.f, 0.f, 0.f);
            if (col + 4 * i < N) sv[i] = __ldg(reinterpret_cast<const float4*>(ep.colsum + col) + i);
          }
        }
      }
      const f32x2 lna2 = f2_pack(ln_a, ln_a), lnb2 = f2_pack(ln_b, ln_b);
      // fused value of the pair (e, e + 1)
      auto value = [&](int e) {
        f32x2 v = f2_pack_u(r[e], r[e + 1]);
        const float4 b4 = bv[e >> 2];
        const f32x2 bb = (e & 2) ? f2_pack(b4.z, b4.w) : f2_pack(b4.x, b4.y);
        if constexpr (LN) {
          const float4 s4 = sv[e >> 2];
          const f32x2 ss = (e & 2) ? f2_pack(s4.z, s4.w) : f2_pack(s4.x, s4.y);
          v = f2_fma(lna2, v, f2_fma(lnb2, ss, bb));  // rstd * acc + (b' - rstd * mean * colsum)
        } else if (has_bias) {  // (dgrad GEMMs have none: warp-uniform)
          v = f2_add(v, bb);
        }
        return v;
      };
      if constexpr (Bf16Fwd<MODE>::value) {
        uint8_t* u = units + (k & 1) * kUnitBytes;
        if (lane == 0) bulk_wait_read<1>();  // the store issued from this unit two boxes ago has read it
        __syncwarp();
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          uint32_t o[4];
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            if constexpr (GeluOnly<MODE>::value) o[q] = pack_bf16_2(quick_gelu2(value(8 * j + 2 * q)));  // (as out1 of the GELU modes)
            else o[q] = pack_bf16_2(value(8 * j + 2 * q));
          }
          *reinterpret_cast<uint4*>(u + unit_slot(lane, j)) = make_uint4(o[0], o[1], o[2], o[3]);
        }
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) { tma_store_2d(mp.o0, u, col, row); bulk_commit(); }
      } else {
        // units {0,1} / {2,3} alternate per box: h and QuickGELU(h)
        uint8_t* uh = units + (k & 1) * 2 * kUnitBytes;
        uint8_t* ug = uh + kUnitBytes;
        if (lane == 0) bulk_wait_read<1>();
        __syncwarp();
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          uint32_t oh[4], og[4];
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            const f32x2 v = value(8 * j + 2 * q);
            oh[q] = pack_bf16_2(v);
            og[q] = pack_bf16_2(quick_gelu2(v));
          }
          *reinterpret_cast<uint4*>(uh + unit_slot(lane, j)) = make_uint4(oh[0], oh[1], oh[2], oh[3]);
          *reinterpret_cast<uint4*>(ug + unit_slot(lane, j)) = make_uint4(og[0], og[1], og[2], og[3]);
        }
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) {
          if (ep.out0 != nullptr) tma_store_2d(mp.o0, uh, col, row);
          tma_store_2d(mp.o1, ug, col, row);
          bulk_commit();  // both stores of the box form one group
        }
      }
    } else if constexpr (DualEpi<MODE>::value) {
      // fp32 box (residual in, out0 out: 32 rows x 128 B, 128B swizzle) + bf16 box (x2 in for the LN backward, out2 out)
      uint8_t* u = units + (k & 1) * 2 * kUnitBytes;
      uint8_t* ub = units + 4 * kUnitBytes + (k & 1) * kUnitBytes;
      if (lane == 0) {
        bulk_wait_read<0>();  // the other buffers' stores (previous box) have been read: refill them for the next box
        prefetch_next(k + 1);
      }
      mbar_wait(&ex_bar[k & 1], (k >> 1) & 1);  // this box's operands have landed
      uint4 rq8[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        rq8[j] = make_uint4(0u, 0u, 0u, 0u);
        if (MODE == EPI_RESID_STATS || has_resid) rq8[j] = *reinterpret_cast<const uint4*>(u + lane * 128 + ((j ^ (lane & 7)) << 4));
      }
      if constexpr (MODE == EPI_RESID_STATS) {
        // x = acc + bias + resid, or the spliced prompt row; statistics of x; x as fp32 and bf16
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          f32x2 v0 = f2_pack_u(r[4 * j], r[4 * j + 1]), v1 = f2_pack_u(r[4 * j + 2], r[4 * j + 3]);
          if (has_bias && col + 4 * j < N) {
            const float4 b4 = __ldg(reinterpret_cast<const float4*>(ep.bias + col) + j);
            v0 = f2_add(v0, f2_pack(b4.x, b4.y));
            v1 = f2_add(v1, f2_pack(b4.z, b4.w));
          }
          v0 = f2_add(v0, f2_pack_u(rq8[j].x, rq8[j].y));
          v1 = f2_add(v1, f2_pack_u(rq8[j].z, rq8[j].w));
          asm("mov.b64 {%0, %1}, %2;" : "=r"(r[4 * j]), "=r"(r[4 * j + 1]) : "l"(v0));
          asm("mov.b64 {%0, %1}, %2;" : "=r"(r[4 * j + 2]), "=r"(r[4 * j + 3]) : "l"(v1));
        }
        if (prow >= 0) {  // deep-prompt splice: the row is replaced verbatim (bit-exact)
          const float4* pp = reinterpret_cast<const float4*>(ep.splice_prompt + static_cast<size_t>(prow) * N + col);
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            if (col + 4 * j < N) {
              const float4 t = __ldg(pp + j);
              r[4 * j] = __float_as_uint(t.x); r[4 * j + 1] = __float_as_uint(t.y);
              r[4 * j + 2] = __float_as_uint(t.z); r[4 * j + 3] = __float_as_uint(t.w);
            }
          }
        }
        f32x2 s2 = f2_pack(0.f, 0.f);
#pragma unroll
        for (int i = 0; i < 16; ++i) s2 = f2_add(s2, f2_pack_u(r[2 * i], r[2 * i + 1]));
        const float sum = f2_hsum(s2), mean = sum * (1.f / 32.f);
        const f32x2 nm2 = f2_pack(-mean, -mean);
        f32x2 q2 = f2_pack(0.f, 0.f);
#pragma unroll
        for (int i = 0; i < 16; ++i) {
          const f32x2 dlt = f2_add(f2_pack_u(r[2 * i], r[2 * i + 1]), nm2);
          q2 = f2_fma(dlt, dlt, q2);
        }
        const float m2 = f2_hsum(q2);
#pragma unroll
        for (int j = 0; j < 8; ++j)
          *reinterpret_cast<uint4*>(u + lane * 128 + ((j ^ (lane & 7)) << 4)) = make_uint4(r[4 * j], r[4 * j + 1], r[4 * j + 2], r[4 * j + 3]);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          uint32_t o[4];
#pragma unroll
          for (int q = 0; q < 4; ++q)
            o[q] = pack_bf16(__uint_as_float(r[8 * j + 2 * q]), __uint_as_float(r[8 * j + 2 * q + 1]));
          *reinterpret_cast<uint4*>(ub + unit_slot(lane, j)) = make_uint4(o[0], o[1], o[2], o[3]);
        }
        if (((col >> 5) & 1) == 0) {
          g_sum = sum; g_m2 = m2; g_mean = mean;
        } else if (trow < M) {  // second box of the 64-column granule: merge (32 + 32 values) and publish
          const float dm = mean - g_mean;
          ep.stats_out[static_cast<size_t>(trow) * (N / kStatSpan) + (col >> 6)] = make_float2(g_sum + sum, g_m2 + m2 + 16.f * dm * dm);
        }
      } else {  // EPI_LN_BWD: out = resid + rstd * acc + a1 * x + a0
        uint4 xq4[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) xq4[j] = *reinterpret_cast<const uint4*>(ub + unit_slot(lane, j));
        const f32x2 a2 = f2_pack(ln_a, ln_a), a1_2 = f2_pack(bw_a1, bw_a1), a0_2 = f2_pack(bw_a0, bw_a0);
        uint32_t ob[4];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const uint32_t w0 = (j & 1) ? xq4[j >> 1].z : xq4[j >> 1].x, w1 = (j & 1) ? xq4[j >> 1].w : xq4[j >> 1].y;
          const f32x2 x0 = f2_pack_u(w0 << 16, w0 & 0xffff0000u), x1 = f2_pack_u(w1 << 16, w1 & 0xffff0000u);
          f32x2 v0 = f2_fma(a2, f2_pack_u(r[4 * j], r[4 * j + 1]), f2_pack_u(rq8[j].x, rq8[j].y));
          f32x2 v1 = f2_fma(a2, f2_pack_u(r[4 * j + 2], r[4 * j + 3]), f2_pack_u(rq8[j].z, rq8[j].w));
          v0 = f2_add(f2_fma(a1_2, x0, v0), a0_2);
          v1 = f2_add(f2_fma(a1_2, x1, v1), a0_2);
          uint4 o;
          asm("mov.b64 {%0, %1}, %2;" : "=r"(o.x), "=r"(o.y) : "l"(v0));
          asm("mov.b64 {%0, %1}, %2;" : "=r"(o.z), "=r"(o.w) : "l"(v1));
          *reinterpret_cast<uint4*>(u + lane * 128 + ((j ^ (lane & 7)) << 4)) = o;
          ob[(j & 1) * 2] = pack_bf16_2(v0);
          ob[(j & 1) * 2 + 1] = pack_bf16_2(v1);
          if (j & 1) *reinterpret_cast<uint4*>(ub + unit_slot(lane, j >> 1)) = make_uint4(ob[0], ob[1], ob[2], ob[3]);
        }
      }
      fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) {
        tma_store_2d(mp.o0, u, col, row);
        if (ep.out2 != nullptr) tma_store_2d(mp.o2, ub, col, row);
        bulk_commit();
      }
    } else if constexpr (F32Epi<MODE>::value) {
      // out0 (fp32) = acc + bias (+ residual): the box is 32 rows x 128 B (two units, 128B TMA swizzle); the residual
      // is TMA-loaded into it one box ahead and rewritten in place (out-proj / c_proj, clip/model.py:299-300)
      uint8_t* u = units + (k & 1) * 2 * kUnitBytes;
      if constexpr (ResidEpi<MODE>::value) {
        if (lane == 0) {
          bulk_wait_read<0>();  // the other buffer's stores (previous box) have been read: refill it for the next box
          prefetch_next(k + 1);
        }
        mbar_wait(&ex_bar[k & 1], (k >> 1) & 1);  // this box's residual has landed
      } else {
        if (lane == 0) bulk_wait_read<1>();
        __syncwarp();
      }
      float4 bv[8];
      if (has_bias && col + 32 <= N) {
        const float4* bp = reinterpret_cast<const float4*>(ep.bias + col);
#pragma unroll
        for (int i = 0; i < 8; ++i) bv[i] = __ldg(bp + i);
      } else {
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          bv[i] = make_float4(0.f, 0.f, 0.f, 0.f);
          if (has_bias && col + 4 * i < N) bv[i] = __ldg(reinterpret_cast<const float4*>(ep.bias + col) + i);
        }
      }
      uint4 rq8[ResidEpi<MODE>::value ? 8 : 1];
      if constexpr (ResidEpi<MODE>::value) {  // read the whole residual row first (see the GELU' branch)
#pragma unroll
        for (int j = 0; j < 8; ++j) rq8[j] = *reinterpret_cast<const uint4*>(u + lane * 128 + ((j ^ (lane & 7)) << 4));
      }
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        uint4* slot = reinterpret_cast<uint4*>(u + lane * 128 + ((j ^ (lane & 7)) << 4));  // 128B swizzle
        f32x2 v0 = f2_pack_u(r[4 * j], r[4 * j + 1]), v1 = f2_pack_u(r[4 * j + 2], r[4 * j + 3]);
        if (has_bias) {
          v0 = f2_add(v0, f2_pack(bv[j].x, bv[j].y));
          v1 = f2_add(v1, f2_pack(bv[j].z, bv[j].w));
        }
        if constexpr (ResidEpi<MODE>::value) {
          const uint4 rq = rq8[j];
          v0 = f2_add(v0, f2_pack_u(rq.x, rq.y));
          v1 = f2_add(v1, f2_pack_u(rq.z, rq.w));
        }
        uint4 o;
        asm("mov.b64 {%0, %1}, %2;" : "=r"(o.x), "=r"(o.y) : "l"(v0));
        asm("mov.b64 {%0, %1}, %2;" : "=r"(o.z), "=r"(o.w) : "l"(v1));
        *slot = o;
      }
      fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) { tma_store_2d(mp.o0, u, col, row); bulk_commit(); }
    } else {  // EPI_GELU_BWD / EPI_GELU_BWD_DOTS
      uint8_t* u = units + (k & 1) * kUnitBytes;
      if (lane == 0) {
        bulk_wait_read<0>();  // the other unit's store (previous box) has been read: it may be refilled
        prefetch_next(k + 1);
      }
      mbar_wait(&ex_bar[k & 1], (k >> 1) & 1);  // this box's pre-activation has landed
      // all four 16 B groups of the row are read before anything is written back: with a load per group the
      // in-place store of group j would order the load of group j + 1 behind it (the compiler cannot prove the
      // slots distinct) and serialise the four dependent chains
      uint4 hq4[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) hq4[j] = *reinterpret_cast<const uint4*>(u + unit_slot(lane, j));
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        uint4* slot = reinterpret_cast<uint4*>(u + unit_slot(lane, j));
        const uint32_t hw[4] = {hq4[j].x, hq4[j].y, hq4[j].z, hq4[j].w};
        uint32_t o[4];
        const bool in_n = col + 8 * j < N;  // (warp-uniform; N % 8 == 0)
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const int e = 8 * j + 2 * q;
          f32x2 v = f2_pack_u(r[e], r[e + 1]);
          if (has_bias && in_n) {  // (dgrad GEMMs have none: warp-uniform)
            const float2 b2 = __ldg(reinterpret_cast<const float2*>(ep.bias + col + e));
            v = f2_add(v, f2_pack(b2.x, b2.y));
          }
          const f32x2 h = f2_pack_u(hw[q] << 16, hw[q] & 0xffff0000u);  // bf16 pair -> fp32 pair
          const f32x2 res = mul_quick_gelu_grad2(v, h);
          if constexpr (MODE == EPI_GELU_BWD_DOTS) {
            if (in_n) {  // partial dots of the row for the fused LayerNorm backward of the next GEMM
              const float4 sb4 = __ldg(reinterpret_cast<const float4*>(ep.sb + col + e));  // (colsum, b') of columns e, e + 1
              dot1 = f2_fma(res, f2_pack(sb4.x, sb4.z), dot1);
              dot2 = f2_fma(res, f2_add(h, f2_pack(-sb4.y, -sb4.w)), dot2);
            }
          }
          o[q] = pack_bf16_2(res);
        }
        *slot = make_uint4(o[0], o[1], o[2], o[3]);
      }
      fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) { tma_store_2d(mp.o0, u, col, row); bulk_commit(); }
    }
    ++k;
  };
  // after the last box of a finished tile
  auto tile_end = [&](int col0) {
    if constexpr (MODE == EPI_GELU_BWD_DOTS) {
      if (trow < M) ep.dots_out[static_cast<size_t>(trow) * ((N + kCols - 1) / kCols) + col0 / kCols] = make_float2(f2_hsum(dot1), f2_hsum(dot2));
      dot1 = f2_pack(0.f, 0.f);
      dot2 = f2_pack(0.f, 0.f);
    }
  };

  // stream-K hand-over of partial accumulators (see the header comment): warp `we` of CTA c owns
  // floats [we * kBoxes * 1024, +kBoxes * 1024) of CTA c's slot; element (box b, 16 B group j, lane) is one uint4
  const size_t slot_floats = static_cast<size_t>(BM) * BN;
  auto slot_of = [&](int cta) { return sk.partials + static_cast<size_t>(cta) * slot_floats + static_cast<size_t>(we) * (kBoxes * kBoxFloats); };
  auto sk_add = [&](uint32_t (&r)[32], int b, int n_contrib) {
    for (int c = 1; c <= n_contrib; ++c) {
      const int cta = TWO ? 2 * (unit - c) + static_cast<int>(rank) : unit - c;
      const uint4* p = reinterpret_cast<const uint4*>(slot_of(cta) + b * kBoxFloats) + lane;
      uint4 v[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) v[j] = __ldcg(p + j * 32);
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        r[4 * j] = __float_as_uint(__uint_as_float(r[4 * j]) + __uint_as_float(v[j].x));
        r[4 * j + 1] = __float_as_uint(__uint_as_float(r[4 * j + 1]) + __uint_as_float(v[j].y));
        r[4 * j + 2] = __float_as_uint(__uint_as_float(r[4 * j + 2]) + __uint_as_float(v[j].z));
        r[4 * j + 3] = __float_as_uint(__uint_as_float(r[4 * j + 3]) + __uint_as_float(v[j].w));
      }
    }
  };

  SegIter it;
  it.init(unit, num_kb, sk);
  Seg sg;
  int acc = 0;
  uint32_t acc_phase = 0;
  while (it.next(sg, unit, unit_stride, num_kb, sk)) {
    int row, col0;
    box_origin(sg.tile, row, col0);
    const int nb = boxes_of(sg.tile);
    if (sg.finish) row_setup(row);  // the row's statistics are in flight while the accumulator is awaited
    mbar_wait(&tmem_full_bar[acc], acc_phase);
    tc_fence_after();
    const uint32_t taddr = tmem_base + (static_cast<uint32_t>(quad * 32) << 16) + static_cast<uint32_t>(acc * BN + half * kCols);
    auto release_acc = [&]() {  // every column this warp needs is in registers: the MMA warp may reuse the buffer
      tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        if constexpr (TWO) mbar_arrive_cluster(&tmem_empty_bar[acc], 0);
        else mbar_arrive(&tmem_empty_bar[acc]);
      }
    };
    if (!sg.finish) {
      // contributor: the raw partial accumulator goes to this CTA's slot, then the warp's flag is raised
      uint32_t ra[32];
      uint4* p = reinterpret_cast<uint4*>(slot_of(static_cast<int>(blockIdx.x))) + lane;
      if (nb == 0) release_acc();
#pragma unroll 1
      for (int b = 0; b < nb; ++b) {
        tmem_ld_32x32(taddr + static_cast<uint32_t>(b * 32), ra);
        tmem_ld_wait_regs(ra);
        if (b + 1 == nb) release_acc();
#pragma unroll
        for (int j = 0; j < 8; ++j) __stcg(p + (b * 8 + j) * 32, make_uint4(ra[4 * j], ra[4 * j + 1], ra[4 * j + 2], ra[4 * j + 3]));
      }
      if (nb > 0) {
        __threadfence();
        __syncwarp();
        if (lane == 0) flag_release(sk.flags + blockIdx.x * 16 + we);
      }
      if (++acc == 2) { acc = 0; acc_phase ^= 1; }
      continue;
    }
    const int n_contrib = nb > 0 ? sg.n_contrib : 0;
    for (int c = 1; c <= n_contrib; ++c) {  // finisher: the same warp of the lower-numbered unit(s) has written its part
      const int cta = TWO ? 2 * (unit - c) + static_cast<int>(rank) : unit - c;
      unsigned* f = sk.flags + cta * 16 + we;
      uint32_t spins = 0;
      while (flag_acquire(f) == 0u) {
        __nanosleep(64);
        if (++spins > (1u << 22)) {
          if (lane == 0) printf("mudpt: stream-K partial of CTA %d never arrived (block %d warp %d)\n", cta, blockIdx.x, warp);
          __trap();
        }
      }
      __syncwarp();
      if (lane == 0) *f = 0u;  // single consumer: leave the flag clear for the next launch
    }
    if constexpr (EW > 8) {
      // 4 warps per scheduler: one accumulator register set, no TMEM prefetch
      uint32_t ra[32];
      if (nb == 0) release_acc();
#pragma unroll 1
      for (int b = 0; b < nb; ++b) {
        tmem_ld_32x32(taddr + static_cast<uint32_t>(b * 32), ra);
        tmem_ld_wait_regs(ra);
        if (b + 1 == nb) release_acc();
        if (n_contrib) sk_add(ra, b, n_contrib);
        process(ra, row, col0 + b * 32);
      }
      if (nb > 0) tile_end(col0);
      if (++acc == 2) { acc = 0; acc_phase ^= 1; }
      continue;
    } else {
      uint32_t ra[32], rb[32];
      if (nb > 0) tmem_ld_32x32(taddr, ra);
      else release_acc();
#pragma unroll 1
      for (int b = 0; b < nb; b += 2) {
        tmem_ld_wait_regs(ra);
        if (b + 1 < nb) tmem_ld_32x32(taddr + static_cast<uint32_t>((b + 1) * 32), rb);
        else release_acc();
        if (n_contrib) sk_add(ra, b, n_contrib);
        process(ra, row, col0 + b * 32);
        if (b + 1 < nb) {
          tmem_ld_wait_regs(rb);
          if (b + 2 < nb) tmem_ld_32x32(taddr + static_cast<uint32_t>((b + 2) * 32), ra);
          else release_acc();
          if (n_contrib) sk_add(rb, b + 1, n_contrib);
          process(rb, row, col0 + (b + 1) * 32);
        }
      }
      if (nb > 0) tile_end(col0);
      if (++acc == 2) { acc = 0; acc_phase ^= 1; }
    }
  }
  if (lane == 0) bulk_wait<0>();  // shared memory must outlive the last store's read; writes complete before exit
}

// ---------------------------------------------------------------------------------------
// The kernel
// ---------------------------------------------------------------------------------------
template <int BN, int MODE, bool TWO>
__global__ void __launch_bounds__(GemmThreads<MODE>::value, 1)
gemm_tn_tcgen05_kernel(const __grid_constant__ CUtensorMap tma_a, const __grid_constant__ CUtensorMap tma_b,
                       const __grid_constant__ CUtensorMap tma_o0, const __grid_constant__ CUtensorMap tma_o1,
                       const __grid_constant__ CUtensorMap tma_ex, const __grid_constant__ CUtensorMap tma_x2,
                       const __grid_constant__ CUtensorMap tma_o2, const GemmEpilogue ep, const SkArgs sk, const int M,
                       const int N, const int K) {
  using Cfg = GemmCfg<BN, MODE, TWO>;
  // CTA pair: rank 0 is the leader (issues the MMAs, owns the "full" and "accumulator drained" barriers)
  const uint32_t rank = TWO ? cluster_ctarank() : 0u;
  constexpr int TM = TWO ? 2 * BM : BM;  // rows of a tile (of the pair)
  const int unit = TWO ? (blockIdx.x >> 1) : blockIdx.x;          // CTA (pair) index = first tile
  const int unit_stride = TWO ? (gridDim.x >> 1) : gridDim.x;
  extern __shared__ uint8_t smem_raw[];
  // 128B-swizzled tiles need 1024 B alignment
  // Pointer arithmetic on the __shared__ array (no integer round trip) keeps the shared address space
  // visible to the compiler, so the epilogue staging accesses compile to STS/LDS, not generic ST/LD.
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint8_t* smem_a = smem;
  uint8_t* smem_b = smem + Cfg::kStages * Cfg::kABytes;
  uint8_t* smem_stage = smem + Cfg::kStages * Cfg::kStageBytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem_stage + Cfg::kStagingBytes);
  uint64_t* full_bar = bars;
  uint64_t* empty_bar = bars + Cfg::kStages;
  uint64_t* tmem_full_bar = bars + 2 * Cfg::kStages;
  uint64_t* tmem_empty_bar = tmem_full_bar + 2;
  constexpr int EPI_WARPS = EpiWarps<MODE>::value;
  uint64_t* extra_bar = tmem_empty_bar + 2;  // [EPI_WARPS][2]: operand boxes of the row epilogues
  uint32_t* tmem_base_slot = reinterpret_cast<uint32_t*>(extra_bar + 2 * EPI_WARPS);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int num_n = (N + BN - 1) / BN;
  const int num_kb = (K + BK - 1) / BK;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tma_a);
    tma_prefetch_desc(&tma_b);
    for (int s = 0; s < Cfg::kStages; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(&tmem_full_bar[a], 1);
      mbar_init(&tmem_empty_bar[a], (TWO ? 2 : 1) * EPI_WARPS);  // one arrive per epilogue warp (of both CTAs)
    }
    for (int a = 0; a < 2 * EPI_WARPS; ++a) mbar_init(&extra_bar[a], 1);
    fence_mbar_init();
  }
  if (warp == 1) {
    if constexpr (TWO) { tmem_alloc_2sm(tmem_base_slot, Cfg::kTmemCols); tmem_relinquish_2sm(); }
    else { tmem_alloc(tmem_base_slot, Cfg::kTmemCols); tmem_relinquish(); }
  }
  tc_fence_before();
  __syncthreads();
  if constexpr (TWO) cluster_sync_all();  // the peer's barriers are initialised before anything signals them
  tc_fence_after();
  const uint32_t tmem_base = *tmem_base_slot;
  // everything above (barriers, TMEM, descriptor prefetch) overlapped the previous kernel's tail
  pdl_wait();
  pdl_trigger();

  if (warp == 0) {
    // ===================== TMA producer =====================
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      SegIter it;
      it.init(unit, num_kb, sk);
      Seg sg;
      while (it.next(sg, unit, unit_stride, num_kb, sk)) {
        const int m_blk = sg.tile / num_n, n_blk = sg.tile - m_blk * num_n;
        const int a_row = m_blk * TM + static_cast<int>(rank) * BM;               // this CTA's 128 rows of A
        const int b_row = n_blk * BN + static_cast<int>(rank) * Cfg::kBRows;     // this CTA's share of B
        for (int kb = sg.kb0; kb < sg.kb1; ++kb) {
          mbar_wait(&empty_bar[stage], phase ^ 1);
          if constexpr (TWO) {
            // both CTAs' loads are credited to the leader's barrier; only the leader arms it
            if (rank == 0) mbar_expect_tx(&full_bar[stage], Cfg::kTxBytes);
            tma_load_2d_2sm(smem_a + stage * Cfg::kABytes, &tma_a, &full_bar[stage], kb * BK, a_row);
            tma_load_2d_2sm(smem_b + stage * Cfg::kBBytes, &tma_b, &full_bar[stage], kb * BK, b_row);
          } else {
            mbar_expect_tx(&full_bar[stage], Cfg::kTxBytes);
            tma_load_2d(smem_a + stage * Cfg::kABytes, &tma_a, &full_bar[stage], kb * BK, a_row);
            tma_load_2d(smem_b + stage * Cfg::kBBytes, &tma_b, &full_bar[stage], kb * BK, b_row);
          }
          if (++stage == Cfg::kStages) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    if (lane == 0 && rank == 0) {
      constexpr uint32_t idesc = make_idesc_bf16(TM, BN);
      int stage = 0;
      uint32_t phase = 0;
      int acc = 0;
      uint32_t acc_phase = 0;
      SegIter it;
      it.init(unit, num_kb, sk);
      Seg sg;
      while (it.next(sg, unit, unit_stride, num_kb, sk)) {
        mbar_wait(&tmem_empty_bar[acc], acc_phase ^ 1);  // epilogue has drained this accumulator
        tc_fence_after();
        const uint32_t tmem_d = tmem_base + static_cast<uint32_t>(acc * BN);
        for (int kb = sg.kb0; kb < sg.kb1; ++kb) {
          mbar_wait(&full_bar[stage], phase);  // TMA bytes have landed
          tc_fence_after();
          const uint64_t da = make_smem_desc_sw128(smem_u32(smem_a + stage * Cfg::kABytes));
          const uint64_t db = make_smem_desc_sw128(smem_u32(smem_b + stage * Cfg::kBBytes));
#pragma unroll
          for (int k = 0; k < BK / 16; ++k) {
            // +32 B per K=16 step inside the 128 B swizzle row (start-address field is >>4)
            const uint32_t accum = static_cast<uint32_t>(kb != sg.kb0 || k != 0);
            if constexpr (TWO)
              umma_bf16_2sm(tmem_d, da + static_cast<uint64_t>(k * 2), db + static_cast<uint64_t>(k * 2), idesc, accum);
            else
              umma_bf16(tmem_d, da + static_cast<uint64_t>(k * 2), db + static_cast<uint64_t>(k * 2), idesc, accum);
          }
          // frees the smem slot (in both CTAs of a pair) once these MMAs retire
          if constexpr (TWO) umma_commit_2sm(&empty_bar[stage], 3); else umma_commit(&empty_bar[stage]);
          if (++stage == Cfg::kStages) { stage = 0; phase ^= 1; }
        }
        // accumulator ready for the epilogue warps (of both CTAs)
        if constexpr (TWO) umma_commit_2sm(&tmem_full_bar[acc], 3); else umma_commit(&tmem_full_bar[acc]);
        if (++acc == 2) { acc = 0; acc_phase ^= 1; }
      }
    }
  } else if constexpr (RowEpi<MODE>::value) {
    // ===================== epilogue (warps 2..), row layout + TMA stores =====================
    const EpiMaps mp{&tma_o0, &tma_o1, &tma_ex, &tma_x2, &tma_o2};
    epilogue_rows<BN, MODE, TWO>(mp, ep, sk, M, N, num_n, num_kb, unit, unit_stride, rank, tmem_base,
                                 smem_stage + (warp - 2) * Cfg::kWarpStaging, extra_bar + (warp - 2) * 2, tmem_full_bar,
                                 tmem_empty_bar, warp, lane);
  } else {
    // ===================== epilogue (warps 2..9), transposing (patch embedding; whole tiles only) =====================
    // Two warps per TMEM lane quadrant (quad = warp % 4); the pair splits the 32-column chunks of the
    // accumulator between them (even / odd), so every SM sub-partition has two epilogue warps to
    // overlap TMEM / shared / global latencies.
    //   Phase A: thread = accumulator row (TMEM lane): 32 fp32 columns -> this warp's staging buffer
    //            (32 rows x 128 B, 16-byte chunks XOR-swizzled by row: conflict-free).
    //   Phase B: 8 lanes per row, lane j owns columns 4j..4j+3, so every global load/store
    //            instruction covers whole 128 B (fp32) / 64 B (bf16) row segments of 4 rows.
    const int num_tiles = sk.dp_tiles;  // (the host never cuts tiles in this mode)
    const int quad = warp & 3;
    const int half = (warp - 2) >> 2;
    uint8_t* stage = smem_stage + (warp - 2) * Cfg::kWarpStaging;
    const int rr0 = lane >> 3, j = lane & 7;
    int acc = 0;
    uint32_t acc_phase = 0;
    constexpr int kChunks = BN / 32;
    for (int tile = unit; tile < num_tiles; tile += unit_stride) {
      const int m_blk = tile / num_n, n_blk = tile - m_blk * num_n;
      const int m_row0 = m_blk * TM + static_cast<int>(rank) * BM;  // first row of this CTA's accumulator
      typedef typename EpiExtra<MODE>::type Ex;
      const int ncol = N - n_blk * BN;  // valid columns in this tile (may exceed BN)
      const int row_base = m_row0 + quad * 32 + rr0;
      int c = half;
      Ex ex[8];
      auto load_extra = [&](Ex(&dst)[8], int chunk) {
        const int col = min(n_blk * BN + chunk * 32 + 4 * j, N - 4);  // clamped: out-of-range lanes never use it
#pragma unroll
        for (int it = 0; it < 8; ++it) dst[it] = epilogue_prefetch<MODE>(ep, min(row_base + it * 4, M - 1), col);
      };
      // the first chunk's operand loads are issued before waiting for the accumulator
      if (c * 32 < ncol) load_extra(ex, c);
      mbar_wait(&tmem_full_bar[acc], acc_phase);
      tc_fence_after();
      const uint32_t taddr = tmem_base + (static_cast<uint32_t>(quad * 32) << 16) + static_cast<uint32_t>(acc * BN);
      uint32_t r[32];
      if (c * 32 < ncol) tmem_ld_32x32(taddr + static_cast<uint32_t>(c * 32), r);
#pragma unroll 1
      for (; c < kChunks && c * 32 < ncol; c += 2) {
        const int col = n_blk * BN + c * 32 + 4 * j;  // this lane's 4 columns in phase B
        const bool has_next = (c + 2 < kChunks) && ((c + 2) * 32 < ncol);
        tmem_ld_wait_regs(r);
#pragma unroll
        for (int k = 0; k < 8; ++k)
          *reinterpret_cast<uint4*>(stage + lane * 128 + (((k ^ lane) & 7) << 4)) =
              make_uint4(r[4 * k], r[4 * k + 1], r[4 * k + 2], r[4 * k + 3]);
        __syncwarp();
        // prefetch the next chunk's accumulator columns while phase B runs
        if (has_next) tmem_ld_32x32(taddr + static_cast<uint32_t>((c + 2) * 32), r);
        if (col < N) {
          float4 bias = make_float4(0.f, 0.f, 0.f, 0.f);
          if (ep.bias != nullptr) bias = *reinterpret_cast<const float4*>(ep.bias + col);
#pragma unroll
          for (int it = 0; it < 8; ++it) {
            const int rr = it * 4 + rr0;
            const int row = m_row0 + quad * 32 + rr;
            float4 v = *reinterpret_cast<const float4*>(stage + rr * 128 + (((j ^ rr) & 7) << 4));
            v.x += bias.x; v.y += bias.y; v.z += bias.z; v.w += bias.w;
            if (row < M) epilogue4<MODE>(ep, row, col, v, ex[it]);
          }
        }
        __syncwarp();
        if (has_next) load_extra(ex, c + 2);
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        if constexpr (TWO) mbar_arrive_cluster(&tmem_empty_bar[acc], 0);  // the leader's MMA thread waits on it
        else mbar_arrive(&tmem_empty_bar[acc]);
      }
      if (++acc == 2) { acc = 0; acc_phase ^= 1; }
    }
  }

  tc_fence_before();
  __syncthreads();
  if constexpr (TWO) cluster_sync_all();  // neither CTA may exit (or free TMEM) while its peer still uses it
  if (warp == 1) {
    tc_fence_after();
    if constexpr (TWO) tmem_dealloc_2sm(tmem_base, Cfg::kTmemCols); else tmem_dealloc(tmem_base, Cfg::kTmemCols);
  }
}

#ifdef MUDPT_BRINGUP
// Bring-up diagnostic only (libmudpt_b200_bringup.so, never the shipped library): a plain
// CUDA-core GEMM with the epilogues of modes 0-5, used to validate the rest of the pipeline
// independently of the tcgen05 path.
template <int MODE>
__global__ void gemm_tn_simt_kernel(const bf16* __restrict__ A, const bf16* __restrict__ B, const GemmEpilogue ep,
                                    int M, int N, int K, int lda, int ldb) {
  const int col = (blockIdx.x * blockDim.x + threadIdx.x) * 8;
  const int row = blockIdx.y;
  if (col >= N || row >= M) return;
  float v[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  const bf16* a = A + static_cast<size_t>(row) * lda;
  for (int k = 0; k < K; ++k) {
    const float av = __bfloat162float(a[k]);
#pragma unroll
    for (int i = 0; i < 8; ++i) v[i] += av * __bfloat162float(B[static_cast<size_t>(col + i) * ldb + k]);
  }
  if (ep.bias != nullptr)
    for (int i = 0; i < 8; ++i) v[i] += ep.bias[col + i];
  epilogue4<MODE>(ep, row, col, make_float4(v[0], v[1], v[2], v[3]), epilogue_prefetch<MODE>(ep, row, col));
  epilogue4<MODE>(ep, row, col + 4, make_float4(v[4], v[5], v[6], v[7]), epilogue_prefetch<MODE>(ep, row, col + 4));
}
static bool g_simt = false;
void gemm_set_bringup_simt(bool on) { g_simt = on; }
#endif

// ---------------------------------------------------------------------------------------
// Host side: tensor maps + launch
// ---------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    // resolved through the runtime so the library has no link-time dependency on libcuda
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  });
  return fn;
}

struct MapKey {
  const void* ptr; int rows, cols, ld, box_rows, box_cols, esize;
  bool operator==(const MapKey& o) const {
    return ptr == o.ptr && rows == o.rows && cols == o.cols && ld == o.ld && box_rows == o.box_rows && box_cols == o.box_cols &&
           esize == o.esize;
  }
};
struct MapKeyHash {
  size_t operator()(const MapKey& k) const {
    size_t h = reinterpret_cast<size_t>(k.ptr);
    h = h * 1000003u ^ static_cast<size_t>(k.rows);
    h = h * 1000003u ^ static_cast<size_t>(k.cols);
    h = h * 1000003u ^ static_cast<size_t>(k.ld);
    h = h * 1000003u ^ static_cast<size_t>(k.box_rows);
    h = h * 1000003u ^ static_cast<size_t>(k.box_cols);
    h = h * 1000003u ^ static_cast<size_t>(k.esize);
    return h;
  }
};
static std::unordered_map<MapKey, CUtensorMap, MapKeyHash> g_maps;
static std::mutex g_maps_mu;

// 2D row-major [rows, cols] (leading dimension ld elements), box = [box_rows, box_cols]: bf16 with box_cols = 64
// and 128B swizzle (MMA operand tiles) or 32 and 64B swizzle (bf16 epilogue boxes); fp32 (esize 4) with box_cols = 32
// and 128B swizzle (fp32 epilogue boxes).
static const char* get_tensor_map(const void* ptr, int rows, int cols, int ld, int box_rows, int box_cols, CUtensorMap* out,
                                  int esize = 2) {
  MapKey key{ptr, rows, cols, ld, box_rows, box_cols, esize};
  std::lock_guard<std::mutex> lk(g_maps_mu);
  auto it = g_maps.find(key);
  if (it != g_maps.end()) { *out = it->second; return nullptr; }
  EncodeTiledFn enc = get_encode_fn();
  if (!enc) return "cuTensorMapEncodeTiled not available (no CUDA driver?)";
  if ((reinterpret_cast<uintptr_t>(ptr) & 15) || (ld % 8)) return "TMA operand must be 16 B aligned with ld % 8 == 0";
  CUtensorMap m;
  cuuint64_t dims[2] = {static_cast<cuuint64_t>(cols), static_cast<cuuint64_t>(rows)};
  const bool f32 = esize == 4;  // fp32 epilogue boxes (32 columns = 128 B rows); everything else is bf16
  cuuint64_t strides[1] = {static_cast<cuuint64_t>(ld) * (f32 ? 4 : 2)};
  cuuint32_t box[2] = {static_cast<cuuint32_t>(box_cols), static_cast<cuuint32_t>(box_rows)};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = enc(&m, f32 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(ptr), dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, box_cols * esize == 128 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B,
                   CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return "cuTensorMapEncodeTiled failed";
  if (g_maps.size() > 4096) g_maps.clear();
  g_maps.emplace(key, m);
  *out = m;
  return nullptr;
}

// 3D bf16 tensor [d2][d1][d0] (d0 contiguous; strides in elements), box [1][box1][box0 = 64] with 128B swizzle:
// one (sequence, head) slice of a token matrix for the attention kernels -- rows past d1 are zero-filled on load
// and clipped on store, so a tile never touches the neighbouring sequence.
const char* tensor_map_3d_bf16(const void* ptr, int d0, int d1, int d2, long long stride1, long long stride2, int box1,
                               CUtensorMap* out) {
  MapKey key{ptr, d1, d0, static_cast<int>(stride1), box1, d2, 3};
  std::lock_guard<std::mutex> lk(g_maps_mu);
  auto it = g_maps.find(key);
  if (it != g_maps.end()) { *out = it->second; return nullptr; }
  EncodeTiledFn enc = get_encode_fn();
  if (!enc) return "cuTensorMapEncodeTiled not available (no CUDA driver?)";
  if ((reinterpret_cast<uintptr_t>(ptr) & 15) || (stride1 % 8) || (stride2 % 8)) return "TMA operand must be 16 B aligned";
  CUtensorMap m;
  cuuint64_t dims[3] = {static_cast<cuuint64_t>(d0), static_cast<cuuint64_t>(d1), static_cast<cuuint64_t>(d2)};
  cuuint64_t strides[2] = {static_cast<cuuint64_t>(stride1) * 2, static_cast<cuuint64_t>(stride2) * 2};
  cuuint32_t box[3] = {64, static_cast<cuuint32_t>(box1), 1};
  cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = enc(&m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<void*>(ptr), dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return "cuTensorMapEncodeTiled (3D) failed";
  if (g_maps.size() > 4096) g_maps.clear();
  g_maps.emplace(key, m);
  *out = m;
  return nullptr;
}

void gemm_clear_tensor_map_cache() {
  std::lock_guard<std::mutex> lk(g_maps_mu);
  g_maps.clear();
}

static bool g_enable_2cta = []{ const char* e = getenv("MUDPT_GEMM_2CTA"); return e ? atoi(e) != 0 : true; }();
// MUDPT_GEMM_SK: 0 = whole tiles only, 1 = cut whenever the tile count is not a multiple of the units, unset = cost model
static const int g_sk_default = []{ const char* e = getenv("MUDPT_GEMM_SK"); return e ? atoi(e) : -1; }();
static int g_sk_mode = g_sk_default;
void gemm_set_stream_k(int mode) { g_sk_mode = mode == -2 ? g_sk_default : mode; }
static int g_num_sms = 0;
static int num_sms() {
  if (g_num_sms == 0) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&g_num_sms, cudaDevAttrMultiProcessorCount, dev);
    if (g_num_sms <= 0) g_num_sms = 148;
  }
  return g_num_sms;
}

static constexpr int kMaxCtas = 160;  // slots / flags are indexed by CTA; 148 SMs on B200
size_t gemm_workspace_partial_bytes() { return static_cast<size_t>(kMaxCtas) * BM * 256 * sizeof(float); }
size_t gemm_workspace_flag_bytes() { return static_cast<size_t>(kMaxCtas) * 16 * sizeof(unsigned); }
static int pick_bn(int N) { return N >= 256 ? 256 : 128; }
int gemm_dots_span(int N) { return pick_bn(N) / (EpiWarps<EPI_GELU_BWD_DOTS>::value / 4); }

// Grouped stream-K plan for `tiles` tiles of `num_kb` k-blocks on `units` units (see the header comment).
// Costs in k-block times (one 64-deep k-block of a tile = 0.46 us on one SM / SM pair at the sustained rate):
//   whole tiles : the remainder costs one more tile-time for everyone: num_kb
//   group of g  : rem * num_kb / g  (imbalance)  +  c * g  (g hand-overs share the L2: measured ~9 us for 74 pair
//                 tiles of 256 KB, i.e. c = 0.29 per pair tile, half of that per single-CTA tile)  +  ~14 (dump, fence,
//                 flag, read-back and the two extra accumulator passes on the last tile's critical path: measured
//                 ~6-8 us whatever g, profiles/r02_gemm_time.txt -- the cut pays for K >= 1536 only)
static SkArgs plan_sk(int tiles, int units, int num_kb, bool pair, const GemmWorkspace* ws, bool allowed) {
  SkArgs a;
  a.dp_tiles = tiles; a.sk_tiles = 0; a.sk_units = 0; a.sk_first = 0;
  a.partials = ws ? ws->partials : nullptr;
  a.flags = ws ? ws->flags : nullptr;
  if (!allowed || ws == nullptr || ws->partials == nullptr || ws->flags == nullptr || g_sk_mode == 0) return a;
  const int rem = tiles % units;
  if (rem == 0) return a;
  const int waves = tiles / units;
  const float c = pair ? 0.29f : 0.145f;
  int g = static_cast<int>(sqrtf(static_cast<float>(rem) * num_kb / c) + 0.5f);
  if (g > units) g = units;
  if (waves == 0) {            // fewer tiles than units: the group would share all of them ...
    // ... with several contributors per tile, read back one after the other by the finisher: measured slower than
    // whole tiles (250 x 512 x 2048: 30.6 against 20.2 us), so only when explicitly forced
    if (g_sk_mode != 1) return a;
    if (g <= rem) return a;    // (nothing to gain from cutting)
    const long long q4 = static_cast<long long>(rem) * num_kb / 4;  // at least 4 k-blocks per unit
    if (g > q4) g = static_cast<int>(q4);
    if (g <= rem) return a;
  } else if (g < 2) {
    g = 2;
  }
  const int sk_tiles = rem + (waves > 0 ? g : 0);
  if (g_sk_mode != 1) {
    // whole tiles: the remainder costs everyone one more tile-time (waves == 0: the one and only tile-time);
    // cut: the group's makespan beyond the full waves
    const float whole = static_cast<float>(num_kb);
    const float cut = static_cast<float>(rem) * num_kb / g + c * g + 14.f;
    if (cut > 0.9f * whole) return a;
  }
  a.dp_tiles = tiles - sk_tiles;
  a.sk_tiles = sk_tiles;
  a.sk_units = g;
  a.sk_first = units - g;
  return a;
}

template <int BN, int MODE, bool TWO>
static const char* launch_one(const CUtensorMap& ta, const CUtensorMap& tb, const CUtensorMap (&te)[5], const GemmEpilogue& ep,
                              int M, int N, int K, cudaStream_t stream, const GemmWorkspace* ws) {
  using Cfg = GemmCfg<BN, MODE, TWO>;
  static bool attr_done = false;
  auto kern = gemm_tn_tcgen05_kernel<BN, MODE, TWO>;
  if (!attr_done) {
    if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::kSmemBytes) != cudaSuccess)
      return "cudaFuncSetAttribute(max dynamic smem) failed";
    attr_done = true;
  }
  constexpr int TM = TWO ? 2 * BM : BM;
  const int tiles = ((M + TM - 1) / TM) * ((N + BN - 1) / BN);
  int units = TWO ? num_sms() / 2 : num_sms();
  if (units * (TWO ? 2 : 1) > kMaxCtas) units = kMaxCtas / (TWO ? 2 : 1);
  const SkArgs sk = plan_sk(tiles, units, (K + BK - 1) / BK, TWO, ws, RowEpi<MODE>::value);
  const int used = sk.sk_tiles > 0 ? units : (tiles < units ? tiles : units);
  const int grid = used * (TWO ? 2 : 1);
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(GemmThreads<MODE>::value);
  cfg.dynamicSmemBytes = Cfg::kSmemBytes;
  cfg.stream = stream;
  cudaLaunchAttribute attr[2];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = TWO ? 2 : 1;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;  // the kernel calls pdl_wait() after its prologue
  attr[1].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 2;
  if (cudaLaunchKernelEx(&cfg, kern, ta, tb, te[0], te[1], te[2], te[3], te[4], ep, sk, M, N, K) != cudaSuccess)
    return launch_status("gemm kernel launch failed");
  count_launch();
  return launch_status("gemm kernel launch failed");
}

template <int MODE>
static const char* launch_mode(const bf16* A, int lda, const bf16* B, int ldb, const GemmEpilogue& ep, int M, int N,
                               int K, cudaStream_t stream, const GemmWorkspace* ws) {
#ifdef MUDPT_BRINGUP
  if (g_simt) {
    if constexpr (MODE <= EPI_PATCH) {
      dim3 grid((N / 8 + 63) / 64, M);
      gemm_tn_simt_kernel<MODE><<<grid, 64, 0, stream>>>(A, B, ep, M, N, K, lda, ldb);
      count_launch();
      return launch_status("simt gemm launch failed");
    } else {
      return "bring-up SIMT GEMM: mode not implemented";
    }
  }
#endif
  // Tile shape: BN = 256 whenever the output is at least that wide (one A row block feeds 256 columns), CTA pairs
  // (256 x 256 pair tiles: a pair tile is two 128 x 256 tiles' worth of work with ~2/3 of the shared-memory operand
  // traffic) whenever there is more than one row block.  The shape is a function of N (and M > 128) only, so the
  // column span of the per-row partials the fused-LayerNorm epilogues exchange is known to the caller; wave
  // quantisation is the work decomposition's problem (stream-K), not the tile shape's.
  int bn = pick_bn(N);
  bool two = g_enable_2cta && bn == 256 && M > BM;
  // Few-row problems (the S gathered CLS / EOT rows of the pruned last block): 256 x 256 pair tiles would leave most
  // of the machine idle while a handful of CTAs walk K alone, so they take 128 x 128 single-CTA tiles (4x the tiles).
  // (Not for EPI_GELU_BWD_DOTS, whose partial-dot span is a function of N alone.)
  if (MODE != EPI_GELU_BWD_DOTS && ((M + 2 * BM - 1) / (2 * BM)) * ((N + 255) / 256) * 4 < num_sms() / 2) {
    bn = 128;
    two = false;
  }
  {  // experiment hook (MUDPT_GEMM_TILE = 1: 128 x 128 single-CTA tiles, 2: 128 x 256 single-CTA, for problems of at most
     // MUDPT_GEMM_TILE_ROWS rows and MUDPT_GEMM_TILE_N columns).  Measured, with 256 x 128 pair tiles as a third variant:
     // every alternative to the 256 x 256 pair tile is slower at the per-rank shapes (profiles/r02_gemm_tile_ab.txt)
    static const int force = getenv("MUDPT_GEMM_TILE") ? atoi(getenv("MUDPT_GEMM_TILE")) : 0;
    static const int force_rows = getenv("MUDPT_GEMM_TILE_ROWS") ? atoi(getenv("MUDPT_GEMM_TILE_ROWS")) : (1 << 30);
    static const int force_n = getenv("MUDPT_GEMM_TILE_N") ? atoi(getenv("MUDPT_GEMM_TILE_N")) : (1 << 30);
    if (force && MODE != EPI_GELU_BWD_DOTS && M <= force_rows && N <= force_n) {
      two = false;
      bn = (force == 1 || N < 256) ? 128 : 256;
    }
  }
  CUtensorMap ta, tb;
  const char* e = get_tensor_map(A, M, K, lda, BM, BK, &ta);
  if (e) return e;
  e = get_tensor_map(B, N, K, ldb, two ? bn / 2 : bn, BK, &tb);
  if (e) return e;
  // epilogue boxes (row-layout modes): out0, out1, operand (residual / saved pre-activation), LN input, out2;
  // unused slots repeat the A map
  CUtensorMap te[5] = {ta, ta, ta, ta, ta};
  if constexpr (F32Epi<MODE>::value) {
    if ((e = get_tensor_map(ep.out0, M, N, ep.ldc, 32, 32, &te[0], 4))) return e;
    if (ResidEpi<MODE>::value && ep.resid != nullptr && (e = get_tensor_map(ep.resid, M, N, ep.ldc, 32, 32, &te[2], 4))) return e;
    if constexpr (DualEpi<MODE>::value) {
      if (ep.out2 != nullptr && (e = get_tensor_map(ep.out2, M, N, ep.ldc, 32, 32, &te[4]))) return e;
      if (MODE == EPI_LN_BWD && (e = get_tensor_map(ep.x2, M, N, ep.ldc, 32, 32, &te[3]))) return e;
    }
  } else if constexpr (RowEpi<MODE>::value) {
    if (ep.out0 != nullptr && (e = get_tensor_map(ep.out0, M, N, ep.ldc, 32, 32, &te[0]))) return e;
    if (GeluFwd<MODE>::value && (e = get_tensor_map(ep.out1, M, N, ep.ldc, 32, 32, &te[1]))) return e;
    if (GeluBwd<MODE>::value && (e = get_tensor_map(ep.aux, M, N, ep.ldc, 32, 32, &te[2]))) return e;
  }
  if (two) return launch_one<256, MODE, true>(ta, tb, te, ep, M, N, K, stream, ws);
  return bn == 256 ? launch_one<256, MODE, false>(ta, tb, te, ep, M, N, K, stream, ws)
                   : launch_one<128, MODE, false>(ta, tb, te, ep, M, N, K, stream, ws);
}

const char* gemm_bf16_tn(const bf16* A, int lda, const bf16* B, int ldb, const GemmEpilogue& ep, int M, int N, int K,
                         cudaStream_t stream, const GemmWorkspace* ws) {
  if (M <= 0 || N <= 0 || K <= 0) return nullptr;
  if (N % 8 != 0 || K % 8 != 0) return "gemm: N and K must be multiples of 8";
  if (ep.ldc % 8 != 0) return "gemm: ldc must be a multiple of 8";
  switch (ep.mode) {
    case EPI_BF16: return launch_mode<EPI_BF16>(A, lda, B, ldb, ep, M, N, K, stream, ws);
    case EPI_F32: return launch_mode<EPI_F32>(A, lda, B, ldb, ep, M, N, K, stream, ws);
    case EPI_RESID_F32:
      if (ep.resid == nullptr) return "gemm: EPI_RESID_F32 needs a residual";
      return launch_mode<EPI_RESID_F32>(A, lda, B, ldb, ep, M, N, K, stream, ws);
    case EPI_GELU: return launch_mode<EPI_GELU>(A, lda, B, ldb, ep, M, N, K, stream, ws);
    case EPI_GELU_ONLY:
      if (ep.out0 == nullptr) return "gemm: EPI_GELU_ONLY needs out0";
      return launch_mode<EPI_GELU_ONLY>(A, lda, B, ldb, ep, M, N, K, stream, ws);
    case EPI_GELU_BWD: return launch_mode<EPI_GELU_BWD>(A, lda, B, ldb, ep, M, N, K, stream, ws);
    case EPI_PATCH: return launch_mode<EPI_PATCH>(A, lda, B, ldb, ep, M, N, K, stream, ws);
    case EPI_LN_BF16:
    case EPI_LN_GELU:
    case EPI_LN_GELU_ONLY:
      if (!ep.ln_stats || !ep.colsum || !ep.bias || ep.ln_parts <= 0 || ep.ln_width <= 0)
        return "gemm: fused LayerNorm needs row statistics, column sums and the folded bias";
      if (ep.mode == EPI_LN_GELU_ONLY) {
        if (ep.out0 == nullptr) return "gemm: EPI_LN_GELU_ONLY needs out0";
        return launch_mode<EPI_LN_GELU_ONLY>(A, lda, B, ldb, ep, M, N, K, stream, ws);
      }
      return ep.mode == EPI_LN_BF16 ? launch_mode<EPI_LN_BF16>(A, lda, B, ldb, ep, M, N, K, stream, ws)
                                    : launch_mode<EPI_LN_GELU>(A, lda, B, ldb, ep, M, N, K, stream, ws);
    case EPI_RESID_STATS:
      if (!ep.resid || !ep.stats_out || !ep.out2) return "gemm: EPI_RESID_STATS needs resid, out2 and stats_out";
      if (N % kStatSpan != 0) return "gemm: EPI_RESID_STATS needs N % 64 == 0";
      if (ep.splice_n > 0 && (!ep.splice_prompt || ep.splice_L <= 0)) return "gemm: bad splice arguments";
      return launch_mode<EPI_RESID_STATS>(A, lda, B, ldb, ep, M, N, K, stream, ws);
    case EPI_LN_BWD:
      if (!ep.ln_stats || !ep.x2 || !ep.dots || ep.ln_parts <= 0 || ep.dot_parts <= 0 || ep.ln_width != N)
        return "gemm: EPI_LN_BWD needs row statistics, the bf16 LN input and the row dots (ln_width == N)";
      return launch_mode<EPI_LN_BWD>(A, lda, B, ldb, ep, M, N, K, stream, ws);
    case EPI_GELU_BWD_DOTS:
      if (!ep.sb || !ep.dots_out) return "gemm: EPI_GELU_BWD_DOTS needs sb and dots_out";
      return launch_mode<EPI_GELU_BWD_DOTS>(A, lda, B, ldb, ep, M, N, K, stream, ws);
    default: return "gemm: unknown epilogue mode";
  }
}

}  // namespace mudpt
