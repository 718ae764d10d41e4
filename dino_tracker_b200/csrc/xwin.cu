// Coarse pass + exact window (see xwin.cuh): kernels and launchers.
#include <cuda_fp16.h>

#include "common.cuh"
#include "corr.cuh"
#include "tcgemm.cuh"
#include "tcgemm2.cuh"
#include "xwin.cuh"

namespace dtk {

int make_tmap_4d(CUtensorMap* map, const void* base, const uint64_t dims[4], const uint64_t strides_bytes[3],
                 const uint32_t box[4], int elem);   // corr_tc.cu

// ====================================================================================================== 1. coarse GEMM
// Epilogue of the single-pass kind::f16 GEMM over the `hi` halves: nothing is stored per token.  Per (map, 256-token tile):
// key1 = bits(max) << 32 | (0x7fffffff - first token holding it), max2 = second largest value (>= 0).  Values are the same
// expression as the exact path, relu(acc / max(|d| |F|, 1e-8)), with a fast division (its error is part of XW_EPS).
struct CoarseEpi {
  const float* rnorms;     // [T][P] 1 / |F[t][p]| (xw_rnorm_kernel; every norm is >= XW_MIN_NORM on this path)
  const float* desc_norm;
  const int* grp_frame;
  const int* grp_row0;
  const int* grp_map0;
  unsigned long long* key1;
  float* max2;
  int n_tiles, P;
  // The epilogue warps have their schedulers (almost) to themselves, so every dependent instruction costs its full latency:
  // the 32 values of a column block are formed as 32 independent chains (all loads first), and the (max, first token, second
  // value) statistics run in four interleaved branch-free accumulators (columns = accumulator mod 4), merged per tile.
  // Per element only u = acc * (1 / |F|) is formed; the row's positive factor 1 / |d| (and the ReLU) are applied to the two
  // statistics at the end of the tile -- multiplication by a positive constant does not change which token holds the maximum.
  struct State { float m1[4], m2[4]; int tok[4]; };
  __device__ __forceinline__ void tile_begin(State& s) const {
#pragma unroll
    for (int a = 0; a < 4; ++a) { s.m1[a] = -INFINITY; s.m2[a] = -INFINITY; s.tok[a] = 0x7fffffff; }
  }
  __device__ __forceinline__ void tile_end(State& s, int g, int r, int nt) const {
    if (nt >= n_tiles) return;   // second half of the last GEMM tile lies completely past the end of the map
    float m1 = s.m1[0], m2 = s.m2[0];
    int tok = s.tok[0];
#pragma unroll
    for (int a = 1; a < 4; ++a) {   // top-2 of the union; equal maxima -> the smaller token (first arg-max)
      m2 = fmaxf(fmaxf(m2, s.m2[a]), fminf(m1, s.m1[a]));
      const bool take = s.m1[a] > m1 || (s.m1[a] == m1 && s.tok[a] < tok);
      tok = take ? s.tok[a] : tok;
      m1 = fmaxf(m1, s.m1[a]);
    }
    const float rdn = __fdividef(1.f, fmaxf(desc_norm[grp_row0[g] + r], XW_MIN_NORM));
    const size_t o = (size_t)(grp_map0[g] + r) * n_tiles + nt;
    key1[o] = ((unsigned long long)__float_as_uint(fmaxf(m1 * rdn, 0.f)) << 32) | (unsigned)(0x7fffffff - tok);
    max2[o] = fmaxf(m2 * rdn, 0.f);
  }
  __device__ __forceinline__ void operator()(State& s, int g, int r, int col0, const float (&f)[32], int ncols) const {
    const float* rn = rnorms + (size_t)grp_frame[g] * P + col0;
    float t[32];
#pragma unroll
    for (int i = 0; i < 32; ++i) t[i] = __ldg(rn + (i < ncols ? i : 0));
#pragma unroll
    for (int i = 0; i < 32; ++i) t[i] = i < ncols ? f[i] * t[i] : -INFINITY;      // columns past the end of the map never win
#pragma unroll
    for (int i = 0; i < 32; ++i) {
      const int a = i & 3;
      const float v = t[i];
      s.m2[a] = fmaxf(s.m2[a], fminf(s.m1[a], v));
      s.tok[a] = v > s.m1[a] ? col0 + i : s.tok[a];      // strict: the first token of this accumulator holding its maximum
      s.m1[a] = fmaxf(s.m1[a], v);
    }
  }
};

// rnorms[i] = 1 / norms[i]; *min_bits = bit pattern of the smallest norm (norms are >= 0: the bit pattern orders like the value)
__global__ void xw_rnorm_kernel(const float* __restrict__ norms, float* __restrict__ rnorms, size_t n, unsigned* __restrict__ min_bits) {
  float mn = INFINITY;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    const float v = norms[i];
    rnorms[i] = __fdiv_rn(1.f, fmaxf(v, XW_MIN_NORM));
    mn = fminf(mn, v);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) mn = fminf(mn, __shfl_xor_sync(0xffffffffu, mn, o));
  if ((threadIdx.x & 31) == 0) atomicMin(min_bits, __float_as_uint(fmaxf(mn, 0.f)));
}

int launch_xw_rnorms(const FeatView& fv, float* rnorms, unsigned* min_bits, cudaStream_t st) {
  const size_t n = (size_t)fv.T * fv.P;
  DTK_CUDA(cudaMemsetAsync(min_bits, 0x7f, sizeof(unsigned), st));   // 0x7f7f7f7f: a huge positive float
  ProfRange pr(PROF_XW_PLAN, st);
  xw_rnorm_kernel<<<148 * 4, 256, 0, st>>>(fv.norms, rnorms, n, min_bits);
  DTK_LAUNCHED();
  return DINOTRK_OK;
}

int launch_xw_coarse(const FeatView& fv, const void* desc_hi, int desc_rows, const float* desc_norm, const int* grp_frame,
                     const int* grp_row0, const int* grp_m, const int* grp_map0, const int* tile_start, int n_groups,
                     int max_tiles, const XwChunk& xc, cudaStream_t st, const float* rnorms) {
  using Cfg = Tc2Cfg<TcMode::F16, 8, false>;
  using Base = TcCfg<TcMode::F16, TC2_BN>;
  static_assert(TC2_BN == 2 * XW_TILE, "coarse keys are per half GEMM tile (8 epilogue warps)");
  CUtensorMap tmA, tmB;
  int rc;
  if ((rc = make_tmap_2d(&tmA, desc_hi, desc_rows, fv.C, 128, Base::kBK, TMAP_F16))) return rc;
  if ((rc = make_tmap_3d(&tmB, fv.hi, fv.T, fv.P, fv.C, TC2_BN / 2, Base::kBK, TMAP_F16))) return rc;
  auto kern = tc_gemm2_kernel<TcMode::F16, CoarseEpi, 8>;
  static PerDev<bool> attr_dev;
  bool& attr = attr_dev.get();
  if (!attr) {
    DTK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::kSmem));
    attr = true;
  }
  TcProblem pb{grp_frame, grp_row0, grp_m, tile_start, n_groups, fv.P, fv.C};
  CoarseEpi epi{rnorms, desc_norm, grp_frame, grp_row0, grp_map0, xc.key1, xc.max2, cdiv(fv.P, XW_TILE), fv.P};
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  const int tiles_bound = max_tiles * cdiv(fv.P, TC2_BN);
  int grid = 2 * (tiles_bound < sms / 2 ? tiles_bound : sms / 2);
  if (grid < 2) grid = 2;
  ProfRange pr(PROF_XW_COARSE, st);
  kern<<<grid, 64 + 32 * 8, Cfg::kSmem, st>>>(tmA, tmA, tmB, tmB, pb, epi);
  DTK_LAUNCHED();
  return DINOTRK_OK;
}

// ====================================================================================================== 2. plan
// (a) one warp per MAP (lane = tile): global coarse maximum, candidate tiles (max1 >= gmax - 2 eps), ambiguity (some tile's
//     SECOND value is also within 2 eps: an arg-max candidate whose token is unknown).  Writes the candidate tokens and
//     pinfo[map] = coarse arg-max token, or -1 - token if the map is ambiguous.
// (b) one warp per CELL: a map fits if every candidate lies within +-XW_SLACK of the lower medians of the unambiguous maps'
//     coarse arg-max row / column.  The cell's box covers the 15 x 15 windows around every fitting candidate: 16 columns
//     (8 box rows per M-part) when those candidates span <= 2 columns, else 21 (6 rows per part); 2..4 parts.
constexpr int PLAN_WARPS = 8;
__global__ void __launch_bounds__(PLAN_WARPS * 32)
xw_cand_kernel(int n_maps, const float* __restrict__ desc_norm, int n_groups, int n_tiles, const unsigned long long* __restrict__ key1,
               const float* __restrict__ max2, int* __restrict__ cand, int* __restrict__ pinfo, int* __restrict__ slow_cnt) {
  const int lane = threadIdx.x & 31;
  const int gw = blockIdx.x * PLAN_WARPS + (threadIdx.x >> 5), nw = gridDim.x * PLAN_WARPS;
  if (gw == 0)   // zero the counters of this chunk (n_groups per-group queue lengths + XW_NCNT chunk totals)
    for (int i = lane; i < n_groups + XW_NCNT; i += 32) slow_cnt[i] = 0;
  for (int map = gw; map < n_maps; map += nw) {
    const unsigned long long* k1 = key1 + (size_t)map * n_tiles;
    const float* k2 = max2 + (size_t)map * n_tiles;
    unsigned long long kk[2] = {0ull, 0ull};
    float v2[2] = {0.f, 0.f};
#pragma unroll
    for (int q = 0; q < 2; ++q) {
      const int t = lane + 32 * q;
      if (t < n_tiles) { kk[q] = __ldg(k1 + t); v2[q] = __ldg(k2 + t); }
    }
    unsigned long long gk = kk[0] > kk[1] ? kk[0] : kk[1];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) { unsigned long long t = __shfl_xor_sync(0xffffffffu, gk, o); gk = t > gk ? t : gk; }
    const float gmax = __uint_as_float((unsigned)(gk >> 32));
    const int ptok = 0x7fffffff - (int)(gk & 0xffffffffu);
    const float th = gmax - 2.f * XW_EPS;
    bool amb = false;
    int ncand = 0;
#pragma unroll
    for (int q = 0; q < 2; ++q) {
      const int t = lane + 32 * q;
      const bool in = t < n_tiles;
      const bool isc = in && __uint_as_float((unsigned)(kk[q] >> 32)) >= th;
      const unsigned cm = __ballot_sync(0xffffffffu, isc);
      amb = amb || __any_sync(0xffffffffu, in && v2[q] >= th);
      const int rank = ncand + __popc(cm & ((1u << lane) - 1u));
      if (isc && rank < XW_MAX_CAND) cand[(size_t)map * XW_MAX_CAND + rank] = 0x7fffffff - (int)(kk[q] & 0xffffffffu);
      ncand += __popc(cm);
    }
    // a (near-)zero map has no meaningful arg-max candidates; a tiny descriptor norm voids the error bound
    amb = amb || ncand > XW_MAX_CAND || !(gmax > 4.f * XW_EPS) || !(desc_norm[map] >= XW_MIN_NORM);
    if (lane >= ncand && lane < XW_MAX_CAND) cand[(size_t)map * XW_MAX_CAND + lane] = -1;
    if (lane == 0) pinfo[map] = amb ? -1 - ptok : ptok;
  }
}

__global__ void __launch_bounds__(PLAN_WARPS * 32)
xw_cell_kernel(XwCells cells, int w, const int* __restrict__ cand, const int* __restrict__ pinfo, int* __restrict__ stat,
               int* __restrict__ cell_of, XwBox* __restrict__ box, int* __restrict__ part_cnt) {
  __shared__ short s_r[PLAN_WARPS][XW_MAX_CELL], s_c[PLAN_WARPS][XW_MAX_CELL];
  __shared__ unsigned char s_ok[PLAN_WARPS][XW_MAX_CELL];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int gw = blockIdx.x * PLAN_WARPS + wid, nw = gridDim.x * PLAN_WARPS;
  for (int cell = gw; cell < cells.n_cells; cell += nw) {
    const int row0 = cells.row0[cell], m = cells.m[cell];
    int nv = 0;
    for (int r = lane; r < m; r += 32) {
      const int pi = __ldg(pinfo + row0 + r);
      const int ptok = pi >= 0 ? pi : -1 - pi;
      s_r[wid][r] = (short)(ptok / w);
      s_c[wid][r] = (short)(ptok - (ptok / w) * w);
      s_ok[wid][r] = pi >= 0 ? 1 : 0;
      nv += pi >= 0 ? 1 : 0;
      cell_of[row0 + r] = cell;
    }
    __syncwarp();
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) nv += __shfl_xor_sync(0xffffffffu, nv, o);
    int med_r = -1, med_c = -1;
    if (nv > 0) {   // lower medians over the unambiguous maps
      const int want = (nv - 1) / 2;
      for (int r = lane; r < m; r += 32) {
        if (!s_ok[wid][r]) continue;
        int rk_r = 0, rk_c = 0;
        const int vr = s_r[wid][r], vc = s_c[wid][r];
        for (int q = 0; q < m; ++q) {
          if (!s_ok[wid][q]) continue;
          rk_r += (s_r[wid][q] < vr) || (s_r[wid][q] == vr && q < r);
          rk_c += (s_c[wid][q] < vc) || (s_c[wid][q] == vc && q < r);
        }
        if (rk_r == want) med_r = vr;
        if (rk_c == want) med_c = vc;
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        med_r = max(med_r, __shfl_xor_sync(0xffffffffu, med_r, o));
        med_c = max(med_c, __shfl_xor_sync(0xffffffffu, med_c, o));
      }
    }
    // bounding rectangle of the fitting maps' candidates (within +-XW_SLACK of the medians: at most 7 x 7 tokens)
    int n_fit = 0, r_lo = INT_MAX, r_hi = INT_MIN, c_lo = INT_MAX, c_hi = INT_MIN;
    for (int r = lane; r < m; r += 32) {
      const int map = row0 + r;
      bool fit = s_ok[wid][r] != 0;
      int mr_lo = INT_MAX, mr_hi = INT_MIN, mc_lo = INT_MAX, mc_hi = INT_MIN;
      if (fit) {
        const int4 cd = __ldg(reinterpret_cast<const int4*>(cand) + map);
        const int ct[4] = {cd.x, cd.y, cd.z, cd.w};
#pragma unroll
        for (int q = 0; q < XW_MAX_CAND; ++q)
          if (ct[q] >= 0) {
            const int tr = ct[q] / w, tc_ = ct[q] - tr * w;
            fit = fit && abs(tr - med_r) <= XW_SLACK && abs(tc_ - med_c) <= XW_SLACK;
            mr_lo = min(mr_lo, tr); mr_hi = max(mr_hi, tr); mc_lo = min(mc_lo, tc_); mc_hi = max(mc_hi, tc_);
          }
      }
      stat[map] = fit ? 0 : 1;
      n_fit += fit ? 1 : 0;
      if (fit) { r_lo = min(r_lo, mr_lo); r_hi = max(r_hi, mr_hi); c_lo = min(c_lo, mc_lo); c_hi = max(c_hi, mc_hi); }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      n_fit += __shfl_xor_sync(0xffffffffu, n_fit, o);
      r_lo = min(r_lo, __shfl_xor_sync(0xffffffffu, r_lo, o)); r_hi = max(r_hi, __shfl_xor_sync(0xffffffffu, r_hi, o));
      c_lo = min(c_lo, __shfl_xor_sync(0xffffffffu, c_lo, o)); c_hi = max(c_hi, __shfl_xor_sync(0xffffffffu, c_hi, o));
    }
    if (lane == 0) {
      XwBox b{0, 0, 0, 0, 0};
      if (n_fit > 0) {   // the rectangle widened by the window's half side (7) on every side: 15..21 rows and columns
        const int height = r_hi - r_lo + 15;
        const bool wide = c_hi - c_lo + 15 > XW_NARROW;
        const int rows = wide ? XW_ROWS_WIDE : XW_ROWS_NARROW;
        b = XwBox{r_lo - 7, c_lo - 7, (short)(wide ? XW_BOX : XW_NARROW), (short)height, (short)((height + rows - 1) / rows)};
        atomicAdd(part_cnt + b.parts - 2, 1);
      }
      box[cell] = b;
    }
    __syncwarp();
  }
}

int launch_xw_plan(const XwCells& cells, const float* desc_norm, int n_groups, const dinotrk_geom& g, const XwChunk& xc,
                   cudaStream_t st, int n_maps) {
  static_assert(XW_MAX_CAND == 4, "candidates are read as one int4");
  const int n_tiles = cdiv(g.h * g.w, XW_TILE);
  DTK_CHECK_ARG(n_tiles <= 64, "exact-window path: token grid too large (%d tiles)", n_tiles);
  DTK_CHECK_ARG(cells.max_m <= XW_MAX_CELL, "exact-window path: cell of %d rows", cells.max_m);
  if (cells.n_cells <= 0 || n_maps <= 0) return DINOTRK_OK;
  ProfRange pr(PROF_XW_PLAN, st);
  int grid = cdiv(n_maps, PLAN_WARPS);
  if (grid > 148 * 8) grid = 148 * 8;
  xw_cand_kernel<<<grid, PLAN_WARPS * 32, 0, st>>>(n_maps, desc_norm, n_groups, n_tiles, xc.key1, xc.max2, xc.cand, xc.pinfo, xc.slow_cnt);
  DTK_LAUNCHED();
  grid = cdiv(cells.n_cells, PLAN_WARPS);
  if (grid > 148 * 8) grid = 148 * 8;
  xw_cell_kernel<<<grid, PLAN_WARPS * 32, 0, st>>>(cells, g.w, xc.cand, xc.pinfo, xc.stat, xc.cell_of, xc.box,
                                                   xc.slow_cnt + n_groups + 2);
  DTK_LAUNCHED();
  return DINOTRK_OK;
}

// ====================================================================================================== 3. exact box GEMM
// Persistent, warp-specialised (same roles as tc_gemm_kernel).  One "tile" = one cell.  The BOX TOKENS are the UMMA M
// operand and the cell's descriptors the N operand (64 or 128 columns): a cell of T = 50 maps fills 50 of 64 columns, where
// descriptors-as-rows filled 50 of 128 rows.  The cell's box (XwBox) comes in M-parts of 128 rows: 8 box rows of a 16-wide
// box (2 or 3 parts) or 6 rows of a 21-wide one (126 of 128 rows, 3 or 4 parts).  D[part][token][map] in TMEM (a slot of
// 4 x NB columns whatever the cell's part count; two cells in flight for NB = 64), split precision (lo*hi + hi*lo + hi*hi
// per K step, in the full-map GEMM's order).  A K-block of the descriptors (hi, lo) is loaded once and used by the cell's
// parts; the box rows arrive as 4-D TMA boxes {64 channels, 16 columns, 8 rows, 1 frame} or {64, 21, 6, 1} of the
// [T][h][w][C] feature video, zero-filled outside the token grid (rows of the last part past the box are computed and
// dropped).  Epilogue: TMEM lane = box token, so for every map the 32 lanes of a warp write consecutive floats of its
// accumulator row -- coalesced without a transpose.
template <int NB>
struct XwCfg {
  static constexpr int kBK = 64;                            // fp16 elements per 128-byte swizzle row
  static constexpr int kTokBytes = 128 * 128;               // hi or lo half of a token tile: 128 rows (126 used by a 21-wide box)
  static constexpr int kTokStage = 2 * kTokBytes, kTokStages = NB == 64 ? 5 : 4;
  static constexpr int kTokTxNarrow = 2 * XW_ROWS_NARROW * XW_NARROW * 128, kTokTxWide = 2 * XW_ROWS_WIDE * XW_BOX * 128;
  static_assert(XW_ROWS_NARROW * XW_NARROW <= 128 && XW_ROWS_WIDE * XW_BOX <= 128, "an M-part is at most 128 tokens");
  static constexpr int kDescBytes = NB * 128;               // one operand half of the descriptor K-block
  static constexpr int kDescStage = 2 * kDescBytes, kDescStages = 2;
  static constexpr int kSmem = kDescStages * kDescStage + kTokStages * kTokStage + 256;
  static constexpr int kAccCols = XW_PARTS * NB, kAccBufs = 512 / kAccCols;
  static constexpr uint32_t kIdesc = tc::make_idesc(0, 128, NB);
};

namespace tc {
__device__ __forceinline__ void tma_load_4d(const CUtensorMap* m, uint64_t* bar, void* dst, int c0, int c1, int c2, int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];\n" ::"r"(
          smem_u32(dst)),
      "l"(m), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}
}  // namespace tc

template <int NB>
__global__ void __launch_bounds__(TC_THREADS, 1)
xw_gemm_kernel(const __grid_constant__ CUtensorMap tmD_hi, const __grid_constant__ CUtensorMap tmD_lo,
               const __grid_constant__ CUtensorMap tmN_hi, const __grid_constant__ CUtensorMap tmN_lo,
               const __grid_constant__ CUtensorMap tmW_hi, const __grid_constant__ CUtensorMap tmW_lo, XwCells cells,
               const XwBox* __restrict__ box, float* __restrict__ xbox, int K) {
  using Cfg = XwCfg<NB>;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw;
  if (tc::smem_u32(smem) & 1023u) __trap();   // no static shared memory in this kernel: the window starts 1 KB-aligned
  uint8_t* t_ring = smem;                                           // token tiles (UMMA A)
  uint8_t* d_ring = smem + Cfg::kTokStages * Cfg::kTokStage;        // descriptor K-blocks (UMMA B)
  uint64_t* bars = reinterpret_cast<uint64_t*>(d_ring + Cfg::kDescStages * Cfg::kDescStage);
  uint64_t* d_full = bars;                          // [2]
  uint64_t* d_empty = d_full + Cfg::kDescStages;    // [2]
  uint64_t* t_full = d_empty + Cfg::kDescStages;    // [kTokStages]
  uint64_t* t_empty = t_full + Cfg::kTokStages;     // [kTokStages]
  uint64_t* tfull = t_empty + Cfg::kTokStages;      // [2]
  uint64_t* tempty = tfull + 2;                     // [2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty + 2);
  static_assert((2 * Cfg::kDescStages + 2 * Cfg::kTokStages + 4) * 8 + 4 <= 256, "barrier block");

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int KB = (K + Cfg::kBK - 1) / Cfg::kBK;

  if (warp == 0 && lane == 0) {
    tc::prefetch_tmap(&tmD_hi); tc::prefetch_tmap(&tmD_lo); tc::prefetch_tmap(&tmN_hi); tc::prefetch_tmap(&tmN_lo);
    tc::prefetch_tmap(&tmW_hi); tc::prefetch_tmap(&tmW_lo);
    for (int s = 0; s < Cfg::kDescStages; ++s) { tc::mbar_init(&d_full[s], 1); tc::mbar_init(&d_empty[s], 1); }
    for (int s = 0; s < Cfg::kTokStages; ++s) { tc::mbar_init(&t_full[s], 1); tc::mbar_init(&t_empty[s], 1); }
    for (int s = 0; s < 2; ++s) { tc::mbar_init(&tfull[s], 1); tc::mbar_init(&tempty[s], 4); }
    tc::mbar_fence_init();
  }
  if (warp == 1) tc::tmem_alloc(tmem_slot, 512);
  tc::fence_before_sync();
  __syncthreads();
  tc::fence_after_sync();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ===================== TMA producer =====================
    if (tc::elect_one()) {
      int ds = 0, dph = 0, ts = 0, tph = 0;
      for (int cell = blockIdx.x; cell < cells.n_cells; cell += gridDim.x) {
        const XwBox bx = box[cell];
        if (bx.parts == 0) continue;               // every map of the cell takes the full-map path
        const bool wide = bx.width == XW_BOX;
        const CUtensorMap* tm_hi = wide ? &tmW_hi : &tmN_hi;
        const CUtensorMap* tm_lo = wide ? &tmW_lo : &tmN_lo;
        const int rows = wide ? XW_ROWS_WIDE : XW_ROWS_NARROW, tx = wide ? Cfg::kTokTxWide : Cfg::kTokTxNarrow;
        const int drow = cells.row0[cell], frame = cells.frame[cell];
        for (int kb = 0; kb < KB; ++kb) {
          const int k0 = kb * Cfg::kBK;
          tc::mbar_wait(&d_empty[ds], dph ^ 1);
          uint8_t* sd = d_ring + ds * Cfg::kDescStage;
          tc::mbar_expect_tx(&d_full[ds], Cfg::kDescStage);
          tc::tma_load_2d(&tmD_hi, &d_full[ds], sd, k0, drow);
          tc::tma_load_2d(&tmD_lo, &d_full[ds], sd + Cfg::kDescBytes, k0, drow);
          if (++ds == Cfg::kDescStages) { ds = 0; dph ^= 1; }
          for (int part = 0; part < bx.parts; ++part) {
            tc::mbar_wait(&t_empty[ts], tph ^ 1);
            uint8_t* st = t_ring + ts * Cfg::kTokStage;
            tc::mbar_expect_tx(&t_full[ts], tx);
            tc::tma_load_4d(tm_hi, &t_full[ts], st, k0, bx.col, bx.row + part * rows, frame);
            tc::tma_load_4d(tm_lo, &t_full[ts], st + Cfg::kTokBytes, k0, bx.col, bx.row + part * rows, frame);
            if (++ts == Cfg::kTokStages) { ts = 0; tph ^= 1; }
          }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    int ds = 0, dph = 0, ts = 0, tph = 0, it = 0;
    for (int cell = blockIdx.x; cell < cells.n_cells; cell += gridDim.x) {
      const int parts = box[cell].parts;
      if (parts == 0) continue;
      const int buf = it % Cfg::kAccBufs, use = it / Cfg::kAccBufs;
      tc::mbar_wait(&tempty[buf], (use & 1) ^ 1);
      tc::fence_after_sync();
      for (int kb = 0; kb < KB; ++kb) {
        tc::mbar_wait(&d_full[ds], dph);
        const uint32_t sd = tc::smem_u32(d_ring + ds * Cfg::kDescStage);
        for (int part = 0; part < parts; ++part) {
          tc::mbar_wait(&t_full[ts], tph);
          tc::fence_after_sync();
          if (tc::elect_one()) {
            const uint32_t st = tc::smem_u32(t_ring + ts * Cfg::kTokStage);
            const uint32_t tmem_d = tmem_base + buf * Cfg::kAccCols + part * NB;
#pragma unroll
            for (int ks = 0; ks < Cfg::kBK / 16; ++ks) {
              const uint32_t koff = ks * 32;
              const uint64_t t_hi = tc::smem_desc_sw128(st + koff), t_lo = tc::smem_desc_sw128(st + Cfg::kTokBytes + koff);
              const uint64_t d_hi = tc::smem_desc_sw128(sd + koff), d_lo = tc::smem_desc_sw128(sd + Cfg::kDescBytes + koff);
              const uint32_t first = (kb == 0 && ks == 0) ? 0u : 1u;
              tc::mma_ss<false>(tmem_d, t_hi, d_lo, Cfg::kIdesc, first);   // desc_lo * tok_hi, desc_hi * tok_lo, desc_hi * tok_hi:
              tc::mma_ss<false>(tmem_d, t_lo, d_hi, Cfg::kIdesc, 1u);      // the product order of tc_gemm_kernel (F16X3)
              tc::mma_ss<false>(tmem_d, t_hi, d_hi, Cfg::kIdesc, 1u);
            }
            tc::mma_commit(&t_empty[ts]);
            if (part == parts - 1) {
              tc::mma_commit(&d_empty[ds]);
              if (kb == KB - 1) tc::mma_commit(&tfull[buf]);
            }
          }
          __syncwarp();
          if (++ts == Cfg::kTokStages) { ts = 0; tph ^= 1; }
        }
        if (++ds == Cfg::kDescStages) { ds = 0; dph ^= 1; }
      }
      ++it;
    }
  } else {
    // ===================== epilogue: TMEM lane = box token -> xbox[map][token], coalesced along the tokens =====================
    const int quad = warp & 3;
    int it = 0;
    for (int cell = blockIdx.x; cell < cells.n_cells; cell += gridDim.x) {
      const XwBox bx = box[cell];
      if (bx.parts == 0) continue;
      const int m = cells.m[cell], map0 = cells.row0[cell];
      const int part_tok = (bx.width == XW_BOX ? XW_ROWS_WIDE : XW_ROWS_NARROW) * bx.width;
      const int buf = it % Cfg::kAccBufs, use = it / Cfg::kAccBufs;
      tc::mbar_wait(&tfull[buf], use & 1);
      tc::fence_after_sync();
      const int tok = quad * 32 + lane;
#pragma unroll 1
      for (int part = 0; part < bx.parts; ++part) {
        const int col = part * part_tok + tok;
        const bool ok = tok < part_tok && col < bx.height * bx.width;
        const uint32_t taddr = tmem_base + ((uint32_t)(quad * 32) << 16) + buf * Cfg::kAccCols + part * NB;
        float* dst = xbox + (size_t)map0 * XW_COLS + col;
#pragma unroll 1
        for (int c = 0; c < NB && c < m; c += 32) {
          uint32_t v[32];
          tc::tmem_ld32(taddr + c, v);
          tc::tmem_ld_wait();
          if (ok) {
#pragma unroll
            for (int i = 0; i < 32; ++i)
              if (c + i < m) dst[(size_t)(c + i) * XW_COLS] = __uint_as_float(v[i]);
          }
        }
      }
      tc::fence_before_sync();
      __syncwarp();
      if (lane == 0) tc::mbar_arrive(&tempty[buf]);
      ++it;
    }
  }

  tc::fence_before_sync();
  __syncthreads();
  if (warp == 1) {
    tc::fence_after_sync();
    tc::tmem_dealloc(tmem_base, 512);
  }
}

int launch_xw_gemm(const FeatView& fv, const dinotrk_geom& g, const void* desc_hi, const void* desc_lo, int desc_rows,
                   const XwCells& cells, const XwChunk& xc, cudaStream_t st) {
  if (cells.n_cells <= 0) return DINOTRK_OK;
  DTK_CHECK_ARG(fv.C % 8 == 0 && cells.max_m <= XW_MAX_CELL, "exact-window GEMM: bad sizes");
  const bool small = cells.max_m <= 64;
  const int nb = small ? 64 : 128;
  CUtensorMap tD_hi, tD_lo, tN_hi, tN_lo, tW_hi, tW_lo;
  int rc;
  if ((rc = make_tmap_2d(&tD_hi, desc_hi, desc_rows, fv.C, nb, 64, TMAP_F16))) return rc;
  if ((rc = make_tmap_2d(&tD_lo, desc_lo, desc_rows, fv.C, nb, 64, TMAP_F16))) return rc;
  const uint64_t dims[4] = {(uint64_t)fv.C, (uint64_t)g.w, (uint64_t)g.h, (uint64_t)fv.T};
  const uint64_t strides[3] = {(uint64_t)fv.C * 2, (uint64_t)g.w * fv.C * 2, (uint64_t)fv.P * fv.C * 2};
  const uint32_t box_n[4] = {64, XW_NARROW, XW_ROWS_NARROW, 1}, box_w[4] = {64, XW_BOX, XW_ROWS_WIDE, 1};
  if ((rc = make_tmap_4d(&tN_hi, fv.hi, dims, strides, box_n, TMAP_F16))) return rc;
  if ((rc = make_tmap_4d(&tN_lo, fv.lo, dims, strides, box_n, TMAP_F16))) return rc;
  if ((rc = make_tmap_4d(&tW_hi, fv.hi, dims, strides, box_w, TMAP_F16))) return rc;
  if ((rc = make_tmap_4d(&tW_lo, fv.lo, dims, strides, box_w, TMAP_F16))) return rc;
  static PerDev<bool> attr_dev;
  bool& attr = attr_dev.get();
  if (!attr) {
    DTK_CUDA(cudaFuncSetAttribute(xw_gemm_kernel<64>, cudaFuncAttributeMaxDynamicSharedMemorySize, XwCfg<64>::kSmem));
    DTK_CUDA(cudaFuncSetAttribute(xw_gemm_kernel<128>, cudaFuncAttributeMaxDynamicSharedMemorySize, XwCfg<128>::kSmem));
    attr = true;
  }
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  const int grid = cells.n_cells < sms ? cells.n_cells : sms;
  ProfRange pr(PROF_XW_GEMM, st);
  if (small)
    xw_gemm_kernel<64><<<grid, TC_THREADS, XwCfg<64>::kSmem, st>>>(tD_hi, tD_lo, tN_hi, tN_lo, tW_hi, tW_lo, cells, xc.box, xc.xbox, fv.C);
  else
    xw_gemm_kernel<128><<<grid, TC_THREADS, XwCfg<128>::kSmem, st>>>(tD_hi, tD_lo, tN_hi, tN_lo, tW_hi, tW_lo, cells, xc.box, xc.xbox, fv.C);
  DTK_LAUNCHED();
  return DINOTRK_OK;
}

// ====================================================================================================== 4. head
// One warp per map.  Exact values v = relu(acc / max(|d| |F|, 1e-8)) (the full-map GEMM's epilogue expression) are formed
// from the raw accumulators of xbox on demand: at the candidates (-> exact first arg-max) and on the 15 x 15 window.  Then
// the refiner on the window (hidden layer 13 x 13 x 16 in two channel halves, logits on 11 x 11), softmax sums, the
// certificate of head.cu with   m_out = max(exact window values outside the 7 x 7 core,
//                                             per tile: (its max token inside the core ? second value : max) + XW_EPS)
// and either the track point or a place in the group's full-map queue.
constexpr int XH_WARPS = 8;
constexpr int XH_MP = 18;      // input window pitch (float2 units, even: 16-byte loads of two positions; 4 row groups -> 4 bank quads)
constexpr int XWM = 15, XWH = 13, XWB = 11;
constexpr int XH_MWIN = 544;   // floats: the 15 x 15 input window with every value stored twice (XWM * XH_MP * 2 = 540)
constexpr int XH_PER_WARP = XH_MWIN + XWH * XWH * 16;      // + hidden window [position][8 channel pairs (c, c + 8)]
constexpr int XH_WTAB = 20 * 16;                           // floats: refiner weights as pairs [w1 k = 0..8 | b1 | w2 k = 0..8 | -][8 pairs]
constexpr int XH_SMEM = (XH_WTAB + XH_WARPS * XH_PER_WARP) * 4;

struct XhParams {
  int h, w, P, n_tiles;
  int stride_px, half_patch, radius2;
  float normW, normH;
  int out_stride, out_mode;
  float P1[16], P2[16];
};

// Window, refiner and softmax sums of one map (one warp).  INTERIOR: the 15 x 15 window lies inside the token grid (no
// zero padding anywhere: the per-position bounds tests drop out -- the common case away from the frame border).
template <bool INTERIOR>
__device__ __forceinline__ void xw_refine(const XhParams& hp, const float2* __restrict__ wtab, float b2w, float2* __restrict__ mm2,
                                          float2* __restrict__ hh2, const float (&wv)[8], int arow, int acol, int lane,
                                          float& zmax, float (&tot)[5]) {
  const int h = hp.h, w = hp.w;
  const int cp = lane & 7, pg = lane >> 3;
  // ---- input window (15 x 15 exact values, zero outside the map; extracted by xw_window_kernel, 16-float rows), every
  // value as the pair (v, v): the packed FMAs below take it straight from one 64-bit shared-memory load ----
#pragma unroll
  for (int q = 0; q < 8; ++q) {
    const int i = lane + 32 * q;
    const int y = i >> 4, x = i & 15;
    if (y < XWM && x < XWM) mm2[y * XH_MP + x] = make_float2(wv[q], wv[q]);
  }
  __syncwarp();
  // ---- refiner on packed fp32 FMAs (FFMA2: two IEEE fp32 FMAs per issue slot; this kernel is issue-bound).  Lane =
  // (channel pair cp = channels (cp, cp + 8), row group pg).  Hidden layer: the lane's two channels on the rows pg, pg + 4,
  // ... of the 13 x 13 window, a 3 x 3 input window sliding along the row (weights in registers), stored [position][pair].
  // Output layer: the SAME lane layout -- the lane forms its two channels' contribution to the logits of box rows pg,
  // pg + 4, pg + 8 (again sliding along the row: 3 new 64-bit shared-memory words per 9 packed FMAs); the pair is folded
  // and the 8 pair lanes of a row group are summed by shuffles.
  {
    float2 w1r[9];
#pragma unroll
    for (int k = 0; k < 9; ++k) w1r[k] = wtab[k * 8 + cp];
    const float2 b1r = wtab[9 * 8 + cp];
    for (int y = pg; y < XWH; y += 4) {
      const int r = arow - 6 + y;
      const bool row_in = r >= 0 && r < h;
      const float2* m0 = mm2 + y * XH_MP;
      // the three input rows of this hidden row, two positions per 16-byte load (positions 15, 16, 17 of a row are padding)
      float2 in0[16], in1[16], in2[16];
#pragma unroll
      for (int x = 0; x < 16; x += 2) {
        const float4 q0 = *reinterpret_cast<const float4*>(m0 + x);
        const float4 q1 = *reinterpret_cast<const float4*>(m0 + XH_MP + x);
        const float4 q2 = *reinterpret_cast<const float4*>(m0 + 2 * XH_MP + x);
        in0[x] = make_float2(q0.x, q0.y); in0[x + 1] = make_float2(q0.z, q0.w);
        in1[x] = make_float2(q1.x, q1.y); in1[x + 1] = make_float2(q1.z, q1.w);
        in2[x] = make_float2(q2.x, q2.y); in2[x + 1] = make_float2(q2.z, q2.w);
      }
#pragma unroll
      for (int x = 0; x < XWH; ++x) {
        // three short chains per output (one per input row) instead of one chain of nine dependent FMAs
        float2 a0 = __ffma2_rn(w1r[0], in0[x], b1r), a1 = __fmul2_rn(w1r[3], in1[x]), a2 = __fmul2_rn(w1r[6], in2[x]);
        a0 = __ffma2_rn(w1r[1], in0[x + 1], a0); a1 = __ffma2_rn(w1r[4], in1[x + 1], a1); a2 = __ffma2_rn(w1r[7], in2[x + 1], a2);
        a0 = __ffma2_rn(w1r[2], in0[x + 2], a0); a1 = __ffma2_rn(w1r[5], in1[x + 2], a1); a2 = __ffma2_rn(w1r[8], in2[x + 2], a2);
        const float2 a = __fadd2_rn(__fadd2_rn(a0, a1), a2);
        const int c = acol - 6 + x;
        const bool in = INTERIOR || (row_in && c >= 0 && c < w);
        hh2[(y * XWH + x) * 8 + cp] = in ? make_float2(fmaxf(a.x, 0.f), fmaxf(a.y, 0.f)) : make_float2(0.f, 0.f);
      }
    }
  }
  __syncwarp();
  float* zb = reinterpret_cast<float*>(mm2);       // the input window is dead: reuse it for the 121 logits
  {
    float2 w2r[9];
#pragma unroll
    for (int k = 0; k < 9; ++k) w2r[k] = wtab[(10 + k) * 8 + cp];
#pragma unroll
    for (int yi = 0; yi < 3; ++yi) {
      const int y = pg + 4 * yi;
      const bool row_ok = y < XWB;                  // (row group 3 has no third row; its lanes still take part in the shuffles)
      const float2* h0 = hh2 + ((row_ok ? y : 0) * XWH) * 8 + cp;
      float2 i00 = h0[0], i01 = h0[8], i10 = h0[XWH * 8], i11 = h0[(XWH + 1) * 8];
      float2 i20 = h0[2 * XWH * 8], i21 = h0[(2 * XWH + 1) * 8];
      float v[12];
      v[11] = 0.f;
#pragma unroll
      for (int x = 0; x < XWB; ++x) {
        const float2 i02 = h0[(x + 2) * 8], i12 = h0[(XWH + x + 2) * 8], i22 = h0[(2 * XWH + x + 2) * 8];
        float2 a0 = __fmul2_rn(w2r[0], i00), a1 = __fmul2_rn(w2r[3], i10), a2 = __fmul2_rn(w2r[6], i20);
        a0 = __ffma2_rn(w2r[1], i01, a0); a1 = __ffma2_rn(w2r[4], i11, a1); a2 = __ffma2_rn(w2r[7], i21, a2);
        a0 = __ffma2_rn(w2r[2], i02, a0); a1 = __ffma2_rn(w2r[5], i12, a1); a2 = __ffma2_rn(w2r[8], i22, a2);
        const float2 a = __fadd2_rn(__fadd2_rn(a0, a1), a2);
        v[x] = a.x + a.y;
        i00 = i01; i01 = i02; i10 = i11; i11 = i12; i20 = i21; i21 = i22;
      }
      // sum over the 8 pair lanes as a reduce-scatter (11 shuffles per row instead of 33): every halving step sends the
      // half of the values the partner will own; afterwards lane cp holds logits 6 b2 + 3 b1 + {2 b0, 1 (b0 = 0 only)}
      const bool b2 = cp & 4, b1 = cp & 2, b0 = cp & 1;
      float u[6], w3[3];
#pragma unroll
      for (int j = 0; j < 6; ++j) {
        const float send = b2 ? v[j] : v[j + 6], keep = b2 ? v[j + 6] : v[j];
        u[j] = keep + __shfl_xor_sync(0xffffffffu, send, 4);
      }
#pragma unroll
      for (int j = 0; j < 3; ++j) {
        const float send = b1 ? u[j] : u[j + 3], keep = b1 ? u[j + 3] : u[j];
        w3[j] = keep + __shfl_xor_sync(0xffffffffu, send, 2);
      }
      const float t0 = (b0 ? w3[2] : w3[0]) + __shfl_xor_sync(0xffffffffu, b0 ? w3[0] : w3[2], 1);
      const float t1 = (b0 ? 0.f : w3[1]) + __shfl_xor_sync(0xffffffffu, b0 ? w3[1] : 0.f, 1);
      const int idx0 = (b2 ? 6 : 0) + (b1 ? 3 : 0) + (b0 ? 2 : 0);
      if (row_ok && idx0 < XWB) zb[y * XWB + idx0] = t0 + b2w;
      if (row_ok && !b0) zb[y * XWB + idx0 + 1] = t1 + b2w;
    }
  }
  __syncwarp();
  // ---- softmax sums on the box / the disc (thread = box pixel) ----
  float z[4];
  bool valid[4], indisc[4];
  float px[4], py[4];
  zmax = -INFINITY;
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    const int p = lane + 32 * q;
    valid[q] = false; indisc[q] = false; z[q] = -INFINITY; px[q] = py[q] = 0.f;
    if (p < XWB * XWB) {
      const int y = p / XWB, x = p - y * XWB;
      const int r = arow - 5 + y, c = acol - 5 + x;
      valid[q] = INTERIOR || (r >= 0 && r < h && c >= 0 && c < w);
      if (valid[q]) {
        z[q] = zb[p];
        const int dr = (r - arow) * hp.stride_px, dc = (c - acol) * hp.stride_px;
        indisc[q] = dr * dr + dc * dc <= hp.radius2;
        px[q] = (float)(hp.half_patch + c * hp.stride_px);
        py[q] = (float)(hp.half_patch + r * hp.stride_px);
      }
    }
    zmax = fmaxf(zmax, z[q]);
  }
  zmax = warp_max(zmax);
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    const float e = valid[q] ? expf(z[q] - zmax) : 0.f;
    tot[0] += e;
    if (indisc[q]) { tot[1] += e; tot[2] = fmaf(px[q], e, tot[2]); tot[3] = fmaf(py[q], e, tot[3]); }
    tot[4] += valid[q] ? 1.f : 0.f;
  }
}

// (a) window extraction: one warp per map, no shared memory, many warps per SM -- every load here is a dependent gather
// (candidates -> box accumulators / token norms), so this part wants parallelism, not registers.  Writes the 15 x 15 exact
// window as [15][16] floats and hin = (exact first arg-max token or -1 for a map the plan queued, m_out bits).
constexpr int XWIN_PITCH = 256;
__global__ void __launch_bounds__(256)
xw_window_kernel(int n_maps, int h, int w, int P, int n_tiles, const float* __restrict__ norms, const float* __restrict__ desc_norm,
                 const int* __restrict__ cell_frame, const int* __restrict__ cell_of, const XwBox* __restrict__ box,
                 const int* __restrict__ stat, const int* __restrict__ cand, const unsigned long long* __restrict__ key1,
                 const float* __restrict__ max2, const float* __restrict__ xbox, float* __restrict__ win, int2* __restrict__ hin) {
  const int lane = threadIdx.x & 31;
  const int gw = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, nw = (gridDim.x * blockDim.x) >> 5;
  for (int map = gw; map < n_maps; map += nw) {
    if (stat[map] != 0) {
      if (lane == 0) hin[map] = make_int2(-1, 0);
      continue;
    }
    const int cell = cell_of[map];
    const XwBox bx = box[cell];
    const float* fn = norms + (size_t)cell_frame[cell] * P;
    const float* xr = xbox + (size_t)map * XW_COLS;
    const float dn = desc_norm[map];
    // exact first arg-max among the candidates (every lane, redundantly: <= 4 loads)
    const int4 cd = __ldg(reinterpret_cast<const int4*>(cand) + map);
    const int ct[4] = {cd.x, cd.y, cd.z, cd.w};
    float best = -1.f;
    int amax = -1;
#pragma unroll
    for (int q = 0; q < XW_MAX_CAND; ++q)
      if (ct[q] >= 0) {
        const int tr = ct[q] / w, tcn = ct[q] - tr * w;
        const float v = fmaxf(__fdiv_rn(__ldg(xr + xw_col(tr - bx.row, tcn - bx.col, bx.width)), fmaxf(__fmul_rn(dn, __ldg(fn + ct[q])), 1e-8f)), 0.f);
        if (v > best || (v == best && ct[q] < amax)) { best = v; amax = ct[q]; }
      }
    const int arow = amax / w, acol = amax - arow * w;
    // coarse bound on everything outside the window, from the tile keys
    float mout = 0.f;
    for (int t = lane; t < n_tiles; t += 32) {
      const unsigned long long k = __ldg(key1 + (size_t)map * n_tiles + t);
      const int tk = 0x7fffffff - (int)(k & 0xffffffffu);
      const int tr = tk / w, tcn = tk - tr * w;
      const bool in_core = abs(tr - arow) <= 3 && abs(tcn - acol) <= 3;
      const float b = in_core ? __ldg(max2 + (size_t)map * n_tiles + t) : __uint_as_float((unsigned)(k >> 32));
      mout = fmaxf(mout, b + XW_EPS);
    }
    // exact window + exact part of m_out
#pragma unroll
    for (int q = 0; q < 8; ++q) {
      const int i = lane + 32 * q;
      const int y = i >> 4, x = i & 15;
      const int r = arow - 7 + y, c = acol - 7 + x;
      float v = 0.f;
      if (y < XWM && x < XWM && r >= 0 && r < h && c >= 0 && c < w) {
        v = fmaxf(__fdiv_rn(__ldg(xr + xw_col(r - bx.row, c - bx.col, bx.width)), fmaxf(__fmul_rn(dn, __ldg(fn + r * w + c)), 1e-8f)), 0.f);
        if (!(abs(r - arow) <= 3 && abs(c - acol) <= 3)) mout = fmaxf(mout, v);
      }
      win[(size_t)map * XWIN_PITCH + i] = v;
    }
    mout = warp_max(mout);
    if (lane == 0) hin[map] = make_int2(amax, __float_as_int(mout));
  }
}

// (b) refiner + softmax sums + certificate: one warp per map; the next map's window (8 coalesced loads per lane) and
// arg-max are in flight while the current map is refined.
__global__ void __launch_bounds__(XH_WARPS * 32, 2)
xw_head_kernel(int n_maps, XhParams hp, dinotrk_head_weights wts, const int* __restrict__ cell_group, const int* __restrict__ grp_map0,
               const int* __restrict__ cell_of, const float* __restrict__ win, const int2* __restrict__ hin,
               const int* __restrict__ out_index, float* __restrict__ out, int* __restrict__ slow_cnt, int* __restrict__ slow_list,
               int n_groups) {
  extern __shared__ __align__(16) float xh_smem[];     // [weights table: 320] then per warp [input window pairs: 544 | hidden window: 2704]
  // (the warp index through a shuffle: the compiler then knows that everything derived from it -- the map index, the
  // loop trip count, the branches on the map's state -- is warp-uniform and keeps the shuffles below plain SHFLs instead
  // of wrapping each in a WARPSYNC.COLLECTIVE sequence)
  const int lane = threadIdx.x & 31, wid = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0);
  float2* wtab = reinterpret_cast<float2*>(xh_smem);
  float2* mm = reinterpret_cast<float2*>(xh_smem + XH_WTAB + wid * XH_PER_WARP);
  float2* hh_ = reinterpret_cast<float2*>(xh_smem + XH_WTAB + wid * XH_PER_WARP + XH_MWIN);
  // refiner weights as channel pairs (c, c + 8) in shared memory: a lane-indexed read of the constant bank serialises over
  // its 8 distinct addresses in the address-divergence unit (55 % busy in the capture before this table existed)
  if (threadIdx.x < 19 * 8) {
    const int k = threadIdx.x >> 3, c = threadIdx.x & 7;
    wtab[threadIdx.x] = k < 9    ? make_float2(wts.w1[c][k], wts.w1[c + 8][k])
                        : k == 9 ? make_float2(wts.b1[c], wts.b1[c + 8])
                                 : make_float2(wts.w2[c][k - 10], wts.w2[c + 8][k - 10]);
  }
  __syncthreads();
  const int h = hp.h, w = hp.w, P = hp.P;
  const int stride = gridDim.x * XH_WARPS;

  int map = blockIdx.x * XH_WARPS + wid;
  float wnext[8];
  int2 hnext = make_int2(-1, 0);
  if (map < n_maps) {
    hnext = __ldg(hin + map);
#pragma unroll
    for (int q = 0; q < 8; ++q) wnext[q] = __ldg(win + (size_t)map * XWIN_PITCH + lane + 32 * q);
  }
  for (; map < n_maps; map += stride) {
    float wv[8];
#pragma unroll
    for (int q = 0; q < 8; ++q) wv[q] = wnext[q];
    const int2 hcur = hnext;
    if (map + stride < n_maps) {
      hnext = __ldg(hin + map + stride);
#pragma unroll
      for (int q = 0; q < 8; ++q) wnext[q] = __ldg(win + (size_t)(map + stride) * XWIN_PITCH + lane + 32 * q);
    }
    const bool slow = hcur.x < 0;
    const int amax = hcur.x;
    const float mout = __int_as_float(hcur.y);
    float zmax = 0.f;
    float tot[5] = {0.f, 0.f, 0.f, 0.f, 0.f};
    if (!slow) {
      const int arow = amax / w, acol = amax - arow * w;
      if (arow >= 7 && arow + 7 < h && acol >= 7 && acol + 7 < w)
        xw_refine<true>(hp, wtab, wts.b2, mm, hh_, wv, arow, acol, lane, zmax, tot);
      else
        xw_refine<false>(hp, wtab, wts.b2, mm, hh_, wv, arow, acol, lane, zmax, tot);
#pragma unroll
      for (int q = 0; q < 5; ++q) tot[q] = warp_sum(tot[q]);
    }
    if (lane == 0) {
      bool certified = false;
      if (!slow) {
        // every logit outside the box:  z <= b2 + sum_o P2_o * relu(b1_o + P1_o * mout)   (head.cu, same certificate)
        float F = wts.b2;
#pragma unroll
        for (int o = 0; o < 16; ++o) F = fmaf(hp.P2[o], fmaxf(fmaf(hp.P1[o], mout, wts.b1[o]), 0.f), F);
        const float rest = ((float)P - tot[4]) * expf(fminf(F - zmax, 80.f));
        certified = tot[1] >= 2e-8f * (tot[0] + rest) && tot[1] > 0.f && isfinite(rest);
      }
      if (certified) {
        const float px_ = __fdiv_rn(tot[2], tot[1]), py_ = __fdiv_rn(tot[3], tot[1]);
        float nx = __fadd_rn(__fmul_rn(2.f, __fdiv_rn(px_, hp.normW)), -1.f);
        float ny = __fadd_rn(__fmul_rn(2.f, __fdiv_rn(py_, hp.normH)), -1.f);
        if (hp.out_mode == 0) {
          nx = __fmul_rn(__fdiv_rn(__fadd_rn(nx, 1.f), 2.f), hp.normW);
          ny = __fmul_rn(__fdiv_rn(__fadd_rn(ny, 1.f), 2.f), hp.normH);
        }
        const size_t oi = (size_t)(out_index ? out_index[map] : map) * hp.out_stride;
        out[oi] = nx; out[oi + 1] = ny;
      } else {
        const int g = cell_group[cell_of[map]];
        const int pos = atomicAdd(slow_cnt + g, 1);
        slow_list[grp_map0[g] + pos] = map;
        atomicAdd(slow_cnt + n_groups, 1);
        if (!slow) atomicAdd(slow_cnt + n_groups + 1, 1);   // (statistics: queued by the certificate, not by the plan)
      }
    }
    __syncwarp();
  }
}

int launch_xw_head(const FeatView& fv, const dinotrk_geom& g, const dinotrk_head_weights& hw, const XwCells& cells,
                   const float* desc_norm, const int* grp_map0, int n_maps, const int* out_index, float* out, int out_stride,
                   int out_mode, const XwChunk& xc, cudaStream_t st, int n_groups) {
  if (n_maps <= 0) return DINOTRK_OK;
  DTK_CHECK_ARG(g.radius <= 5 * g.stride, "exact-window path: disc radius %d exceeds 5 tokens", g.radius);
  XhParams hp;
  hp.h = g.h; hp.w = g.w; hp.P = g.h * g.w; hp.n_tiles = cdiv(hp.P, XW_TILE);
  hp.stride_px = g.stride; hp.half_patch = g.patch / 2; hp.radius2 = g.radius * g.radius;
  hp.normW = (float)(g.W - 1); hp.normH = (float)(g.H - 1);
  hp.out_stride = out_stride; hp.out_mode = out_mode;
  for (int o = 0; o < 16; ++o) {
    float p1 = 0.f, p2 = 0.f;
    for (int k = 0; k < 9; ++k) { p1 += hw.w1[o][k] > 0.f ? hw.w1[o][k] : 0.f; p2 += hw.w2[o][k] > 0.f ? hw.w2[o][k] : 0.f; }
    hp.P1[o] = p1 * (1.f + 1e-6f); hp.P2[o] = p2 * (1.f + 1e-6f);
  }
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  int grid = cdiv(n_maps, XH_WARPS);
  if (grid > sms * 2) grid = sms * 2;
  static PerDev<bool> attr_dev;
  bool& attr = attr_dev.get();
  if (!attr) {
    DTK_CUDA(cudaFuncSetAttribute(xw_head_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, XH_SMEM));
    attr = true;
  }
  ProfRange pr(PROF_XW_HEAD, st);
  {
    int wgrid = cdiv(n_maps, 8);
    if (wgrid > sms * 8) wgrid = sms * 8;
    xw_window_kernel<<<wgrid, 256, 0, st>>>(n_maps, g.h, g.w, hp.P, hp.n_tiles, fv.norms, desc_norm, cells.frame, xc.cell_of, xc.box,
                                            xc.stat, xc.cand, xc.key1, xc.max2, xc.xbox, xc.win, xc.hin);
    DTK_LAUNCHED();
  }
  xw_head_kernel<<<grid, XH_WARPS * 32, XH_SMEM, st>>>(n_maps, hp, hw, cells.group, grp_map0, xc.cell_of, xc.win, xc.hin, out_index,
                                                 out, xc.slow_cnt, xc.slow_list, n_groups);
  DTK_LAUNCHED();
  return DINOTRK_OK;
}

// ====================================================================================================== 5. full-map queue
// One block per queued map: copies its descriptor (fp32 + fp16 hi / lo), norm and output slot to compact row b; block 0
// also writes the compact group arrays.  Rows of a group keep their queue order (arbitrary, results do not depend on it).
__global__ void __launch_bounds__(128)
xw_compact_kernel(const float4* __restrict__ desc, const uint4* __restrict__ dhi, const uint4* __restrict__ dlo,
                  const float* __restrict__ desc_norm, const int* __restrict__ out_index, int C, const int* __restrict__ grp_frame,
                  const int* __restrict__ grp_map0, int n_groups, const int* __restrict__ slow_cnt,
                  const int* __restrict__ slow_list, float4* __restrict__ c_desc, uint4* __restrict__ c_hi, uint4* __restrict__ c_lo,
                  float* __restrict__ c_norm, int* __restrict__ c_out_index, int* __restrict__ cgrp, int gcap, int row_base,
                  int grp_base) {
  __shared__ int s_g, s_pos;
  const int bb = blockIdx.x;
  if (threadIdx.x == 0) {
    int pre = 0, gsel = -1, psel = 0;
    for (int g = 0; g < n_groups; ++g) {
      const int c = slow_cnt[g];
      if (bb == 0) {
        cgrp[grp_base + g] = grp_frame[g]; cgrp[gcap + grp_base + g] = row_base + pre; cgrp[2 * gcap + grp_base + g] = c;
        cgrp[3 * gcap + grp_base + g] = row_base + pre;
      }
      if (gsel < 0 && bb < pre + c) { gsel = g; psel = bb - pre; }
      pre += c;
    }
    s_g = gsel; s_pos = psel;
  }
  __syncthreads();
  if (s_g < 0) return;
  const int b = row_base + bb;
  const int src = slow_list[grp_map0[s_g] + s_pos];
  if (desc != nullptr)   // (the fp32 copy only feeds the non-tensor GEMMs)
    for (int i = threadIdx.x; i < C / 4; i += blockDim.x) c_desc[(size_t)b * (C / 4) + i] = desc[(size_t)src * (C / 4) + i];
  if (dhi != nullptr)
    for (int i = threadIdx.x; i < C / 8; i += blockDim.x) {
      c_hi[(size_t)b * (C / 8) + i] = dhi[(size_t)src * (C / 8) + i];
      c_lo[(size_t)b * (C / 8) + i] = dlo[(size_t)src * (C / 8) + i];
    }
  if (threadIdx.x == 0) { c_norm[b] = desc_norm[src]; c_out_index[b] = out_index[src]; }
}

int launch_xw_compact(const float* desc, const void* desc_hi, const void* desc_lo, const float* desc_norm,
                      const int* out_index, int C, const int* grp_frame, const int* grp_map0, int n_groups, int n_slow,
                      const XwChunk& xc, float* c_desc, void* c_hi, void* c_lo, float* c_norm, int* c_out_index, int* cgrp,
                      int gcap, cudaStream_t st, int row_base, int grp_base) {
  if (n_slow <= 0) return DINOTRK_OK;
  ProfRange pr(PROF_MISC, st);
  xw_compact_kernel<<<n_slow, 128, 0, st>>>(reinterpret_cast<const float4*>(desc), reinterpret_cast<const uint4*>(desc_hi),
                                            reinterpret_cast<const uint4*>(desc_lo), desc_norm, out_index, C, grp_frame, grp_map0,
                                            n_groups, xc.slow_cnt, xc.slow_list, reinterpret_cast<float4*>(c_desc),
                                            reinterpret_cast<uint4*>(c_hi), reinterpret_cast<uint4*>(c_lo), c_norm, c_out_index, cgrp,
                                            gcap, row_base, grp_base);
  DTK_LAUNCHED();
  return DINOTRK_OK;
}

size_t xw_chunk_bytes(int chunk_maps, int max_cells, int n_tiles, int gcap) {
  const size_t ch = (size_t)chunk_maps;
  size_t b = 0;
  b += align_up(ch * n_tiles * 8, 256) + align_up(ch * n_tiles * 4, 256);              // key1, max2
  b += align_up(ch * XW_MAX_CAND * 4, 256) + 4 * align_up(ch * 4, 256);                // cand, stat, pinfo, cell_of, slow_list
  b += align_up((size_t)max_cells * sizeof(XwBox), 256);                               // box
  b += align_up(ch * XW_COLS * 4, 256);                                                // xbox
  b += align_up(ch * 256 * 4, 256) + align_up(ch * 8, 256);                            // win, hin
  b += align_up((size_t)(gcap + XW_NCNT) * 4, 256);                                    // slow_cnt
  return b + 2048;
}

}  // namespace dtk
