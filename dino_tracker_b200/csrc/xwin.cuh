// Coarse pass + exact window: the anchor phase's correlation + head without ever writing a correlation map.
// Internal interface of xwin.cu (not part of the C ABI).
//
//   models/tracker.py:158-180 + models/networks/tracker_head.py:68-121 produce, per (descriptor, frame) map, ONE point:
//   the disc-masked soft-argmax around the map's arg-max.  That point depends on (i) which token is the arg-max,
//   (ii) the map values on the 15 x 15 window around it (11 x 11 logits <- 13 x 13 hidden <- 15 x 15 inputs) and (iii) an
//   upper bound on everything else (certificate that the stability branch, tracker_head.py:87-94, stays off).
//
//   1. coarse GEMM   one kind::f16 pass over the fp16 `hi` halves (1/3 of the split-precision work), epilogue keeps per
//                    map and 256-token tile only (largest value, its first token, second largest value); |coarse - exact|
//                    <= XW_EPS for every token (fp16 rounding of both operands + TMEM accumulation, see DESIGN.md).
//   2. plan          per map: the tokens that can be the exact arg-max (coarse >= max - 2 XW_EPS); a map whose candidates
//                    are not all tile maxima is "ambiguous".  Maps come in CELLS = the <= 128 source frames of one (query,
//                    anchor frame) pair: their arg-maxes cluster around the query's position in the anchor frame.  A map
//                    fits if its candidates lie within +-XW_SLACK of the cell's median arg-max; the cell's box is the
//                    bounding rectangle of the fitting maps' candidates widened by 7 tokens on every side (so it holds every
//                    fitting map's 15 x 15 window): 15..21 rows by 16 columns (column extent <= 1) or 21 columns.
//   3. exact GEMM    per cell, the fp32-faithful split-precision contraction (lo*hi + hi*lo + hi*hi, same operation
//                    sequence as the full-map GEMM) of the cell's descriptors against the box's tokens only (at most 441,
//                    5.4 % of the map; 240..256 for a cell whose members agree to one token).  Raw accumulators go to a
//                    [map][448] buffer, row-major with the cell's box width as pitch (1.8 KB per map instead of 32 KB).
//   4. head          two kernels, one warp per map each: (a) exact arg-max among the candidates + the exact 15 x 15 window
//                    + m_out (dependent gathers: many warps per SM), (b) refiner, softmax sums on the 11 x 11 box, certificate
//                    with the bound from (1); writes the track point.
//   Maps that are ambiguous, do not fit their cell's box or fail the certificate are queued and re-done by the full-map
//   path (split-precision GEMM over all tokens + head kernels of head.cu) -- results never depend on the coarse values.
#pragma once
#include "common.cuh"
#include "corr.cuh"

namespace dtk {

constexpr float XW_EPS = 1.1e-3f;     // bound on |coarse - exact| in cosine units (2^-10 + accumulation, rounded up)
constexpr int XW_BOX = 21;            // largest box side (tokens): windows of maps whose candidates lie within +-3 of the centre
constexpr int XW_SLACK = 3;
constexpr int XW_NARROW = 16;         // box width when the fitting candidates span <= 2 columns
// One UMMA M-part = 128 rows: 8 box rows of a 16-wide box (128 tokens) or 6 rows of a 21-wide one (126 tokens)
constexpr int XW_ROWS_NARROW = 8, XW_ROWS_WIDE = 6;
constexpr int XW_PARTS = 4;           // most parts of a box (21 x 21: ceil(21 / 6)); a cell's TMEM slot holds XW_PARTS x NB columns
constexpr int XW_COLS = 448;                                     // accumulator row pitch per map (<= 441 box tokens, row-major)
constexpr int XW_MAX_CELL = 128;      // maps (source frames) per cell = UMMA N (64 or 128)
constexpr int XW_MAX_CAND = 4;
constexpr float XW_MIN_NORM = 1e-4f;  // the coarse pass forms acc / (|d| |F|) without the reference's max(|d| |F|, 1e-8) clamp: both
                                      // norms must be >= 1e-4 (smaller descriptor norms -> ambiguous map, smaller token norms
                                      // anywhere in the video -> the whole call takes the full-map pipeline)
constexpr int XW_TILE = 128;          // tokens per coarse key (the coarse GEMM's 8 epilogue warps cover 128 columns each)
constexpr int XW_NCNT = 2 + (XW_PARTS - 1);   // chunk counters after the per-group queue lengths (see XwChunk::slow_cnt)

// column of box token (by, bx) in a map's accumulator row (box of `width` columns)
__host__ __device__ inline int xw_col(int by, int bx, int width) { return by * width + bx; }

struct __align__(16) XwBox {   // a cell's token box: first row and column, width (16 or 21), height (15..21), M-parts
  int row, col;                 // (2..4; 0: no map of the cell fits, the cell is skipped)
  short width, height, parts;
};

struct XwChunk {          // device buffers of one chunk in flight (all sized for chunk_maps maps)
  unsigned long long* key1;   // [maps][n_tiles]  coarse maximum of a XW_TILE-token tile << 32 | (0x7fffffff - first token)
  float* max2;                // [maps][n_tiles]  second largest coarse value of the tile
  int* cand;                  // [maps][XW_MAX_CAND] candidate tokens (-1 = none)
  int* pinfo;                 // [maps] coarse arg-max token, or -1 - token for an ambiguous map (plan scratch)
  int* stat;                  // [maps] 0: exact-window path, 1: full-map path
  int* cell_of;               // [maps] cell index
  XwBox* box;                 // [cells] token box; parts = 0: no map of the cell fits, every map takes the full-map path
  float* xbox;                // [maps][XW_COLS] raw split-precision accumulators of the box tokens
  float* win;                 // [maps][256] exact 15 x 15 windows ([15][16] floats, zero outside the map)
  int2* hin;                  // [maps] (exact first arg-max token or -1, bits of m_out)
  int* slow_cnt;              // [n_groups + XW_NCNT] per group count of queued maps; [n_groups] = total, [n_groups + 1] =
                              // queued by the certificate, [n_groups + 2 + i] = cells whose box has 2 + i parts
  int* slow_list;             // [maps] group g's queue lives at [grp_map0[g], grp_map0[g] + slow_cnt[g])
};

struct XwCells {          // host-planned, device-resident description of a chunk's cells
  const int* row0;     // [cells] first descriptor row (= first map) of the cell
  const int* m;        // [cells] rows
  const int* frame;    // [cells] anchor frame
  const int* group;    // [cells] group index (for the slow queues)
  int n_cells, max_m;
};

size_t xw_chunk_bytes(int chunk_maps, int max_cells, int n_tiles, int gcap);
// Coarse GEMM over the chunk's groups (tile_start: prefix of ceil(m / 256) per group, all groups wide).
int launch_xw_coarse(const FeatView& fv, const void* desc_hi, int desc_rows, const float* desc_norm, const int* grp_frame,
                     const int* grp_row0, const int* grp_m, const int* grp_map0, const int* tile_start, int n_groups,
                     int max_tiles, const XwChunk& xc, cudaStream_t st, const float* rnorms);
// rnorms = 1 / |F| for the coarse epilogue; *min_bits = bit pattern of the smallest token norm of the video
int launch_xw_rnorms(const FeatView& fv, float* rnorms, unsigned* min_bits, cudaStream_t st);
int launch_xw_plan(const XwCells& cells, const float* desc_norm, int n_groups, const dinotrk_geom& g, const XwChunk& xc,
                   cudaStream_t st, int n_maps);
int launch_xw_gemm(const FeatView& fv, const dinotrk_geom& g, const void* desc_hi, const void* desc_lo, int desc_rows,
                   const XwCells& cells, const XwChunk& xc, cudaStream_t st);
int launch_xw_head(const FeatView& fv, const dinotrk_geom& g, const dinotrk_head_weights& hw, const XwCells& cells,
                   const float* desc_norm, const int* grp_map0, int n_maps, const int* out_index, float* out, int out_stride,
                   int out_mode, const XwChunk& xc, cudaStream_t st, int n_groups);
// Appends the queued maps' descriptor rows (fp32 optional, hi, lo, norm, out_index) to compact arrays at row_base and their
// group arrays ([frame | row0 | m | map0] x gcap, entries grp_base ..) to cgrp.  n_slow = host copy of slow_cnt[n_groups].
int launch_xw_compact(const float* desc, const void* desc_hi, const void* desc_lo, const float* desc_norm,
                      const int* out_index, int C, const int* grp_frame, const int* grp_map0, int n_groups, int n_slow,
                      const XwChunk& xc, float* c_desc, void* c_hi, void* c_lo, float* c_norm, int* c_out_index, int* cgrp,
                      int gcap, cudaStream_t st, int row_base = 0, int grp_base = 0);

}  // namespace dtk
