/*
 * dinotrk.h -- C ABI of libdinotrk.so, the B200 (sm_100a) implementation of the
 * DINO-Tracker inference hot path.
 *
 * The reference (AssafSinger94/dino-tracker) has no FFI layer: its boundary is the Python
 * class surface of models/tracker.py + models/model_inference.py (SURVEY.md 8b).  The host
 * mirror of that surface lives in dino_tracker_b200/ and reaches the kernels only through
 * the entry points declared here (ctypes; see INTEGRATION.md).  Every entry point
 *   - is extern "C", takes raw device pointers, sizes and a cudaStream_t (as void*);
 *   - never allocates device memory: big scratch is a caller-provided workspace whose size
 *     comes from the matching *_workspace_bytes query;
 *   - only enqueues work on `stream` unless stated otherwise ("syncs" below);
 *   - returns 0 on success or a negative code; dinotrk_last_error() gives the message
 *     (thread-local).
 *
 * Layouts.  "tpc" = token-major feature video  [T][P][C] fp32, P = h*w tokens row-major
 * (r*w + c), C contiguous: the ViT's natural output order, K-major for every contraction
 * and coalesced for bilinear descriptor sampling.  "chw" = the reference's T x C x h x w
 * (models/tracker.py:64-71).  Pixel coordinates are in the model frame (x in [0,W-1]).
 */
#ifndef DINOTRK_H_
#define DINOTRK_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DINOTRK_VERSION 100

#define DINOTRK_OK 0
#define DINOTRK_EINVAL (-22)
#define DINOTRK_ECUDA (-5)
#define DINOTRK_ENOMEM (-12)

/* Video / token-grid geometry.  h = 1 + (H - patch) / stride, w likewise
 * (models/extractor.py:171-177); radius = TrackerHead.argmax_radius (tracker_head.py:47). */
typedef struct dinotrk_geom {
  int H, W, patch, stride, radius;
  int h, w;
} dinotrk_geom;

/* Refiner weights AFTER the spatial-sum normalisation of models/networks/conv_norm.py:34-46
 * (done once per weight load on the host): w1[16][9], b1[16], w2[16][9] (out=1, in=16), b2. */
typedef struct dinotrk_head_weights {
  float w1[16][9];
  float b1[16];
  float w2[16][9];
  float b2;
} dinotrk_head_weights;

/* A cached feature video.  tpc [T][P][C] and norms [T][P] are required.  hi / lo (optional, both or
 * neither): the fp16 split of tpc ([T][P][C] halves each, x = hi + lo) produced by dinotrk_split_fp16; when
 * present the wide correlation groups run on the tcgen05 tensor cores (3-pass split precision,
 * fp32-faithful), otherwise on the exact-fp32 FFMA GEMM.  C must then be a multiple of 8. */
typedef struct dinotrk_features {
  const float* tpc;
  const float* norms;
  const void* hi;
  const void* lo;
  int T, C;
} dinotrk_features;

int dinotrk_version(void);
const char* dinotrk_last_error(void);
/* Fills *g from (H, W, patch, stride, radius); returns DINOTRK_EINVAL on bad sizes. */
int dinotrk_make_geom(int H, int W, int patch, int stride, int radius, dinotrk_geom* g);

/* ---- feature cache (models/tracker.py:64-71,131-135) --------------------------------- */
/* chw [T][C][P] -> tpc [T][P][C] and per-token L2 norms [T][P]
 * (frame_embeddings_set.norm(dim=1), models/tracker.py:162). */
int dinotrk_pack_features(const float* chw, float* tpc, float* norms, int T, int C, int P,
                          void* stream);
int dinotrk_unpack_features(const float* tpc, float* chw, int T, int C, int P, void* stream);
int dinotrk_token_norms(const float* tpc, float* norms, int T, int C, int P, void* stream);
/* x = hi + lo with hi = rn_fp16(x), lo = rn_fp16(x - hi) (fp16 arrays of n elements); n % 4 == 0. */
int dinotrk_split_fp16(const float* x, void* hi, void* lo, size_t n, void* stream);

/* ---- descriptor sampling (models/tracker.py:77-111, utils.py:75-101) ------------------- */
/* points [B][3] = (x_px, y_px, set_index) ; frames_set [N] int32 = frame of each set slot.
 * Reproduces normalize_points_for_sampling + the 5-D grid_sample (border, align_corners),
 * including the fp32 temporal-weight leak.  points_normalized != 0: x,y already in [-1,1]
 * (Tracker.sample_embeddings semantics).  out desc [B][C], desc_norm [B] (may be NULL). */
int dinotrk_sample_descriptors(const float* tpc, int T, int C, const dinotrk_geom* g,
                               const float* points, int B, const int* frames_set, int N,
                               int points_normalized, float* desc, float* desc_norm,
                               void* stream);

/* ---- correlation + head (models/tracker.py:158-180, tracker_head.py:107-121) ----------- */
/* Generic grouped form.  Group k (k < n_groups) correlates descriptor rows
 * [row0[k], row0[k] + m[k]) of `desc` with every token of frame frame[k]; its maps are
 * numbered map0[k] + r.  For map j the (x, y) result is written to out[out_index[j] * out_stride
 * + {0,1}] (out_index == NULL: j).  out_mode 0: pixels (after RangeNormalizer.unnormalize,
 * models/model_inference.py:52), 1: normalised [-1,1] (Tracker.forward).
 * group arrays are device int32[n_groups]; total_maps = sum m.  Syncs: no. */
size_t dinotrk_corr_track_workspace_bytes(int total_maps, int n_groups, int C, const dinotrk_geom* g);
int dinotrk_corr_track(const dinotrk_features* feat, const dinotrk_geom* g,
                       const dinotrk_head_weights* hw, const float* desc, const float* desc_norm,
                       const int* grp_frame, const int* grp_row0, const int* grp_m,
                       const int* grp_map0, int n_groups, int total_maps, int max_group_m,
                       const int* out_index, float* out, int out_stride, int out_mode,
                       void* workspace, size_t workspace_bytes, void* stream);

/* Correlation maps only (ReLU'd cosine maps, [total_maps][map_stride] fp32,
 * map_stride = dinotrk_map_stride(g)) -- the volume the fused path never keeps. */
int dinotrk_map_stride(const dinotrk_geom* g);
size_t dinotrk_corr_maps_workspace_bytes(int total_maps, int n_groups, int C);
int dinotrk_corr_maps(const dinotrk_features* feat, const dinotrk_geom* g,
                      const float* desc, const float* desc_norm, const int* grp_frame,
                      const int* grp_row0, const int* grp_m, const int* grp_map0, int n_groups,
                      int total_maps, int max_group_m, float* maps, void* workspace,
                      size_t workspace_bytes, void* stream);
/* Head only: maps -> (x, y) (tracker_head.py:107-121).  aux (may be NULL) receives per map
 * {argmax index, fallback flag} as int32[2].  scratch: device int32[n_maps + 1] enabling the windowed
 * fast path (exact refiner on the 11x11 box around the arg-max + certified absence of the stability
 * branch; uncertified maps go to the full-map kernel); NULL: full-map kernel for every map. */
int dinotrk_head(const float* maps, int n_maps, const dinotrk_geom* g,
                 const dinotrk_head_weights* hw, const int* out_index, float* out,
                 int out_stride, int out_mode, int* aux, int* scratch, void* stream);

/* ---- training: reverse pass of the tracker forward (dino_tracker.py:405-429, models/tracker.py:170-180,303-325) -- */
/* The forward of a training step is dinotrk_sample_descriptors + dinotrk_corr_maps + dinotrk_head (with aux) on the
 * frame set's embeddings, with desc / desc_norm / maps / aux kept.  Given grad_out [B][2] = d loss / d coords (the
 * normalised output of Tracker.forward), row j of points / desc / maps / aux / tgt_frame / grad_out describing map j:
 *   grad_w   float[305] += d loss / d (w1[16][9] | b1[16] | w2[16][9] | b2), w1 / w2 the NORMALISED refiner weights of
 *            dinotrk_head_weights (the spatial-sum normalisation of conv_norm.py:34-46 stays with the caller's autograd);
 *   grad_tpc [T][P][C] += d loss / d feat->tpc, through the target maps (tracker.py:158-169) and through the sampled
 *            source descriptors (tracker.py:96-111); NULL: embeddings without gradient (cached refined features).
 * points [B][3] = (x_px, y_px, set slot) and frames_set [N] as given to dinotrk_sample_descriptors; tgt_frame [B] =
 * the FRAME (index into feat) each map correlates against.  arg-max and disc mask carry no gradient (as in autograd).
 * Accumulates with atomics: the caller zeroes grad_w / grad_tpc.  Syncs: no. */
size_t dinotrk_track_backward_workspace_bytes(int B, int C, const dinotrk_geom* g);
int dinotrk_track_backward(const dinotrk_features* feat, const dinotrk_geom* g, const dinotrk_head_weights* hw,
                           const float* points, const int* frames_set, int N, const float* desc,
                           const float* desc_norm, const int* tgt_frame, const float* maps, const int* aux,
                           const float* grad_out, int B, float* grad_w, float* grad_tpc, void* workspace,
                           size_t workspace_bytes, void* stream);

/* Reverse pass of dinotrk_sample_descriptors alone (the contrastive losses sample refined embeddings with a graph,
 * dino_tracker.py:215-220): grad_tpc [T][P][C] += the trilinear weights of every point times grad_desc [B][C]. */
int dinotrk_sample_backward(int T, int C, const dinotrk_geom* g, const float* points, int B, const int* frames_set,
                            int N, int points_normalized, const float* grad_desc, float* grad_tpc, void* stream);

/* ---- inference driver (models/model_inference.py:97-216) ------------------------------- */
/* query_points [N][3] (x, y, t) px; frame_batch = the reference's --batch-size (0 = whole
 * video).  Outputs: traj [N][T][3] (x, y, t); cos_sims [N][T]; anchors [N][T(a)][T(i)][2] valid
 * where cos_sims[n][a] >= anchor_th; occ [N][T] uint8.  Any of the last three may be NULL only
 * together with stop_after < 3 / 2 / 1.  Phases 0 = trajectories (compute_trajectories),
 * 1 = cos-sims, 2 = anchors, 3 = occlusion; phases start_phase..stop_after run (0..3 = infer), and
 * the outputs of earlier phases are then inputs.  SYNCS the stream once when phase 2 runs (reads
 * the per-frame anchor counts back to size the anchor work lists). */
size_t dinotrk_infer_workspace_bytes(int T, int C, const dinotrk_geom* g, int N, int chunk_maps);
/* Host-only helper (no GPU needed): the chunk plan dinotrk_infer uses.  kind 0 = trajectory phase (items = every
 * (frame, query row) pair), kind 1 = anchor phase (anchor_counts[a] * T items per anchor frame a).  Chunks hold
 * <= chunk_maps correlation maps; inside a chunk the items of one target frame form a group.  Outputs (either may be
 * NULL to just count): groups [n_chunks][5][T + 2] int32 = per chunk {frame, first descriptor row, rows m, first map,
 * first item} x group; meta [n_chunks][4] = {maps used, largest m, number of groups, 1 if no group is thin};
 * *n_chunks.  dinotrk_infer_max_chunks bounds n_chunks (and sizes dinotrk_infer's workspace). */
size_t dinotrk_infer_max_chunks(int T, int N, int chunk_maps);
int dinotrk_infer_plan(int kind, int T, int N, const int* anchor_counts, int chunk_maps, int* groups, int* meta,
                       int max_chunks, int* n_chunks);
/* Phase 2 pipelining across CUDA streams (process-wide; results are identical in every mode):
 * 0 = everything on the caller's stream; 1 (default) = the descriptor sampling of chunk k+1 runs on an
 * internal side stream under the correlation GEMM of chunk k; 2 = the head's fast path as well;
 * -1 = back to the default / the DTK_OVERLAP environment variable.  All side-stream work is joined back
 * into the caller's stream before dinotrk_infer returns.  The side streams and their events are one set per
 * process (one process per GPU): with mode >= 1 do not run dinotrk_infer from two host threads at once. */
int dinotrk_infer_set_overlap(int mode);
/* Pipeline of the anchor re-tracking phase (process-wide):
 *  1 = coarse pass + exact window: one single-pass fp16 GEMM keeps per map and 256-token tile only (max, its token, second
 *      value); the fp32-faithful split-precision contraction is then evaluated only on a 21 x 21 token box around the
 *      arg-max of each (query, anchor frame) cell, and a warp-per-map head consumes those values -- no correlation map is
 *      ever written.  Maps whose arg-max cannot be resolved from the coarse pass (near ties), that leave their cell's box
 *      or that fail the head's certificate are re-done by pipeline 0; no result depends on a coarse value.
 *  0 = full maps: split-precision GEMM over all tokens into chunk buffers + the head kernels (the round-1 pipeline).
 * -1 (default) = 1 when the feature struct carries fp16 hi / lo halves (tensor path), unless the trajectory phase just
 *      showed that the head's certificate fails for more than a quarter of the maps (ill-conditioned refiner weights);
 *      the DTK_XW environment variable (0 / 1) overrides.
 * dinotrk_infer_last_stats (n >= 4 slots): {anchor-phase maps, maps finished by the exact-window path, maps re-done by the
 * full-map path, pipeline used[, of the re-done maps: those queued by the head's certificate rather than by the plan[,
 * exact-window cells whose token box took 2, 3, 4 GEMM parts]]} of the last dinotrk_infer call that ran the anchor phase
 * (n >= 5 returns the certificate count, n >= 8 also the part counts). */
int dinotrk_infer_set_path(int path);
int dinotrk_infer_last_stats(long long* out, int n);
int dinotrk_infer(const dinotrk_features* feat, const dinotrk_geom* g,
                  const dinotrk_head_weights* hw, const float* query_points, int N,
                  float anchor_th, float cos_th, int frame_batch, int start_phase, int stop_after,
                  int chunk_maps,
                  float* traj, float* cos_sims, float* anchors, uint8_t* occ,
                  void* workspace, size_t workspace_bytes, void* stream);
/* Piecewise entry points behind ModelInference.compute_* (same arithmetic as dinotrk_infer). */
int dinotrk_traj_cos_sims(const float* tpc, int T, int C, const dinotrk_geom* g,
                          const float* traj, const float* query_points, int N, float* cos_sims,
                          void* workspace, size_t workspace_bytes, void* stream);
int dinotrk_occlusion(const float* traj, const float* cos_sims, const float* anchors, int N, int T,
                      float anchor_th, float cos_th, uint8_t* occ, void* stream);

/* ---- Delta-DINO refinement (models/tracker.py:113-135, delta_dino.py:8-61, models/utils.py:7-45) */
/* frames [B][3][H][W] raw RGB in [0,1]; channels[5] = {3, c1, c2, c3, C} (c* multiples of 4);
 * wgt[l] = conv l weights with BatchNorm(eval) folded in, K-major [C_out][5][5][C_in_pad]
 * (C_in_pad = 4 for l = 0, else C_in); bias[l] [C_out] likewise folded.  dino_tpc [B][h*w][C];
 * ixs[w] / iys[h] = un-normalised clipped CNN-grid sampling coordinates of the token columns / rows
 * (models/utils.py:31-43).  Writes refined_tpc [B][h*w][C] = dino + aligned residual and
 * (optional) per-token norms [B][h*w]. */
size_t dinotrk_delta_workspace_bytes(int B, int H, int W, const int* channels);
int dinotrk_delta_refine(const float* frames, int B, int H, int W, const int* channels,
                         const float* const* wgt, const float* const* bias, const float* dino_tpc,
                         const float* ixs, const float* iys, int h, int w, float* refined_tpc,
                         float* norms, void* workspace, size_t workspace_bytes, void* stream);

/* Frame-sharded multi-GPU variant (SURVEY.md 8e, config 4): as dinotrk_delta_refine, and every refined row is ALSO
 * stored into the same slot of each peer GPU's full feature video -- peer_bases[k] (HOST array of n_peers <= 8 device
 * pointers mapped with dinotrk_peer_open) + (first_frame * h*w + row) * C -- by the producing kernel itself
 * (stores over NVLink to mapped peer memory): the all-gather is fused into the delta-DINO epilogue.  The caller
 * synchronises the ranks afterwards (stream sync + barrier) before reading remote frames. */
int dinotrk_delta_refine_allgather(const float* frames, int B, int H, int W, const int* channels,
                                   const float* const* wgt, const float* const* bias, const float* dino_tpc,
                                   const float* ixs, const float* iys, int h, int w, float* refined_tpc,
                                   float* norms, void* workspace, size_t workspace_bytes,
                                   float* const* peer_bases, int n_peers, size_t first_frame, void* stream);
/* Tensor-core variant: the four convolutions run as explicit-im2col (fp16 hi/lo split on the fly) + tcgen05
 * split-precision GEMMs (fp32-faithful).  wgt_hi[l] / wgt_lo[l]: fp16 split (dinotrk_split_fp16) of the folded K-major
 * weights [C_out][Kp], Kp = 25 * C_in_pad rounded up to 8; channel counts multiples of 8.  peer_bases / n_peers /
 * first_frame as in dinotrk_delta_refine_allgather (n_peers = 0: single GPU). */
int dinotrk_delta_refine_tc(const float* frames, int B, int H, int W, const int* channels,
                            const void* const* wgt_hi, const void* const* wgt_lo, const float* const* bias,
                            const float* dino_tpc, const float* ixs, const float* iys, int h, int w,
                            float* refined_tpc, float* norms, void* workspace, size_t workspace_bytes,
                            float* const* peer_bases, int n_peers, size_t first_frame, void* stream);
/* Peer-mapped buffers for the above (one process per GPU, one node): cudaMalloc + CUDA IPC handle (64 bytes). */
int dinotrk_peer_alloc(size_t bytes, void** ptr, unsigned char* handle64);
int dinotrk_peer_open(const unsigned char* handle64, void** ptr);
int dinotrk_peer_close(void* ptr);
int dinotrk_peer_free(void* ptr);

/* ---- DINOv2 ViT feature extractor (utils.py:32-72, models/extractor.py:41-85,137-150) -------------- */
typedef struct dinotrk_vit_config {
  int depth, dim, heads;   /* ViT-L/14: 24, 1024, 16; ViT-B/14: 12, 768, 12 (head dim 64) */
  int tap_layer;           /* 0-based block whose output (before the final norm) is returned; 15 in the shipped config */
  int patch, stride;       /* 14, 7 */
  int attn_materialized;   /* 0: fused tcgen05 attention (fp16 q/k/v/p, scores stay on the SM); 1: TF32 scores through a
                              workspace (tensor-core GEMM -> softmax -> tensor-core GEMM), validation path */
  int gemm_f16;            /* 1: linear layers on the kind::f16 pipe -- patch_w and the qkv / proj / fc1 / fc2 weight matrices
                              are passed as fp16 arrays, activations are written in fp16 by the producing epilogue;
                              0 (or attn_materialized): fp32 arrays, TF32 MMAs */
  int gemm_pair;           /* with gemm_f16: 1 = linear layers on CTA pairs (tcgen05 cta_group::2, 256 x 256 tiles, each SM
                              stages half of the weight tile), 0 = single-CTA 128 x 256 tiles */
} dinotrk_vit_config;
/* Device fp32 (weight matrices fp16 when gemm_f16).  patch_w: patch-embedding conv weight flattened K-major
 * [dim][Kp], Kp = 3*patch*patch zero-padded to a multiple of 4 (fp32) / 8 (fp16) elements; cls_pos [dim] =
 * cls_token + pos_embed[0]; pos [h*w][dim] = bicubic-interpolated patch position embedding (extractor.py:57-85);
 * blocks: HOST array of depth x 14 device pointers in the order norm1.w, norm1.b, qkv.w [3D][D], qkv.b, proj.w,
 * proj.b, ls1.gamma, norm2.w, norm2.b, fc1.w [4D][D], fc1.b, fc2.w [D][4D], fc2.b, ls2.gamma. */
typedef struct dinotrk_vit_weights {
  const void* patch_w; const float* patch_b; const float* cls_pos; const float* pos;
  const float* const* blocks;
} dinotrk_vit_weights;
size_t dinotrk_vit_workspace_bytes(const dinotrk_vit_config* c, const dinotrk_geom* g, int B);
/* frames [B][3][H][W] RGB in [0,1] -> out_tpc [B][h*w][dim] (token-major features of block tap_layer). */
int dinotrk_vit_forward(const float* frames, int B, const dinotrk_geom* g, const dinotrk_vit_config* c,
                        const dinotrk_vit_weights* wt, float* out_tpc, void* workspace,
                        size_t workspace_bytes, void* stream);
/* The attention of one ViT block on its own (the fused tcgen05 kernel of dinotrk_vit_forward; head dim 64):
 * q16 [B*heads][N1][64] fp16 ALREADY multiplied by 64^-1/2 * log2(e), k16 [B*heads][N1][64] fp16,
 * vT16 [B*heads][64][N1p] fp16 (v transposed, row pitch N1p >= N1, a multiple of 8);
 * out [B*N1][heads*64] fp32 = softmax(q k^T) v with head h in columns [64 h, 64 h + 64)
 * (the layout of the reference's attn output before `proj`, dinov2 attention.py). */
int dinotrk_vit_attention(const void* q16, const void* k16, const void* vT16, int B, int heads, int N1, int N1p,
                          float* out, void* stream);

/* ---- best buddies (preprocessing_dino_bb/extract_dino_best_buddies.py:12-54) ------------------------ */
/* For every ordered pair k (source frame pair_src[k], target frame pair_tgt[k]; device int32[n_pairs]):
 * nn_idx[k][n] = argmax_m cos(F_src[n], F_tgt[m]) (first maximum), nn_cos[k][n] = that cosine (exact fp32,
 * clamp 1e-8 on the norm product).  The affinity matrix runs through the tcgen05 split-fp16 GEMM and never
 * leaves TMEM; candidates are re-evaluated in exact fp32.  feat->hi / lo are required. */
size_t dinotrk_best_buddies_workspace_bytes(int n_pairs, int P);
int dinotrk_best_buddies_pairs(const dinotrk_features* feat, const dinotrk_geom* g, const int* pair_src,
                               const int* pair_tgt, int n_pairs, int* nn_idx, float* nn_cos,
                               void* workspace, size_t workspace_bytes, void* stream);
/* mutual[k][n] = (nn_ts[k][nn_st[k][n]] == n): source token n of pair k is a best buddy. */
int dinotrk_bb_mutual(const int* nn_st, const int* nn_ts, int n_pairs, int P, uint8_t* mutual, void* stream);
/* Peak filter of the best-buddy pairs (preprocessing_dino_bb/compute_dino_bb_nms.py:12-66, get_bb_sim_indices): maps =
 * [n_maps][dinotrk_map_stride] similarity maps of the source points against the target frame (dinotrk_corr_maps). Per map:
 * peak_affs[2] = the two largest values that survive box NMS (boxes of +-box_size px around the token centres, greedy,
 * IoU threshold, restricted to the `topk` largest values), r = second / first. */
int dinotrk_bb_nms(const float* maps, int n_maps, const dinotrk_geom* g, float box_size, float iou_thresh, int topk,
                   float* peak_affs, float* r, void* stream);

/* ---- per-kernel-class device timing (CUDA events on the launching stream; bench.py roofline) ------ */
int dinotrk_profile_classes(void);
const char* dinotrk_profile_class_name(int cls);
void dinotrk_profile_enable(int on);
/* Waits for the recorded events; ms[cls] / launches[cls] accumulate since the previous collect. */
int dinotrk_profile_collect(double* ms, unsigned long long* launches, int n);

/* number of kernel launches issued by this library since load (bench.py's gpu_launches) */
unsigned long long dinotrk_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif /* DINOTRK_H_ */
