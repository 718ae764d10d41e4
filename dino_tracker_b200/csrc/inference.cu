// Inference driver on the device: trajectories, trajectory cosine similarities, anchor re-tracking and
// occlusion (models/model_inference.py:8-216) + the generic grouped correlation/head entry point behind
// Tracker.forward (models/tracker.py:303-325).
//
// The reference walks query points and anchor frames in Python, one model() call per (query, anchor):
// each call gathers (T+1) x C x h x w twice and runs a B x N einsum.  Here every phase is a handful of
// launches over work lists grouped by target frame:
//   A  trajectories : descriptors s_n (N of them)          x every frame t        -> traj[n][t]
//   B  cos-sims     : d[n][i] sampled along the trajectory . d[n][t_q]            -> cos[n][i]
//   C  anchors      : for every anchor frame a, descriptors e[n][i] (a in A_n)    -> anchors[n][a][i]
//   D  occlusion    : lower medians over anchors, threshold, OR with cos < th     -> occ[n][i]
#include <algorithm>
#include <vector>

#include "common.cuh"
#include "corr.cuh"
#include "sample.cuh"
#include "xwin.cuh"

namespace dtk {

constexpr int TC2_BM_ROWS = 256;   // M tile of the CTA-pair GEMM (tcgemm2.cuh: TC2_BM)

// ---------------------------------------------------------------------------------- phase A helpers
// descriptors of the query points: frames_set = [t_q, s..e-1], set index 0 (model_inference.py:8-34)
__global__ void sample_query_kernel(const float* __restrict__ tpc, int T, int C, int P, int h, int w, PointAffine pa,
                                    const float* __restrict__ qp, float* __restrict__ desc, float* __restrict__ dnorm) {
  int n = blockIdx.x;
  float x = __fadd_rn(__fmul_rn(pa.aw, qp[n * 3 + 0]), pa.bw);
  float y = __fadd_rn(__fmul_rn(pa.ah, qp[n * 3 + 1]), pa.bh);
  int tq = (int)qp[n * 3 + 2];
  tq = min(max(tq, 0), T - 1);
  // set index 0 of a set with N >= 2 slots: t_n = -1 exactly -> slot 0 with weight 1, slot 1 with weight 0.
  // The weight-0 corner is skipped (0 * finite), so only frame t_q contributes.
  TriCorners c = tri_setup(x, y, 0.f, 2, h, w);
  sample_point(tpc, C, P, c, tq, -1, desc + (size_t)n * C, dnorm + n);
}

// out_index / t column for phase A maps of one chunk: map j -> group k -> (n, t)
__global__ void index_traj_kernel(const int* __restrict__ grp_frame, const int* __restrict__ grp_row0,
                                  const int* __restrict__ grp_map0, int n_groups, int n_maps, int T,
                                  int* __restrict__ out_index, float* __restrict__ traj) {
  int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= n_maps) return;
  int lo = 0, hi = n_groups - 1;
  while (lo < hi) {
    int mid = (lo + hi + 1) >> 1;
    if (grp_map0[mid] <= j) lo = mid; else hi = mid - 1;
  }
  int n = grp_row0[lo] + (j - grp_map0[lo]);
  int t = grp_frame[lo];
  out_index[j] = n * T + t;
  traj[((size_t)n * T + t) * 3 + 2] = (float)t;
}

// ---------------------------------------------------------------------------------- phase B
// cos[n][i] = F.cosine_similarity(d[n][t_q], d[n][i]) with d sampled from the full T-frame set
// (model_inference.py:110-126): x / max(|x|, eps) . y / max(|y|, eps), eps = 1e-8.
__global__ void traj_cos_kernel(const float* __restrict__ tpc, int T, int C, int P, int h, int w, PointAffine pa,
                                const float* __restrict__ traj, const float* __restrict__ qp,
                                float* __restrict__ cos_out) {
  extern __shared__ __align__(16) float sm[];  // dq[C], di[C]
  __shared__ float nrm[2];
  __shared__ float red[SAMPLE_THREADS / 32];
  const int n = blockIdx.y, i = blockIdx.x;
  int tq = (int)qp[n * 3 + 2];
  tq = min(max(tq, 0), T - 1);
  for (int which = 0; which < 2; ++which) {
    const float* pt = traj + ((size_t)n * T + (which == 0 ? tq : i)) * 3;
    float x = __fadd_rn(__fmul_rn(pa.aw, pt[0]), pa.bw);
    float y = __fadd_rn(__fmul_rn(pa.ah, pt[1]), pa.bh);
    TriCorners c = tri_setup(x, y, pt[2], T, h, w);  // frames_set = identity over the T frames
    sample_point(tpc, C, P, c, c.z0, c.z1, sm + which * C, nrm + which);
    __syncthreads();
  }
  const float nq = fmaxf(nrm[0], 1e-8f), ni = fmaxf(nrm[1], 1e-8f);
  float acc = 0.f;
  for (int c = threadIdx.x; c < C; c += SAMPLE_THREADS) acc = fmaf(__fdiv_rn(sm[c], nq), __fdiv_rn(sm[C + c], ni), acc);
  acc = warp_sum(acc);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    float s = 0.f;
    for (int k = 0; k < SAMPLE_THREADS / 32; ++k) s += red[k];
    cos_out[(size_t)n * T + i] = s;
  }
}

// ---------------------------------------------------------------------------------- phase C helpers
// per anchor frame a: ordered list of the query points n with cos[n][a] >= th, and its length
__global__ void anchor_lists_kernel(const float* __restrict__ cos_sims, int N, int T, float th,
                                    int* __restrict__ cnt, int* __restrict__ qlist) {
  const int a = blockIdx.x;
  __shared__ int base;
  __shared__ int wcount[32];
  if (threadIdx.x == 0) base = 0;
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
  for (int n0 = 0; n0 < N; n0 += blockDim.x) {
    int n = n0 + threadIdx.x;
    bool v = n < N && cos_sims[(size_t)n * T + a] >= th;
    unsigned bal = __ballot_sync(0xffffffffu, v);
    if (lane == 0) wcount[warp] = __popc(bal);
    __syncthreads();
    int off = base;
    for (int k = 0; k < warp; ++k) off += wcount[k];
    if (v) qlist[(size_t)a * N + off + __popc(bal & ((1u << lane) - 1))] = n;
    __syncthreads();
    if (threadIdx.x == 0) {
      int tot = 0;
      for (int k = 0; k < nw; ++k) tot += wcount[k];
      base += tot;
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) cnt[a] = base;
}

// descriptors of one chunk of anchor work items.  Group k of the chunk covers items
// [grp_item0[k], grp_item0[k] + grp_m[k]) of anchor frame grp_frame[k]; item u = (query slot u / T, frame u % T).
// Source point traj[n][i] lives in frame i; frames_set = [a, i0..e-1] (model_inference.py:138-143).
__global__ void sample_anchor_kernel(const float* __restrict__ tpc, int T, int C, int P, int h, int w, PointAffine pa,
                                     const float* __restrict__ traj, const int* __restrict__ qlist, int N,
                                     const int* __restrict__ grp_frame, const int* __restrict__ grp_map0,
                                     const int* __restrict__ grp_item0, int n_groups, int frame_batch,
                                     float* __restrict__ desc, float* __restrict__ dnorm, int* __restrict__ out_index,
                                     __half* __restrict__ desc_hi, __half* __restrict__ desc_lo) {
  const int j = blockIdx.x;
  int lo = 0, hi = n_groups - 1;
  while (lo < hi) {
    int mid = (lo + hi + 1) >> 1;
    if (grp_map0[mid] <= j) lo = mid; else hi = mid - 1;
  }
  const int a = grp_frame[lo];
  const int u = grp_item0[lo] + (j - grp_map0[lo]);
  const int slot = u / T, i = u - slot * T;
  const int n = qlist[(size_t)a * N + slot];
  const int i0 = (i / frame_batch) * frame_batch, e = min(i0 + frame_batch, T);
  const int Nset = e - i0 + 1;
  const float* pt = traj + ((size_t)n * T + i) * 3;
  float x = __fadd_rn(__fmul_rn(pa.aw, pt[0]), pa.bw);
  float y = __fadd_rn(__fmul_rn(pa.ah, pt[1]), pa.bh);
  TriCorners c = tri_setup(x, y, (float)(i - i0 + 1), Nset, h, w);
  int f0 = c.z0 == 0 ? a : i0 + c.z0 - 1;
  int f1 = c.z1 < 0 ? -1 : (c.z1 == 0 ? a : i0 + c.z1 - 1);
  sample_point(tpc, C, P, c, f0, f1, desc + (size_t)j * C, dnorm + j, desc_hi ? desc_hi + (size_t)j * C : nullptr,
               desc_lo ? desc_lo + (size_t)j * C : nullptr);
  if (threadIdx.x == 0) out_index[j] = (n * T + a) * T + i;
}

// The descriptor of work item (n, i, a) -- trajectory point traj[n][i] sampled from the frame set [a, i0..e-1] at slot
// i - i0 + 1 -- does not depend on the anchor frame a unless the fp32 round trip of the slot index (utils.py:96-99) leaks
// weight onto slot 0.  So every (n, i) is sampled ONCE (fp16 hi / lo halves + norm, what the tensor-path GEMMs consume) and
// flagged if slot 0 takes part; per chunk, unflagged items are row copies, flagged ones are sampled as before.
__global__ void sample_unique_kernel(const float* __restrict__ tpc, int T, int C, int P, int h, int w, PointAffine pa,
                                     const float* __restrict__ traj, int frame_batch, __half* __restrict__ u_hi,
                                     __half* __restrict__ u_lo, float* __restrict__ u_norm, int* __restrict__ u_flag) {
  const int u = blockIdx.x;                 // n * T + i
  const int i = u % T;
  const int i0 = (i / frame_batch) * frame_batch, e = min(i0 + frame_batch, T);
  const float* pt = traj + (size_t)u * 3;
  float x = __fadd_rn(__fmul_rn(pa.aw, pt[0]), pa.bw);
  float y = __fadd_rn(__fmul_rn(pa.ah, pt[1]), pa.bh);
  TriCorners c = tri_setup(x, y, (float)(i - i0 + 1), e - i0 + 1, h, w);
  bool slot0 = false;
#pragma unroll
  for (int k = 0; k < 4; ++k) slot0 = slot0 || (c.z0 == 0 && c.tok[k] >= 0 && c.wxy[k][0] != 0.f);
  if (threadIdx.x == 0) u_flag[u] = slot0 ? 1 : 0;
  if (slot0) return;                        // depends on the anchor frame: sampled per work item
  const int f0 = i0 + c.z0 - 1;
  const int f1 = c.z1 < 0 ? -1 : i0 + c.z1 - 1;
  sample_point(tpc, C, P, c, f0, f1, nullptr, u_norm + u, u_hi + (size_t)u * C, u_lo + (size_t)u * C);
}

// descriptors (fp16 hi / lo + norm) and output slots of one chunk of anchor work items, from the unique samples
__global__ void gather_anchor_kernel(const float* __restrict__ tpc, int T, int C, int P, int h, int w, PointAffine pa,
                                     const float* __restrict__ traj, const int* __restrict__ qlist, int N,
                                     const int* __restrict__ grp_frame, const int* __restrict__ grp_map0,
                                     const int* __restrict__ grp_item0, int n_groups, int frame_batch,
                                     const __half* __restrict__ u_hi, const __half* __restrict__ u_lo,
                                     const float* __restrict__ u_norm, const int* __restrict__ u_flag,
                                     float* __restrict__ dnorm, int* __restrict__ out_index, __half* __restrict__ desc_hi,
                                     __half* __restrict__ desc_lo) {
  const int j = blockIdx.x;
  int lo = 0, hi = n_groups - 1;
  while (lo < hi) {
    int mid = (lo + hi + 1) >> 1;
    if (grp_map0[mid] <= j) lo = mid; else hi = mid - 1;
  }
  const int a = grp_frame[lo];
  const int uu = grp_item0[lo] + (j - grp_map0[lo]);
  const int slot = uu / T, i = uu - slot * T;
  const int n = qlist[(size_t)a * N + slot];
  const size_t u = (size_t)n * T + i;
  if (threadIdx.x == 0) out_index[j] = (n * T + a) * T + i;
  if (!u_flag[u]) {
    const uint4* sh = reinterpret_cast<const uint4*>(u_hi + u * C);
    const uint4* sl = reinterpret_cast<const uint4*>(u_lo + u * C);
    uint4* dh = reinterpret_cast<uint4*>(desc_hi + (size_t)j * C);
    uint4* dl = reinterpret_cast<uint4*>(desc_lo + (size_t)j * C);
    for (int k = threadIdx.x; k < C / 8; k += blockDim.x) { dh[k] = __ldg(sh + k); dl[k] = __ldg(sl + k); }
    if (threadIdx.x == 0) dnorm[j] = u_norm[u];
    return;
  }
  const int i0 = (i / frame_batch) * frame_batch, e = min(i0 + frame_batch, T);
  const float* pt = traj + u * 3;
  float x = __fadd_rn(__fmul_rn(pa.aw, pt[0]), pa.bw);
  float y = __fadd_rn(__fmul_rn(pa.ah, pt[1]), pa.bh);
  TriCorners c = tri_setup(x, y, (float)(i - i0 + 1), e - i0 + 1, h, w);
  int f0 = c.z0 == 0 ? a : i0 + c.z0 - 1;
  int f1 = c.z1 < 0 ? -1 : (c.z1 == 0 ? a : i0 + c.z1 - 1);
  sample_point(tpc, C, P, c, f0, f1, nullptr, dnorm + j, desc_hi + (size_t)j * C, desc_lo + (size_t)j * C);
}

// ---------------------------------------------------------------------------------- phase D
// model_inference.py:169-177.  One block per query point, one warp per column i.
// D[a][i] = |anchors[n][a][i] - traj[n][a]| for a in A_n; med[i] = lower median over a
// (torch.median: sorted position (M-1)/2); th = max_{i in A_n} med[i];
// occ[i] = med[i] > th || cos[n][i] < cos_th.
constexpr int OCC_THREADS = 256;
__global__ void occlusion_kernel(const float* __restrict__ traj, const float* __restrict__ cos_sims,
                                 const float* __restrict__ anchors, int T, float anchor_th, float cos_th,
                                 uint8_t* __restrict__ occ) {
  extern __shared__ float sm[];  // med[T] | alist[T] | ax[T] | ay[T] | col[nwarps][T]
  float* med = sm;
  int* alist = reinterpret_cast<int*>(sm + T);
  float* ax = sm + 2 * T;
  float* ay = sm + 3 * T;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = OCC_THREADS / 32;
  float* col = sm + 4 * T + warp * T;
  __shared__ int M;
  __shared__ float th_s;
  const int n = blockIdx.x;
  if (threadIdx.x == 0) {
    int m = 0;
    for (int a = 0; a < T; ++a)
      if (cos_sims[(size_t)n * T + a] >= anchor_th) {
        alist[m] = a;
        ax[m] = traj[((size_t)n * T + a) * 3 + 0];
        ay[m] = traj[((size_t)n * T + a) * 3 + 1];
        ++m;
      }
    M = m;
  }
  __syncthreads();
  const int m = M, want = (m - 1) / 2;
  for (int i = warp; i < T; i += nw) {
    for (int p = lane; p < m; p += 32) {
      const float* g = anchors + (((size_t)n * T + alist[p]) * T + i) * 2;
      float dx = __fsub_rn(g[0], ax[p]), dy = __fsub_rn(g[1], ay[p]);
      col[p] = sqrtf(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)));
    }
    __syncwarp();
    for (int p = lane; p < m; p += 32) {
      const float dp = col[p];
      int rank = 0;
      for (int q = 0; q < m; ++q) {
        float dq = col[q];
        rank += (dq < dp) || (dq == dp && q < p);
      }
      if (rank == want) med[i] = dp;
    }
    __syncwarp();
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    float th = -INFINITY;
    for (int p = 0; p < m; ++p) th = fmaxf(th, med[alist[p]]);
    th_s = th;
  }
  __syncthreads();
  for (int i = threadIdx.x; i < T; i += blockDim.x)
    occ[(size_t)n * T + i] = (m > 0 && (med[i] > th_s || cos_sims[(size_t)n * T + i] < cos_th)) ? 1 : 0;
}

struct GroupBuf {  // host mirror of the per-chunk group arrays: [frame | row0 | m | map0 | item0] x cap
  std::vector<int> v;
  int cap, n;
  explicit GroupBuf(int c) : v((size_t)5 * c), cap(c), n(0) {}
  void clear() { n = 0; }
  void push(int frame, int row0, int m, int map0, int item0) {
    v[n] = frame; v[cap + n] = row0; v[2 * cap + n] = m; v[3 * cap + n] = map0; v[4 * cap + n] = item0; ++n;
  }
};

// ---- chunk planning (host only) ---------------------------------------------------------------------------------
// A phase's work items are cut into chunks of <= ch correlation maps; inside a chunk, items of the same target
// frame form one group = [frame | first descriptor row | number of rows m | first map | first item] (GroupBuf order).
//   kind 0 (trajectories): items = (frame t, query row n), t-major; descriptor rows are the N query rows.
//   kind 1 (anchors): items of anchor frame a = cnt[a] * T pairs (slot, i), a-major; descriptor rows are per chunk.
struct ChunkMeta { int used, maxm, n_groups; bool no_thin; };
// align: anchor-phase chunks are cut at multiples of `align` items per frame (T for the exact-window path: whole cells).
// first_cap > 0: capacity of the first anchor-phase chunk only (the probe chunk of the exact-window pipeline).
static void plan_chunks(int kind, int T, int N, const int* cnt, int ch_all, int gcap, std::vector<ChunkMeta>& metas,
                        std::vector<int>& plan_host, int align = 1, int first_cap = 0) {
  int ch = ch_all;
  metas.clear(); plan_host.clear();
  GroupBuf gb(gcap);
  auto commit_chunk = [&](int used, int maxm) {
    bool no_thin = true;
    for (int k = 0; k < gb.n; ++k) no_thin = no_thin && gb.v[2 * gb.cap + k] > STREAM_MAX_M;
    metas.push_back(ChunkMeta{used, maxm, gb.n, no_thin});
    plan_host.insert(plan_host.end(), gb.v.begin(), gb.v.end());
  };
  if (kind == 0) {
    int t = 0, row = 0;  // next work item: (frame t, query row)
    while (t < T) {
      gb.clear();
      int used = 0, maxm = 0;
      while (t < T && used < ch && gb.n < gcap) {
        int m = N - row;
        if (m > ch - used) m = ch - used;
        gb.push(t, row, m, used, 0);
        used += m; row += m;
        if (m > maxm) maxm = m;
        if (row == N) { row = 0; ++t; }
      }
      commit_chunk(used, maxm);
    }
  } else {
    int a = 0;
    long long item = 0;  // next work item: anchor frame a, item index within a (slot * T + i)
    while (a < T) {
      gb.clear();
      int used = 0, maxm = 0;
      ch = (metas.empty() && first_cap > 0 && first_cap < ch_all) ? first_cap : ch_all;
      while (a < T && used < ch && gb.n < gcap) {
        long long tot = (long long)cnt[a] * T;
        long long m = tot - item;
        if (m > ch - used) {
          m = (long long)((ch - used) / align) * align;
          if (m == 0 && used > 0) break;            // chunk full up to the alignment
          if (m == 0) m = align;                    // (ch >= align is guaranteed by the caller)
        }
        if (m > 0) {
          gb.push(a, used, (int)m, used, (int)item);
          used += (int)m; item += m;
          if ((int)m > maxm) maxm = (int)m;
        }
        if (item >= tot) { item = 0; ++a; }
      }
      if (used == 0) break;
      commit_chunk(used, maxm);
    }
  }
}

// ---- cells of the exact-window path (xwin.cuh): the <= 128 source frames of one (query slot, anchor frame) ----
struct CellPlan {
  std::vector<int> v;               // per chunk: [row0 | m | frame | group] x (cells of the chunk), chunks back to back
  std::vector<size_t> first;        // first cell of chunk k in v's cell numbering (size chunks + 1)
  std::vector<int> tiles;           // per chunk: (gcap + 1) prefix of ceil(m / 256) per group (coarse GEMM)
  int max_m = 0;
};
static void plan_cells(int T, int gcap, const std::vector<ChunkMeta>& metas, const std::vector<int>& plan_host, CellPlan& cp) {
  const int nb = (T + XW_MAX_CELL - 1) / XW_MAX_CELL, rb = (T + nb - 1) / nb;
  cp.v.clear(); cp.first.assign(1, 0); cp.tiles.clear(); cp.max_m = 0;
  std::vector<int> r0, mm, fr, gr;
  for (size_t k = 0; k < metas.size(); ++k) {
    const int* gb = plan_host.data() + k * 5 * gcap;
    r0.clear(); mm.clear(); fr.clear(); gr.clear();
    int pre = 0;
    for (int g = 0; g < metas[k].n_groups; ++g) {
      const int frame = gb[g], row0 = gb[gcap + g], m = gb[2 * gcap + g];
      cp.tiles.push_back(pre);
      pre += (m + TC2_BM_ROWS - 1) / TC2_BM_ROWS;
      for (int s0 = 0; s0 < m; s0 += T)
        for (int b = 0; b < T; b += rb) {
          const int cm = std::min(rb, T - b);
          r0.push_back(row0 + s0 + b); mm.push_back(cm); fr.push_back(frame); gr.push_back(g);
          cp.max_m = std::max(cp.max_m, cm);
        }
    }
    for (int g = metas[k].n_groups; g <= gcap; ++g) cp.tiles.push_back(pre);
    const size_t n = r0.size();
    cp.v.insert(cp.v.end(), r0.begin(), r0.end());
    cp.v.insert(cp.v.end(), mm.begin(), mm.end());
    cp.v.insert(cp.v.end(), fr.begin(), fr.end());
    cp.v.insert(cp.v.end(), gr.begin(), gr.end());
    cp.first.push_back(cp.first.back() + n);
  }
}

// auxiliary stream + events of the phase-C pipeline (one set per process; DTK_OVERLAP=0 disables the overlap)
struct InferAsync {
  int mode;                 // 1: sampling overlapped with the GEMMs (default); 2: sampling and the head fast path
  cudaStream_t aux, aux2;   // head stream, sampling stream
  cudaEvent_t fork, join, sample[2], gemm[2], head[2];
  int head_ctas_per_sm;
};
static int g_overlap_mode = -1;   // -1: DTK_OVERLAP or the default (1); see dinotrk_infer_set_overlap
struct InferAsyncSlot { InferAsync ia; int state; };   // state 0: not created, 1: ready, -1: creation failed
static InferAsync* infer_async() {
  static PerDev<InferAsyncSlot> slots;   // streams and events belong to the device they were created on
  InferAsyncSlot& slot = slots.get();
  InferAsync& ia = slot.ia;
  int& state = slot.state;
  int mode = g_overlap_mode;
  if (mode < 0) {
    const char* e = getenv("DTK_OVERLAP");
    mode = e ? atoi(e) : 1;
  }
  if (mode <= 0) return nullptr;
  if (state == 0) {
    state = -1;
    const char* hc = getenv("DTK_HEAD_OVERLAP_CTAS");
    ia.head_ctas_per_sm = hc ? atoi(hc) : 2;
    if (cudaStreamCreateWithFlags(&ia.aux, cudaStreamNonBlocking) != cudaSuccess) return nullptr;
    if (cudaStreamCreateWithFlags(&ia.aux2, cudaStreamNonBlocking) != cudaSuccess) return nullptr;
    cudaEvent_t* evs[] = {&ia.fork, &ia.join, &ia.sample[0], &ia.sample[1], &ia.gemm[0], &ia.gemm[1], &ia.head[0], &ia.head[1]};
    for (cudaEvent_t* ev : evs)
      if (cudaEventCreateWithFlags(ev, cudaEventDisableTiming) != cudaSuccess) return nullptr;
    state = 1;
  }
  if (state != 1) return nullptr;
  ia.mode = mode;
  return &ia;
}

// events, pinned counters and selection of the exact-window pipeline (one set per device)
constexpr int XW_RING = 4;
constexpr int XW_PROBE_MAPS = 4096;   // size of the probe chunk (automatic pipeline choice)
struct XwAsync {
  int state;                                   // 0: not created, 1: ready, -1: failed
  cudaEvent_t sample[XW_RING], done[XW_RING], freed[XW_RING];
  int* host_cnt;                               // pinned: [XW_RING][XW_NCNT] chunk counters (XwChunk::slow_cnt from [n_groups])
                                               // + [16] phase-A uncertified counts + the smallest token norm
};
static XwAsync* xw_async() {
  static PerDev<XwAsync> slots;
  XwAsync& xa = slots.get();
  if (xa.state == 0) {
    xa.state = -1;
    for (int k = 0; k < XW_RING; ++k) {
      if (cudaEventCreateWithFlags(&xa.sample[k], cudaEventDisableTiming) != cudaSuccess) return nullptr;
      if (cudaEventCreateWithFlags(&xa.done[k], cudaEventDisableTiming) != cudaSuccess) return nullptr;
      if (cudaEventCreateWithFlags(&xa.freed[k], cudaEventDisableTiming) != cudaSuccess) return nullptr;
    }
    if (cudaHostAlloc(&xa.host_cnt, (XW_NCNT * XW_RING + 16 + 4) * sizeof(int), cudaHostAllocDefault) != cudaSuccess) return nullptr;
    xa.state = 1;
  }
  return xa.state == 1 ? &xa : nullptr;
}
static int g_xw_path = -1;                     // -1: automatic (DTK_XW or on), 0: full-map path only, 1: exact-window path
// anchor-phase maps | on the exact-window path | queued | path used | queued by the certificate | exact-window cells whose box
// has 2, 3, 4 M-parts
constexpr int INFER_NSTATS = 5 + (XW_PARTS - 1);
static long long g_infer_stats[INFER_NSTATS] = {};

}  // namespace dtk

using namespace dtk;

extern "C" {

int dinotrk_infer_set_path(int path) {
  DTK_CHECK_ARG(path >= -1 && path <= 1, "infer_set_path: -1 (automatic), 0 (full-map GEMM + head) or 1 (coarse pass + exact window)");
  g_xw_path = path;
  return DINOTRK_OK;
}

int dinotrk_infer_last_stats(long long* out, int n) {
  DTK_CHECK_ARG(out && n >= 4, "infer_last_stats: need at least 4 slots");
  for (int i = 0; i < (n < INFER_NSTATS ? n : INFER_NSTATS); ++i) out[i] = g_infer_stats[i];
  return DINOTRK_OK;
}

static int infer_chunk_maps(int chunk_maps) { return chunk_maps > 0 ? chunk_maps : 4096; }
// chunks of the anchor phase hold whole (query, anchor frame) cells of T maps: never smaller than T
static int infer_chunk_eff(int chunk_maps, int T) { const int c = infer_chunk_maps(chunk_maps); return c > T ? c : T; }
// upper bound on the number of chunks of one phase (phase C has the most work items: N * T * T)
// (anchor-phase chunks are cut at whole cells of T maps: a full chunk holds at least the largest multiple of T <= ch)
static size_t infer_max_chunks(int T, int N, size_t ch) {
  size_t cap = (ch / (size_t)T) * (size_t)T;
  if (cap < (size_t)T) cap = T;
  return ((size_t)N * T * T + cap - 1) / cap + 2;
}

// (planner entry point: plain chunks of `chunk_maps` maps, cut anywhere)
size_t dinotrk_infer_max_chunks(int T, int N, int chunk_maps) {
  const size_t ch = (size_t)infer_chunk_maps(chunk_maps);
  return ((size_t)N * T * T + ch - 1) / ch + 2;
}

int dinotrk_infer_plan(int kind, int T, int N, const int* anchor_counts, int chunk_maps, int* groups, int* meta,
                       int max_chunks, int* n_chunks) {
  DTK_CHECK_ARG((kind == 0 || kind == 1) && T > 0 && N >= 0 && n_chunks, "infer_plan: bad arguments");
  DTK_CHECK_ARG(kind == 0 || anchor_counts, "infer_plan: kind 1 needs the per-frame anchor counts");
  const int ch = infer_chunk_maps(chunk_maps), gcap = T + 2;
  std::vector<ChunkMeta> metas;
  std::vector<int> plan_host;
  plan_chunks(kind, T, N, anchor_counts, ch, gcap, metas, plan_host);
  *n_chunks = (int)metas.size();
  DTK_CHECK_ARG((int)metas.size() <= max_chunks || (!groups && !meta), "infer_plan: %zu chunks, room for %d", metas.size(), max_chunks);
  if (groups) std::copy(plan_host.begin(), plan_host.end(), groups);
  if (meta)
    for (size_t k = 0; k < metas.size(); ++k) {
      meta[4 * k] = metas[k].used; meta[4 * k + 1] = metas[k].maxm; meta[4 * k + 2] = metas[k].n_groups;
      meta[4 * k + 3] = metas[k].no_thin ? 1 : 0;
    }
  return DINOTRK_OK;
}

int dinotrk_infer_set_overlap(int mode) {
  DTK_CHECK_ARG(mode >= -1 && mode <= 2, "infer_set_overlap: mode must be -1 (default / DTK_OVERLAP), 0, 1 or 2");
  g_overlap_mode = mode;
  return DINOTRK_OK;
}

size_t dinotrk_corr_track_workspace_bytes(int total_maps, int n_groups, int C, const dinotrk_geom* g) {
  if (!g) return 0;
  return align_up((size_t)total_maps * dinotrk_map_stride(g) * sizeof(float), 256) + corr_plan_bytes(n_groups) +
         corr_tc_workspace_bytes(total_maps, C) + align_up((size_t)(total_maps + 1) * 4, 256) + 1024;
}

int dinotrk_corr_track(const dinotrk_features* feat, const dinotrk_geom* g,
                       const dinotrk_head_weights* hw, const float* desc, const float* desc_norm,
                       const int* grp_frame, const int* grp_row0, const int* grp_m, const int* grp_map0,
                       int n_groups, int total_maps, int max_group_m, const int* out_index, float* out,
                       int out_stride, int out_mode, void* workspace, size_t workspace_bytes, void* stream) {
  DTK_CHECK_ARG(feat && feat->tpc && feat->norms && g && hw && desc && desc_norm && grp_frame && grp_row0 && grp_m &&
                grp_map0 && out, "corr_track: null pointer");
  const int C = feat->C;
  DTK_CHECK_ARG(feat->T > 0 && C > 0 && C % 4 == 0 && n_groups >= 0 && total_maps >= 0, "corr_track: bad sizes");
  DTK_CHECK_ARG((feat->hi == nullptr) == (feat->lo == nullptr), "corr_track: hi and lo must be given together");
  DTK_CHECK_ARG(workspace && workspace_bytes >= dinotrk_corr_track_workspace_bytes(total_maps, n_groups, C, g),
                "corr_track: workspace too small");
  if (total_maps == 0) return DINOTRK_OK;
  Arena ar(workspace, workspace_bytes);
  const int ms = dinotrk_map_stride(g);
  float* maps = ar.take<float>((size_t)total_maps * ms);
  int* plan = ar.take<int>(n_groups + 1);
  float* split = ar.take<float>(corr_tc_workspace_bytes(total_maps, C) / 4);
  int* hscratch = ar.take<int>(total_maps + 1);
  cudaStream_t st = (cudaStream_t)stream;
  int rc = launch_corr_maps(make_view(*feat, *g), desc, total_maps, desc_norm, grp_frame, grp_row0, grp_m, grp_map0,
                            n_groups, total_maps, max_group_m, maps, ms, plan, split, st);
  if (rc) return rc;
  return launch_head(maps, total_maps, ms, *g, *hw, out_index, out, out_stride, out_mode, nullptr, hscratch, st);
}


size_t dinotrk_infer_workspace_bytes(int T, int C, const dinotrk_geom* g, int N, int chunk_maps) {
  if (!g) return 0;
  const size_t ch = infer_chunk_eff(chunk_maps, T), ms = dinotrk_map_stride(g);
  const int gcap = T + 2;
  size_t b = 0;
  b += align_up((size_t)N * C * 4, 256) + align_up((size_t)N * 4, 256);   // descA, normA
  size_t c = 0;                                                            // per chunk buffer set (two: pipelining)
  c += align_up(ch * ms * 4, 256);                                         // maps chunk
  c += align_up(ch * C * 4, 256) + align_up(ch * 4, 256);                  // descC, normC
  c += align_up((size_t)(gcap + 1) * 4, 256);                              // GEMM tile plan
  c += corr_tc_workspace_bytes((int)(ch > (size_t)N ? ch : (size_t)N), C) + 256;  // fp16 split of the descriptors
  c += align_up((ch + 1) * 4, 256);                                        // head: list of uncertified maps
  c += align_up(ch * (size_t)cdiv(g->h * g->w, CORR_TILE) * 8, 256);       // tile keys of the chunk's maps
  b += 2 * c;
  b += 4 * align_up(ch * 4, 256);                                          // out_index ring
  b += align_up(infer_max_chunks(T, N, ch) * 5 * gcap * 4, 256);           // group arrays of every chunk of a phase
  b += align_up((size_t)T * 4, 256) + align_up((size_t)T * N * 4, 256);    // cnt, qlist
  // exact-window pipeline: ring of XW_RING chunk sets (descriptors fp32 + fp16 hi/lo, norms, out_index, keys, boxes),
  // the cells of every chunk of the phase, coarse-GEMM tile prefixes, compact group arrays of the full-map queue
  const size_t chx = ch;
  const int nb = (T + XW_MAX_CELL - 1) / XW_MAX_CELL;
  const size_t max_cells_chunk = chx + 2;                                  // cells have >= 1 row
  size_t x = 0;
  x += align_up(chx * 4, 256) + corr_tc_workspace_bytes((int)chx, C) + 256 + align_up(chx * 4, 256);   // norms, hi / lo, out_index
  x += xw_chunk_bytes((int)chx, (int)max_cells_chunk, cdiv(g->h * g->w, XW_TILE), gcap);
  b += XW_RING * x;
  b += 2 * align_up((size_t)N * T * C * 2, 256) + 2 * align_up((size_t)N * T * 4, 256);   // unique descriptors (hi, lo, norm, flag)
  b += align_up((size_t)T * g->h * g->w * 4, 256) + 256;                                  // reciprocal token norms, smallest norm
  b += align_up((size_t)N * T * nb * 16 + 64, 256);                         // cells of all chunks
  b += align_up(infer_max_chunks(T, N, ch) * (gcap + 1) * 4, 256);         // coarse tile prefixes per chunk
  {
    const size_t sg = std::min<size_t>(infer_max_chunks(T, N, ch) * (size_t)gcap, 16384);
    b += align_up(4 * sg * 4, 256) + align_up((sg + 1) * 4, 256) + align_up(64 * 4, 256);   // queue group arrays + tile plan, phase-A counters
  }
  return b + 16384;
}

int dinotrk_traj_cos_sims(const float* tpc, int T, int C, const dinotrk_geom* g, const float* traj,
                          const float* query_points, int N, float* cos_sims, void* workspace,
                          size_t workspace_bytes, void* stream) {
  (void)workspace; (void)workspace_bytes;
  DTK_CHECK_ARG(tpc && g && traj && query_points && cos_sims, "traj_cos_sims: null pointer");
  DTK_CHECK_ARG(T > 0 && C > 0 && C % 4 == 0 && N >= 0, "traj_cos_sims: bad sizes");
  if (N == 0) return DINOTRK_OK;
  size_t smem = (size_t)2 * C * sizeof(float);
  static PerDev<size_t> attr_dev;
  size_t& attr = attr_dev.get();
  if (smem > 48 * 1024 && smem > attr) {
    DTK_CUDA(cudaFuncSetAttribute(traj_cos_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    attr = smem;
  }
  ProfRange pr(PROF_COS, (cudaStream_t)stream);
  traj_cos_kernel<<<dim3(T, N), SAMPLE_THREADS, smem, (cudaStream_t)stream>>>(
      tpc, T, C, g->h * g->w, g->h, g->w, make_point_affine(*g), traj, query_points, cos_sims);
  DTK_LAUNCHED();
  return DINOTRK_OK;
}

int dinotrk_occlusion(const float* traj, const float* cos_sims, const float* anchors, int N, int T,
                      float anchor_th, float cos_th, uint8_t* occ, void* stream) {
  DTK_CHECK_ARG(traj && cos_sims && anchors && occ && N >= 0 && T > 0, "occlusion: bad args");
  if (N == 0) return DINOTRK_OK;
  size_t smem = (size_t)(4 + OCC_THREADS / 32) * T * sizeof(float);
  DTK_CHECK_ARG(smem <= 200 * 1024, "occlusion: T=%d too large", T);
  static PerDev<size_t> attr_dev;
  size_t& attr = attr_dev.get();
  if (smem > 48 * 1024 && smem > attr) {
    DTK_CUDA(cudaFuncSetAttribute(occlusion_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    attr = smem;
  }
  ProfRange pr(PROF_OCCLUSION, (cudaStream_t)stream);
  occlusion_kernel<<<N, OCC_THREADS, smem, (cudaStream_t)stream>>>(traj, cos_sims, anchors, T, anchor_th, cos_th, occ);
  DTK_LAUNCHED();
  return DINOTRK_OK;
}

int dinotrk_infer(const dinotrk_features* feat, const dinotrk_geom* g,
                  const dinotrk_head_weights* hw, const float* query_points, int N, float anchor_th, float cos_th,
                  int frame_batch, int start_phase, int stop_after, int chunk_maps, float* traj, float* cos_sims,
                  float* anchors,
                  uint8_t* occ, void* workspace, size_t workspace_bytes, void* stream) {
  DTK_CHECK_ARG(feat && feat->tpc && feat->norms && g && hw && query_points && traj, "infer: null pointer");
  const float* tpc = feat->tpc;
  const int T = feat->T, C = feat->C;
  DTK_CHECK_ARG(T > 0 && C > 0 && C % 4 == 0 && N >= 0, "infer: bad sizes");
  DTK_CHECK_ARG((feat->hi == nullptr) == (feat->lo == nullptr), "infer: hi and lo must be given together");
  const FeatView fv = make_view(*feat, *g);
  DTK_CHECK_ARG(start_phase >= 0 && start_phase <= stop_after && stop_after <= 3,
                "infer: need 0 <= start_phase <= stop_after <= 3");
  DTK_CHECK_ARG((stop_after < 1 || cos_sims) && (stop_after < 2 || anchors) && (stop_after < 3 || occ),
                "infer: missing output buffer for the requested phases");
  DTK_CHECK_ARG(workspace && workspace_bytes >= dinotrk_infer_workspace_bytes(T, C, g, N, chunk_maps),
                "infer: workspace too small (%zu < %zu)", workspace_bytes,
                dinotrk_infer_workspace_bytes(T, C, g, N, chunk_maps));
  if (N == 0) return DINOTRK_OK;
  cudaStream_t st = (cudaStream_t)stream;
  const int P = g->h * g->w, ms = dinotrk_map_stride(g);
  const int ch = infer_chunk_eff(chunk_maps, T);
  const int fb = frame_batch > 0 ? (frame_batch < T ? frame_batch : T) : T;
  const int gcap = T + 2;
  const PointAffine pa = make_point_affine(*g);

  Arena ar(workspace, workspace_bytes);
  float* descA = ar.take<float>((size_t)N * C);
  float* normA = ar.take<float>(N);
  struct ChunkBufs {   // everything one chunk in flight owns
    float* maps; float* desc; float* norm; int* plan; float* split; int* hscratch; unsigned long long* tkeys;
  } cb[2];
  int* out_index_ring[4];   // written by the sampler of chunk k, read by both head kernels of chunk k (the second one late)
  for (int k = 0; k < 2; ++k) {
    cb[k].maps = ar.take<float>((size_t)ch * ms);
    cb[k].desc = ar.take<float>((size_t)ch * C);
    cb[k].norm = ar.take<float>(ch);
    cb[k].plan = ar.take<int>(gcap + 1);
    cb[k].split = ar.take<float>(corr_tc_workspace_bytes(ch > N ? ch : N, C) / 4);
    cb[k].hscratch = ar.take<int>(ch + 1);
    cb[k].tkeys = ar.take<unsigned long long>((size_t)ch * cdiv(P, CORR_TILE));
  }
  for (int k = 0; k < 4; ++k) out_index_ring[k] = ar.take<int>(ch);
  const size_t max_chunks = infer_max_chunks(T, N, (size_t)ch);
  int* d_groups = ar.take<int>(max_chunks * 5 * gcap);
  int* d_cnt = ar.take<int>(T);
  int* d_qlist = ar.take<int>((size_t)T * N);
  struct XwSet { float* norm; float* split; int* out_index; XwChunk xc; } xr[XW_RING];
  const int n_tiles_map = cdiv(P, XW_TILE);     // coarse keys per map
  __half* u_hi = ar.take<__half>((size_t)N * T * C);
  __half* u_lo = ar.take<__half>((size_t)N * T * C);
  float* u_norm = ar.take<float>((size_t)N * T);
  int* u_flag = ar.take<int>((size_t)N * T);
  float* d_rnorms = ar.take<float>((size_t)T * P);
  unsigned* d_minnorm = ar.take<unsigned>(4);
  for (int k = 0; k < XW_RING; ++k) {
    xr[k].norm = ar.take<float>(ch);
    xr[k].split = ar.take<float>(corr_tc_workspace_bytes(ch, C) / 4);
    xr[k].out_index = ar.take<int>(ch);
    XwChunk& x = xr[k].xc;
    x.key1 = ar.take<unsigned long long>((size_t)ch * n_tiles_map);
    x.max2 = ar.take<float>((size_t)ch * n_tiles_map);
    x.cand = ar.take<int>((size_t)ch * XW_MAX_CAND);
    x.stat = ar.take<int>(ch);
    x.pinfo = ar.take<int>(ch);
    x.cell_of = ar.take<int>(ch);
    x.slow_list = ar.take<int>(ch);
    x.box = ar.take<XwBox>((size_t)ch + 2);
    x.xbox = ar.take<float>((size_t)ch * XW_COLS);
    x.win = ar.take<float>((size_t)ch * 256);
    x.hin = ar.take<int2>(ch);
    x.slow_cnt = ar.take<int>(gcap + XW_NCNT);
  }
  const int cell_nb = (T + XW_MAX_CELL - 1) / XW_MAX_CELL;
  int* d_cells = ar.take<int>((size_t)N * T * cell_nb * 4 + 16);
  int* d_tiles = ar.take<int>(max_chunks * (gcap + 1));
  const int sg_cap = (int)std::min<size_t>(max_chunks * (size_t)gcap, 16384);   // groups of the accumulated full-map queue
  int* d_cgrp = ar.take<int>((size_t)4 * sg_cap);
  int* d_splan = ar.take<int>((size_t)sg_cap + 1);
  int* d_cntA = ar.take<int>(64);
  DTK_CHECK_ARG(ar.ok(), "infer: workspace arena overflow");
  const bool tensor = fv.tensor();   // tensor-core GEMM: tile keys for the head, fp16 split fused into the samplers

  // The chunks of a phase are planned on the host in one go and their group arrays uploaded with ONE copy, so the
  // per-chunk launches below never block the host (a pageable cudaMemcpyAsync per chunk would).
  std::vector<ChunkMeta> metas;
  std::vector<int> plan_host;
  auto upload_plan = [&]() -> int {
    DTK_CHECK_ARG(metas.size() <= max_chunks, "infer: chunk plan exceeds its bound (%zu > %zu)", metas.size(), max_chunks);
    if (!plan_host.empty())
      DTK_CUDA(cudaMemcpyAsync(d_groups, plan_host.data(), plan_host.size() * sizeof(int), cudaMemcpyHostToDevice, st));
    return DINOTRK_OK;
  };
  struct Grp { const int *f, *r, *m, *map0, *item; };
  auto grp_of = [&](size_t k) {
    const int* b = d_groups + k * 5 * gcap;
    return Grp{b, b + gcap, b + 2 * gcap, b + 3 * gcap, b + 4 * gcap};
  };

  int n_chunks_A = 0;
  long long maps_A = 0;
  // ---- phase A: trajectories -------------------------------------------------------------------
  if (start_phase <= 0) {
    NvtxRange nv("dinotrk.infer.A.trajectories");
    {
      ProfRange pr(PROF_SAMPLE, st);
      sample_query_kernel<<<N, SAMPLE_THREADS, 0, st>>>(tpc, T, C, P, g->h, g->w, pa, query_points, descA, normA);
      DTK_LAUNCHED();
    }
    if (tensor) {   // the query descriptors are reused by every chunk: split them once (layout of desc_rows = N)
      for (int k = 0; k < 2; ++k) {
        char* a_hi = reinterpret_cast<char*>(cb[k].split);
        int rc = launch_split_f16(descA, a_hi, a_hi + align_up((size_t)N * C * 2, 256), (size_t)N * C, st);
        if (rc) return rc;
      }
    }
    plan_chunks(0, T, N, nullptr, ch, gcap, metas, plan_host);
    int rc = upload_plan();
    if (rc) return rc;
    for (size_t k = 0; k < metas.size(); ++k) {
      const ChunkMeta& cm = metas[k];
      const ChunkBufs& b = cb[k & 1];
      const Grp gp = grp_of(k);
      {
        ProfRange pr(PROF_MISC, st);
        index_traj_kernel<<<cdiv(cm.used, 256), 256, 0, st>>>(gp.f, gp.r, gp.map0, cm.n_groups, cm.used, T, out_index_ring[k & 3], traj);
        DTK_LAUNCHED();
      }
      CorrAssist as;
      as.tkeys = tensor ? b.tkeys : nullptr; as.zero_word = b.hscratch; as.split_ready = tensor; as.no_thin = cm.no_thin;
      rc = launch_corr_maps(fv, descA, N, normA, gp.f, gp.r, gp.m, gp.map0, cm.n_groups, cm.used, cm.maxm, b.maps, ms, b.plan,
                            b.split, st, as);
      if (rc) return rc;
      rc = launch_head(b.maps, cm.used, ms, *g, *hw, out_index_ring[k & 3], traj, 3, 0, nullptr, b.hscratch, st, as.tkeys, true);
      if (rc) return rc;
      if (k < 16)   // uncertified maps of this chunk: the anchor phase chooses its pipeline from their share
        DTK_CUDA(cudaMemcpyAsync(d_cntA + k, b.hscratch, sizeof(int), cudaMemcpyDeviceToDevice, st));
    }
    n_chunks_A = (int)std::min<size_t>(metas.size(), 16);
    maps_A = (long long)N * T;
  }
  if (stop_after < 1) return DINOTRK_OK;

  // ---- phase B: cosine similarities along the trajectories --------------------------------------
  if (start_phase <= 1) {
    NvtxRange nv("dinotrk.infer.B.cos_sims");
    int rc = dinotrk_traj_cos_sims(tpc, T, C, g, traj, query_points, N, cos_sims, nullptr, 0, stream);
    if (rc) return rc;
  }
  if (stop_after < 2) return DINOTRK_OK;

  // ---- phase C: anchor re-tracking ---------------------------------------------------------------
  // Three streams: the caller's stream runs the correlation GEMMs back to back; one auxiliary stream samples the
  // descriptors of chunk k+1, another runs the head of chunk k, both while the GEMM of chunk k+1 owns the tensor cores
  // (the head kernel is then launched with one CTA per SM so that it fits next to the GEMM's ~200 KB of shared memory;
  // the rare full-map head launches cannot co-reside and simply wait for the GEMM's CTAs to retire).
  if (start_phase <= 2) {
    NvtxRange nv("dinotrk.infer.C.anchors");
    {
      ProfRange pr(PROF_ANCHOR_LIST, st);
      anchor_lists_kernel<<<T, 256, 0, st>>>(cos_sims, N, T, anchor_th, d_cnt, d_qlist);
      DTK_LAUNCHED();
    }
    std::vector<int> cnt(T);
    // pipeline of the anchor phase: coarse pass + exact window (xwin.cuh) on the tensor path, unless disabled
    bool use_xw = tensor && g->radius <= 5 * g->stride && n_tiles_map <= 64;
    int pathsel = g_xw_path;
    if (pathsel < 0) { const char* e = getenv("DTK_XW"); if (e) pathsel = atoi(e) != 0 ? 1 : 0; }
    if (pathsel == 0) use_xw = false;
    XwAsync* xa = use_xw ? xw_async() : nullptr;
    if (!xa) use_xw = false;
    if (xa) {   // reciprocal token norms for the coarse epilogue + the smallest norm of the video (the host reads it below)
      int rcn = launch_xw_rnorms(fv, d_rnorms, d_minnorm, st);
      if (rcn) return rcn;
      DTK_CUDA(cudaMemcpyAsync(xa->host_cnt + XW_NCNT * XW_RING + 16, d_minnorm, sizeof(unsigned), cudaMemcpyDeviceToHost, st));
    }
    if (xa && n_chunks_A > 0)
      DTK_CUDA(cudaMemcpyAsync(xa->host_cnt + XW_NCNT * XW_RING, d_cntA, (size_t)n_chunks_A * sizeof(int), cudaMemcpyDeviceToHost, st));
    DTK_CUDA(cudaMemcpyAsync(cnt.data(), d_cnt, (size_t)T * sizeof(int), cudaMemcpyDeviceToHost, st));
    DTK_CUDA(cudaStreamSynchronize(st));  // the one host sync: sizes of the anchor work lists
    if (use_xw) {   // a (near-)zero token anywhere voids the coarse pass's error bound (xwin.cuh: XW_MIN_NORM)
      float mn;
      memcpy(&mn, xa->host_cnt + XW_NCNT * XW_RING + 16, sizeof(float));
      if (!(mn >= XW_MIN_NORM)) use_xw = false;
    }
    if (use_xw && pathsel < 0 && n_chunks_A > 0) {
      // head weights the certificate cannot handle send (almost) every map to the full-map kernels anyway: the trajectory
      // phase just showed it; skip the exact-window attempt then.  (Depends on the weights and the video only.)
      long long unc = 0;
      for (int k = 0; k < n_chunks_A; ++k) unc += xa->host_cnt[XW_NCNT * XW_RING + k];
      if (unc * 4 > maps_A) use_xw = false;
    }
    long long maps_C = 0;
    for (int a = 0; a < T; ++a) maps_C += (long long)cnt[a] * T;
    for (long long& v : g_infer_stats) v = 0;
    g_infer_stats[0] = maps_C; g_infer_stats[3] = use_xw ? 1 : 0;
    size_t k0 = 0;            // first chunk of the full-map pipeline (> 0 after an exact-window probe)
    bool planned = false;
    if (use_xw) {
      // automatic mode: the first chunk is a small probe; if the head's certificate sends more than a quarter of it to the
      // full-map queue (refiner weights whose outside-the-box logit bound needs the exact map), the rest of the phase runs
      // the full-map pipeline directly.  The probe is the same set of work items for every chunk size >= XW_PROBE_MAPS.
      const bool probing = pathsel < 0;
      const int probe_cap = std::max(T, (XW_PROBE_MAPS / T) * T);
      plan_chunks(1, T, N, cnt.data(), ch, gcap, metas, plan_host, T, probing ? probe_cap : 0);
      int rc = upload_plan();
      if (rc) return rc;
      planned = true;
      CellPlan cp;
      plan_cells(T, gcap, metas, plan_host, cp);
      DTK_CHECK_ARG(cp.first.back() * 4 <= (size_t)N * T * cell_nb * 4 + 16, "infer: cell plan exceeds its bound");
      if (!cp.v.empty()) DTK_CUDA(cudaMemcpyAsync(d_cells, cp.v.data(), cp.v.size() * sizeof(int), cudaMemcpyHostToDevice, st));
      if (!cp.tiles.empty()) DTK_CUDA(cudaMemcpyAsync(d_tiles, cp.tiles.data(), cp.tiles.size() * sizeof(int), cudaMemcpyHostToDevice, st));
      InferAsync* ia = infer_async();
      const bool ovl = ia != nullptr && metas.size() > 1;
      cudaStream_t sb = ovl ? ia->aux2 : st;   // sampling stream
      if (ovl) {
        DTK_CUDA(cudaEventRecord(ia->fork, st));
        DTK_CUDA(cudaStreamWaitEvent(sb, ia->fork, 0));
      }
      auto hi_of = [&](const XwSet& x, int rows) { (void)rows; return reinterpret_cast<char*>(x.split); };
      auto lo_of = [&](const XwSet& x, int rows) { return reinterpret_cast<char*>(x.split) + align_up((size_t)rows * C * 2, 256); };
      auto cells_of = [&](size_t k) {
        XwCells c;
        const int n = (int)(cp.first[k + 1] - cp.first[k]);
        const int* base = d_cells + 4 * cp.first[k];
        c.row0 = base; c.m = base + n; c.frame = base + 2 * n; c.group = base + 3 * n; c.n_cells = n; c.max_m = cp.max_m;
        return c;
      };
      auto enqueue_sample_x = [&](size_t k) -> int {
        const ChunkMeta& cm = metas[k];
        const XwSet& x = xr[k % XW_RING];
        const Grp gp = grp_of(k);
        if (ovl && k >= XW_RING) DTK_CUDA(cudaStreamWaitEvent(sb, xa->freed[k % XW_RING], 0));   // chunk k - 4 is through
        {
          ProfRange pr(PROF_SAMPLE, sb);
          gather_anchor_kernel<<<cm.used, SAMPLE_THREADS, 0, sb>>>(tpc, T, C, P, g->h, g->w, pa, traj, d_qlist, N, gp.f, gp.map0,
                                                                  gp.item, cm.n_groups, fb, u_hi, u_lo, u_norm, u_flag, x.norm,
                                                                  x.out_index, reinterpret_cast<__half*>(hi_of(x, cm.used)),
                                                                  reinterpret_cast<__half*>(lo_of(x, cm.used)));
          DTK_LAUNCHED();
        }
        if (ovl) DTK_CUDA(cudaEventRecord(xa->sample[k % XW_RING], sb));
        return DINOTRK_OK;
      };
      // Full-map queue.  The queued maps of chunk j (the host knows how many once the chunk's head has run) are appended to
      // ONE compact descriptor array (buffer set cb[0]); the queue is worked off -- split-precision GEMM over all tokens on
      // 128-row tiles + the head kernels of head.cu -- when it is full and at the end of the phase.
      int q_rows = 0, q_groups = 0;
      auto flush = [&]() -> int {
        if (q_rows == 0) return DINOTRK_OK;
        const ChunkBufs& b = cb[0];
        CorrAssist as;
        as.tkeys = b.tkeys; as.zero_word = b.hscratch; as.split_ready = true; as.no_thin = true; as.all_wide = true; as.small_tiles = true;
        int rc2 = launch_corr_maps(fv, nullptr, ch, b.norm, d_cgrp, d_cgrp + sg_cap, d_cgrp + 2 * sg_cap, d_cgrp + 3 * sg_cap, q_groups,
                                   q_rows, q_rows, b.maps, ms, d_splan, b.split, st, as);
        if (rc2) return rc2;
        rc2 = launch_head(b.maps, q_rows, ms, *g, *hw, out_index_ring[0], anchors, 2, 0, nullptr, b.hscratch, st, b.tkeys, true);
        q_rows = q_groups = 0;
        return rc2;
      };
      auto finish = [&](size_t j) -> int {
        DTK_CUDA(cudaEventSynchronize(xa->done[j % XW_RING]));
        const int* hc = xa->host_cnt + XW_NCNT * (j % XW_RING);
        const int n_slow = hc[0];
        for (int i = 1; i < XW_NCNT; ++i) g_infer_stats[3 + i] += hc[i];   // queued by the certificate, cells by part count
        const ChunkMeta& cm = metas[j];
        const XwSet& x = xr[j % XW_RING];
        const Grp gp = grp_of(j);
        DTK_CHECK_ARG(n_slow >= 0 && n_slow <= cm.used, "infer: corrupt full-map queue (%d of %d)", n_slow, cm.used);
        g_infer_stats[1] += cm.used - n_slow; g_infer_stats[2] += n_slow;
        if (n_slow > 0) {
          if (q_rows + n_slow > ch || q_groups + cm.n_groups > sg_cap) {
            int rc2 = flush();
            if (rc2) return rc2;
          }
          const ChunkBufs& b = cb[0];
          char* c_hi = reinterpret_cast<char*>(b.split);
          char* c_lo = c_hi + align_up((size_t)ch * C * 2, 256);          // layout of a descriptor array of `ch` rows
          int rc2 = launch_xw_compact(nullptr, hi_of(x, cm.used), lo_of(x, cm.used), x.norm, x.out_index, C, gp.f, gp.map0, cm.n_groups,
                                      n_slow, x.xc, nullptr, c_hi, c_lo, b.norm, out_index_ring[0], d_cgrp, sg_cap, st, q_rows, q_groups);
          if (rc2) return rc2;
          q_rows += n_slow; q_groups += cm.n_groups;
        }
        DTK_CUDA(cudaEventRecord(xa->freed[j % XW_RING], st));
        return DINOTRK_OK;
      };
      {   // every (query, source frame) descriptor once; the per-chunk kernels copy rows
        ProfRange pr(PROF_SAMPLE, st);
        sample_unique_kernel<<<N * T, SAMPLE_THREADS, 0, st>>>(tpc, T, C, P, g->h, g->w, pa, traj, fb, u_hi, u_lo, u_norm, u_flag);
        DTK_LAUNCHED();
      }
      if (ovl) {   // (the fork above was recorded before this launch: make the sampling stream wait for it)
        DTK_CUDA(cudaEventRecord(ia->fork, st));
        DTK_CUDA(cudaStreamWaitEvent(sb, ia->fork, 0));
      }
      if (!metas.empty() && (rc = enqueue_sample_x(0))) return rc;
      size_t n_finished = 0, k_end = metas.size();
      for (size_t k = 0; k < metas.size(); ++k) {
        const ChunkMeta& cm = metas[k];
        const XwSet& x = xr[k % XW_RING];
        const Grp gp = grp_of(k);
        const XwCells cells = cells_of(k);
        if (ovl) DTK_CUDA(cudaStreamWaitEvent(st, xa->sample[k % XW_RING], 0));
        if ((rc = launch_xw_coarse(fv, hi_of(x, cm.used), cm.used, x.norm, gp.f, gp.r, gp.m, gp.map0, d_tiles + k * (gcap + 1),
                                   cm.n_groups, cm.used / TC2_BM_ROWS + cm.n_groups, x.xc, st, d_rnorms))) return rc;
        if ((rc = launch_xw_plan(cells, x.norm, cm.n_groups, *g, x.xc, st, cm.used))) return rc;
        if ((rc = launch_xw_gemm(fv, *g, hi_of(x, cm.used), lo_of(x, cm.used), cm.used, cells, x.xc, st))) return rc;
        if ((rc = launch_xw_head(fv, *g, *hw, cells, x.norm, gp.map0, cm.used, x.out_index, anchors, 2, 0, x.xc, st, cm.n_groups)))
          return rc;
        DTK_CUDA(cudaMemcpyAsync(xa->host_cnt + XW_NCNT * (k % XW_RING), x.xc.slow_cnt + cm.n_groups, XW_NCNT * sizeof(int),
                                 cudaMemcpyDeviceToHost, st));
        DTK_CUDA(cudaEventRecord(xa->done[k % XW_RING], st));
        if (k == 0 && probing && metas.size() > 1) {   // the probe: wait for it, look at the certificate's verdicts
          if ((rc = finish(0))) return rc;
          n_finished = 1;
          if (g_infer_stats[4] * 4 > (long long)cm.used) { k_end = 1; break; }
        }
        if (k + 1 < metas.size() && (rc = enqueue_sample_x(k + 1))) return rc;
        while (n_finished + 2 <= k)
          if ((rc = finish(n_finished++))) return rc;
      }
      while (n_finished < k_end)
        if ((rc = finish(n_finished++))) return rc;
      if ((rc = flush())) return rc;
      if (ovl) {
        DTK_CUDA(cudaEventRecord(ia->join, sb));
        DTK_CUDA(cudaStreamWaitEvent(st, ia->join, 0));
      }
      if (k_end == metas.size()) {
        if (stop_after < 3) return DINOTRK_OK;
        NvtxRange nvd("dinotrk.infer.D.occlusion");
        return dinotrk_occlusion(traj, cos_sims, anchors, N, T, anchor_th, cos_th, occ, stream);
      }
      k0 = k_end;                       // switched: chunks k0.. on the full-map pipeline below (same plan)
      g_infer_stats[3] = 0;
    }
    if (!planned) {
      plan_chunks(1, T, N, cnt.data(), ch, gcap, metas, plan_host);
      int rc0 = upload_plan();
      if (rc0) return rc0;
    }
    int rc = DINOTRK_OK;
    InferAsync* ia = infer_async();
    const bool ovl = ia != nullptr && metas.size() > k0 + 1;
    cudaStream_t sa = (ovl && ia->mode >= 2) ? ia->aux : st;    // head stream
    cudaStream_t sb = ovl ? ia->aux2 : st;   // sampling stream
    if (ovl) {
      DTK_CUDA(cudaEventRecord(ia->fork, st));
      DTK_CUDA(cudaStreamWaitEvent(sa, ia->fork, 0));
      DTK_CUDA(cudaStreamWaitEvent(sb, ia->fork, 0));
    }
    auto enqueue_sample = [&](size_t k) -> int {   // descriptors of chunk k (buffer set k & 1)
      const ChunkMeta& cm = metas[k];
      const ChunkBufs& b = cb[k & 1];
      const Grp gp = grp_of(k);
      if (ovl && k >= k0 + 2) DTK_CUDA(cudaStreamWaitEvent(sb, ia->gemm[k & 1], 0));   // GEMM k-2 read the descriptors of this set
      {
        ProfRange pr(PROF_SAMPLE, sb);
        // the split layout of launch_corr_gemm_tc for desc_rows = used: hi rows, then lo rows at the next 256-byte boundary
        __half* c_hi = tensor ? reinterpret_cast<__half*>(b.split) : nullptr;
        __half* c_lo = tensor ? reinterpret_cast<__half*>(reinterpret_cast<char*>(b.split) + align_up((size_t)cm.used * C * 2, 256))
                              : nullptr;
        sample_anchor_kernel<<<cm.used, SAMPLE_THREADS, 0, sb>>>(tpc, T, C, P, g->h, g->w, pa, traj, d_qlist, N, gp.f, gp.map0,
                                                                gp.item, cm.n_groups, fb, b.desc, b.norm, out_index_ring[k & 3], c_hi, c_lo);
        DTK_LAUNCHED();
      }
      if (ovl) DTK_CUDA(cudaEventRecord(ia->sample[k & 1], sb));
      return DINOTRK_OK;
    };
    // the full-map head of chunk j (usually an empty list) runs on the GEMM stream between two GEMMs: it needs ~70 KB of
    // shared memory per CTA and could not co-reside with a GEMM anyway
    auto head_full = [&](size_t j) -> int {
      const ChunkBufs& b = cb[j & 1];
      if (ovl) DTK_CUDA(cudaStreamWaitEvent(st, ia->head[j & 1], 0));   // fast head of chunk j (its list is complete)
      return launch_head(b.maps, metas[j].used, ms, *g, *hw, out_index_ring[j & 3], anchors, 2, 0, nullptr, b.hscratch, st,
                         tensor ? b.tkeys : nullptr, true, 0, 2);
    };
    if (k0 < metas.size() && (rc = enqueue_sample(k0))) return rc;
    for (size_t k = k0; k < metas.size(); ++k) {
      const ChunkMeta& cm = metas[k];
      const ChunkBufs& b = cb[k & 1];
      const Grp gp = grp_of(k);
      if (ovl) DTK_CUDA(cudaStreamWaitEvent(st, ia->sample[k & 1], 0));
      if (k >= k0 + 2 && (rc = head_full(k - 2))) return rc;   // last reader of maps / keys / list of this buffer set
      CorrAssist as;
      as.tkeys = tensor ? b.tkeys : nullptr; as.zero_word = b.hscratch; as.split_ready = tensor; as.no_thin = cm.no_thin;
      rc = launch_corr_maps(fv, b.desc, cm.used, b.norm, gp.f, gp.r, gp.m, gp.map0, cm.n_groups, cm.used, cm.maxm, b.maps, ms,
                            b.plan, b.split, st, as);
      if (rc) return rc;
      if (ovl) DTK_CUDA(cudaEventRecord(ia->gemm[k & 1], st));
      if (k + 1 < metas.size() && (rc = enqueue_sample(k + 1))) return rc;
      if (ovl) DTK_CUDA(cudaStreamWaitEvent(sa, ia->gemm[k & 1], 0));
      rc = launch_head(b.maps, cm.used, ms, *g, *hw, out_index_ring[k & 3], anchors, 2, 0, nullptr, b.hscratch, sa, as.tkeys, true,
                       (ovl && ia->mode >= 2) ? ia->head_ctas_per_sm : 0, 1);
      if (rc) return rc;
      if (ovl) DTK_CUDA(cudaEventRecord(ia->head[k & 1], sa));
    }
    for (size_t j = std::max(k0, metas.size() >= 2 ? metas.size() - 2 : 0); j < metas.size(); ++j)
      if ((rc = head_full(j))) return rc;
    if (ovl) {
      DTK_CUDA(cudaEventRecord(ia->join, sa));
      DTK_CUDA(cudaStreamWaitEvent(st, ia->join, 0));
    }
  }
  if (stop_after < 3) return DINOTRK_OK;

  // ---- phase D: occlusion --------------------------------------------------------------------------
  NvtxRange nvd("dinotrk.infer.D.occlusion");
  return dinotrk_occlusion(traj, cos_sims, anchors, N, T, anchor_th, cos_th, occ, stream);
}

}  // extern "C"
