// Stage 1: sample points along rays, exact nearest posed-vertex search within the 5 cm cull radius
// (per-sub-cell candidate lists, common.cuh: NnLists; uniform grid, 27-cell neighbourhood where a sub-cell has no list), ordered
// compaction of the survivors.
// Replaces renderer.py:299-321 (sample_stratified, SMPL-space transform, knn_points #1, mask, boolean-index
// compaction).  Index bookkeeping is bit-exact against oracle/port.py (see its header for the rounding order).
#include "common.cuh"

namespace sherf {

// Search the 27-cell neighbourhood of q's cell for the nearest vertex; returns best squared distance and id
// under the lexicographic (d2, id) order = "smallest index wins ties".
__device__ __forceinline__ void nn_27(const GridDesc& g, const int* __restrict__ cell_start, const float4* __restrict__ gv,
                                      float qx, float qy, float qz, int cx, int cy, int cz, float& best, int& best_id) {
  const int x0 = max(cx - 1, 0), x1 = min(cx + 1, g.dim[0] - 1);
  for (int z = max(cz - 1, 0); z <= min(cz + 1, g.dim[2] - 1); ++z) {
    for (int y = max(cy - 1, 0); y <= min(cy + 1, g.dim[1] - 1); ++y) {
      const int row = (z * g.dim[1] + y) * g.dim[0];
      const int b = cell_start[row + x0], e = cell_start[row + x1 + 1];
      for (int k = b; k < e; ++k) {
        const float4 v = gv[k];
        const float d2 = dist2_xyz(qx, qy, qz, v.x, v.y, v.z);
        const int id = __float_as_int(v.w);
        if (d2 < best || (d2 == best && id < best_id)) { best = d2; best_id = id; }
      }
    }
  }
}

// The cull runs in two kernels so that the nearest-vertex search is load balanced: in a one-warp-per-ray formulation only the lanes
// whose sample falls into an occupied cell search (7.6 of 32 on average at 512x512x64, profiles/r1_q), the rest of the warp idles.
//   k_cull_candidates : one warp per ray, lane per sample: depth -> SMPL-space query -> grid cell -> occupancy byte (with lists: the
//                       sub-cell's candidate byte); candidates are appended to a queue (one atomicAdd per warp pass), all others get
//                       vid = -1
//   k_cull_search     : one thread per candidate: exact search over the sub-cell's list (27-cell search without one), 5 cm test,
//                       per-ray survivor count (atomicAdd)
// Candidates of a ray are contiguous in the queue, so neighbouring threads search neighbouring cells (similar trip counts).
// Both kernels derive q with the same exactly-rounded operations, so the result is bit-identical to the single-kernel form.
__device__ __forceinline__ void cull_query(const FrameConst& fc, const float* __restrict__ origins, const float* __restrict__ dirs, int n,
                                           float t, float q[3]) {
  float p[3];
  p[0] = __fsub_rn(mul_add_sep(t, dirs[n * 3], origins[n * 3]), fc.Th_tgt[0]);
  p[1] = __fsub_rn(mul_add_sep(t, dirs[n * 3 + 1], origins[n * 3 + 1]), fc.Th_tgt[1]);
  p[2] = __fsub_rn(mul_add_sep(t, dirs[n * 3 + 2], origins[n * 3 + 2]), fc.Th_tgt[2]);
  rowvec_mat3(p, fc.R_tgt, q);
}

__global__ void __launch_bounds__(256) k_cull_candidates(const float* __restrict__ origins, const float* __restrict__ dirs,
                                                         const float* __restrict__ nearv, const float* __restrict__ farv, int N, int S,
                                                         const FrameConst* __restrict__ fcp, const unsigned char* __restrict__ occ,
                                                         const float* __restrict__ depths, int* __restrict__ sample_vid,
                                                         int* __restrict__ ray_count, int* __restrict__ queue, int* __restrict__ queue_count,
                                                         int write_all, const NnLists nl) {
  __shared__ FrameConst fc;
  for (int i = threadIdx.x; i < (int)(sizeof(FrameConst) / 4); i += blockDim.x) ((int*)&fc)[i] = ((const int*)fcp)[i];
  __syncthreads();
  const int lane = threadIdx.x & 31;
  const int n = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (n >= N) return;
  const float nr = nearv[n], fr = farv[n];
  const GridDesc& g = fc.g1;
  if (lane == 0) ray_count[n] = 0;
  // Conservative parameter interval [t0, t1] in which the ray can be inside the cull grid's box (slab test in SMPL space, box grown by
  // 1 mm to cover the fp32 rounding of the exactly-rounded query below): a sample outside it cannot fall into a grid cell, so it is a
  // non-candidate without transforming it.  ~85 % of the rays of a 512x512 view miss the box altogether; when nobody reads the dense
  // per-sample ids of such rays (no debug taps, no fine pass: k_compact skips rays without survivors) their -1 entries are not even written.
  float t0 = -3.0e38f, t1 = 3.0e38f;
  {
    float po[3] = {origins[n * 3] - fc.Th_tgt[0], origins[n * 3 + 1] - fc.Th_tgt[1], origins[n * 3 + 2] - fc.Th_tgt[2]};
    float pd[3] = {dirs[n * 3], dirs[n * 3 + 1], dirs[n * 3 + 2]}, qo[3], qd[3];
    rowvec_mat3(po, fc.R_tgt, qo);
    rowvec_mat3(pd, fc.R_tgt, qd);
    const float tmag = fmaxf(fabsf(nr), fabsf(fr));
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      const float margin = 1.0e-3f + 1.0e-5f * (fabsf(qo[k]) + tmag * fabsf(qd[k]));
      const float lo = g.origin[k] - margin, hi = g.origin[k] + (float)g.dim[k] * g.cell + margin;
      if (fabsf(qd[k]) < 1.0e-12f) {
        if (qo[k] < lo || qo[k] > hi) { t0 = 1.f; t1 = 0.f; }
      } else {
        const float a = (lo - qo[k]) / qd[k], b = (hi - qo[k]) / qd[k];
        t0 = fmaxf(t0, fminf(a, b));
        t1 = fminf(t1, fmaxf(a, b));
      }
    }
    const float slack = 1.0e-5f * (fabsf(t0) + fabsf(t1)) + 1.0e-6f;
    t0 -= slack; t1 += slack;
  }
  const bool ray_misses = !(t0 <= t1) || t1 < fminf(nr, fr) || t0 > fmaxf(nr, fr);
  if (ray_misses && !write_all && !depths) return;           // stratified depths lie in [near, far]: nothing of this ray can be a candidate
  for (int i0 = 0; i0 < S; i0 += 32) {
    const int i = i0 + lane;
    bool cand = false;
    if (i < S) {
      const float t = depths ? depths[(size_t)n * S + i] : sample_depth(nr, fr, i, S);   // fine pass: importance-sampled depths
      float q[3];
      if (t < t0 || t > t1) { sample_vid[(size_t)n * S + i] = -1; }
      else {
      cull_query(fc, origins, dirs, n, t, q);
      if (nl.cand) {
        // sub-cell byte: 0 for an empty cull list (no vertex within 5 cm of the sub-cell) as for an unoccupied coarse cell
        int cell, sub;
        cand = nnl_cell(g, q[0], q[1], q[2], cell, sub) && nl.cand[cell * kNnlSub3 + sub];
      } else {
        const int cx = grid_coord(q[0], g.origin[0], g.inv_cell, g.dim[0]);
        const int cy = grid_coord(q[1], g.origin[1], g.inv_cell, g.dim[1]);
        const int cz = grid_coord(q[2], g.origin[2], g.inv_cell, g.dim[2]);
        cand = cx >= 0 && cx < g.dim[0] && cy >= 0 && cy < g.dim[1] && cz >= 0 && cz < g.dim[2] && occ[(cz * g.dim[1] + cy) * g.dim[0] + cx];
      }
      if (!cand) sample_vid[(size_t)n * S + i] = -1;
      }
    }
    const unsigned m = __ballot_sync(0xffffffffu, cand);
    if (m) {
      int base = 0;
      if (lane == 0) base = atomicAdd(queue_count, __popc(m));
      base = __shfl_sync(0xffffffffu, base, 0);
      if (cand) queue[base + __popc(m & ((1u << lane) - 1u))] = n * S + i;
    }
  }
}

// (256, 4): without a minimum occupancy ptxas capped the list form at 32 registers and spilled 128 bytes per thread
__global__ void __launch_bounds__(256, 4) k_cull_search(const float* __restrict__ origins, const float* __restrict__ dirs,
                                                     const float* __restrict__ nearv, const float* __restrict__ farv, int S,
                                                     const FrameConst* __restrict__ fcp, const int* __restrict__ cell_start,
                                                     const float4* __restrict__ gv, float thr, const float* __restrict__ depths,
                                                     const int* __restrict__ queue, const int* __restrict__ queue_count,
                                                     int* __restrict__ sample_vid, int* __restrict__ ray_count, const NnLists nl,
                                                     int* __restrict__ cand_out) {
  __shared__ FrameConst fc;
  for (int i = threadIdx.x; i < (int)(sizeof(FrameConst) / 4); i += blockDim.x) ((int*)&fc)[i] = ((const int*)fcp)[i];
  __syncthreads();
  const GridDesc& g = fc.g1;
  const int count = *queue_count;
  if (cand_out && blockIdx.x == 0 && threadIdx.x == 0) *cand_out = count;
  for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < count; j += gridDim.x * blockDim.x) {
    const int s = queue[j];
    const int n = s / S, i = s - n * S;
    const float t = depths ? depths[s] : sample_depth(nearv[n], farv[n], i, S);
    float q[3];
    cull_query(fc, origins, dirs, n, t, q);
    float best = 3.0e38f;
    int bid = 0x7fffffff;
    const float qx = q[0], qy = q[1], qz = q[2];
    const int li = nl.slot ? nnl_index(g, nl.slot, qx, qy, qz) : -1;
    const int ln = li >= 0 ? nl.len[li] : -1;
    if (ln >= 0) {
      const float4* e = nl.ent + (size_t)li * kNnlCap;
      for (int k = 0; k < ln; ++k) {
        const float4 v = e[k];
        const float d2 = dist2_xyz(qx, qy, qz, v.x, v.y, v.z);
        const int id = __float_as_int(v.w);
        if (d2 < best || (d2 == best && id < bid)) { best = d2; bid = id; }
      }
    } else {                                 // no list (occupied cell without a slot, overflowing sub-cell): the grid search
      const int cx = grid_coord(q[0], g.origin[0], g.inv_cell, g.dim[0]);
      const int cy = grid_coord(q[1], g.origin[1], g.inv_cell, g.dim[1]);
      const int cz = grid_coord(q[2], g.origin[2], g.inv_cell, g.dim[2]);
      nn_27(g, cell_start, gv, qx, qy, qz, cx, cy, cz, best, bid);
    }
    const int vid = best < thr ? bid : -1;
    sample_vid[s] = vid;
    if (vid >= 0) atomicAdd(&ray_count[n], 1);
  }
}

// Exclusive scan of ray_count[0..N) -> ray_start[0..N] in two coalesced passes over 1024-ray blocks.
__global__ void __launch_bounds__(1024) k_ray_block_sums(const int* __restrict__ cnt, int N, int* __restrict__ bsum) {
  __shared__ int red[32];
  const int i = blockIdx.x * 1024 + threadIdx.x;
  int v = i < N ? cnt[i] : 0;
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  if (threadIdx.x < 32) {
    int x = red[threadIdx.x];
    for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
    if (threadIdx.x == 0) bsum[blockIdx.x] = x;
  }
}

__global__ void __launch_bounds__(1024) k_scan_rays(const int* __restrict__ cnt, const int* __restrict__ bsum, int nblocks, int N,
                                                    int* __restrict__ start, int64_t* total_out) {
  __shared__ int red[32];
  __shared__ int warp_off[32];
  __shared__ int block_off;
  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  // offset of this block = sum of the preceding block sums (nblocks is small: N / 1024)
  int pre = 0;
  for (int b = tid; b < (int)blockIdx.x; b += 1024) pre += bsum[b];
  for (int o = 16; o > 0; o >>= 1) pre += __shfl_xor_sync(0xffffffffu, pre, o);
  if (lane == 0) red[w] = pre;
  __syncthreads();
  if (tid < 32) {
    int x = red[tid];
    for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
    if (tid == 0) block_off = x;
  }
  __syncthreads();
  const int i = blockIdx.x * 1024 + tid;
  const int v = i < N ? cnt[i] : 0;
  int incl = v;
  for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += t; }
  __syncthreads();
  if (lane == 31) red[w] = incl;
  __syncthreads();
  if (tid < 32) {
    const int x = red[tid];
    int y = x;
    for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(0xffffffffu, y, o); if (tid >= o) y += t; }
    warp_off[tid] = y - x;
  }
  __syncthreads();
  const int excl = block_off + warp_off[w] + incl - v;
  if (i < N) start[i] = excl;
  if (i == N - 1) { start[N] = excl + v; *total_out = excl + v; }
}

// Ordered scatter: point_sample[pos] = n*S+i, point_vid[pos] = vid, pos ascending in row-major sample order.
__global__ void __launch_bounds__(256) k_compact(const int* __restrict__ sample_vid, const int* __restrict__ ray_start, int N, int S,
                                                 int* __restrict__ point_sample, int* __restrict__ point_vid) {
  const int lane = threadIdx.x & 31;
  const int n = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (n >= N) return;
  int pos = ray_start[n];
  if (ray_start[n + 1] == pos) return;
  for (int i0 = 0; i0 < S; i0 += 32) {
    const int i = i0 + lane;
    const int vid = (i < S) ? sample_vid[(size_t)n * S + i] : -1;
    const unsigned m = __ballot_sync(0xffffffffu, vid >= 0);
    if (vid >= 0) {
      const int p = pos + __popc(m & ((1u << lane) - 1u));
      point_sample[p] = n * S + i;
      point_vid[p] = vid;
    }
    pos += __popc(m);
  }
}

int run_exclusive_scan(const int* cnt, int n, int* block_sums, int* start, int64_t* total_dev, cudaStream_t st) {
  const int nb = ceil_div(n, 1024);
  k_ray_block_sums<<<nb, 1024, 0, st>>>(cnt, n, block_sums);
  SHERF_LAUNCH_CHECK();
  k_scan_rays<<<nb, 1024, 0, st>>>(cnt, block_sums, nb, n, start, total_dev);
  SHERF_LAUNCH_CHECK();
  return SHERF_OK;
}

#define RC_SCAN(x) do { int _rc = (x); if (_rc) return _rc; } while (0)

int run_cull(const SherfRays& rays, int S, const float* depths, const FrameTables& ft, int* sample_vid, int* ray_count, int* block_sums,
             int* ray_start, int64_t* total_dev, int* point_sample, int* point_vid, cudaStream_t st, int write_all) {
  const int N = rays.n_rays;
  const float thr = (float)(0.05 * 0.05);        // `distance < 0.05 ** 2` compares in fp32 (renderer.py:318-319)
  // candidate queue = point_sample (written by k_compact only after the search), its counter = the first word of total_dev
  int* queue = point_sample;
  int* queue_count = reinterpret_cast<int*>(total_dev);
  SHERF_CUDA_OK(cudaMemsetAsync(queue_count, 0, sizeof(int), st));
  k_cull_candidates<<<ceil_div(N, 8), 256, 0, st>>>(rays.origins, rays.dirs, rays.near_, rays.far_, N, S, ft.fc, ft.g1_occ, depths,
                                                    sample_vid, ray_count, queue, queue_count, write_all, ft.lists(0));
  SHERF_LAUNCH_CHECK();
  k_cull_search<<<148 * 8, 256, 0, st>>>(rays.origins, rays.dirs, rays.near_, rays.far_, S, ft.fc, ft.g1_cell_start, ft.g1_verts, thr, depths,
                                         queue, queue_count, sample_vid, ray_count, ft.lists(0), ft.nnl_on ? ft.nnl_count + 2 : nullptr);
  SHERF_LAUNCH_CHECK();
  RC_SCAN(run_exclusive_scan(ray_count, N, block_sums, ray_start, total_dev, st));
  k_compact<<<ceil_div(N, 8), 256, 0, st>>>(sample_vid, ray_start, N, S, point_sample, point_vid);
  SHERF_LAUNCH_CHECK();
  return SHERF_OK;
}

}  // namespace sherf
