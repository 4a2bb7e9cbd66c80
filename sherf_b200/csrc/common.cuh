// Shared device/host definitions of the sherf_b200 render path (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stddef.h>
#include <string.h>
#include "../../include/sherf_b200.h"

namespace sherf {

constexpr int kJoints = 24;
constexpr int kPoseFeat = 207;          // 23 * 9
constexpr float kPi2 = 1.57079632679489661923f;   // torch.pi * 0.5 rounded to fp32 (renderer.py:897)

// Uniform grid over a vertex set (exact K=1 NN search; replaces pytorch3d knn_points call sites
// renderer.py:315,564,627).  Cell linear index = (z*dim[1] + y)*dim[0] + x.
struct GridDesc {
  float origin[3];
  float inv_cell;
  float cell;
  int dim[3];
  int ncell;
};

// Candidate lists of the exact nearest-vertex searches.  Every coarse cell that has a vertex in its 27-neighbourhood gets a slot (up to
// kNnlSlots per grid); each of its kNnlSub^3 sub-cells B holds up to kNnlCap vertices: every v with dmin(B, v) <= U(B) = d(centre(B), v*)
// + half-diagonal(B) for a vertex v* near the centre (and, in the cull grid, dmin(B, v) < 5 cm), both with a conservative slack.  The
// nearest vertex of any q in B and every vertex tied with it satisfy that test, so the lexicographic (d2, id) minimum over the list is
// the global one.  Queries without a list (no slot, more than the capacity) take the grid search.
constexpr int kNnlSub = 2;
constexpr int kNnlSub3 = kNnlSub * kNnlSub * kNnlSub;
constexpr int kNnlCap = 64;
constexpr int kNnlSlots = 6144;

struct NnLists {
  const int* slot;      // [maxcell] coarse cell -> slot; -1: no vertex in its 27-neighbourhood, -2: occupied but no slot left
  const int* len;       // [kNnlSlots * kNnlSub3] list length of a sub-cell, -1: more than the capacity
  const float4* ent;    // [kNnlSlots * kNnlSub3][kNnlCap] (x, y, z, id bits)
  const unsigned char* cand;   // cull grid only, [maxcell * kNnlSub3]: 0 = an empty list or no vertex in the 27-neighbourhood
};

// Coarse cell (grid_coord's) and sub-cell of q; false outside the grid.  The sub-cell is the fractional part of the same grid
// coordinate (t - floor(t) and the power-of-two scale are exact), so q lies in the sub-cell up to the rounding of t.
__device__ __forceinline__ bool nnl_cell(const GridDesc& g, float qx, float qy, float qz, int& cell, int& sub) {
  const float tx = (qx - g.origin[0]) * g.inv_cell, ty = (qy - g.origin[1]) * g.inv_cell, tz = (qz - g.origin[2]) * g.inv_cell;
  const int cx = (int)floorf(tx), cy = (int)floorf(ty), cz = (int)floorf(tz);
  if (cx < 0 || cx >= g.dim[0] || cy < 0 || cy >= g.dim[1] || cz < 0 || cz >= g.dim[2]) return false;
  cell = (cz * g.dim[1] + cy) * g.dim[0] + cx;
  const int sx = min((int)((tx - (float)cx) * (float)kNnlSub), kNnlSub - 1);
  const int sy = min((int)((ty - (float)cy) * (float)kNnlSub), kNnlSub - 1);
  const int sz = min((int)((tz - (float)cz) * (float)kNnlSub), kNnlSub - 1);
  sub = (sz * kNnlSub + sy) * kNnlSub + sx;
  return true;
}

// List index (slot * kNnlSub3 + sub-cell) of the sub-cell that holds q, or -1 (q outside the grid), -2 (no vertex in the coarse cell's
// 27-neighbourhood), -3 (occupied coarse cell without a slot)
__device__ __forceinline__ int nnl_index(const GridDesc& g, const int* __restrict__ slot, float qx, float qy, float qz) {
  int cell, sub;
  if (!nnl_cell(g, qx, qy, qz, cell, sub)) return -1;
  const int sl = slot[cell];
  return sl < 0 ? sl - 1 : sl * kNnlSub3 + sub;
}

// Per-vertex piecewise-affine warp record.  Blend weights come from the single nearest vertex
// (renderer.py:565,628), so the blended LBS matrices depend on the vertex id only.
//   p  = Rinv * (p - t);  d = Rinv * d
//   p  = p + s0*off0;  p = p + s1*off1;  p = p + s2*off2      (applied in this order)
//   p  = Af_R * p + Af_t;  d = Af_R * d
struct __align__(16) VertexWarp {
  float Rinv[9];
  float t[3];
  float off0[3];
  float off1[3];
  float off2[3];
  float Af[12];      // rows of the forward 3x4
  float pad[3];
};
static_assert(sizeof(VertexWarp) == 36 * 4, "VertexWarp must be 144 B");

struct FrameConst {
  float R_tgt[9], Th_tgt[3];        // input_data['params'] R, Th          renderer.py:307-308
  float Rinv_obs[9], Th_obs[3];     // inverse(obs R), obs Th              renderer.py:681-682
  float camR[9], camT[3], camK[9];  // observation camera                  renderer.py:686-699
  float twb_min[3], twb_max[3];     // t_world_bounds                      renderer.py:239
  float spb_min[3];                 // obs_sp_input['bounds'][0,0]         renderer.py:548
  float out_sh[3];                  // z,y,x as floats                     renderer.py:552
  GridDesc g1, g3;
  int dmin_bits, dmax_bits;         // ordered-int encodings of the global depth clamp range
  float dmin, dmax;
};

__host__ __device__ inline int float_to_ordered(float f) {
#ifdef __CUDA_ARCH__
  int i = __float_as_int(f);
#else
  int i; memcpy(&i, &f, 4);
#endif
  return i >= 0 ? i : i ^ 0x7fffffff;
}
__device__ inline float ordered_to_float(int i) { return __int_as_float(i >= 0 ? i : i ^ 0x7fffffff); }

// ---- exactly-rounded building blocks for the index bookkeeping (see oracle/port.py header) ----
__device__ __forceinline__ float sample_depth(float nearv, float farv, int i, int S) {
  float step = __fdiv_rn((float)i, (float)(S - 1));                       // math_utils.py:107
  return __fadd_rn(nearv, __fmul_rn(step, __fsub_rn(farv, nearv)));       // math_utils.py:116
}
__device__ __forceinline__ float mul_add_sep(float a, float b, float c) { // fl(c + fl(a*b)), no contraction
  return __fadd_rn(c, __fmul_rn(a, b));
}
// row-vector times 3x3 (row-major M), k-ordered FMA chain = what torch's CPU sgemm does for K=3
__device__ __forceinline__ void rowvec_mat3(const float p[3], const float* __restrict__ M, float out[3]) {
#pragma unroll
  for (int j = 0; j < 3; ++j)
    out[j] = __fmaf_rn(p[2], M[6 + j], __fmaf_rn(p[1], M[3 + j], __fmul_rn(p[0], M[j])));
}
__device__ __forceinline__ float dist2_xyz(float qx, float qy, float qz, float vx, float vy, float vz) {
  float dx = __fsub_rn(qx, vx), dy = __fsub_rn(qy, vy), dz = __fsub_rn(qz, vz);
  return __fadd_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)), __fmul_rn(dz, dz));
}
__device__ __forceinline__ int grid_coord(float x, float origin, float inv_cell, int dim) {
  int c = (int)floorf((x - origin) * inv_cell);
  return c;   // may be outside [0,dim)
}

__device__ __forceinline__ void mat3_vec(const float* __restrict__ M, const float v[3], float out[3]) {
#pragma unroll
  for (int i = 0; i < 3; ++i) out[i] = M[3 * i] * v[0] + M[3 * i + 1] * v[1] + M[3 * i + 2] * v[2];
}

// launch accounting / errors (host)
struct LaunchCounter { int64_t n = 0; };
extern thread_local LaunchCounter g_launches;
void set_error(const char* fmt, ...);
// true while the host-side weight plans are being rebuilt for blobs that are already packed in the arena (no pack kernel is launched)
extern thread_local bool g_pack_plan_only;

#define SHERF_CUDA_OK(expr)                                                              \
  do {                                                                                   \
    cudaError_t _e = (expr);                                                             \
    if (_e != cudaSuccess) {                                                             \
      ::sherf::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
      return SHERF_E_CUDA;                                                               \
    }                                                                                    \
  } while (0)

#define SHERF_LAUNCH_CHECK()                                                             \
  do {                                                                                   \
    ::sherf::g_launches.n++;                                                             \
    cudaError_t _e = cudaGetLastError();                                                 \
    if (_e != cudaSuccess) {                                                             \
      ::sherf::set_error("kernel launch failed: %s (%s:%d)", cudaGetErrorString(_e), __FILE__, __LINE__); \
      return SHERF_E_CUDA;                                                               \
    }                                                                                    \
  } while (0)

inline int ceil_div(int64_t a, int64_t b) { return (int)((a + b - 1) / b); }

// ---- stage entry points (defined in the .cu files) ----
struct FrameTables {           // device pointers carved out of the scratch arena
  FrameConst* fc;
  float* A;                    // [3][24][16] target, canonical, obs LBS transforms
  float* joints;               // [3][24][3]
  float* posefeat;             // [3][207]
  float* poff;                 // [3][V][3] pose offsets (target, canonical, obs)
  float* soff;                 // [2][V][3] shape offsets (target shapes, obs shapes)
  float* verts_smpl;           // [V][3]
  VertexWarp* T1;              // [V] target -> canonical
  VertexWarp* T3;              // [V] canonical -> observation (SMPL space)
  int* g1_cell_start;          // [maxcell+1]
  int* g3_cell_start;
  int* g_cursor;               // [2][maxcell] per-cell vertex counts (histogram, then scatter cursors)
  int* g_block_sums;           // [2][maxcell/1024 + 2] scan scratch, one per grid (the grids are built on different streams)
  int64_t* g_total;            // [2] scan totals (unused)
  float4* g1_verts;            // [V] (x,y,z,id bits) sorted by cell
  float4* g3_verts;
  unsigned char* g1_occ;       // [maxcell] 27-neighbourhood occupancy
  int maxcell;
  // candidate lists of the cull grid (0) and of the canonical grid (1); nnl_on = 0 (or null buffers): the grid searches only
  int nnl_on;
  int nnl_cap;                 // list capacity used by the build (<= kNnlCap)
  int* nnl_slot[2];            // [maxcell]
  int* nnl_slot_cell[2];       // [kNnlSlots] slot -> coarse cell
  int* nnl_count;              // [4] slots taken per grid, cull candidates of the last cull
  int* nnl_len[2];             // [kNnlSlots * kNnlSub3]
  float4* nnl_ent[2];          // [kNnlSlots * kNnlSub3 * kNnlCap]
  unsigned char* nnl_cand;     // [maxcell * kNnlSub3] candidate byte per sub-cell of the cull grid
  NnLists lists(int g) const {
    return nnl_on ? NnLists{nnl_slot[g], nnl_len[g], nnl_ent[g], g == 0 ? nnl_cand : nullptr} : NnLists{nullptr, nullptr, nullptr, nullptr};
  }
};
// SHERF_NN_LEGACY=1: grid searches only; SHERF_NN_LIST_CAP=k: list capacity k (1..kNnlCap), read on every call
bool nn_lists_enabled();
int nn_list_cap();

int run_prologue_frame(const SherfFrame& frame, const FrameTables& ft, cudaStream_t st);
int run_prologue_cull(const SherfSmplModel& smpl, const SherfFrame& frame, const SherfRays& rays, const SherfOptions& opts,
                      const FrameTables& ft, cudaStream_t st);
int run_prologue_tables(const SherfSmplModel& smpl, const SherfFrame& frame, const FrameTables& ft, cudaStream_t st);
int run_lbs_only(const SherfSmplModel& smpl, const SherfPose& pose, float* A_out, float* joints_tmp, float* pf_tmp, cudaStream_t st);
int run_depth_range(const SherfRays& rays, FrameConst* fc, cudaStream_t st);
// exclusive scan of cnt[0..n) -> start[0..n] (start[n] = total, also written to *total_dev); block_sums: n/1024 + 2 ints of scratch
int run_exclusive_scan(const int* cnt, int n, int* block_sums, int* start, int64_t* total_dev, cudaStream_t st);

}  // namespace sherf
