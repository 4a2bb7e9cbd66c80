// Per-frame prologue: SMPL kinematic chain, pose/shape offsets, per-vertex warp tables, uniform
// grids for the exact nearest-vertex searches, global depth range.  O(V) + O(N) work, a few tiny
// kernels per frame.  Replaces renderer.py:76-157 (called 4x per forward by the reference) and the
// per-point blend / inverse / offset gathers of renderer.py:565-615 and :628-682 by per-VERTEX tables.
#include "common.cuh"
#include <limits.h>

namespace sherf {

// ---------------------------------------------------------------------------------------------
// joints[s][j] = J_regressor[j] . (v_template + shapedirs . beta_s)        renderer.py:138,146
__global__ void k_joints(const float* __restrict__ vt, const float* __restrict__ sd, const float* __restrict__ jr,
                         const float* __restrict__ b0, const float* __restrict__ b1, const float* __restrict__ b2,
                         int V, float* __restrict__ joints) {
  const int j = blockIdx.x, s = blockIdx.y;
  const float* beta = s == 0 ? b0 : (s == 1 ? b1 : b2);
  float b[10];
#pragma unroll
  for (int k = 0; k < 10; ++k) b[k] = beta[k];
  float acc[3] = {0.f, 0.f, 0.f};
  for (int v = threadIdx.x; v < V; v += blockDim.x) {
    float w = jr[(size_t)j * V + v];
    if (w != 0.f) {
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        const float* row = sd + ((size_t)v * 3 + c) * 10;
        float off = 0.f;
#pragma unroll
        for (int k = 0; k < 10; ++k) off += row[k] * b[k];
        acc[c] += w * (vt[v * 3 + c] + off);
      }
    }
  }
  __shared__ float red[3][32];
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    float x = acc[c];
    for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
    if ((threadIdx.x & 31) == 0) red[c][threadIdx.x >> 5] = x;
  }
  __syncthreads();
  if (threadIdx.x < 3) {
    float x = 0.f;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) x += red[threadIdx.x][w];
    joints[(s * kJoints + j) * 3 + threadIdx.x] = x;
  }
}

struct Parents { int p[kJoints]; };

// Rodrigues + kinematic chain -> A[s][24][16], pose feature pf[s][207].   renderer.py:76-126, :582-583
__global__ void k_chain(const float* __restrict__ p0, const float* __restrict__ p1, const float* __restrict__ p2,
                        const float* __restrict__ joints, Parents par, float* __restrict__ A, float* __restrict__ pf) {
  const int s = blockIdx.x, j = threadIdx.x;
  const float* poses = s == 0 ? p0 : (s == 1 ? p1 : p2);
  __shared__ float loc[kJoints][12];
  __shared__ float wor[kJoints][12];
  const float* jt = joints + s * kJoints * 3;
  if (j < kJoints) {
    float rx = poses[3 * j], ry = poses[3 * j + 1], rz = poses[3 * j + 2];
    float ax = rx + 1e-8f, ay = ry + 1e-8f, az = rz + 1e-8f;
    float angle = sqrtf(ax * ax + ay * ay + az * az);
    float kx = rx / angle, ky = ry / angle, kz = rz / angle;
    float c = cosf(angle), sn = sinf(angle);
    float K[9] = {0.f, -kz, ky, kz, 0.f, -kx, -ky, kx, 0.f};
    float KK[9];
#pragma unroll
    for (int r = 0; r < 3; ++r)
#pragma unroll
      for (int q = 0; q < 3; ++q) KK[r * 3 + q] = K[r * 3] * K[q] + K[r * 3 + 1] * K[3 + q] + K[r * 3 + 2] * K[6 + q];
    float R[9];
#pragma unroll
    for (int e = 0; e < 9; ++e) R[e] = ((e % 4 == 0) ? 1.f : 0.f) + sn * K[e] + (1.f - c) * KK[e];
    int pj = par.p[j];
#pragma unroll
    for (int r = 0; r < 3; ++r) {
      loc[j][r * 4 + 0] = R[r * 3 + 0];
      loc[j][r * 4 + 1] = R[r * 3 + 1];
      loc[j][r * 4 + 2] = R[r * 3 + 2];
      loc[j][r * 4 + 3] = (j == 0) ? jt[r] : (jt[j * 3 + r] - jt[pj * 3 + r]);
    }
    if (j >= 1) {
#pragma unroll
      for (int e = 0; e < 9; ++e) pf[s * kPoseFeat + (j - 1) * 9 + e] = R[e] - ((e % 4 == 0) ? 1.f : 0.f);
    }
  }
  __syncthreads();
  if (j == 0) {
    for (int e = 0; e < 12; ++e) wor[0][e] = loc[0][e];
    for (int i = 1; i < kJoints; ++i) {
      const float* P = wor[par.p[i]];
      const float* L = loc[i];
      for (int r = 0; r < 3; ++r) {
        for (int q = 0; q < 4; ++q) {
          float x = P[r * 4] * L[q] + P[r * 4 + 1] * L[4 + q] + P[r * 4 + 2] * L[8 + q];
          if (q == 3) x += P[r * 4 + 3];
          wor[i][r * 4 + q] = x;
        }
      }
    }
  }
  __syncthreads();
  if (j < kJoints) {
    float* out = A + (s * kJoints + j) * 16;
#pragma unroll
    for (int r = 0; r < 3; ++r) {
      float rel = wor[j][r * 4] * jt[j * 3] + wor[j][r * 4 + 1] * jt[j * 3 + 1] + wor[j][r * 4 + 2] * jt[j * 3 + 2];
      out[r * 4 + 0] = wor[j][r * 4 + 0];
      out[r * 4 + 1] = wor[j][r * 4 + 1];
      out[r * 4 + 2] = wor[j][r * 4 + 2];
      out[r * 4 + 3] = wor[j][r * 4 + 3] - rel;
    }
    out[12] = 0.f; out[13] = 0.f; out[14] = 0.f; out[15] = 1.f;
  }
}

// poff[s][row] = posedirs[row,:] . pf[s];  soff[{0,1}][row] = shapedirs[row,:] . beta_{target,obs}
// one warp per row (row = v*3+c).                                  renderer.py:584,591,602,652,658,668
__global__ void k_offsets(const float* __restrict__ posedirs, const float* __restrict__ shapedirs,
                          const float* __restrict__ pf, const float* __restrict__ beta_t, const float* __restrict__ beta_o,
                          int rows, float* __restrict__ poff, float* __restrict__ soff) {
  __shared__ float spf[3 * kPoseFeat];
  for (int i = threadIdx.x; i < 3 * kPoseFeat; i += blockDim.x) spf[i] = pf[i];
  __syncthreads();
  const int lane = threadIdx.x & 31;
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= rows) return;
  const float* pr = posedirs + (size_t)row * kPoseFeat;
  float a0 = 0.f, a1 = 0.f, a2 = 0.f;
  for (int k = lane; k < kPoseFeat; k += 32) {
    float x = pr[k];
    a0 += x * spf[k];
    a1 += x * spf[kPoseFeat + k];
    a2 += x * spf[2 * kPoseFeat + k];
  }
  float s0 = 0.f, s1 = 0.f;
  if (lane < 10) {
    float x = shapedirs[(size_t)row * 10 + lane];
    s0 = x * beta_t[lane];
    s1 = x * beta_o[lane];
  }
  for (int o = 16; o > 0; o >>= 1) {
    a0 += __shfl_xor_sync(0xffffffffu, a0, o);
    a1 += __shfl_xor_sync(0xffffffffu, a1, o);
    a2 += __shfl_xor_sync(0xffffffffu, a2, o);
    s0 += __shfl_xor_sync(0xffffffffu, s0, o);
    s1 += __shfl_xor_sync(0xffffffffu, s1, o);
  }
  if (lane == 0) {
    poff[row] = a0;
    poff[rows + row] = a1;
    poff[2 * rows + row] = a2;
    soff[row] = s0;
    soff[rows + row] = s1;
  }
}

__device__ inline void inv3(const float* m, float* o) {
  float a = m[0], b = m[1], c = m[2], d = m[3], e = m[4], f = m[5], g = m[6], h = m[7], i = m[8];
  float A = e * i - f * h, B = -(d * i - f * g), C = d * h - e * g;
  float det = a * A + b * B + c * C;
  float r = 1.f / det;
  o[0] = A * r; o[1] = -(b * i - c * h) * r; o[2] = (b * f - c * e) * r;
  o[3] = B * r; o[4] = (a * i - c * g) * r;  o[5] = -(a * f - c * d) * r;
  o[6] = C * r; o[7] = -(a * h - b * g) * r; o[8] = (a * e - b * d) * r;
}

__global__ void k_frame_const(SherfFrame fr, float3 out_sh, FrameConst* fc) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  for (int e = 0; e < 9; ++e) { fc->R_tgt[e] = fr.target.R[e]; fc->camR[e] = fr.obs_R[e]; fc->camK[e] = fr.obs_K[e]; }
  float ro[9];
  for (int e = 0; e < 9; ++e) ro[e] = fr.obs.R[e];
  inv3(ro, fc->Rinv_obs);
  for (int e = 0; e < 3; ++e) {
    fc->Th_tgt[e] = fr.target.Th[e];
    fc->Th_obs[e] = fr.obs.Th[e];
    fc->camT[e] = fr.obs_T[e];
    fc->twb_min[e] = fr.t_world_bounds[e];
    fc->twb_max[e] = fr.t_world_bounds[3 + e];
    fc->spb_min[e] = fr.sp_bounds[e];
  }
  fc->out_sh[0] = out_sh.x; fc->out_sh[1] = out_sh.y; fc->out_sh[2] = out_sh.z;
  fc->dmin_bits = INT_MAX;
  fc->dmax_bits = INT_MIN;
}

// thread per vertex: blend the 24 rigid transforms with the vertex's skinning weights, invert,
// and store both warp records; also the posed vertices in SMPL space (bit-exact, renderer.py:314).
__global__ void k_vertex_tables(const float* __restrict__ weights, const float* __restrict__ A, const float* __restrict__ poff,
                                const float* __restrict__ soff, const float* __restrict__ vertices, const FrameConst* __restrict__ fc,
                                int V, VertexWarp* __restrict__ T1, VertexWarp* __restrict__ T3, float* __restrict__ verts_smpl) {
  __shared__ float sA[3 * kJoints * 12];
  for (int i = threadIdx.x; i < 3 * kJoints * 12; i += blockDim.x) sA[i] = A[(i / 12) * 16 + (i % 12)];
  __syncthreads();
  const int v = blockIdx.x * blockDim.x + threadIdx.x;
  if (v >= V) return;
  float w[kJoints];
  float wsum = 0.f;
#pragma unroll
  for (int j = 0; j < kJoints; ++j) { w[j] = weights[(size_t)v * kJoints + j]; wsum += w[j]; }
  const int rows = 3 * V;
  // ---- T1: target -> canonical (renderer.py:565-615) ----
  {
    float At[12], Ab[12];
#pragma unroll
    for (int e = 0; e < 12; ++e) { At[e] = 0.f; Ab[e] = 0.f; }
#pragma unroll
    for (int j = 0; j < kJoints; ++j)
#pragma unroll
      for (int e = 0; e < 12; ++e) { At[e] += w[j] * sA[(0 * kJoints + j) * 12 + e]; Ab[e] += w[j] * sA[(1 * kJoints + j) * 12 + e]; }
    VertexWarp r;
    float R3[9] = {At[0], At[1], At[2], At[4], At[5], At[6], At[8], At[9], At[10]};
    inv3(R3, r.Rinv);
    r.t[0] = At[3]; r.t[1] = At[7]; r.t[2] = At[11];
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      r.off0[c] = -poff[0 * rows + v * 3 + c];
      r.off1[c] = -soff[0 * rows + v * 3 + c];
      r.off2[c] = poff[1 * rows + v * 3 + c];
    }
#pragma unroll
    for (int e = 0; e < 12; ++e) r.Af[e] = Ab[e];
    r.pad[0] = r.pad[1] = r.pad[2] = 0.f;
    T1[v] = r;
  }
  // ---- T3: canonical -> observation pose, renormalised weights (renderer.py:628-678) ----
  {
    float Ab[12], Ao[12];
#pragma unroll
    for (int e = 0; e < 12; ++e) { Ab[e] = 0.f; Ao[e] = 0.f; }
#pragma unroll
    for (int j = 0; j < kJoints; ++j) {
      float wn = w[j] / wsum;
#pragma unroll
      for (int e = 0; e < 12; ++e) { Ab[e] += wn * sA[(1 * kJoints + j) * 12 + e]; Ao[e] += wn * sA[(2 * kJoints + j) * 12 + e]; }
    }
    VertexWarp r;
    float R3[9] = {Ab[0], Ab[1], Ab[2], Ab[4], Ab[5], Ab[6], Ab[8], Ab[9], Ab[10]};
    inv3(R3, r.Rinv);
    r.t[0] = Ab[3]; r.t[1] = Ab[7]; r.t[2] = Ab[11];
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      r.off0[c] = -poff[1 * rows + v * 3 + c];
      r.off1[c] = soff[1 * rows + v * 3 + c];
      r.off2[c] = poff[2 * rows + v * 3 + c];
    }
#pragma unroll
    for (int e = 0; e < 12; ++e) r.Af[e] = Ao[e];
    r.pad[0] = r.pad[1] = r.pad[2] = 0.f;
    T3[v] = r;
  }
  if (verts_smpl) {
    float p[3], o[3];
#pragma unroll
    for (int c = 0; c < 3; ++c) p[c] = __fsub_rn(vertices[v * 3 + c], fc->Th_tgt[c]);
    rowvec_mat3(p, fc->R_tgt, o);
    verts_smpl[v * 3 + 0] = o[0]; verts_smpl[v * 3 + 1] = o[1]; verts_smpl[v * 3 + 2] = o[2];
  }
}

// posed vertices in SMPL space, (vertices - Th) @ R (bit-exact, renderer.py:314): all the cull needs from the body
__global__ void __launch_bounds__(256) k_verts_smpl(const float* __restrict__ vertices, const FrameConst* __restrict__ fc, int V,
                                                    float* __restrict__ verts_smpl) {
  const int v = blockIdx.x * blockDim.x + threadIdx.x;
  if (v >= V) return;
  float p[3], o[3];
#pragma unroll
  for (int c = 0; c < 3; ++c) p[c] = __fsub_rn(vertices[v * 3 + c], fc->Th_tgt[c]);
  rowvec_mat3(p, fc->R_tgt, o);
  verts_smpl[v * 3 + 0] = o[0]; verts_smpl[v * 3 + 1] = o[1]; verts_smpl[v * 3 + 2] = o[2];
}

// ---------------------------------------------------------------------------------------------
// Uniform grids over the posed (g = 0, cell >= cull radius) and the canonical (g = 1) vertices: bbox -> cell size -> counting sort
// of the vertices by cell -> 27-neighbourhood occupancy bytes for the cull grid.  Five small kernels instead of one block per
// grid: the single-block form spent 190 us (profiles/r1_q: 55 % of its stalls on the 27 byte stores per vertex of the dilation,
// the rest on serial passes over the cells by one SM) on the critical path in front of the cull.
__global__ void __launch_bounds__(1024) k_grid_setup(const float* __restrict__ verts_smpl, const float* __restrict__ t_vertices, int V,
                                                      int maxcell, float min_cell, FrameConst* fc, int g0, int* nslots) {
  const int g = g0 + blockIdx.x;
  if (nslots && threadIdx.x == 0) nslots[g] = 0;              // list slots of this grid are counted by k_grid_occupancy
  const float* P = g == 0 ? verts_smpl : t_vertices;
  GridDesc* gd = g == 0 ? &fc->g1 : &fc->g3;
  const int tid = threadIdx.x, nt = blockDim.x;
  __shared__ float smin[3][32], smax[3][32];
  float mn[3] = {3.0e38f, 3.0e38f, 3.0e38f}, mx[3] = {-3.0e38f, -3.0e38f, -3.0e38f};
  for (int v = tid; v < V; v += nt)
#pragma unroll
    for (int c = 0; c < 3; ++c) { float x = P[v * 3 + c]; mn[c] = fminf(mn[c], x); mx[c] = fmaxf(mx[c], x); }
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    for (int o = 16; o > 0; o >>= 1) {
      mn[c] = fminf(mn[c], __shfl_xor_sync(0xffffffffu, mn[c], o));
      mx[c] = fmaxf(mx[c], __shfl_xor_sync(0xffffffffu, mx[c], o));
    }
    if ((tid & 31) == 0) { smin[c][tid >> 5] = mn[c]; smax[c][tid >> 5] = mx[c]; }
  }
  __syncthreads();
  if (tid == 0) {
    GridDesc sg;
    float lo[3], hi[3];
    for (int c = 0; c < 3; ++c) {
      lo[c] = smin[c][0]; hi[c] = smax[c][0];
      for (int w = 1; w < nt / 32; ++w) { lo[c] = fminf(lo[c], smin[c][w]); hi[c] = fmaxf(hi[c], smax[c][w]); }
    }
    float cell = min_cell;
    int d[3];
    for (int it = 0; it < 64; ++it) {
      long long n = 1;
      for (int c = 0; c < 3; ++c) { d[c] = (int)floorf((hi[c] - lo[c]) / cell) + 3; n *= d[c]; }   // one pad cell each side
      if (n <= maxcell) break;
      cell *= 1.1f;
    }
    for (int c = 0; c < 3; ++c) { sg.origin[c] = lo[c] - cell; sg.dim[c] = d[c]; }
    sg.cell = cell;
    sg.inv_cell = 1.f / cell;
    sg.ncell = d[0] * d[1] * d[2];
    *gd = sg;
  }
}

__device__ __forceinline__ int vertex_cell(const GridDesc& sg, float x, float y, float z) {
  const int cx = min(max(grid_coord(x, sg.origin[0], sg.inv_cell, sg.dim[0]), 0), sg.dim[0] - 1);
  const int cy = min(max(grid_coord(y, sg.origin[1], sg.inv_cell, sg.dim[1]), 0), sg.dim[1] - 1);
  const int cz = min(max(grid_coord(z, sg.origin[2], sg.inv_cell, sg.dim[2]), 0), sg.dim[2] - 1);
  return (cz * sg.dim[1] + cy) * sg.dim[0] + cx;
}

// histogram of the vertices over the cells; blockIdx.y selects the grid.  counts: [2][maxcell], zeroed by the caller
__global__ void __launch_bounds__(256) k_grid_count(const float* __restrict__ verts_smpl, const float* __restrict__ t_vertices, int V,
                                                    const FrameConst* __restrict__ fc, int* __restrict__ counts, int maxcell, int g0) {
  const int g = g0 + blockIdx.y, v = blockIdx.x * blockDim.x + threadIdx.x;
  if (v >= V) return;
  const float* P = g == 0 ? verts_smpl : t_vertices;
  const GridDesc sg = g == 0 ? fc->g1 : fc->g3;
  atomicAdd(&counts[(size_t)g * maxcell + vertex_cell(sg, P[v * 3], P[v * 3 + 1], P[v * 3 + 2])], 1);
}

// counting-sort scatter: the order of the vertices inside a cell is arbitrary, which the searches do not depend on (they take the
// lexicographic minimum of (d2, id))
__global__ void __launch_bounds__(256) k_grid_scatter(const float* __restrict__ verts_smpl, const float* __restrict__ t_vertices, int V,
                                                      const FrameConst* __restrict__ fc, int* __restrict__ counts, int maxcell,
                                                      const int* __restrict__ g1_start, const int* __restrict__ g3_start,
                                                      float4* __restrict__ g1_verts, float4* __restrict__ g3_verts, int g0) {
  const int g = g0 + blockIdx.y, v = blockIdx.x * blockDim.x + threadIdx.x;
  if (v >= V) return;
  const float* P = g == 0 ? verts_smpl : t_vertices;
  const GridDesc sg = g == 0 ? fc->g1 : fc->g3;
  const float x = P[v * 3], y = P[v * 3 + 1], z = P[v * 3 + 2];
  const int cell = vertex_cell(sg, x, y, z);
  const int pos = (g == 0 ? g1_start : g3_start)[cell] + atomicSub(&counts[(size_t)g * maxcell + cell], 1) - 1;
  (g == 0 ? g1_verts : g3_verts)[pos] = make_float4(x, y, z, __int_as_float(v));
}

// occupancy of a cell = "some vertex lies in its 27-neighbourhood" (cells of a row are contiguous in cell_start): the cull grid's byte
// and, when the candidate lists are built, the list slot of the cell (nnl_slot / nnl_slot_cell, counted in *nslots, one atomic per warp)
// and the cull grid's sub-cell candidate bytes (1 for every sub-cell of an occupied cell; k_nnl_build clears those with empty lists)
__global__ void __launch_bounds__(256) k_grid_occupancy(const FrameConst* __restrict__ fc, int g, const int* __restrict__ start,
                                                        unsigned char* __restrict__ occ, int* __restrict__ slot, int* __restrict__ slot_cell,
                                                        int* __restrict__ nslots, unsigned char* __restrict__ cand) {
  const GridDesc sg = g == 0 ? fc->g1 : fc->g3;
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= sg.ncell) return;
  const int x = c % sg.dim[0], t = c / sg.dim[0], y = t % sg.dim[1], z = t / sg.dim[1];
  const int x0 = max(x - 1, 0), x1 = min(x + 1, sg.dim[0] - 1);
  bool any = false;
  for (int zz = max(z - 1, 0); zz <= min(z + 1, sg.dim[2] - 1); ++zz)
    for (int yy = max(y - 1, 0); yy <= min(y + 1, sg.dim[1] - 1); ++yy) {
      const int row = (zz * sg.dim[1] + yy) * sg.dim[0];
      any |= start[row + x1 + 1] > start[row + x0];
    }
  if (occ) occ[c] = any ? 1 : 0;
  if (cand) *reinterpret_cast<uint2*>(cand + (size_t)c * kNnlSub3) = any ? make_uint2(0x01010101u, 0x01010101u) : make_uint2(0u, 0u);
  if (slot) {
    const unsigned act = __activemask(), m = __ballot_sync(act, any);
    const int lane = threadIdx.x & 31, leader = __ffs(act) - 1;
    int base = 0;
    if (lane == leader && m) base = atomicAdd(nslots, __popc(m));
    base = __shfl_sync(act, base, leader);
    int s = -1;
    if (any) {
      s = base + __popc(m & ((1u << lane) - 1u));
      if (s < kNnlSlots) slot_cell[s] = c;
      else s = -2;
    }
    slot[c] = s;
  }
}

// Candidate lists (common.cuh: NnLists), one warp per slotted coarse cell, all kNnlSub^3 = 8 sub-cells at once (the cell's vertex
// neighbourhood is read once).  Box B = the sub-cell grown by 1e-4 of a coarse cell on every side (covers the rounding of the queries'
// grid coordinates).  U = d(centre, v*) + half-diagonal(B) with v* the vertex of the 27-neighbourhood nearest to the centre; the list
// takes every v with dmin(B, v) <= lim = U (1 + 1e-4) + 1e-4 cell, lim capped at `cut` in the cull grid (5 cm with the same slack).
// Vertices with dmin(B, v) <= lim lie in the (2r+1)^3 block of cells around B when lim < r cells; r = 1 or 2, beyond that (and beyond
// `cap` entries) the sub-cell is marked -1 and its queries take the grid search.  cand (cull grid): 0 for the sub-cells with empty lists.
__global__ void __launch_bounds__(256) k_nnl_build(const FrameConst* __restrict__ fc, int g, const int* __restrict__ start,
                                                   const float4* __restrict__ gv, const int* __restrict__ slot_cell,
                                                   const int* __restrict__ nslots, int cap, float cut, int* __restrict__ len,
                                                   float4* __restrict__ ent, unsigned char* __restrict__ cand) {
  static_assert(kNnlSub == 2, "one bit per axis selects the sub-cell");
  const GridDesc sg = g == 0 ? fc->g1 : fc->g3;
  const int lane = threadIdx.x & 31;
  const int ns = min(*nslots, kNnlSlots);
  const float f = sg.cell * 0.5f, eps = 1.0e-4f * sg.cell;
  for (int sl = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; sl < ns; sl += (gridDim.x * blockDim.x) >> 5) {
    const int c = slot_cell[sl];
    const int cx = c % sg.dim[0], t = c / sg.dim[0], cy = t % sg.dim[1], cz = t / sg.dim[1];
    const int cc[3] = {cx, cy, cz};
    float lo[3][2], hi[3][2], ctr[3][2];                     // per axis and sub-cell coordinate
#pragma unroll
    for (int k = 0; k < 3; ++k)
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        lo[k][h] = sg.origin[k] + (float)cc[k] * sg.cell + (float)h * f - eps;
        hi[k][h] = lo[k][h] + f + 2.f * eps;
        ctr[k][h] = 0.5f * (lo[k][h] + hi[k][h]);
      }
    // v* of every sub-cell: nearest vertex of the 27-neighbourhood to its centre (the coarse cell is occupied, so there is one)
    float dc[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) dc[i] = 3.0e38f;
    for (int zz = max(cz - 1, 0); zz <= min(cz + 1, sg.dim[2] - 1); ++zz)
      for (int yy = max(cy - 1, 0); yy <= min(cy + 1, sg.dim[1] - 1); ++yy) {
        const int row = (zz * sg.dim[1] + yy) * sg.dim[0];
        const int b = start[row + max(cx - 1, 0)], e = start[row + min(cx + 1, sg.dim[0] - 1) + 1];
        for (int k = b + lane; k < e; k += 32) {
          const float4 v = gv[k];
          float d[3][2];
#pragma unroll
          for (int h = 0; h < 2; ++h) {
            d[0][h] = (v.x - ctr[0][h]) * (v.x - ctr[0][h]);
            d[1][h] = (v.y - ctr[1][h]) * (v.y - ctr[1][h]);
            d[2][h] = (v.z - ctr[2][h]) * (v.z - ctr[2][h]);
          }
#pragma unroll
          for (int i = 0; i < 8; ++i) dc[i] = fminf(dc[i], d[0][i & 1] + d[1][(i >> 1) & 1] + d[2][i >> 2]);
        }
      }
    float lim2[8];
    int rmax = 0, rbits = 0;                                   // bit i: sub-cell i has a usable bound
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      float x = dc[i];
      for (int o = 16; o > 0; o >>= 1) x = fminf(x, __shfl_xor_sync(0xffffffffu, x, o));
      float lim = (sqrtf(x) + 1.7320508f * (0.5f * f + eps)) * 1.0001f + eps;
      if (cut > 0.f) lim = fminf(lim, cut);
      const int r = lim < 0.999f * sg.cell ? 1 : (lim < 1.999f * sg.cell ? 2 : 0);
      rmax = max(rmax, r);
      rbits |= r > 0 ? 1 << i : 0;
      lim2[i] = r > 0 ? lim * lim : -1.f;
    }
    int n[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) n[i] = 0;
    float4* out = ent + (size_t)sl * kNnlSub3 * kNnlCap;
    for (int zz = max(cz - rmax, 0); zz <= min(cz + rmax, sg.dim[2] - 1); ++zz)
      for (int yy = max(cy - rmax, 0); yy <= min(cy + rmax, sg.dim[1] - 1); ++yy) {
        const int row = (zz * sg.dim[1] + yy) * sg.dim[0];
        const int b = start[row + max(cx - rmax, 0)], e = start[row + min(cx + rmax, sg.dim[0] - 1) + 1];
        for (int k0 = b; k0 < e; k0 += 32) {
          const int k = k0 + lane;
          const float4 v = k < e ? gv[k] : make_float4(3.0e38f, 3.0e38f, 3.0e38f, 0.f);
          float o[3][2];
#pragma unroll
          for (int h = 0; h < 2; ++h) {
            const float ox = fmaxf(fmaxf(lo[0][h] - v.x, v.x - hi[0][h]), 0.f);
            const float oy = fmaxf(fmaxf(lo[1][h] - v.y, v.y - hi[1][h]), 0.f);
            const float oz = fmaxf(fmaxf(lo[2][h] - v.z, v.z - hi[2][h]), 0.f);
            o[0][h] = ox * ox; o[1][h] = oy * oy; o[2][h] = oz * oz;
          }
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const bool take = k < e && o[0][i & 1] + o[1][(i >> 1) & 1] + o[2][i >> 2] <= lim2[i];
            const unsigned m = __ballot_sync(0xffffffffu, take);
            const int pos = n[i] + __popc(m & ((1u << lane) - 1u));
            if (take && pos < cap) out[i * kNnlCap + pos] = v;
            n[i] += __popc(m);
          }
        }
      }
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      if (lane == i) {
        const int l = ((rbits >> i) & 1) && n[i] <= cap ? n[i] : -1;
        len[sl * kNnlSub3 + i] = l;
        if (cand) cand[(size_t)c * kNnlSub3 + i] = l != 0;
      }
    }
  }
}

// global min / max over all sample depths = over rays of {t_0, t_{S-1}} (t is monotone in i)   ray_marcher.py:57
__global__ void k_depth_range(const float* __restrict__ nearv, const float* __restrict__ farv, int N, int S, FrameConst* fc) {
  int lo = INT_MAX, hi = INT_MIN;
  for (int n = blockIdx.x * blockDim.x + threadIdx.x; n < N; n += gridDim.x * blockDim.x) {
    float a = sample_depth(nearv[n], farv[n], 0, S), b = sample_depth(nearv[n], farv[n], S - 1, S);
    int ia = float_to_ordered(a), ib = float_to_ordered(b);
    lo = min(lo, min(ia, ib));
    hi = max(hi, max(ia, ib));
  }
  for (int o = 16; o > 0; o >>= 1) {
    lo = min(lo, __shfl_xor_sync(0xffffffffu, lo, o));
    hi = max(hi, __shfl_xor_sync(0xffffffffu, hi, o));
  }
  if ((threadIdx.x & 31) == 0) { atomicMin(&fc->dmin_bits, lo); atomicMax(&fc->dmax_bits, hi); }
}

__global__ void k_set_depth_range(FrameConst* fc, float lo, float hi) {
  fc->dmin_bits = float_to_ordered(lo);
  fc->dmax_bits = float_to_ordered(hi);
}

// ---------------------------------------------------------------------------------------------
static Parents make_parents(const SherfSmplModel& smpl) {
  Parents p;
  for (int j = 0; j < kJoints; ++j) p.p[j] = (j == 0) ? 0 : smpl.parents[j];
  return p;
}

int run_lbs_only(const SherfSmplModel& smpl, const SherfPose& pose, float* A_out, float* joints_tmp, float* pf_tmp, cudaStream_t st) {
  k_joints<<<dim3(kJoints, 1), 256, 0, st>>>(smpl.v_template, smpl.shapedirs, smpl.j_regressor, pose.shapes, pose.shapes,
                                             pose.shapes, smpl.n_verts, joints_tmp);
  SHERF_LAUNCH_CHECK();
  k_chain<<<1, 32, 0, st>>>(pose.poses, pose.poses, pose.poses, joints_tmp, make_parents(smpl), A_out, pf_tmp);
  SHERF_LAUNCH_CHECK();
  return SHERF_OK;
}

int run_depth_range(const SherfRays& rays, FrameConst* fc, cudaStream_t st) {
  k_depth_range<<<min(ceil_div(rays.n_rays, 256), 1184), 256, 0, st>>>(rays.near_, rays.far_, rays.n_rays, rays.n_samples, fc);
  SHERF_LAUNCH_CHECK();
  return SHERF_OK;
}

// counting-sort build of one grid (g = 0: posed vertices / cull grid with occupancy bytes, g = 1: canonical vertices) on `st`
static int build_grid(int g, const SherfFrame& fr, const FrameTables& ft, int V, cudaStream_t st) {
  int* counts = ft.g_cursor + (size_t)g * ft.maxcell;
  int* bsums = ft.g_block_sums + (size_t)g * (ft.maxcell / 1024 + 2);
  const bool lists = ft.nnl_on != 0;
  k_grid_setup<<<1, 1024, 0, st>>>(ft.verts_smpl, fr.t_vertices, V, ft.maxcell, 0.0505f, ft.fc, g, lists ? ft.nnl_count : nullptr);
  SHERF_LAUNCH_CHECK();
  SHERF_CUDA_OK(cudaMemsetAsync(counts, 0, sizeof(int) * (size_t)ft.maxcell, st));
  k_grid_count<<<dim3(ceil_div(V, 256), 1), 256, 0, st>>>(ft.verts_smpl, fr.t_vertices, V, ft.fc, ft.g_cursor, ft.maxcell, g);
  SHERF_LAUNCH_CHECK();
  // exclusive scan over all maxcell slots (cells beyond ncell hold 0 vertices): cell_start[c], cell_start[maxcell] = V
  int rc = run_exclusive_scan(counts, ft.maxcell, bsums, g == 0 ? ft.g1_cell_start : ft.g3_cell_start, ft.g_total + g, st);
  if (rc) return rc;
  k_grid_scatter<<<dim3(ceil_div(V, 256), 1), 256, 0, st>>>(ft.verts_smpl, fr.t_vertices, V, ft.fc, ft.g_cursor, ft.maxcell, ft.g1_cell_start,
                                                           ft.g3_cell_start, ft.g1_verts, ft.g3_verts, g);
  SHERF_LAUNCH_CHECK();
  if (g == 0 || lists) {
    k_grid_occupancy<<<ceil_div(ft.maxcell, 256), 256, 0, st>>>(ft.fc, g, g == 0 ? ft.g1_cell_start : ft.g3_cell_start, g == 0 ? ft.g1_occ : nullptr,
                                                                lists ? ft.nnl_slot[g] : nullptr, ft.nnl_slot_cell[g], ft.nnl_count + g,
                                                                lists && g == 0 ? ft.nnl_cand : nullptr);
    SHERF_LAUNCH_CHECK();
  }
  if (lists) {
    // the cull lists keep only what can pass the cull's 5 cm test (run_cull: d2 < 0.05^2 in fp32), with the same slack as the bound
    const float cut = g == 0 ? 0.05f * 1.0001f + 1.0e-5f : 0.f;
    k_nnl_build<<<148 * 8, 256, 0, st>>>(ft.fc, g, g == 0 ? ft.g1_cell_start : ft.g3_cell_start, g == 0 ? ft.g1_verts : ft.g3_verts,
                                         ft.nnl_slot_cell[g], ft.nnl_count + g, ft.nnl_cap, cut, ft.nnl_len[g], ft.nnl_ent[g],
                                         g == 0 ? ft.nnl_cand : nullptr);
    SHERF_LAUNCH_CHECK();
  }
  return SHERF_OK;
}

// The per-frame work is split by what consumes it, so that the two halves can run on different streams (api.cu):
//   run_prologue_frame  : FrameConst (everything else reads it)
//   run_prologue_cull   : what the cull stage needs -- posed vertices in SMPL space, the cull grid, the global depth range
//   run_prologue_tables : what only the warp + gather stage needs -- SMPL chain of the three pose sets, pose / shape offsets,
//                         per-vertex warp tables, the canonical-vertex grid
int run_prologue_frame(const SherfFrame& fr, const FrameTables& ft, cudaStream_t st) {
  // consumers copy the whole struct to shared memory before the later stages have filled their part (grid descriptors, depth range):
  // define every byte first
  SHERF_CUDA_OK(cudaMemsetAsync(ft.fc, 0, sizeof(FrameConst), st));
  k_frame_const<<<1, 32, 0, st>>>(fr, make_float3((float)fr.out_sh[0], (float)fr.out_sh[1], (float)fr.out_sh[2]), ft.fc);
  SHERF_LAUNCH_CHECK();
  return SHERF_OK;
}

int run_prologue_cull(const SherfSmplModel& smpl, const SherfFrame& fr, const SherfRays& rays, const SherfOptions& opts,
                      const FrameTables& ft, cudaStream_t st) {
  const int V = smpl.n_verts;
  k_verts_smpl<<<ceil_div(V, 256), 256, 0, st>>>(fr.vertices, ft.fc, V, ft.verts_smpl);
  SHERF_LAUNCH_CHECK();
  int rc = build_grid(0, fr, ft, V, st);
  if (rc) return rc;
  if (opts.use_external_clamp) {
    k_set_depth_range<<<1, 1, 0, st>>>(ft.fc, opts.depth_clamp_min, opts.depth_clamp_max);
    SHERF_LAUNCH_CHECK();
  } else {
    rc = run_depth_range(rays, ft.fc, st);
    if (rc) return rc;
  }
  return SHERF_OK;
}

int run_prologue_tables(const SherfSmplModel& smpl, const SherfFrame& fr, const FrameTables& ft, cudaStream_t st) {
  const int V = smpl.n_verts;
  k_joints<<<dim3(kJoints, 3), 256, 0, st>>>(smpl.v_template, smpl.shapedirs, smpl.j_regressor, fr.target.shapes,
                                             fr.canonical.shapes, fr.obs.shapes, V, ft.joints);
  SHERF_LAUNCH_CHECK();
  k_chain<<<3, 32, 0, st>>>(fr.target.poses, fr.canonical.poses, fr.obs.poses, ft.joints, make_parents(smpl), ft.A, ft.posefeat);
  SHERF_LAUNCH_CHECK();
  k_offsets<<<ceil_div(3 * V, 8), 256, 0, st>>>(smpl.posedirs, smpl.shapedirs, ft.posefeat, fr.target.shapes, fr.obs.shapes,
                                                3 * V, ft.poff, ft.soff);
  SHERF_LAUNCH_CHECK();
  k_vertex_tables<<<ceil_div(V, 128), 128, 0, st>>>(smpl.weights, ft.A, ft.poff, ft.soff, fr.vertices, ft.fc, V, ft.T1, ft.T3, nullptr);
  SHERF_LAUNCH_CHECK();
  return build_grid(1, fr, ft, V, st);
}

}  // namespace sherf
