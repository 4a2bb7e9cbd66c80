// Stage 2: per surviving point -- inverse-LBS warp to canonical space, canonical -> observation warp
// (exact unbounded nearest canonical vertex), projection, and the three hierarchical feature gathers.
// One warp per point, lane = channel, so every tap is one coalesced 128 B line of a channels-last copy
// of the feature tensor.  Replaces renderer.py:323-350 (minus conv1d_projection) and :402 (sample_from_planes).
#include "common.cuh"
#include "stages.cuh"
#include <cstdlib>

namespace sherf {

// [C][M] (channel-major, the reference's NCHW/NCDHW) -> [M][C] channels-last; 32x32 smem tiles.  All the feature tensors of a
// forward (3 planes, 2-D feature map, 3 volume levels) go through ONE launch: block b belongs to job j with blk0[j] <= b < blk0[j+1].
struct ClJobs { const float* in[8]; float* out[8]; int C[8]; long long M[8]; int blk0[9]; int vec[8]; int n; };

// Tile = 32 channels x 128 positions.  vec jobs (M % 4 == 0, C % 4 == 0, 16-byte aligned bases): 128-bit loads along M and 128-bit
// stores along C (four times the bytes in flight per thread of the scalar form, which reached 2.7 TB/s); other jobs: scalar accesses.
__global__ void __launch_bounds__(256) k_to_channels_last(const ClJobs J) {
  __shared__ float tile[32][129];
  int j = 0;
  while (j + 1 < J.n && (int)blockIdx.x >= J.blk0[j + 1]) ++j;
  const float* __restrict__ in = J.in[j];
  float* __restrict__ out = J.out[j];
  const int C = J.C[j];
  const int64_t M = J.M[j];
  const int cblocks = (C + 31) / 32;
  const int lb = (int)blockIdx.x - J.blk0[j];
  const int64_t m0 = (int64_t)(lb / cblocks) * 128;
  const int c0 = (lb % cblocks) * 32;
  const int tid = threadIdx.x;
  if (J.vec[j]) {
#pragma unroll
    for (int k = 0; k < 4; ++k) {                            // 32 rows (channels) x 32 float4 along M
      const int idx = tid + 256 * k, r = idx >> 5, q = idx & 31;
      const int c = c0 + r;
      const int64_t m = m0 + 4 * q;
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (c < C && m < M) v = __ldg(reinterpret_cast<const float4*>(in + (size_t)c * M + m));
      tile[r][4 * q] = v.x; tile[r][4 * q + 1] = v.y; tile[r][4 * q + 2] = v.z; tile[r][4 * q + 3] = v.w;
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < 4; ++k) {                            // 128 positions x 8 float4 along C
      const int idx = tid + 256 * k, mm = idx >> 3, q = idx & 7;
      const int64_t m = m0 + mm;
      const int c = c0 + 4 * q;
      if (c < C && m < M)
        *reinterpret_cast<float4*>(out + (size_t)m * C + c) = make_float4(tile[4 * q][mm], tile[4 * q + 1][mm], tile[4 * q + 2][mm], tile[4 * q + 3][mm]);
    }
  } else {
    const int tx = tid & 31, ty = tid >> 5;                  // 32 x 8
    for (int sub = 0; sub < 4; ++sub) {
#pragma unroll
      for (int r = ty; r < 32; r += 8) {
        const int c = c0 + r;
        const int64_t m = m0 + 32 * sub + tx;
        tile[r][32 * sub + tx] = (c < C && m < M) ? in[(size_t)c * M + m] : 0.f;
      }
    }
    __syncthreads();
    for (int sub = 0; sub < 4; ++sub) {
#pragma unroll
      for (int r = ty; r < 32; r += 8) {
        const int64_t m = m0 + 32 * sub + r;
        const int c = c0 + tx;
        if (c < C && m < M) out[(size_t)m * C + c] = tile[tx][32 * sub + r];
      }
    }
  }
}

int run_to_channels_last_multi(int n, const float* const* in, float* const* out, const int* C, const int64_t* M, cudaStream_t st) {
  if (n <= 0 || n > 8) { set_error("internal: %d channels-last jobs", n); return SHERF_E_INVALID; }
  ClJobs J;
  J.n = n;
  int64_t blocks = 0;
  for (int j = 0; j < n; ++j) {
    J.in[j] = in[j]; J.out[j] = out[j]; J.C[j] = C[j]; J.M[j] = M[j];
    J.vec[j] = (M[j] % 4 == 0 && C[j] % 4 == 0 && ((uintptr_t)in[j] & 15) == 0 && ((uintptr_t)out[j] & 15) == 0) ? 1 : 0;
    J.blk0[j] = (int)blocks;
    blocks += ((M[j] + 127) / 128) * ((C[j] + 31) / 32);
  }
  J.blk0[n] = (int)blocks;
  if (blocks >= (1LL << 31)) { set_error("feature tensors too large for one layout launch"); return SHERF_E_INVALID; }
  k_to_channels_last<<<(unsigned)blocks, 256, 0, st>>>(J);
  SHERF_LAUNCH_CHECK();
  return SHERF_OK;
}

__device__ __forceinline__ void warp_lexmin(float& d, int& id) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    float od = __shfl_xor_sync(0xffffffffu, d, o);
    int oi = __shfl_xor_sync(0xffffffffu, id, o);
    if (od < d || (od == d && oi < id)) { d = od; id = oi; }
  }
}

// Exact K=1 search, no radius bound (renderer.py:627): box of Chebyshev radius r around the query's cell, one lane per
// cell of the box; r doubles until every unsearched cell is provably farther than the best hit.
__device__ int nn_unbounded(const GridDesc& g, const int* __restrict__ cell_start, const float4* __restrict__ gv,
                            float qx, float qy, float qz, int lane) {
  const int cx = min(max(grid_coord(qx, g.origin[0], g.inv_cell, g.dim[0]), 0), g.dim[0] - 1);
  const int cy = min(max(grid_coord(qy, g.origin[1], g.inv_cell, g.dim[1]), 0), g.dim[1] - 1);
  const int cz = min(max(grid_coord(qz, g.origin[2], g.inv_cell, g.dim[2]), 0), g.dim[2] - 1);
  float best = 3.0e38f;
  int bid = 0x7fffffff;
  for (int r = 1;; r *= 2) {
    const int x0 = max(cx - r, 0), x1 = min(cx + r, g.dim[0] - 1);
    const int y0 = max(cy - r, 0), y1 = min(cy + r, g.dim[1] - 1);
    const int z0 = max(cz - r, 0), z1 = min(cz + r, g.dim[2] - 1);
    const int nx = x1 - x0 + 1, ny = y1 - y0 + 1, ncells = nx * ny * (z1 - z0 + 1);
    for (int cc = lane; cc < ncells; cc += 32) {
      const int xx = x0 + cc % nx, t = cc / nx;
      const int cell = ((z0 + t / ny) * g.dim[1] + (y0 + t % ny)) * g.dim[0] + xx;
      const int b = cell_start[cell], e = cell_start[cell + 1];
      for (int k = b; k < e; ++k) {
        const float4 v = gv[k];
        const float d2 = dist2_xyz(qx, qy, qz, v.x, v.y, v.z);
        const int id = __float_as_int(v.w);
        if (d2 < best || (d2 == best && id < bid)) { best = d2; bid = id; }
      }
    }
    warp_lexmin(best, bid);
    // distance from q to the nearest face of the searched box that still has grid cells behind it
    float m = 3.0e38f;
    if (cx - r > 0) m = fminf(m, qx - (g.origin[0] + (float)(cx - r) * g.cell));
    if (cx + r < g.dim[0] - 1) m = fminf(m, (g.origin[0] + (float)(cx + r + 1) * g.cell) - qx);
    if (cy - r > 0) m = fminf(m, qy - (g.origin[1] + (float)(cy - r) * g.cell));
    if (cy + r < g.dim[1] - 1) m = fminf(m, (g.origin[1] + (float)(cy + r + 1) * g.cell) - qy);
    if (cz - r > 0) m = fminf(m, qz - (g.origin[2] + (float)(cz - r) * g.cell));
    if (cz + r < g.dim[2] - 1) m = fminf(m, (g.origin[2] + (float)(cz + r + 1) * g.cell) - qz);
    if (m > 1.0e38f) break;                       // whole grid searched
    const float ms = m - 1.0e-4f * g.cell;        // guard band for fp32 rounding of d2 / face positions
    if (ms > 0.f && best < ms * ms) break;
  }
  return bid;
}

__device__ __forceinline__ void apply_warp(const VertexWarp* __restrict__ Tp, float p[3], float d[3], bool with_dir) {
  // broadcast loads: every lane reads the same 144 B record
  const float4* r4 = reinterpret_cast<const float4*>(Tp);
  float w[36];
#pragma unroll
  for (int i = 0; i < 9; ++i) { float4 v = r4[i]; w[4 * i] = v.x; w[4 * i + 1] = v.y; w[4 * i + 2] = v.z; w[4 * i + 3] = v.w; }
  float a[3] = {p[0] - w[9], p[1] - w[10], p[2] - w[11]};
  float c[3];
  mat3_vec(w, a, c);
#pragma unroll
  for (int k = 0; k < 3; ++k) { c[k] = c[k] + w[12 + k]; c[k] = c[k] + w[15 + k]; c[k] = c[k] + w[18 + k]; }
  const float* Af = w + 21;
#pragma unroll
  for (int k = 0; k < 3; ++k) p[k] = (Af[4 * k] * c[0] + Af[4 * k + 1] * c[1] + Af[4 * k + 2] * c[2]) + Af[4 * k + 3];
  if (with_dir) {
    float e[3];
    mat3_vec(w, d, e);
#pragma unroll
    for (int k = 0; k < 3; ++k) d[k] = Af[4 * k] * e[0] + Af[4 * k + 1] * e[1] + Af[4 * k + 2] * e[2];
  }
}

__global__ void __launch_bounds__(256) k_point_gather(const GatherParams P) {
  __shared__ FrameConst fc;
  for (int i = threadIdx.x; i < (int)(sizeof(FrameConst) / 4); i += blockDim.x) ((int*)&fc)[i] = ((const int*)P.fc)[i];
  __syncthreads();
  const int lane = threadIdx.x & 31;
  const int warps_total = gridDim.x * (blockDim.x >> 5);
  for (int lp = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); lp < P.np; lp += warps_total) {
    const int64_t gp = P.p0 + lp;
    const int s = P.point_sample[gp];
    const int n = s / P.S, i = s - n * P.S;
    // ---- re-derive the SMPL-space query exactly as the cull did (renderer.py:304-310) ----
    const float t = P.depths ? P.depths[s] : sample_depth(P.nearv[n], P.farv[n], i, P.S);
    float dray[3] = {P.dirs[n * 3], P.dirs[n * 3 + 1], P.dirs[n * 3 + 2]};
    float pw[3], q[3], vd[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) pw[k] = __fsub_rn(mul_add_sep(t, dray[k], P.origins[n * 3 + k]), fc.Th_tgt[k]);
    rowvec_mat3(pw, fc.R_tgt, q);
    rowvec_mat3(dray, fc.R_tgt, vd);
    // ---- target -> canonical (renderer.py:558-621) ----
    float can[3] = {q[0], q[1], q[2]}, cdir[3] = {vd[0], vd[1], vd[2]};
    apply_warp(P.T1 + P.point_vid[gp], can, cdir, true);
    // ---- canonical -> observation -> pixel (renderer.py:623-704) ----
    const int vid3 = nn_unbounded(fc.g3, P.g3_start, P.g3_verts, can[0], can[1], can[2], lane);
    float ps[3] = {can[0], can[1], can[2]}, dummy[3] = {0.f, 0.f, 0.f};
    apply_warp(P.T3 + vid3, ps, dummy, false);
    float world[3], cam[3], pix[3];
#pragma unroll
    for (int k = 0; k < 3; ++k)
      world[k] = (ps[0] * fc.Rinv_obs[k] + ps[1] * fc.Rinv_obs[3 + k] + ps[2] * fc.Rinv_obs[6 + k]) + fc.Th_obs[k];
    mat3_vec(fc.camR, world, cam);
#pragma unroll
    for (int k = 0; k < 3; ++k) cam[k] += fc.camT[k];
    mat3_vec(fc.camK, cam, pix);
    const float zz = pix[2] + 1e-5f;
    const float u = pix[0] / zz, v = pix[1] / zz;

    float* comb = P.comb + (size_t)lp * 288;
    float* f3 = P.f3raw + (size_t)lp * 192;
    float* dbgf = (P.dbg_feat && gp < P.dbg_feat_max) ? P.dbg_feat + (size_t)gp * 384 : nullptr;

    // ================= lane-parallel tap setup: every lane prepares ONE 2-D tap and ONE 3-D tap =================
    // set A (2-D): lanes 0-11 tri-plane (plane k = lane/4), 12-15 observation feature map, 16-19 observation image;
    //              corner = lane & 3 in grid_sample's accumulation order nw, ne, sw, se                 renderer.py:234-243,331-340
    // set B (3-D): lanes 0-23 pyramid level lane/8, corner = lane & 7 (bit0 x, bit1 y, bit2 z)          renderer.py:544-556,762-797
    int offA = -1; float wA = 0.f;
    {
      float cn[3];
#pragma unroll
      for (int k = 0; k < 3; ++k) cn[k] = 2.f * (can[k] - fc.twb_min[k]) / (fc.twb_max[k] - fc.twb_min[k]) - 1.f;
      const float gx = 2.0f * u / (float)P.img_w - 1.0f, gy = 2.0f * v / (float)P.img_h - 1.0f;
      const int grp = lane >> 2;                                   // 0..2 planes, 3 feature map, 4 image
      float ix, iy; int W, H, C;
      if (grp < 3) {                                                // align_corners=False
        const float px = grp == 2 ? cn[2] : cn[0], py = grp == 1 ? cn[2] : cn[1];
        W = P.plane_w; H = P.plane_h; C = 32;
        ix = ((px + 1.f) * (float)W - 1.f) * 0.5f; iy = ((py + 1.f) * (float)H - 1.f) * 0.5f;
      } else if (grp == 3) {                                        // align_corners=True, uv normalised by the IMAGE size
        W = P.feat_w; H = P.feat_h; C = P.feat_ch;
        ix = (gx + 1.f) * 0.5f * (float)(W - 1); iy = (gy + 1.f) * 0.5f * (float)(H - 1);
      } else {
        W = P.img_w; H = P.img_h; C = 1;
        ix = (gx + 1.f) * 0.5f * (float)(W - 1); iy = (gy + 1.f) * 0.5f * (float)(H - 1);
      }
      const float fx = floorf(ix), fy = floorf(iy);
      const int cxb = lane & 1, cyb = (lane >> 1) & 1;
      const int xx = (int)fx + cxb, yy = (int)fy + cyb;
      const float wx = cxb ? ix - fx : (fx + 1.f) - ix, wy = cyb ? iy - fy : (fy + 1.f) - iy;
      wA = wx * wy;
      if (lane < 20 && xx >= 0 && xx < W && yy >= 0 && yy < H) offA = (yy * W + xx) * C;
    }
    int offB = -1; float wB = 0.f;
    {
      const int l = lane >> 3;
      const int D = l == 0 ? P.vol_d[0] : (l == 1 ? P.vol_d[1] : P.vol_d[2]);
      const int H = l == 0 ? P.vol_h[0] : (l == 1 ? P.vol_h[1] : P.vol_h[2]);
      const int W = l == 0 ? P.vol_w[0] : (l == 1 ? P.vol_w[1] : P.vol_w[2]);
      const int C = l == 0 ? P.vol_ch[0] : (l == 1 ? P.vol_ch[1] : P.vol_ch[2]);
      float gn[3];   // normalised (x, y, z); dhw axis 2-k holds coordinate k, out_sh is (z,y,x)
#pragma unroll
      for (int k = 0; k < 3; ++k) gn[k] = ((can[k] - fc.spb_min[k]) / 0.005f) / fc.out_sh[2 - k] * 2.f - 1.f;
      const float ix = (gn[0] + 1.f) * 0.5f * (float)(W - 1), iy = (gn[1] + 1.f) * 0.5f * (float)(H - 1),
                  iz = (gn[2] + 1.f) * 0.5f * (float)(D - 1);
      const float fx = floorf(ix), fy = floorf(iy), fz = floorf(iz);
      const int bx = lane & 1, by = (lane >> 1) & 1, bz = (lane >> 2) & 1;
      const int xx = (int)fx + bx, yy = (int)fy + by, zz2 = (int)fz + bz;
      const float wx = bx ? ix - fx : (fx + 1.f) - ix, wy = by ? iy - fy : (fy + 1.f) - iy, wz = bz ? iz - fz : (fz + 1.f) - iz;
      wB = wx * wy * wz;
      if (lane < 24 && xx >= 0 && xx < W && yy >= 0 && yy < H && zz2 >= 0 && zz2 < D) offB = ((zz2 * H + yy) * W + xx) * C;
    }

    // ================= gathers: lane = channel; tap offsets / weights arrive by shuffle =================
    // ---- tri-planes ----
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      const float* base = P.planes_cl + (size_t)k * P.plane_h * P.plane_w * 32 + lane;
      float acc = 0.f;
#pragma unroll
      for (int t = 0; t < 4; ++t) {
        const int off = __shfl_sync(0xffffffffu, offA, 4 * k + t);
        const float w = __shfl_sync(0xffffffffu, wA, 4 * k + t);
        const float val = off >= 0 ? __ldg(base + off) : 0.f;
        acc = t == 0 ? val * w : acc + val * w;
      }
      comb[k * 96 + lane] = acc;
      if (dbgf) dbgf[k * 32 + lane] = acc;
    }
    // ---- pixel-aligned 2-D features + rgb positional encoding ----
    {
      float f0 = 0.f, f1 = 0.f, rgbc = 0.f;
#pragma unroll
      for (int t = 0; t < 4; ++t) {
        const int off = __shfl_sync(0xffffffffu, offA, 12 + t);
        const float w = __shfl_sync(0xffffffffu, wA, 12 + t);
        const float v0 = off >= 0 ? __ldg(P.feat_cl + off + lane) : 0.f;
        const float v1 = off >= 0 ? __ldg(P.feat_cl + off + 32 + lane) : 0.f;
        f0 = t == 0 ? v0 * w : f0 + v0 * w;
        f1 = t == 0 ? v1 * w : f1 + v1 * w;
        const int offi = __shfl_sync(0xffffffffu, offA, 16 + t);
        const float wi = __shfl_sync(0xffffffffu, wA, 16 + t);
        const float vi = (lane < 3 && offi >= 0) ? __ldg(P.img + (size_t)lane * P.img_h * P.img_w + offi) : 0.f;
        rgbc = t == 0 ? vi * wi : rgbc + vi * wi;
      }
      // rgb_enc (num_freqs=5) truncated to its first 32 outputs (renderer.py:339, :900-916)
      const int e = lane - 3;
      const int m = e >= 0 ? e / 3 : 0, c = e >= 0 ? e - 3 * m : lane;
      const float xc = __shfl_sync(0xffffffffu, rgbc, c);
      const float enc = lane < 3 ? xc : sinf(__fadd_rn((m & 1) ? kPi2 : 0.f, __fmul_rn(xc, (float)(1 << (m >> 1)))));
      comb[0 * 96 + 32 + lane] = f0;
      comb[1 * 96 + 32 + lane] = f1;
      comb[2 * 96 + 32 + lane] = enc;
      if (dbgf) { dbgf[96 + lane] = f0; dbgf[128 + lane] = f1; dbgf[160 + lane] = enc; }
    }
    // ---- 3-D pyramid ----
    {
      int coff = 0;
#pragma unroll
      for (int l = 0; l < 3; ++l) {
        int off[8]; float w[8];
#pragma unroll
        for (int t = 0; t < 8; ++t) { off[t] = __shfl_sync(0xffffffffu, offB, 8 * l + t); w[t] = __shfl_sync(0xffffffffu, wB, 8 * l + t); }
        const float* vol = P.vol_cl[l] + lane;
#pragma unroll
        for (int gsel = 0; gsel < 3; ++gsel) {
          if (gsel <= l) {                                          // level l has 32*(l+1) channels
            float acc = 0.f;
#pragma unroll
            for (int t = 0; t < 8; ++t) {
              const float val = off[t] >= 0 ? __ldg(vol + off[t] + 32 * gsel) : 0.f;
              acc += val * w[t];
            }
            f3[coff + 32 * gsel + lane] = acc;
            if (dbgf) dbgf[192 + coff + 32 * gsel + lane] = acc;
          }
        }
        coff += 32 * (l + 1);
      }
    }
    if (lane < 8) {
      float gval = 0.f;   // select chain instead of dynamic indexing (keeps the vectors in registers)
      if (lane == 0) gval = can[0]; else if (lane == 1) gval = can[1]; else if (lane == 2) gval = can[2];
      else if (lane == 3) gval = cdir[0]; else if (lane == 4) gval = cdir[1]; else if (lane == 5) gval = cdir[2];
      P.geo[(size_t)lp * 8 + lane] = gval;
    }
    if (lane == 0 && gp < P.dbg_max) {
      if (P.dbg_vid3) P.dbg_vid3[gp] = vid3;
      if (P.dbg_can) { P.dbg_can[gp * 3] = can[0]; P.dbg_can[gp * 3 + 1] = can[1]; P.dbg_can[gp * 3 + 2] = can[2]; }
      if (P.dbg_cdir) { P.dbg_cdir[gp * 3] = cdir[0]; P.dbg_cdir[gp * 3 + 1] = cdir[1]; P.dbg_cdir[gp * 3 + 2] = cdir[2]; }
      if (P.dbg_uv) { P.dbg_uv[gp * 2] = u; P.dbg_uv[gp * 2 + 1] = v; }
    }
  }
}


// =====================================================================================================================
// 4 points per warp: lanes [8g, 8g+8) own point g; lane l8 = lane & 7 owns channels 4*l8 .. 4*l8+3 of every 32-channel
// group (one 16-byte load per tap).  All geometry / tap-setup instructions therefore serve four points at once.
// Same arithmetic (and the same operation order per point) as the one-point-per-warp kernel above.
// =====================================================================================================================
__device__ __forceinline__ void grp_lexmin(float& d, int& id) {      // reduce over the 8 lanes of a point group
#pragma unroll
  for (int o = 4; o > 0; o >>= 1) {
    const float od = __shfl_xor_sync(0xffffffffu, d, o);
    const int oi = __shfl_xor_sync(0xffffffffu, id, o);
    if (od < d || (od == d && oi < id)) { d = od; id = oi; }
  }
}

// Exact K=1 search seeded with an upper bound: the canonical position of the point's nearest POSED vertex (knn #1) is almost always
// within a few centimetres of the canonical point, so d2(q, t_vertices[seed]) bounds the answer and only the cells that intersect the
// ball of that radius need to be visited (typically 8-18 instead of 27 cells of 5 cm, and never a second, 125-cell round).  Any vertex
// that beats or ties the seed lies inside the box [q - r, q + r], r = sqrt(d2_seed) (+ guard for the fp32 rounding of d2 and of the
// cell coordinates), and the vertex cells are clamped exactly like the box, so the lexicographic (d2, id) minimum is unchanged.
// With candidate lists (common.cuh: NnLists) the 8 lanes scan the list of the point's sub-cell instead, where it has one.
__device__ int nn_seeded8(const GridDesc& g, const int* __restrict__ cell_start, const float4* __restrict__ gv, const NnLists& nl,
                          const float* __restrict__ t_vertices, float qx, float qy, float qz, int l8, int seed) {
  const int li = nl.slot ? nnl_index(g, nl.slot, qx, qy, qz) : -1;
  const int ln = li >= 0 ? nl.len[li] : -1;
  if (ln > 0) {
    float best = 3.0e38f;
    int bid = 0x7fffffff;
    const float4* e = nl.ent + (size_t)li * kNnlCap;
    for (int k = l8; k < ln; k += 8) {
      const float4 v = e[k];
      const float d2 = dist2_xyz(qx, qy, qz, v.x, v.y, v.z);
      const int id = __float_as_int(v.w);
      if (d2 < best || (d2 == best && id < bid)) { best = d2; bid = id; }
    }
    grp_lexmin(best, bid);
    return bid;
  }
  float best = dist2_xyz(qx, qy, qz, t_vertices[seed * 3], t_vertices[seed * 3 + 1], t_vertices[seed * 3 + 2]);
  int bid = seed;
  const float rb = sqrtf(best) * 1.0001f + 1.0e-4f * g.cell;
  const int x0 = min(max(grid_coord(qx - rb, g.origin[0], g.inv_cell, g.dim[0]), 0), g.dim[0] - 1);
  const int x1 = min(max(grid_coord(qx + rb, g.origin[0], g.inv_cell, g.dim[0]), 0), g.dim[0] - 1);
  const int y0 = min(max(grid_coord(qy - rb, g.origin[1], g.inv_cell, g.dim[1]), 0), g.dim[1] - 1);
  const int y1 = min(max(grid_coord(qy + rb, g.origin[1], g.inv_cell, g.dim[1]), 0), g.dim[1] - 1);
  const int z0 = min(max(grid_coord(qz - rb, g.origin[2], g.inv_cell, g.dim[2]), 0), g.dim[2] - 1);
  const int z1 = min(max(grid_coord(qz + rb, g.origin[2], g.inv_cell, g.dim[2]), 0), g.dim[2] - 1);
  const int nx = x1 - x0 + 1, ny = y1 - y0 + 1, ncells = nx * ny * (z1 - z0 + 1);
  for (int cc = l8; cc < ncells; cc += 8) {
    const int xx = x0 + cc % nx, t = cc / nx;
    const int cell = ((z0 + t / ny) * g.dim[1] + (y0 + t % ny)) * g.dim[0] + xx;
    const int b = cell_start[cell], e = cell_start[cell + 1];
    for (int k = b; k < e; ++k) {
      const float4 v = gv[k];
      const float d2 = dist2_xyz(qx, qy, qz, v.x, v.y, v.z);
      const int id = __float_as_int(v.w);
      if (d2 < best || (d2 == best && id < bid)) { best = d2; bid = id; }
    }
  }
  grp_lexmin(best, bid);
  return bid;
}

__device__ int nn_unbounded8(const GridDesc& g, const int* __restrict__ cell_start, const float4* __restrict__ gv, float qx, float qy,
                             float qz, int l8, bool active) {
  const int cx = min(max(grid_coord(qx, g.origin[0], g.inv_cell, g.dim[0]), 0), g.dim[0] - 1);
  const int cy = min(max(grid_coord(qy, g.origin[1], g.inv_cell, g.dim[1]), 0), g.dim[1] - 1);
  const int cz = min(max(grid_coord(qz, g.origin[2], g.inv_cell, g.dim[2]), 0), g.dim[2] - 1);
  float best = 3.0e38f;
  int bid = 0x7fffffff;
  (void)active;            // inactive groups shadow a valid point and must still produce a valid vertex id
  bool done = false;
  for (int r = 1; __any_sync(0xffffffffu, !done); r *= 2) {
    if (!done) {
      const int x0 = max(cx - r, 0), x1 = min(cx + r, g.dim[0] - 1);
      const int y0 = max(cy - r, 0), y1 = min(cy + r, g.dim[1] - 1);
      const int z0 = max(cz - r, 0), z1 = min(cz + r, g.dim[2] - 1);
      const int nx = x1 - x0 + 1, ny = y1 - y0 + 1, ncells = nx * ny * (z1 - z0 + 1);
      for (int cc = l8; cc < ncells; cc += 8) {
        const int xx = x0 + cc % nx, t = cc / nx;
        const int cell = ((z0 + t / ny) * g.dim[1] + (y0 + t % ny)) * g.dim[0] + xx;
        const int b = cell_start[cell], e = cell_start[cell + 1];
        for (int k = b; k < e; ++k) {
          const float4 v = gv[k];
          const float d2 = dist2_xyz(qx, qy, qz, v.x, v.y, v.z);
          const int id = __float_as_int(v.w);
          if (d2 < best || (d2 == best && id < bid)) { best = d2; bid = id; }
        }
      }
    }
    grp_lexmin(best, bid);
    if (!done) {
      float m = 3.0e38f;
      if (cx - r > 0) m = fminf(m, qx - (g.origin[0] + (float)(cx - r) * g.cell));
      if (cx + r < g.dim[0] - 1) m = fminf(m, (g.origin[0] + (float)(cx + r + 1) * g.cell) - qx);
      if (cy - r > 0) m = fminf(m, qy - (g.origin[1] + (float)(cy - r) * g.cell));
      if (cy + r < g.dim[1] - 1) m = fminf(m, (g.origin[1] + (float)(cy + r + 1) * g.cell) - qy);
      if (cz - r > 0) m = fminf(m, qz - (g.origin[2] + (float)(cz - r) * g.cell));
      if (cz + r < g.dim[2] - 1) m = fminf(m, (g.origin[2] + (float)(cz + r + 1) * g.cell) - qz);
      const float ms = m - 1.0e-4f * g.cell;
      if (m > 1.0e38f || (ms > 0.f && best < ms * ms)) done = true;
    }
  }
  return bid;
}

// BWD = true turns the kernel into the ADJOINT of its three gathers (backward.cu): the warps, the knn #3 and the tap offsets / weights are
// recomputed exactly as in the forward, P.comb / P.f3raw are READ as dL/d(comb) / dL/d(f3raw) and every tap adds weight x gradient into
// the channels-last gradient grids P.g_* with one 16-byte vector reduction per lane and tap (red.global.add.v4.f32).
__device__ __forceinline__ void red_add4(float* p, const float4& g, float w) {
  atomicAdd(reinterpret_cast<float4*>(p), make_float4(g.x * w, g.y * w, g.z * w, g.w * w));
}

template <bool DBG, bool BWD>
__global__ void __launch_bounds__(256) k_point_gather4(const GatherParams P) {
  __shared__ FrameConst fc;
  for (int i = threadIdx.x; i < (int)(sizeof(FrameConst) / 4); i += blockDim.x) ((int*)&fc)[i] = ((const int*)P.fc)[i];
  __syncthreads();
  const int lane = threadIdx.x & 31, l8 = lane & 7, gbase = lane & 24;
  const int groups_total = gridDim.x * (blockDim.x >> 3);
  const int niter = (P.np + groups_total - 1) / groups_total;
  for (int it = 0; it < niter; ++it) {
    const int lp_raw = it * groups_total + blockIdx.x * (blockDim.x >> 3) + (threadIdx.x >> 3);
    const bool active = lp_raw < P.np;
    const int lp = active ? lp_raw : P.np - 1;               // inactive groups shadow the last point and store nothing
    const int64_t gp = P.p0 + lp;
    const int s = P.point_sample[gp];
    const int n = s / P.S, i = s - n * P.S;
    const float t = P.depths ? P.depths[s] : sample_depth(P.nearv[n], P.farv[n], i, P.S);
    float dray[3] = {P.dirs[n * 3], P.dirs[n * 3 + 1], P.dirs[n * 3 + 2]};
    float pw[3], q[3], vd[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) pw[k] = __fsub_rn(mul_add_sep(t, dray[k], P.origins[n * 3 + k]), fc.Th_tgt[k]);
    rowvec_mat3(pw, fc.R_tgt, q);
    rowvec_mat3(dray, fc.R_tgt, vd);
    float can[3] = {q[0], q[1], q[2]}, cdir[3] = {vd[0], vd[1], vd[2]};
    apply_warp(P.T1 + P.point_vid[gp], can, cdir, true);
    const int vid3 = P.t_vertices ? nn_seeded8(fc.g3, P.g3_start, P.g3_verts, BWD ? NnLists{nullptr, nullptr, nullptr, nullptr} : P.nl3, P.t_vertices, can[0], can[1], can[2], l8, P.point_vid[gp])
                                  : nn_unbounded8(fc.g3, P.g3_start, P.g3_verts, can[0], can[1], can[2], l8, active);
    float ps[3] = {can[0], can[1], can[2]}, dummy[3] = {0.f, 0.f, 0.f};
    apply_warp(P.T3 + vid3, ps, dummy, false);
    float world[3], cam[3], pix[3];
#pragma unroll
    for (int k = 0; k < 3; ++k)
      world[k] = (ps[0] * fc.Rinv_obs[k] + ps[1] * fc.Rinv_obs[3 + k] + ps[2] * fc.Rinv_obs[6 + k]) + fc.Th_obs[k];
    mat3_vec(fc.camR, world, cam);
#pragma unroll
    for (int k = 0; k < 3; ++k) cam[k] += fc.camT[k];
    mat3_vec(fc.camK, cam, pix);
    const float zz = pix[2] + 1e-5f;
    const float u = pix[0] / zz, v = pix[1] / zz;

    // ---- tap setup: lane l8 prepares taps l8, l8+8, l8+16 of set A (20 taps) and of set B (24 taps) ----
    float cn[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) cn[k] = 2.f * (can[k] - fc.twb_min[k]) / (fc.twb_max[k] - fc.twb_min[k]) - 1.f;
    const float gx = 2.0f * u / (float)P.img_w - 1.0f, gy = 2.0f * v / (float)P.img_h - 1.0f;
    float gn[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) gn[k] = ((can[k] - fc.spb_min[k]) / 0.005f) / fc.out_sh[2 - k] * 2.f - 1.f;
    int offA[3], offB[3];
    float wA[3], wB[3];
#pragma unroll
    for (int sl = 0; sl < 3; ++sl) {
      const int tA = l8 + 8 * sl;                              // 0..23 (20..23 unused)
      {
        const int grp = tA >> 2;
        float ix, iy; int W, H, C;
        if (grp < 3) {
          const float px = grp == 2 ? cn[2] : cn[0], py = grp == 1 ? cn[2] : cn[1];
          W = P.plane_w; H = P.plane_h; C = 32;
          ix = ((px + 1.f) * (float)W - 1.f) * 0.5f; iy = ((py + 1.f) * (float)H - 1.f) * 0.5f;
        } else if (grp == 3) {
          W = P.feat_w; H = P.feat_h; C = P.feat_ch;
          ix = (gx + 1.f) * 0.5f * (float)(W - 1); iy = (gy + 1.f) * 0.5f * (float)(H - 1);
        } else {
          W = P.img_w; H = P.img_h; C = 1;
          ix = (gx + 1.f) * 0.5f * (float)(W - 1); iy = (gy + 1.f) * 0.5f * (float)(H - 1);
        }
        const float fx = floorf(ix), fy = floorf(iy);
        const int cxb = tA & 1, cyb = (tA >> 1) & 1;
        const int xx = (int)fx + cxb, yy = (int)fy + cyb;
        const float wx = cxb ? ix - fx : (fx + 1.f) - ix, wy = cyb ? iy - fy : (fy + 1.f) - iy;
        wA[sl] = wx * wy;
        offA[sl] = (tA < 20 && xx >= 0 && xx < W && yy >= 0 && yy < H) ? (yy * W + xx) * C : -1;
      }
      {
        const int tB = l8 + 8 * sl;                            // 0..23: level sl, corner l8
        const int l = sl;
        const int D = P.vol_d[l], H = P.vol_h[l], W = P.vol_w[l], C = P.vol_ch[l];
        const float ix = (gn[0] + 1.f) * 0.5f * (float)(W - 1), iy = (gn[1] + 1.f) * 0.5f * (float)(H - 1),
                    iz = (gn[2] + 1.f) * 0.5f * (float)(D - 1);
        const float fx = floorf(ix), fy = floorf(iy), fz = floorf(iz);
        const int bx = tB & 1, by = (tB >> 1) & 1, bz = (tB >> 2) & 1;
        const int xx = (int)fx + bx, yy = (int)fy + by, zz2 = (int)fz + bz;
        const float wx = bx ? ix - fx : (fx + 1.f) - ix, wy = by ? iy - fy : (fy + 1.f) - iy, wz = bz ? iz - fz : (fz + 1.f) - iz;
        wB[sl] = wx * wy * wz;
        offB[sl] = (xx >= 0 && xx < W && yy >= 0 && yy < H && zz2 >= 0 && zz2 < D) ? ((zz2 * H + yy) * W + xx) * C : -1;
      }
    }
    auto tapA = [&](int tix, int& off, float& w) {             // tap tix of this point's set A (tix is compile-time after unrolling)
      off = __shfl_sync(0xffffffffu, offA[tix >> 3], gbase + (tix & 7));
      w = __shfl_sync(0xffffffffu, wA[tix >> 3], gbase + (tix & 7));
    };
    float* comb = P.comb + (size_t)lp * 288;
    float* f3 = P.f3raw + (size_t)lp * 192;
    float* dbgf = (DBG && P.dbg_feat && gp < P.dbg_feat_max) ? P.dbg_feat + (size_t)gp * 384 : nullptr;
    const int c4 = 4 * l8;

    // ---- tri-planes ----
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      if (BWD) {
        if (P.g_planes_cl) {
          float* gb = P.g_planes_cl + (size_t)k * P.plane_h * P.plane_w * 32 + c4;
          const float4 g = *reinterpret_cast<const float4*>(comb + k * 96 + c4);
#pragma unroll
          for (int tp = 0; tp < 4; ++tp) {
            int off; float w;
            tapA(4 * k + tp, off, w);
            if (active && off >= 0) red_add4(gb + off, g, w);
          }
        }
        continue;
      }
      const float* base = P.planes_cl + (size_t)k * P.plane_h * P.plane_w * 32 + c4;
      float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
      for (int tp = 0; tp < 4; ++tp) {
        int off; float w;
        tapA(4 * k + tp, off, w);
        const float4 val = off >= 0 ? __ldg(reinterpret_cast<const float4*>(base + off)) : make_float4(0.f, 0.f, 0.f, 0.f);
        if (tp == 0) { acc.x = val.x * w; acc.y = val.y * w; acc.z = val.z * w; acc.w = val.w * w; }
        else { acc.x += val.x * w; acc.y += val.y * w; acc.z += val.z * w; acc.w += val.w * w; }
      }
      if (active) *reinterpret_cast<float4*>(comb + k * 96 + c4) = acc;
      if (DBG && dbgf && active) *reinterpret_cast<float4*>(dbgf + k * 32 + c4) = acc;
    }
    // ---- pixel-aligned 2-D features + rgb positional encoding ----
    if (BWD) {
      if (P.g_feat_cl) {
        const float4 g0 = *reinterpret_cast<const float4*>(comb + 0 * 96 + 32 + c4), g1 = *reinterpret_cast<const float4*>(comb + 1 * 96 + 32 + c4);
#pragma unroll
        for (int tp = 0; tp < 4; ++tp) {
          int off; float w;
          tapA(12 + tp, off, w);
          if (active && off >= 0) { red_add4(P.g_feat_cl + off + c4, g0, w); red_add4(P.g_feat_cl + off + 32 + c4, g1, w); }
        }
      }
    } else {
      float4 f0 = make_float4(0.f, 0.f, 0.f, 0.f), f1 = f0;
      float rgbc = 0.f;
#pragma unroll
      for (int tp = 0; tp < 4; ++tp) {
        int off; float w;
        tapA(12 + tp, off, w);
        const float4 v0 = off >= 0 ? __ldg(reinterpret_cast<const float4*>(P.feat_cl + off + c4)) : make_float4(0.f, 0.f, 0.f, 0.f);
        const float4 v1 = off >= 0 ? __ldg(reinterpret_cast<const float4*>(P.feat_cl + off + 32 + c4)) : make_float4(0.f, 0.f, 0.f, 0.f);
        if (tp == 0) { f0.x = v0.x * w; f0.y = v0.y * w; f0.z = v0.z * w; f0.w = v0.w * w; f1.x = v1.x * w; f1.y = v1.y * w; f1.z = v1.z * w; f1.w = v1.w * w; }
        else { f0.x += v0.x * w; f0.y += v0.y * w; f0.z += v0.z * w; f0.w += v0.w * w; f1.x += v1.x * w; f1.y += v1.y * w; f1.z += v1.z * w; f1.w += v1.w * w; }
        int offi; float wi;
        tapA(16 + tp, offi, wi);
        const float vi = (l8 < 3 && offi >= 0) ? __ldg(P.img + (size_t)l8 * P.img_h * P.img_w + offi) : 0.f;
        rgbc = tp == 0 ? vi * wi : rgbc + vi * wi;
      }
      // rgb_enc outputs 4*l8 .. 4*l8+3 of the 32 kept ones: [r,g,b, sin(..) ...]                     renderer.py:339,900-916
      const float r0 = __shfl_sync(0xffffffffu, rgbc, gbase + 0), r1 = __shfl_sync(0xffffffffu, rgbc, gbase + 1),
                  r2 = __shfl_sync(0xffffffffu, rgbc, gbase + 2);
      float enc[4];
#pragma unroll
      for (int e4 = 0; e4 < 4; ++e4) {
        const int o = c4 + e4;
        if (o < 3) enc[e4] = o == 0 ? r0 : (o == 1 ? r1 : r2);
        else {
          const int e = o - 3, m = e / 3, c = e - 3 * m;
          const float xc = c == 0 ? r0 : (c == 1 ? r1 : r2);
          enc[e4] = sinf(__fadd_rn((m & 1) ? kPi2 : 0.f, __fmul_rn(xc, (float)(1 << (m >> 1)))));
        }
      }
      if (active) {
        *reinterpret_cast<float4*>(comb + 0 * 96 + 32 + c4) = f0;
        *reinterpret_cast<float4*>(comb + 1 * 96 + 32 + c4) = f1;
        *reinterpret_cast<float4*>(comb + 2 * 96 + 32 + c4) = make_float4(enc[0], enc[1], enc[2], enc[3]);
        if (DBG && dbgf) {
          *reinterpret_cast<float4*>(dbgf + 96 + c4) = f0;
          *reinterpret_cast<float4*>(dbgf + 128 + c4) = f1;
          *reinterpret_cast<float4*>(dbgf + 160 + c4) = make_float4(enc[0], enc[1], enc[2], enc[3]);
        }
      }
    }
    // ---- 3-D pyramid ----
    {
      int coff = 0;
#pragma unroll
      for (int l = 0; l < 3; ++l) {
        int off[8]; float w[8];
#pragma unroll
        for (int tp = 0; tp < 8; ++tp) { off[tp] = __shfl_sync(0xffffffffu, offB[l], gbase + tp); w[tp] = __shfl_sync(0xffffffffu, wB[l], gbase + tp); }
        const float* vol = P.vol_cl[l] + c4;
        if (BWD) {
          if (P.g_vol_cl[l]) {
#pragma unroll
            for (int gsel = 0; gsel < 3; ++gsel) {
              if (gsel <= l) {
                const float4 g = *reinterpret_cast<const float4*>(f3 + coff + 32 * gsel + c4);
#pragma unroll
                for (int tp = 0; tp < 8; ++tp)
                  if (active && off[tp] >= 0) red_add4(P.g_vol_cl[l] + c4 + off[tp] + 32 * gsel, g, w[tp]);
              }
            }
          }
          coff += 32 * (l + 1);
          continue;
        }
#pragma unroll
        for (int gsel = 0; gsel < 3; ++gsel) {
          if (gsel <= l) {
            float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
            for (int tp = 0; tp < 8; ++tp) {
              const float4 val = off[tp] >= 0 ? __ldg(reinterpret_cast<const float4*>(vol + off[tp] + 32 * gsel)) : make_float4(0.f, 0.f, 0.f, 0.f);
              acc.x += val.x * w[tp]; acc.y += val.y * w[tp]; acc.z += val.z * w[tp]; acc.w += val.w * w[tp];
            }
            if (active) *reinterpret_cast<float4*>(f3 + coff + 32 * gsel + c4) = acc;
            if (DBG && dbgf && active) *reinterpret_cast<float4*>(dbgf + 192 + coff + 32 * gsel + c4) = acc;
          }
        }
        coff += 32 * (l + 1);
      }
    }
    if (active && !BWD) {
      float gval = 0.f;
      if (l8 == 0) gval = can[0]; else if (l8 == 1) gval = can[1]; else if (l8 == 2) gval = can[2];
      else if (l8 == 3) gval = cdir[0]; else if (l8 == 4) gval = cdir[1]; else if (l8 == 5) gval = cdir[2];
      P.geo[(size_t)lp * 8 + l8] = gval;
      if (DBG && l8 == 0 && gp < P.dbg_max) {
        if (P.dbg_vid3) P.dbg_vid3[gp] = vid3;
        if (P.dbg_can) { P.dbg_can[gp * 3] = can[0]; P.dbg_can[gp * 3 + 1] = can[1]; P.dbg_can[gp * 3 + 2] = can[2]; }
        if (P.dbg_cdir) { P.dbg_cdir[gp * 3] = cdir[0]; P.dbg_cdir[gp * 3 + 1] = cdir[1]; P.dbg_cdir[gp * 3 + 2] = cdir[2]; }
        if (P.dbg_uv) { P.dbg_uv[gp * 2] = u; P.dbg_uv[gp * 2 + 1] = v; }
      }
    }
  }
}


int run_point_gather(const GatherParams& P, cudaStream_t st) {
  if (P.np <= 0) return SHERF_OK;
  const bool dbg = P.dbg_feat || P.dbg_vid3 || P.dbg_can || P.dbg_cdir || P.dbg_uv;
  if (getenv("SHERF_GATHER_V1")) {
    const int blocks = min(ceil_div(P.np, 8), 148 * 16);
    k_point_gather<<<blocks, 256, 0, st>>>(P);
  } else {
    const int blocks = min(ceil_div(P.np, 32), 148 * 8);
    if (dbg) k_point_gather4<true, false><<<blocks, 256, 0, st>>>(P);
    else k_point_gather4<false, false><<<blocks, 256, 0, st>>>(P);
  }
  SHERF_LAUNCH_CHECK();
  return SHERF_OK;
}

// Adjoint of the three gathers: P.comb = dL/d(comb) [np][288], P.f3raw = dL/d(f3raw) [np][192]; P.g_* = channels-last gradient grids
// (accumulated into; NULL = that input needs no gradient).  F.grid_sample's backward w.r.t. its input, renderer.py:243,333,790-797.
int run_point_scatter(const GatherParams& P, cudaStream_t st) {
  if (P.np <= 0) return SHERF_OK;
  const int blocks = min(ceil_div(P.np, 32), 148 * 8);
  k_point_gather4<false, true><<<blocks, 256, 0, st>>>(P);
  SHERF_LAUNCH_CHECK();
  return SHERF_OK;
}

}  // namespace sherf
