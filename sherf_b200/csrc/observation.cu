// Observation preparation ("vertex-feature splat", SURVEY.md 8f rank 1): what TriPlaneGenerator.synthesis does once per observation
// image before it calls the renderer (triplane.py:105-137):
//   * project the observation-pose SMPL vertices into the observation camera and mark the camera-facing ones
//     (renderer.projection with faces, renderer.py:686-704; compute_normal / normalize_v3, renderer.py:40-63),
//   * sample the 2-D feature map and the image at the vertex pixels (F.grid_sample, align_corners=True, triplane.py:115-118),
//     rgb positional encoding truncated to 32 (:122), concat -> Conv1d(96,32,1) (:123-124), zero the back-facing vertices (:126),
//   * warp the vertices to the canonical ("big") pose (coarse_deform_target2c on the vertices themselves, :129-132),
//   * voxelise them at 5 mm inside the canonical box (prepare_sp_input, :174-217).
// The result is the SparseConvTensor of triplane.py:137 (features [V,32], indices [V,4]) that sherf_sparse_encode consumes.
#include "common.cuh"
#include "stages.cuh"
#include <climits>

namespace sherf {

struct ObsConst {
  float bounds[6];     // min xyz, max xyz of the canonical vertices -+ 0.05        triplane.py:177-186
  int out_sh[3];       // z, y, x                                                    triplane.py:199-201
};

// single block: bounds of the canonical vertices and the voxel-grid shape
__global__ void k_obs_bounds(const float* __restrict__ t_vertices, int V, ObsConst* __restrict__ oc, float* __restrict__ bounds_out) {
  __shared__ float smin[3][32], smax[3][32];
  float lo[3] = {3.0e38f, 3.0e38f, 3.0e38f}, hi[3] = {-3.0e38f, -3.0e38f, -3.0e38f};
  for (int v = threadIdx.x; v < V; v += blockDim.x)
#pragma unroll
    for (int k = 0; k < 3; ++k) { const float x = t_vertices[v * 3 + k]; lo[k] = fminf(lo[k], x); hi[k] = fmaxf(hi[k], x); }
#pragma unroll
  for (int k = 0; k < 3; ++k)
    for (int o = 16; o > 0; o >>= 1) { lo[k] = fminf(lo[k], __shfl_xor_sync(0xffffffffu, lo[k], o)); hi[k] = fmaxf(hi[k], __shfl_xor_sync(0xffffffffu, hi[k], o)); }
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (lane == 0)
#pragma unroll
    for (int k = 0; k < 3; ++k) { smin[k][w] = lo[k]; smax[k][w] = hi[k]; }
  __syncthreads();
  if (threadIdx.x == 0) {
    const int nw = blockDim.x >> 5;
    for (int k = 0; k < 3; ++k) {
      float a = smin[k][0], b = smax[k][0];
      for (int i = 1; i < nw; ++i) { a = fminf(a, smin[k][i]); b = fmaxf(b, smax[k][i]); }
      a = __fsub_rn(a, 0.05f); b = __fadd_rn(b, 0.05f);                 // big_box = True
      oc->bounds[k] = a; oc->bounds[3 + k] = b;
      bounds_out[k] = a; bounds_out[3 + k] = b;
    }
    for (int k = 0; k < 3; ++k) {                                         // dhw = xyz[2,1,0]
      const float ext = __fdiv_rn(__fsub_rn(oc->bounds[3 + (2 - k)], oc->bounds[2 - k]), 0.005f);
      const int c = (int)ceilf(ext);
      oc->out_sh[k] = (c | 31) + 1;
    }
  }
}

// thread per vertex: camera-space position, pixel, the reference's (non-accumulating) vertex normal, visibility; SMPL-space point
__global__ void k_obs_geometry(const float* __restrict__ verts, int V, const float* __restrict__ camR, const float* __restrict__ camT,
                               const float* __restrict__ camK, const int* __restrict__ faces, const int* __restrict__ last_face,
                               const float* __restrict__ Rsm, const float* __restrict__ Th, float* __restrict__ uv,
                               unsigned char* __restrict__ vmask, float* __restrict__ verts_smpl) {
  const int v = blockIdx.x * blockDim.x + threadIdx.x;
  if (v >= V) return;
  const float p[3] = {verts[v * 3], verts[v * 3 + 1], verts[v * 3 + 2]};
  float cam[3];
#pragma unroll
  for (int i = 0; i < 3; ++i) cam[i] = (camR[3 * i] * p[0] + camR[3 * i + 1] * p[1] + camR[3 * i + 2] * p[2]) + camT[i];
  // `norm[:, faces[:, k]] += n` does NOT accumulate over repeated indices (index_put semantics): for each corner slot k the LAST face
  // that lists the vertex there wins (sequential CPU order; renderer.py:58-60).  last_face[k][v] is that face or -1.
  float nrm[3] = {0.f, 0.f, 0.f};
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    const int f = last_face[k * V + v];
    if (f < 0) continue;
    const int i0 = faces[f * 3], i1 = faces[f * 3 + 1], i2 = faces[f * 3 + 2];
    const float a[3] = {verts[i1 * 3] - verts[i0 * 3], verts[i1 * 3 + 1] - verts[i0 * 3 + 1], verts[i1 * 3 + 2] - verts[i0 * 3 + 2]};
    const float b[3] = {verts[i2 * 3] - verts[i0 * 3], verts[i2 * 3 + 1] - verts[i0 * 3 + 1], verts[i2 * 3 + 2] - verts[i0 * 3 + 2]};
    float n[3] = {__fsub_rn(__fmul_rn(a[1], b[2]), __fmul_rn(a[2], b[1])), __fsub_rn(__fmul_rn(a[2], b[0]), __fmul_rn(a[0], b[2])),
                  __fsub_rn(__fmul_rn(a[0], b[1]), __fmul_rn(a[1], b[0]))};
    float len = sqrtf(__fadd_rn(__fadd_rn(__fmul_rn(n[0], n[0]), __fmul_rn(n[1], n[1])), __fmul_rn(n[2], n[2])));
    if (len < 1e-8f) len = 1e-8f;
#pragma unroll
    for (int c = 0; c < 3; ++c) nrm[c] = __fadd_rn(nrm[c], __fdiv_rn(n[c], len));
  }
  {
    float len = sqrtf(__fadd_rn(__fadd_rn(__fmul_rn(nrm[0], nrm[0]), __fmul_rn(nrm[1], nrm[1])), __fmul_rn(nrm[2], nrm[2])));
    if (len < 1e-8f) len = 1e-8f;
#pragma unroll
    for (int c = 0; c < 3; ++c) nrm[c] = __fdiv_rn(nrm[c], len);
  }
  float ncam[3];
#pragma unroll
  for (int i = 0; i < 3; ++i) ncam[i] = camR[3 * i] * nrm[0] + camR[3 * i + 1] * nrm[1] + camR[3 * i + 2] * nrm[2];
  vmask[v] = ((ncam[0] * cam[0] + ncam[1] * cam[1]) + ncam[2] * cam[2]) < 0.f ? 1 : 0;
  float pix[3];
#pragma unroll
  for (int i = 0; i < 3; ++i) pix[i] = camK[3 * i] * cam[0] + camK[3 * i + 1] * cam[1] + camK[3 * i + 2] * cam[2];
  const float zz = pix[2] + 1e-5f;
  uv[v * 2] = pix[0] / zz;
  uv[v * 2 + 1] = pix[1] / zz;
  float pw[3] = {__fsub_rn(p[0], Th[0]), __fsub_rn(p[1], Th[1]), __fsub_rn(p[2], Th[2])}, q[3];
  rowvec_mat3(pw, Rsm, q);
  verts_smpl[v * 3] = q[0]; verts_smpl[v * 3 + 1] = q[1]; verts_smpl[v * 3 + 2] = q[2];
}

// thread per vertex: exact nearest vertex of the set to itself (0 distance; a duplicated position resolves to the smallest index like
// every other knn of the path), per-vertex warp to the canonical pose, 5 mm voxel coordinate.
__global__ void __launch_bounds__(256) k_obs_canonical(const float* __restrict__ verts_smpl, int V, const VertexWarp* __restrict__ T1,
                                                       const ObsConst* __restrict__ oc, float* __restrict__ can_out,
                                                       int* __restrict__ coord) {
  __shared__ float sv[256 * 3];
  const int v = blockIdx.x * blockDim.x + threadIdx.x;
  const bool ok = v < V;
  const float qx = ok ? verts_smpl[v * 3] : 0.f, qy = ok ? verts_smpl[v * 3 + 1] : 0.f, qz = ok ? verts_smpl[v * 3 + 2] : 0.f;
  float best = 3.0e38f;
  int bid = 0;
  for (int base = 0; base < V; base += 256) {
    __syncthreads();
    const int n = min(256, V - base);
    for (int i = threadIdx.x; i < n * 3; i += blockDim.x) sv[i] = verts_smpl[base * 3 + i];
    __syncthreads();
    for (int j = 0; j < n; ++j) {
      const float d2 = dist2_xyz(qx, qy, qz, sv[j * 3], sv[j * 3 + 1], sv[j * 3 + 2]);
      if (d2 < best) { best = d2; bid = base + j; }                       // ascending scan + strict '<' = smallest index on ties
    }
  }
  if (!ok) return;
  float p[3] = {qx, qy, qz}, dummy[3] = {0.f, 0.f, 0.f};
  {
    const float* w = reinterpret_cast<const float*>(T1 + bid);
    const float a[3] = {p[0] - w[9], p[1] - w[10], p[2] - w[11]};
    float c[3];
    mat3_vec(w, a, c);
#pragma unroll
    for (int k = 0; k < 3; ++k) { c[k] = c[k] + w[12 + k]; c[k] = c[k] + w[15 + k]; c[k] = c[k] + w[18 + k]; }
    const float* Af = w + 21;
#pragma unroll
    for (int k = 0; k < 3; ++k) p[k] = (Af[4 * k] * c[0] + Af[4 * k + 1] * c[1] + Af[4 * k + 2] * c[2]) + Af[4 * k + 3];
    (void)dummy;
  }
  if (can_out) { can_out[v * 3] = p[0]; can_out[v * 3 + 1] = p[1]; can_out[v * 3 + 2] = p[2]; }
  coord[v * 4] = 0;                                                       // batch index (per-GPU batch is 1)
#pragma unroll
  for (int k = 0; k < 3; ++k)                                             // (z, y, x) = round((xyz[2-k] - min) / 0.005), half to even
    coord[v * 4 + 1 + k] = (int)rintf(__fdiv_rn(__fsub_rn(p[2 - k], oc->bounds[2 - k]), 0.005f));
}

// warp per vertex: bilinear taps (align_corners=True, zeros padding) of the NCHW feature map and image, rgb positional encoding
// (5 octaves, first 32 outputs), Conv1d(96, 32, 1) with lane = output channel, masked by the visibility.
__global__ void __launch_bounds__(256) k_obs_features(const float* __restrict__ uv, const unsigned char* __restrict__ vmask, int V,
                                                      const float* __restrict__ feat, int fc_, int fh, int fw, const float* __restrict__ img,
                                                      int ih, int iw, const float* __restrict__ Wp, const float* __restrict__ bp,
                                                      float* __restrict__ out) {
  __shared__ float sW[32 * 97];
  __shared__ float sx[8][96];
  for (int i = threadIdx.x; i < 32 * 96; i += blockDim.x) sW[(i / 96) * 97 + (i % 96)] = Wp[i];
  __syncthreads();
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int v = blockIdx.x * 8 + wid;
  if (v >= V) return;
  const float gx = 2.0f * uv[v * 2] / (float)iw - 1.0f, gy = 2.0f * uv[v * 2 + 1] / (float)ih - 1.0f;
  auto bilinear = [&](const float* __restrict__ plane, int H, int W) -> float {
    const float ix = (gx + 1.f) * 0.5f * (float)(W - 1), iy = (gy + 1.f) * 0.5f * (float)(H - 1);
    const float fx = floorf(ix), fy = floorf(iy);
    const int x0 = (int)fx, y0 = (int)fy;
    float acc = 0.f;
#pragma unroll
    for (int t = 0; t < 4; ++t) {                                          // nw, ne, sw, se: grid_sample's accumulation order
      const int cx = t & 1, cy = t >> 1;
      const int xx = x0 + cx, yy = y0 + cy;
      const float w = (cx ? ix - fx : (fx + 1.f) - ix) * (cy ? iy - fy : (fy + 1.f) - iy);
      const float val = (xx >= 0 && xx < W && yy >= 0 && yy < H) ? __ldg(plane + (size_t)yy * W + xx) : 0.f;
      acc = t == 0 ? val * w : acc + val * w;
    }
    return acc;
  };
  sx[wid][lane] = bilinear(feat + (size_t)lane * fh * fw, fh, fw);
  sx[wid][32 + lane] = bilinear(feat + (size_t)(32 + lane) * fh * fw, fh, fw);
  const float rgbc = lane < 3 ? bilinear(img + (size_t)lane * ih * iw, ih, iw) : 0.f;
  {
    const int e = lane - 3;
    const int m = e >= 0 ? e / 3 : 0, c = e >= 0 ? e - 3 * m : lane;
    const float xc = __shfl_sync(0xffffffffu, rgbc, c);
    sx[wid][64 + lane] = lane < 3 ? xc : sinf(__fadd_rn((m & 1) ? kPi2 : 0.f, __fmul_rn(xc, (float)(1 << (m >> 1)))));
  }
  __syncwarp();
  float acc = 0.f;
  for (int k = 0; k < 96; ++k) acc += sW[lane * 97 + k] * sx[wid][k];
  acc += bp[lane];
  out[(size_t)v * 32 + lane] = vmask[v] ? acc : 0.f;
}

size_t observation_scratch_bytes(int V, int maxcell) {
  size_t b = 4096;
  b += sizeof(FrameConst) + sizeof(ObsConst) + 512;
  b += sizeof(float) * (3 * kJoints * 16 + 3 * kJoints * 3 + 3 * kPoseFeat) + 1024;
  b += sizeof(float) * ((size_t)3 * V * 3 + (size_t)2 * V * 3 + (size_t)V * 3 + (size_t)V * 2) + 2048;
  b += sizeof(VertexWarp) * (size_t)2 * V + 512;
  b += sizeof(int) * ((size_t)2 * (maxcell + 1) + (size_t)2 * maxcell + (size_t)2 * (maxcell / 1024 + 2)) + 2048;
  b += sizeof(float4) * (size_t)2 * V + sizeof(int64_t) * 2 + (size_t)maxcell + 1024;
  b += (size_t)V + 256;
  return b;
}

int run_prepare_observation(const SherfSmplModel& smpl, const SherfObservation& ob, float* vert_feat, int32_t* coord, uint8_t* vmask_out,
                            float* bounds_out, int32_t* out_sh_host, float* can_out, void* scratch, size_t scratch_bytes, cudaStream_t st) {
  const int V = smpl.n_verts;
  constexpr int kMaxCell = 1 << 18;
  if (scratch_bytes < observation_scratch_bytes(V, kMaxCell)) { set_error("scratch arena too small for sherf_prepare_observation"); return SHERF_E_SCRATCH; }
  char* base = (char*)scratch;
  size_t off = 0;
  auto take = [&](size_t bytes) -> void* { off = (off + 255) & ~(size_t)255; void* p = base + off; off += bytes; return p; };
  { const size_t mis = ((size_t)base) & 255; if (mis) base += 256 - mis; }
  FrameTables ft{};
  ft.fc = (FrameConst*)take(sizeof(FrameConst));
  ObsConst* oc = (ObsConst*)take(sizeof(ObsConst));
  ft.A = (float*)take(sizeof(float) * 3 * kJoints * 16);
  ft.joints = (float*)take(sizeof(float) * 3 * kJoints * 3);
  ft.posefeat = (float*)take(sizeof(float) * 3 * kPoseFeat);
  ft.poff = (float*)take(sizeof(float) * (size_t)3 * V * 3);
  ft.soff = (float*)take(sizeof(float) * (size_t)2 * V * 3);
  ft.verts_smpl = (float*)take(sizeof(float) * (size_t)V * 3);
  float* uv = (float*)take(sizeof(float) * (size_t)V * 2);
  ft.T1 = (VertexWarp*)take(sizeof(VertexWarp) * (size_t)V);
  ft.T3 = (VertexWarp*)take(sizeof(VertexWarp) * (size_t)V);
  ft.g1_cell_start = (int*)take(sizeof(int) * (kMaxCell + 1));
  ft.g3_cell_start = (int*)take(sizeof(int) * (kMaxCell + 1));
  ft.g_cursor = (int*)take(sizeof(int) * (size_t)2 * kMaxCell);
  ft.g_block_sums = (int*)take(sizeof(int) * (size_t)2 * (kMaxCell / 1024 + 2));
  ft.g_total = (int64_t*)take(sizeof(int64_t) * 2);
  ft.g1_verts = (float4*)take(sizeof(float4) * (size_t)V);
  ft.g3_verts = (float4*)take(sizeof(float4) * (size_t)V);
  ft.g1_occ = (unsigned char*)take(kMaxCell);
  ft.maxcell = kMaxCell;
  ft.nnl_on = 0;                     // this path has no nearest-vertex queries
  unsigned char* vmask = vmask_out ? vmask_out : (unsigned char*)take(V);

  // the render path's per-vertex warp tables with the OBSERVATION pose in the "target" slot: T1[v] = observation SMPL space ->
  // canonical pose for points whose nearest vertex is v (renderer.py:558-621 applied to the vertices, triplane.py:132)
  SherfFrame fr;
  memset(&fr, 0, sizeof(fr));
  fr.target = ob.obs; fr.canonical = ob.canonical; fr.obs = ob.obs;
  fr.vertices = ob.obs_vertices; fr.t_vertices = ob.t_vertices;
  fr.obs_K = ob.obs_K; fr.obs_R = ob.obs_R; fr.obs_T = ob.obs_T;
  k_obs_bounds<<<1, 1024, 0, st>>>(ob.t_vertices, V, oc, bounds_out);
  SHERF_LAUNCH_CHECK();
  fr.t_world_bounds = bounds_out; fr.sp_bounds = bounds_out;              // read by k_frame_const only; not used on this path
  int rc = run_prologue_frame(fr, ft, st);
  if (rc) return rc;
  rc = run_prologue_tables(smpl, fr, ft, st);
  if (rc) return rc;
  k_obs_geometry<<<ceil_div(V, 128), 128, 0, st>>>(ob.obs_vertices, V, ob.obs_R, ob.obs_T, ob.obs_K, ob.faces, ob.last_face, ob.obs.R, ob.obs.Th,
                                                  uv, vmask, ft.verts_smpl);
  SHERF_LAUNCH_CHECK();
  k_obs_canonical<<<ceil_div(V, 256), 256, 0, st>>>(ft.verts_smpl, V, ft.T1, oc, can_out, coord);
  SHERF_LAUNCH_CHECK();
  k_obs_features<<<ceil_div(V, 8), 256, 0, st>>>(uv, vmask, V, ob.obs_feat, ob.feat_ch, ob.feat_h, ob.feat_w, ob.obs_img, ob.img_h, ob.img_w,
                                                ob.proj_w, ob.proj_b, vert_feat);
  SHERF_LAUNCH_CHECK();
  SHERF_CUDA_OK(cudaMemcpyAsync(out_sh_host, oc->out_sh, sizeof(int) * 3, cudaMemcpyDeviceToHost, st));
  SHERF_CUDA_OK(cudaStreamSynchronize(st));                               // out_sh sizes the caller's volumes: once per observation
  return SHERF_OK;
}


// ---- backward of the vertex features (SURVEY.md 8 f2): what autograd derives through triplane.py:115-126 --------------------------------
// out[v] = mask[v] (Wp [f64(uv_v) | pe32(rgb(uv_v))] + bp).  Gradients: Wp, bp (TriPlaneGenerator.conv1d_projection) and the 2-D feature
// map (bilinear adjoint = F.grid_sample's backward, red.add like torch).  The image and the vertex pixels are data.  Blocks stride over
// groups of 8 vertices (warp per vertex) and keep their share of dWp in registers: one atomicAdd per entry and block.
constexpr int kObsBwdBlocks = 64;
__global__ void __launch_bounds__(256) k_obs_features_bwd(const float* __restrict__ uv, const unsigned char* __restrict__ vmask, int V,
                                                          const float* __restrict__ feat, int fh, int fw, const float* __restrict__ img, int ih, int iw,
                                                          const float* __restrict__ Wp, const float* __restrict__ g_out, float* __restrict__ g_Wp,
                                                          float* __restrict__ g_bp, float* __restrict__ g_feat) {
  __shared__ float sW[32 * 97];
  __shared__ float sx[8][96];
  __shared__ float sg[8][32];
  for (int i = threadIdx.x; i < 32 * 96; i += blockDim.x) sW[(i / 96) * 97 + (i % 96)] = Wp[i];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  float accW[12], accB = 0.f;                          // entries threadIdx.x + 256 e of the [32][96] matrix; bias: threads < 32
#pragma unroll
  for (int e = 0; e < 12; ++e) accW[e] = 0.f;
  for (int v0 = blockIdx.x * 8; v0 < V; v0 += gridDim.x * 8) {
    __syncthreads();
    const int v = v0 + wid;
    float g = 0.f;
    if (v < V) {
      const float gx = 2.0f * uv[v * 2] / (float)iw - 1.0f, gy = 2.0f * uv[v * 2 + 1] / (float)ih - 1.0f;
      auto taps = [&](int H, int W, int (&xx)[4], int (&yy)[4], float (&w)[4]) {
        const float ix = (gx + 1.f) * 0.5f * (float)(W - 1), iy = (gy + 1.f) * 0.5f * (float)(H - 1);
        const float fx = floorf(ix), fy = floorf(iy);
#pragma unroll
        for (int t = 0; t < 4; ++t) {
          const int cx = t & 1, cy = t >> 1;
          xx[t] = (int)fx + cx; yy[t] = (int)fy + cy;
          w[t] = (cx ? ix - fx : (fx + 1.f) - ix) * (cy ? iy - fy : (fy + 1.f) - iy);
          if (xx[t] < 0 || xx[t] >= W || yy[t] < 0 || yy[t] >= H) w[t] = 0.f, xx[t] = 0, yy[t] = 0;
        }
      };
      int fxx[4], fyy[4], ixx[4], iyy[4];
      float fwt[4], iwt[4];
      taps(fh, fw, fxx, fyy, fwt);
      taps(ih, iw, ixx, iyy, iwt);
      auto bil = [&](const float* __restrict__ plane, int W, const int (&xx)[4], const int (&yy)[4], const float (&w)[4]) {
        float a = 0.f;
#pragma unroll
        for (int t = 0; t < 4; ++t) a += w[t] * __ldg(plane + (size_t)yy[t] * W + xx[t]);
        return a;
      };
      sx[wid][lane] = bil(feat + (size_t)lane * fh * fw, fw, fxx, fyy, fwt);
      sx[wid][32 + lane] = bil(feat + (size_t)(32 + lane) * fh * fw, fw, fxx, fyy, fwt);
      const float rgbc = lane < 3 ? bil(img + (size_t)lane * ih * iw, iw, ixx, iyy, iwt) : 0.f;
      {
        const int e = lane - 3;
        const int m = e >= 0 ? e / 3 : 0, c = e >= 0 ? e - 3 * m : lane;
        const float xc = __shfl_sync(0xffffffffu, rgbc, c);
        sx[wid][64 + lane] = lane < 3 ? xc : sinf(__fadd_rn((m & 1) ? kPi2 : 0.f, __fmul_rn(xc, (float)(1 << (m >> 1)))));
      }
      g = vmask[v] ? g_out[(size_t)v * 32 + lane] : 0.f;
      // d f64[k] = sum_out Wp[out][k] g[out]  ->  bilinear adjoint into the feature map
      if (g_feat) {
        float d0 = 0.f, d1 = 0.f;
        for (int o = 0; o < 32; ++o) {
          const float go = __shfl_sync(0xffffffffu, g, o);
          d0 = fmaf(sW[o * 97 + lane], go, d0);
          d1 = fmaf(sW[o * 97 + 32 + lane], go, d1);
        }
#pragma unroll
        for (int t = 0; t < 4; ++t)
          if (fwt[t] != 0.f) {
            atomicAdd(g_feat + ((size_t)lane * fh + fyy[t]) * fw + fxx[t], fwt[t] * d0);
            atomicAdd(g_feat + ((size_t)(32 + lane) * fh + fyy[t]) * fw + fxx[t], fwt[t] * d1);
          }
      }
    } else {
      sx[wid][lane] = 0.f; sx[wid][32 + lane] = 0.f; sx[wid][64 + lane] = 0.f;
    }
    sg[wid][lane] = g;
    __syncthreads();
#pragma unroll
    for (int e = 0; e < 12; ++e) {
      const int idx = threadIdx.x + 256 * e, o = idx / 96, k = idx - o * 96;
      float a = 0.f;
#pragma unroll
      for (int q = 0; q < 8; ++q) a = fmaf(sg[q][o], sx[q][k], a);
      accW[e] += a;
    }
    if (threadIdx.x < 32) {
#pragma unroll
      for (int q = 0; q < 8; ++q) accB += sg[q][threadIdx.x];
    }
  }
  if (g_Wp)
#pragma unroll
    for (int e = 0; e < 12; ++e) atomicAdd(g_Wp + threadIdx.x + 256 * e, accW[e]);
  if (g_bp && threadIdx.x < 32) atomicAdd(g_bp + threadIdx.x, accB);
}

int run_prepare_observation_backward(const SherfSmplModel& smpl, const SherfObservation& ob, const float* g_vert_feat, float* g_proj_w, float* g_proj_b,
                                     float* g_obs_feat, void* scratch, size_t scratch_bytes, cudaStream_t st) {
  const int V = smpl.n_verts;
  char* base = (char*)scratch;
  { const size_t mis = ((size_t)base) & 255; if (mis) base += 256 - mis; }
  size_t off = 0;
  auto take = [&](size_t bytes) -> void* { off = (off + 255) & ~(size_t)255; void* p = base + off; off += bytes; return p; };
  float* uv = (float*)take(sizeof(float) * (size_t)V * 2);
  float* verts_smpl = (float*)take(sizeof(float) * (size_t)V * 3);
  unsigned char* vmask = (unsigned char*)take(V);
  if (off + 512 > scratch_bytes) { set_error("scratch arena too small for sherf_prepare_observation_backward"); return SHERF_E_SCRATCH; }
  k_obs_geometry<<<ceil_div(V, 128), 128, 0, st>>>(ob.obs_vertices, V, ob.obs_R, ob.obs_T, ob.obs_K, ob.faces, ob.last_face, ob.obs.R, ob.obs.Th,
                                                  uv, vmask, verts_smpl);
  SHERF_LAUNCH_CHECK();
  if (g_proj_w) SHERF_CUDA_OK(cudaMemsetAsync(g_proj_w, 0, sizeof(float) * 32 * 96, st));
  if (g_proj_b) SHERF_CUDA_OK(cudaMemsetAsync(g_proj_b, 0, sizeof(float) * 32, st));
  if (g_obs_feat) SHERF_CUDA_OK(cudaMemsetAsync(g_obs_feat, 0, sizeof(float) * (size_t)ob.feat_ch * ob.feat_h * ob.feat_w, st));
  k_obs_features_bwd<<<kObsBwdBlocks, 256, 0, st>>>(uv, vmask, V, ob.obs_feat, ob.feat_h, ob.feat_w, ob.obs_img, ob.img_h, ob.img_w, ob.proj_w,
                                                   g_vert_feat, g_proj_w, g_proj_b, g_obs_feat);
  SHERF_LAUNCH_CHECK();
  return SHERF_OK;
}

}  // namespace sherf
