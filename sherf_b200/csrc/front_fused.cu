// The "front" kernel of the point stages: warp + gather + feature fusion in ONE kernel, nothing in between touches HBM.
//   renderer.py:323-350  inverse-LBS warp to canonical space, canonical -> observation warp, projection, pixel-aligned 2-D gather,
//                        3-D pyramid gather, conv1d_projection 192 -> 96
//   renderer.py:402,423-424  tri-plane gather, conv1d_reprojection 96 -> 32 over [tri_k | f2d_k | f3d_k], k = 0..2
// Output: the three 32-channel tokens of every surviving point (384 B) + its canonical position / direction (32 B).  The gathered
// features (1.5 KB per point through HBM in round 1: 770 MB written by the gather + 810 MB read back by the fusion kernel per 524 288
// points, profiles/r1_ab) now go from the gather lanes' registers straight into the tensor-core operand slots in shared memory.
//
// One CTA = one 128-point tile at a time, 16 warps, TWO CTAs per SM (one CTA's gather overlaps the other's MMA / epilogue phases).
//   gather : FOUR lanes per point (lane l4 owns channels 8*l4..8*l4+7 of every 32-channel group: two 16-byte loads per tap), so a warp
//            covers 8 points and the 16 warps exactly one 128-point tile -- every per-point instruction (geometry, tap set-up, shuffles,
//            address arithmetic) serves 8 points (the kernel is instruction-issue bound, not memory bound: with the tap loads, the MMAs
//            and the knn-#3 search knocked out it still took 73 % of its time, profiles/README.md r2 knock-outs).  The tile is produced
//            in twelve 32-channel CHUNKS (six of the 3-D pyramid, three tri-planes, two feature-map halves, the rgb encoding); a chunk's
//            values are split into bf16 hi / lo and stored as the K-major no-swizzle UMMA operand (one 16-byte core-matrix row per lane
//            and part: conflict-free with LBO = 2080).
//   MMA    : bf16 split products a_hi*w_hi + a_lo*w_hi + a_hi*w_lo on tcgen05 kind::f16, fp32 accumulators in TMEM; chunk c's MMAs
//            run while chunk c+1 is gathered (two operand slots; projection weights stream through a two-stage TMA ring, 12 KB per
//            chunk from L2; reprojection weights resident).  Warp 0 issues (after producing its own part of the chunk).
//   E1     : projected 3-D feature = D1 + bias -> bf16 hi (shared memory) / lo (TMEM) operand of the reprojection; never leaves the SM.
//   E2     : tokens = D2 + bias -> global.
#include "common.cuh"
#include "stages.cuh"
#include "umma.cuh"
#include <cuda_bf16.h>
#include <cstdlib>

namespace sherf {

namespace fr {
constexpr uint32_t kLboA = 2080;                          // streamed operand chunks: 8-byte stores from the gather lanes are conflict-free
constexpr uint32_t kChunkHalf = 4 * kLboA;                // hi (or lo) part of one 32-channel chunk: 4 core-matrix columns
constexpr uint32_t kChunk = 2 * kChunkHalf;
constexpr int kSlots = 3;                                  // operand slots: a producer may run two chunks ahead of the slowest warp of the CTA
constexpr uint32_t kLboF = 2048;                          // projected 3-D feature (16-byte stores, thread = row: conflict-free without padding)
constexpr uint32_t kF3d = kSlots * kChunk;                // 12 core-matrix columns (96 channels), hi part
constexpr uint32_t kWr = kF3d + 12 * kLboF;               // reprojection weights: 3 source blocks x (hi 2048 B | lo 2048 B)
constexpr uint32_t kWrBlock = 4096;
constexpr uint32_t kWp = kWr + 3 * kWrBlock;              // projection weight ring: 2 stages x (hi 6144 B | lo 6144 B)
constexpr uint32_t kWpStage = 12288;
constexpr uint32_t kSmemBytes = kWp + 2 * kWpStage;
constexpr uint32_t kD1 = 0, kD2 = 96, kF3dLo = 192;       // tensor-memory columns (256 allocated)
constexpr int kThreads = 512;
}  // namespace fr

struct FrontArgs {
  GatherParams G;
  const unsigned char* wblob;          // 6 projection chunks (hi | lo), then 3 reprojection blocks (hi | lo)
  const float *bp, *br;                // conv1d_projection bias [96], conv1d_reprojection bias [32]
  float* tok;                          // [np][3][32]
  int knock;                           // diagnostics only (SHERF_FRONT_KNOCK): 1 no knn-#3 search, 2 no tap loads, 4 no MMAs, 8 no phase A geometry
};

__device__ __forceinline__ void fr_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(umma::smem_u32(bar)) : "memory");
}

__device__ __forceinline__ void fr_apply_warp(const VertexWarp* __restrict__ Tp, float p[3], float d[3], bool with_dir) {
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

__device__ __forceinline__ void fr_grp_lexmin(float& d, int& id) {      // over the 4 lanes of a point
#pragma unroll
  for (int o = 2; o > 0; o >>= 1) {
    const float od = __shfl_xor_sync(0xffffffffu, d, o);
    const int oi = __shfl_xor_sync(0xffffffffu, id, o);
    if (od < d || (od == d && oi < id)) { d = od; id = oi; }
  }
}

// exact K=1 search over the canonical vertices, 4 lanes per point: over the candidate list of the point's sub-cell (lane l4 takes entries
// l4, l4 + 4, ...), or, where the sub-cell has no list, over the grid cells within the distance of the seed, the nearest posed vertex
// (gather.cu: nn_seeded8)
__device__ __forceinline__ int fr_nn_seeded4(const GridDesc& g, const int* __restrict__ cell_start, const float4* __restrict__ gv,
                                             const NnLists& nl, const float* __restrict__ t_vertices, float qx, float qy, float qz, int l4,
                                             int seed) {
  const int li = nl.slot ? nnl_index(g, nl.slot, qx, qy, qz) : -1;
  const int ln = li >= 0 ? nl.len[li] : -1;
  if (ln > 0) {
    float best = 3.0e38f;
    int bid = 0x7fffffff;
    const float4* e = nl.ent + (size_t)li * kNnlCap;
    for (int k = l4; k < ln; k += 4) {
      const float4 v = e[k];
      const float d2 = dist2_xyz(qx, qy, qz, v.x, v.y, v.z);
      const int id = __float_as_int(v.w);
      if (d2 < best || (d2 == best && id < bid)) { best = d2; bid = id; }
    }
    fr_grp_lexmin(best, bid);
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
  for (int cc = l4; cc < ncells; cc += 4) {
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
  fr_grp_lexmin(best, bid);
  return bid;
}

template <bool DBG>
__global__ void __launch_bounds__(fr::kThreads, 2) k_front_fused(const FrontArgs a) {
  extern __shared__ __align__(128) unsigned char smem[];
  __shared__ FrameConst fc;
  __shared__ __align__(8) uint64_t a_full[fr::kSlots], a_free[fr::kSlots], w_full[2], w_free[2], acc1, acc2, f3d_ready;
  __shared__ uint32_t tmem_base_s;
  __shared__ float s_bp[96], s_br[32];
  __shared__ float s_pt[128][6];      // per point: gn xyz | cn xyz (see phase A)
  const GatherParams& P = a.G;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, l4 = lane & 3, gbase = lane & 28;
  const int c8 = 8 * l4;

  for (int i = tid; i < (int)(sizeof(FrameConst) / 4); i += blockDim.x) ((int*)&fc)[i] = ((const int*)P.fc)[i];
  if (tid == 0) {
    for (int b = 0; b < fr::kSlots; ++b) { umma::mbar_init(&a_full[b], fr::kThreads); umma::mbar_init(&a_free[b], 1); }
    for (int b = 0; b < 2; ++b) { umma::mbar_init(&w_full[b], 1); umma::mbar_init(&w_free[b], 1); }
    umma::mbar_init(&acc1, 1); umma::mbar_init(&acc2, 1); umma::mbar_init(&f3d_ready, fr::kThreads);
    umma::fence_mbar_init();
  }
  if (warp == 0) umma::tmem_alloc(&tmem_base_s, 256);
  for (int i = tid; i < (int)(3 * fr::kWrBlock / 16); i += blockDim.x)
    reinterpret_cast<uint4*>(smem + fr::kWr)[i] = __ldg(reinterpret_cast<const uint4*>(a.wblob + 6 * fr::kWpStage) + i);
  if (tid < 96) s_bp[tid] = a.bp[tid];
  if (tid < 32) s_br[tid] = a.br[tid];
  umma::fence_proxy_async_smem();
  umma::tc_fence_before_sync();
  __syncthreads();
  umma::tc_fence_after_sync();
  const uint32_t tmem_base = tmem_base_s;
  const uint32_t sbase = umma::smem_u32(smem);
  const int np = resolve_np(P.np, P.dc);
  const int ntiles = (np + 127) / 128;
  const uint32_t el = umma::elect_one();                   // warp 0 stays converged in the issue code; one lane issues
  const int gi = warp * 8 + (lane >> 2);                   // lane group = row 0..127 of the tile
  // E1 / E2 role of this thread: TMEM lane quarter = warp & 3, 24-column group = warp >> 2
  const int erow = 32 * (warp & 3) + lane, ecg = warp >> 2;
  const uint32_t etb = tmem_base + ((uint32_t)(32 * (warp & 3)) << 16);

  if (warp == 0 && lane == 0 && (int)blockIdx.x < ntiles) {          // projection weight chunks 0, 1 of the first tile
    for (int s = 0; s < 2; ++s) {
      umma::mbar_arrive_expect_tx(&w_full[s], fr::kWpStage);
      umma::bulk_g2s(smem + fr::kWp + s * fr::kWpStage, a.wblob + (size_t)s * fr::kWpStage, fr::kWpStage, &w_full[s]);
    }
  }

  // split products of one 32-channel block: D[:, dcol:+N] (+)= A * W^T, A hi from shared memory, A lo from shared or tensor memory
  auto gemm32 = [&](uint32_t a_hi_addr, uint32_t a_lbo, bool lo_in_tmem, uint32_t a_lo, uint32_t w_hi_addr, uint32_t w_lo_addr, int N, uint32_t dcol,
                    uint32_t acc0) {
    const uint32_t idesc = umma::make_idesc_bf16(128, N);
    const uint32_t w_lbo = (uint32_t)N * 16u;
    const uint64_t ah0 = umma::make_smem_desc(a_hi_addr, a_lbo, 128u);
    const uint64_t al0 = umma::make_smem_desc(a_lo, a_lbo, 128u);
    const uint64_t wh0 = umma::make_smem_desc(w_hi_addr, w_lbo, 128u);
    const uint64_t wl0 = umma::make_smem_desc(w_lo_addr, w_lbo, 128u);
    const uint64_t da = (uint64_t)((2u * a_lbo) >> 4), dw = (uint64_t)((2u * w_lbo) >> 4);
#pragma unroll
    for (int st = 0; st < 2; ++st) {
      const uint32_t acc = st == 0 ? acc0 : 1u;
      if (lo_in_tmem) umma::mma_bf16_ts_e(tmem_base + dcol, tmem_base + a_lo + (uint32_t)st * 8u, wh0 + (uint64_t)st * dw, idesc, acc, el);
      else umma::mma_bf16_ss_e(tmem_base + dcol, al0 + (uint64_t)st * da, wh0 + (uint64_t)st * dw, idesc, acc, el);
      umma::mma_bf16_ss_e(tmem_base + dcol, ah0 + (uint64_t)st * da, wl0 + (uint64_t)st * dw, idesc, 1u, el);
      umma::mma_bf16_ss_e(tmem_base + dcol, ah0 + (uint64_t)st * da, wh0 + (uint64_t)st * dw, idesc, 1u, el);
    }
  };

  uint32_t ti = 0;                                          // tile iteration of this CTA (barrier phase bookkeeping)
  for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x, ++ti) {
    const bool has_next = tile + (int)gridDim.x < ntiles;
    // =========================== phase A: geometry of this lane group's point (row gi of the tile) ===========================
    // The per-point coordinates every later chunk needs -- 3-D grid coordinates gn (renderer.py:544-556), tri-plane coordinates cn
    // (renderer.py:218-243), observation pixel uv (renderer.py:686-704) -- go to shared memory (s_pt[row][8]); the chunk loop reloads
    // what it needs, so nothing of a point stays in registers between chunks.
    bool act;
    int64_t gpt;
    float pu, pv;                                            // observation pixel of the point (used by chunk 9's tap set-up)
    {
      const int lp_raw = tile * 128 + gi;
      act = lp_raw < np;
      const int lp = act ? lp_raw : np - 1;                  // rows beyond the list shadow the last point; nothing of them is stored
      const int64_t gp = P.p0 + lp;
      gpt = gp;
      const int s = P.point_sample[gp];
      const int n = s / P.S, i = s - n * P.S;
      const float t = P.depths ? P.depths[s] : sample_depth(P.nearv[n], P.farv[n], i, P.S);
      float dray[3] = {P.dirs[n * 3], P.dirs[n * 3 + 1], P.dirs[n * 3 + 2]};
      float pw[3], q[3], vd[3];
#pragma unroll
      for (int k = 0; k < 3; ++k) pw[k] = __fsub_rn(mul_add_sep(t, dray[k], P.origins[n * 3 + k]), fc.Th_tgt[k]);
      rowvec_mat3(pw, fc.R_tgt, q);
      rowvec_mat3(dray, fc.R_tgt, vd);
      float cn[3] = {q[0], q[1], q[2]}, cdir[3] = {vd[0], vd[1], vd[2]};
      const int vid1 = P.point_vid[gp];
      if (!(a.knock & 8)) fr_apply_warp(P.T1 + vid1, cn, cdir, true);                  // target -> canonical   renderer.py:558-621
      const int vid3 = (a.knock & 1) ? vid1 : fr_nn_seeded4(fc.g3, P.g3_start, P.g3_verts, P.nl3, P.t_vertices, cn[0], cn[1], cn[2], l4, vid1);
      float ps[3] = {cn[0], cn[1], cn[2]}, dummy[3] = {0.f, 0.f, 0.f};
      fr_apply_warp(P.T3 + vid3, ps, dummy, false);                                    // canonical -> observation   renderer.py:623-684
      float world[3], cam[3], pix[3];
#pragma unroll
      for (int k = 0; k < 3; ++k) world[k] = (ps[0] * fc.Rinv_obs[k] + ps[1] * fc.Rinv_obs[3 + k] + ps[2] * fc.Rinv_obs[6 + k]) + fc.Th_obs[k];
      mat3_vec(fc.camR, world, cam);
#pragma unroll
      for (int k = 0; k < 3; ++k) cam[k] += fc.camT[k];
      mat3_vec(fc.camK, cam, pix);                                                     // renderer.py:686-704
      const float zz = pix[2] + 1e-5f;
      const float u = pix[0] / zz, v = pix[1] / zz;
      {
        // s_pt[row] = gn xyz | cn xyz with gn_k = ((can_k - bounds_min_k) / 0.005) / out_sh[2-k] * 2 - 1 and
        // cn_k = 2 (can_k - lo_k) / (hi_k - lo_k) - 1.  Lane l4 < 3 writes gn_l4 and cn_l4.
        const int k3 = l4 < 3 ? l4 : 0;
        const float ck = k3 == 0 ? cn[0] : (k3 == 1 ? cn[1] : cn[2]);
        const float gnv = ((ck - fc.spb_min[k3]) / 0.005f) / fc.out_sh[2 - k3] * 2.f - 1.f;
        const float cnv = 2.f * (ck - fc.twb_min[k3]) / (fc.twb_max[k3] - fc.twb_min[k3]) - 1.f;
        if (l4 < 3) { s_pt[gi][l4] = gnv; s_pt[gi][3 + l4] = cnv; }
        pu = u; pv = v;
      }
      if (act) {
        if (l4 < 3) {
          P.geo[(size_t)lp * 8 + l4] = l4 == 0 ? cn[0] : (l4 == 1 ? cn[1] : cn[2]);
          P.geo[(size_t)lp * 8 + 3 + l4] = l4 == 0 ? cdir[0] : (l4 == 1 ? cdir[1] : cdir[2]);
        } else {
          P.geo[(size_t)lp * 8 + 6] = 0.f;
          P.geo[(size_t)lp * 8 + 7] = 0.f;
        }
        if (DBG && l4 == 0 && gp < P.dbg_max) {
          if (P.dbg_vid3) P.dbg_vid3[gp] = vid3;
          if (P.dbg_can) { P.dbg_can[gp * 3] = cn[0]; P.dbg_can[gp * 3 + 1] = cn[1]; P.dbg_can[gp * 3 + 2] = cn[2]; }
          if (P.dbg_cdir) { P.dbg_cdir[gp * 3] = cdir[0]; P.dbg_cdir[gp * 3 + 1] = cdir[1]; P.dbg_cdir[gp * 3 + 2] = cdir[2]; }
          if (P.dbg_uv) { P.dbg_uv[gp * 2] = u; P.dbg_uv[gp * 2 + 1] = v; }
        }
      }
    }
    __syncwarp();                                            // s_pt rows of this lane group are read back by the same 4 lanes

    // =========================== the twelve chunks: ONE loop body (compact code: the unrolled form was 24 500 instructions) ===========================
    //   c = 0..5  3-D pyramid (level, 32-channel group) = (0,0) (1,0) (1,1) (2,0) (2,1) (2,2)   renderer.py:544-556,762-797
    //   c = 6..8  tri-plane k = c - 6 (align_corners=False)                                     renderer.py:234-243
    //   c = 9,10  2-D feature map channels 0-31 / 32-63, c = 11 rgb encoding (align_corners=True, uv normalised by the IMAGE size) renderer.py:331-340
    // Tap registers: lane l4 holds taps l4 and l4 + 4 of the current 8-tap set (3-D), or tap l4 of a 4-tap set (2-D) in slot 0.
    int offT[2] = {-1, -1}, offI = -1;
    float wT[2] = {0.f, 0.f}, wI = 0.f;
    const float* pt = s_pt[gi];
#pragma unroll 1
    for (int c = 0; c < 12; ++c) {
      // ---- tap setup where a new sample set starts ----
      if (c == 0 || c == 1 || c == 3) {
        const int l = c == 0 ? 0 : (c == 1 ? 1 : 2);
        const int D = P.vol_d[l], Hh = P.vol_h[l], Ww = P.vol_w[l], C = P.vol_ch[l];
        const float ix = (pt[0] + 1.f) * 0.5f * (float)(Ww - 1), iy = (pt[1] + 1.f) * 0.5f * (float)(Hh - 1), iz = (pt[2] + 1.f) * 0.5f * (float)(D - 1);
        const float fx = floorf(ix), fy = floorf(iy), fz = floorf(iz);
        const int bx = l4 & 1, by = (l4 >> 1) & 1;             // corner index = l4 + 4 * slot: bit0 x, bit1 y, bit2 z (= slot)
        const int xx = (int)fx + bx, yy = (int)fy + by;
        const float wxy = (bx ? ix - fx : (fx + 1.f) - ix) * (by ? iy - fy : (fy + 1.f) - iy);
        const bool inxy = xx >= 0 && xx < Ww && yy >= 0 && yy < Hh;
#pragma unroll
        for (int sl = 0; sl < 2; ++sl) {
          const int zz2 = (int)fz + sl;
          wT[sl] = wxy * (sl ? iz - fz : (fz + 1.f) - iz);
          offT[sl] = (inxy && zz2 >= 0 && zz2 < D) ? ((zz2 * Hh + yy) * Ww + xx) * C : -1;
        }
      } else if (c >= 6 && c <= 8) {
        const int k = c - 6;
        const int Ww = P.plane_w, Hh = P.plane_h;
        const float px = k == 2 ? pt[5] : pt[3], py = k == 1 ? pt[5] : pt[4];
        const float ix = ((px + 1.f) * (float)Ww - 1.f) * 0.5f, iy = ((py + 1.f) * (float)Hh - 1.f) * 0.5f;
        const float fx = floorf(ix), fy = floorf(iy);
        const int cxb = l4 & 1, cyb = (l4 >> 1) & 1;
        const int xx = (int)fx + cxb, yy = (int)fy + cyb;
        wT[0] = (cxb ? ix - fx : (fx + 1.f) - ix) * (cyb ? iy - fy : (fy + 1.f) - iy);
        offT[0] = (xx >= 0 && xx < Ww && yy >= 0 && yy < Hh) ? (yy * Ww + xx) * 32 : -1;
      } else if (c == 9) {
        const float gx = 2.0f * pu / (float)P.img_w - 1.0f, gy = 2.0f * pv / (float)P.img_h - 1.0f;
        const int cxb = l4 & 1, cyb = (l4 >> 1) & 1;
        {
          const int Ww = P.feat_w, Hh = P.feat_h;
          const float ix = (gx + 1.f) * 0.5f * (float)(Ww - 1), iy = (gy + 1.f) * 0.5f * (float)(Hh - 1);
          const float fx = floorf(ix), fy = floorf(iy);
          const int xx = (int)fx + cxb, yy = (int)fy + cyb;
          wT[0] = (cxb ? ix - fx : (fx + 1.f) - ix) * (cyb ? iy - fy : (fy + 1.f) - iy);
          offT[0] = (xx >= 0 && xx < Ww && yy >= 0 && yy < Hh) ? (yy * Ww + xx) * P.feat_ch : -1;
        }
        {
          const int Ww = P.img_w, Hh = P.img_h;
          const float ix = (gx + 1.f) * 0.5f * (float)(Ww - 1), iy = (gy + 1.f) * 0.5f * (float)(Hh - 1);
          const float fx = floorf(ix), fy = floorf(iy);
          const int xx = (int)fx + cxb, yy = (int)fy + cyb;
          wI = (cxb ? ix - fx : (fx + 1.f) - ix) * (cyb ? iy - fy : (fy + 1.f) - iy);
          offI = (xx >= 0 && xx < Ww && yy >= 0 && yy < Hh) ? (yy * Ww + xx) : -1;
        }
      }
      // ---- operand slot b = c % 3, used for the (ti * 4 + c / 3)-th time: wait until the MMAs that read it three chunks ago have completed ----
      const int b = c % fr::kSlots;
      const uint32_t u = ti * 4u + (uint32_t)(c / fr::kSlots);
      umma::mbar_wait_backoff(&a_free[b], (u & 1u) ^ 1u);
      if (warp == 0 && c >= 2 && c <= 7 && (c <= 5 || has_next)) {
        // projection-weight stage ws = c & 1 is refilled once the MMAs of the chunk that used it last (two chunks ago) have completed:
        // with this tile's chunk c, or the next tile's chunk 0 / 1 (predicated issue, no lane branch)
        const int ws = c & 1, wc = c <= 5 ? c : c - 6;
        const uint32_t fill = c <= 5 ? ti * 3u + (uint32_t)(c >> 1) : (ti + 1u) * 3u;
        umma::mbar_wait(&w_free[ws], (fill - 1u) & 1u);
        umma::mbar_arrive_expect_tx_e(&w_full[ws], fr::kWpStage, el);
        umma::bulk_g2s_e(smem + fr::kWp + ws * fr::kWpStage, a.wblob + (size_t)wc * fr::kWpStage, fr::kWpStage, &w_full[ws], el);
      }
      unsigned char* buf = smem + (uint32_t)b * fr::kChunk;
      // ---- gather the chunk's 32 channels of the point: 4 lanes x 2 float4 per tap ----
      const float* src;
      int dbg_col;
      if (c < 6) { const int l = c == 0 ? 0 : (c < 3 ? 1 : 2); src = P.vol_cl[l] + 32 * (c - (l == 0 ? 0 : (l == 1 ? 1 : 3))); dbg_col = 192 + 32 * c; }
      else if (c < 9) { src = P.planes_cl + (size_t)(c - 6) * P.plane_h * P.plane_w * 32; dbg_col = 32 * (c - 6); }
      else { src = P.feat_cl + 32 * (c - 9); dbg_col = 96 + 32 * (c - 9); }
      src += c8;
      float4 acc0 = make_float4(0.f, 0.f, 0.f, 0.f), acc1v = make_float4(0.f, 0.f, 0.f, 0.f);      // channels c8 .. c8+3 and c8+4 .. c8+7
      if (c < 11) {
        // taps in grid_sample's accumulation order (tap t sits in lane t & 3, register slot t >> 2); the four loads-pairs of a half set are
        // issued back to back before the blend
#pragma unroll
        for (int hs = 0; hs < 2; ++hs) {
          if (hs == 0 || c < 6) {                               // 2-D sets have four taps only
            int off[4]; float w[4];
#pragma unroll
            for (int tp = 0; tp < 4; ++tp) {
              off[tp] = __shfl_sync(0xffffffffu, hs ? offT[1] : offT[0], gbase + tp);
              w[tp] = __shfl_sync(0xffffffffu, hs ? wT[1] : wT[0], gbase + tp);
            }
            float4 v0[4], v1[4];
#pragma unroll
            for (int tp = 0; tp < 4; ++tp) {
              const bool ok = off[tp] >= 0 && !(a.knock & 2);
              v0[tp] = ok ? __ldg(reinterpret_cast<const float4*>(src + off[tp])) : make_float4(0.f, 0.f, 0.f, 0.f);
              v1[tp] = ok ? __ldg(reinterpret_cast<const float4*>(src + off[tp]) + 1) : make_float4(0.f, 0.f, 0.f, 0.f);
            }
#pragma unroll
            for (int tp = 0; tp < 4; ++tp) {
              if (tp == 0 && hs == 0 && c >= 6) {               // the 2-D form starts from the first product, the 3-D form from zero
                acc0.x = v0[0].x * w[0]; acc0.y = v0[0].y * w[0]; acc0.z = v0[0].z * w[0]; acc0.w = v0[0].w * w[0];
                acc1v.x = v1[0].x * w[0]; acc1v.y = v1[0].y * w[0]; acc1v.z = v1[0].z * w[0]; acc1v.w = v1[0].w * w[0];
              } else {
                acc0.x += v0[tp].x * w[tp]; acc0.y += v0[tp].y * w[tp]; acc0.z += v0[tp].z * w[tp]; acc0.w += v0[tp].w * w[tp];
                acc1v.x += v1[tp].x * w[tp]; acc1v.y += v1[tp].y * w[tp]; acc1v.z += v1[tp].z * w[tp]; acc1v.w += v1[tp].w * w[tp];
              }
            }
          }
        }
      } else {
        float rgbc = 0.f;
#pragma unroll
        for (int tp = 0; tp < 4; ++tp) {
          const int offi = __shfl_sync(0xffffffffu, offI, gbase + tp);
          const float wi = __shfl_sync(0xffffffffu, wI, gbase + tp);
          const float vi = (l4 < 3 && offi >= 0) ? __ldg(P.img + (size_t)l4 * P.img_h * P.img_w + offi) : 0.f;
          rgbc = tp == 0 ? vi * wi : rgbc + vi * wi;
        }
        // rgb_enc outputs 8*l4 .. 8*l4+7 of the 32 kept ones: [r, g, b, sin(..) ...]                        renderer.py:339,900-916
        const float r0 = __shfl_sync(0xffffffffu, rgbc, gbase + 0), r1 = __shfl_sync(0xffffffffu, rgbc, gbase + 1),
                    r2 = __shfl_sync(0xffffffffu, rgbc, gbase + 2);
        float enc[8];
#pragma unroll
        for (int e8 = 0; e8 < 8; ++e8) {
          const int o = c8 + e8;
          if (o < 3) enc[e8] = o == 0 ? r0 : (o == 1 ? r1 : r2);
          else {
            const int e = o - 3, m = e / 3, cc = e - 3 * m;
            const float xc = cc == 0 ? r0 : (cc == 1 ? r1 : r2);
            enc[e8] = sinf(__fadd_rn((m & 1) ? kPi2 : 0.f, __fmul_rn(xc, (float)(1 << (m >> 1)))));
          }
        }
        acc0 = make_float4(enc[0], enc[1], enc[2], enc[3]);
        acc1v = make_float4(enc[4], enc[5], enc[6], enc[7]);
        dbg_col = 160;
      }
      {                                                        // 8 channels of row gi -> one 16-byte core-matrix row of the hi part and of the lo part
        uint4 h, l;
        umma::split_bf16x2(acc0.x, acc0.y, h.x, l.x);
        umma::split_bf16x2(acc0.z, acc0.w, h.y, l.y);
        umma::split_bf16x2(acc1v.x, acc1v.y, h.z, l.z);
        umma::split_bf16x2(acc1v.z, acc1v.w, h.w, l.w);
        unsigned char* dst = buf + (size_t)l4 * fr::kLboA + (size_t)gi * 16;
        *reinterpret_cast<uint4*>(dst) = h;
        *reinterpret_cast<uint4*>(dst + fr::kChunkHalf) = l;
      }
      if (DBG && P.dbg_feat && act && gpt < P.dbg_feat_max) {
        float4* d4 = reinterpret_cast<float4*>(P.dbg_feat + (size_t)gpt * 384 + dbg_col + c8);
        d4[0] = acc0; d4[1] = acc1v;
      }
      // ---- hand the chunk over ----
      umma::fence_proxy_async_smem();
      umma::tc_fence_before_sync();
      fr_arrive(&a_full[b]);
      // MMA issue, ROTATING over the warps (chunk c -> warp c): the issuer has to wait until all 512 threads have delivered the chunk; with a
      // fixed issuer that warp was always the slowest of the CTA and every other warp spun on a_free behind it (r2f profile: 10 % of all
      // executed instructions were that spin).  tcgen05 ordering across the issuing threads is carried by the fence::before_thread_sync /
      // mbarrier / fence::after_thread_sync chain every chunk hand-over already has.
      if (warp == c) {                                         // warp-uniform branch; one elected lane issues
        umma::mbar_wait(&a_full[b], u & 1u);
        const uint32_t a_hi = sbase + (uint32_t)b * fr::kChunk, a_lo = a_hi + fr::kChunkHalf;
        if (c < 6) {
          const int ws = c & 1;
          umma::mbar_wait(&w_full[ws], (ti * 3u + (uint32_t)(c >> 1)) & 1u);
          umma::tc_fence_after_sync();
          const uint32_t w_hi = sbase + fr::kWp + (uint32_t)ws * fr::kWpStage;
          if (!(a.knock & 4)) gemm32(a_hi, fr::kLboA, false, a_lo, w_hi, w_hi + fr::kWpStage / 2, 96, fr::kD1, c == 0 ? 0u : 1u);
          umma::mma_commit_e(&a_free[b], el);
          umma::mma_commit_e(&w_free[ws], el);
          if (c == 5) umma::mma_commit_e(&acc1, el);
        } else {
          umma::tc_fence_after_sync();
          const int tt = (c - 6) % 3, sblk = c < 9 ? 0 : 1;     // tri_t -> source block 0 (first MMA of token t), f2d_t -> block 1
          if (c == 9) {                                         // all three tokens are initialised: add the projected 3-D feature (source block 2)
            umma::mbar_wait(&f3d_ready, ti & 1u);
            umma::tc_fence_after_sync();
            const uint32_t w2 = sbase + fr::kWr + 2u * fr::kWrBlock;
#pragma unroll 1
            for (int t3 = 0; t3 < 3; ++t3)
              gemm32(sbase + fr::kF3d + (uint32_t)(4 * t3) * fr::kLboF, fr::kLboF, true, fr::kF3dLo + (uint32_t)(16 * t3), w2, w2 + fr::kWrBlock / 2, 32,
                     fr::kD2 + (uint32_t)(32 * t3), 1u);
          }
          const uint32_t wb = sbase + fr::kWr + (uint32_t)sblk * fr::kWrBlock;
          if (!(a.knock & 4)) gemm32(a_hi, fr::kLboA, false, a_lo, wb, wb + fr::kWrBlock / 2, 32, fr::kD2 + (uint32_t)(32 * tt), c < 9 ? 0u : 1u);
          umma::mma_commit_e(&a_free[b], el);
          if (c == 11) umma::mma_commit_e(&acc2, el);
        }
      }
      if (c == 6) {
        // =========================== E1: projected 3-D feature -> reprojection operand (on-chip only) ===========================
        umma::mbar_wait(&acc1, ti & 1u);
        umma::tc_fence_after_sync();
#pragma unroll
        for (int i = 0; i < 3; ++i) {
          const int c0 = 24 * ecg + 8 * i;
          uint32_t d[8];
          umma::tmem_ld8(etb + fr::kD1 + (uint32_t)c0, d);
          umma::tmem_ld_wait();
          uint4 h; uint32_t lo[4];
          umma::split_bf16x2(__uint_as_float(d[0]) + s_bp[c0], __uint_as_float(d[1]) + s_bp[c0 + 1], h.x, lo[0]);
          umma::split_bf16x2(__uint_as_float(d[2]) + s_bp[c0 + 2], __uint_as_float(d[3]) + s_bp[c0 + 3], h.y, lo[1]);
          umma::split_bf16x2(__uint_as_float(d[4]) + s_bp[c0 + 4], __uint_as_float(d[5]) + s_bp[c0 + 5], h.z, lo[2]);
          umma::split_bf16x2(__uint_as_float(d[6]) + s_bp[c0 + 6], __uint_as_float(d[7]) + s_bp[c0 + 7], h.w, lo[3]);
          *reinterpret_cast<uint4*>(smem + fr::kF3d + (size_t)(c0 >> 3) * fr::kLboF + erow * 16) = h;
          umma::tmem_st4(etb + fr::kF3dLo + (uint32_t)(c0 >> 1), lo);
        }
        umma::tmem_st_wait();
        umma::fence_proxy_async_smem();
        umma::tc_fence_before_sync();
        fr_arrive(&f3d_ready);
      }
    }
    // =========================== E2: tokens = D2 + bias -> global ===========================
    {
      umma::mbar_wait(&acc2, ti & 1u);
      umma::tc_fence_after_sync();
      const int m = tile * 128 + erow;
      uint32_t d[3][8];
#pragma unroll
      for (int i = 0; i < 3; ++i) umma::tmem_ld8(etb + fr::kD2 + (uint32_t)(24 * ecg + 8 * i), d[i]);
      umma::tmem_ld_wait();
      umma::tc_fence_before_sync();
      if (m < np) {
        float4* dst = reinterpret_cast<float4*>(a.tok + (size_t)m * 96 + 24 * ecg);
#pragma unroll
        for (int i = 0; i < 3; ++i) {
          const int c0 = (24 * ecg + 8 * i) & 31;               // bias index: column within the 32-channel token
          dst[2 * i] = make_float4(__uint_as_float(d[i][0]) + s_br[c0], __uint_as_float(d[i][1]) + s_br[c0 + 1], __uint_as_float(d[i][2]) + s_br[c0 + 2],
                                   __uint_as_float(d[i][3]) + s_br[c0 + 3]);
          dst[2 * i + 1] = make_float4(__uint_as_float(d[i][4]) + s_br[c0 + 4], __uint_as_float(d[i][5]) + s_br[c0 + 5], __uint_as_float(d[i][6]) + s_br[c0 + 6],
                                       __uint_as_float(d[i][7]) + s_br[c0 + 7]);
        }
      }
    }
    __syncwarp();                                            // every lane has read its s_pt rows before the next tile overwrites them
  }
  umma::tc_fence_before_sync();
  __syncthreads();
  if (warp == 0) umma::tmem_dealloc(tmem_base, 256);
}

// ---------------------------------------------------------------------------------------------------------------------
// blob: 6 x [hi: 4 kg x 96 rows x 8 bf16 | lo] (projection chunk c = input channels 32c .. 32c+31), then 3 x [hi: 4 kg x 32 rows x 8 | lo]
// (reprojection source block s = input channels 32s .. 32s+31: tri | f2d | f3d)
__global__ void k_pack_front(const float* __restrict__ wp, const float* __restrict__ wr, __nv_bfloat16* __restrict__ blob) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  constexpr int kProjHalf = 4 * 96 * 8, kReHalf = 4 * 32 * 8;
  if (i < 6 * kProjHalf) {
    const int c = i / kProjHalf, r = i % kProjHalf;
    const int e = r & 7, n = (r >> 3) % 96, kg = (r >> 3) / 96;
    const float v = wp[n * 192 + 32 * c + 8 * kg + e];
    const __nv_bfloat16 h = __float2bfloat16_rn(v);
    blob[c * 2 * kProjHalf + r] = h;
    blob[c * 2 * kProjHalf + kProjHalf + r] = __float2bfloat16_rn(v - __bfloat162float(h));
  } else if (i < 6 * kProjHalf + 3 * kReHalf) {
    const int j = i - 6 * kProjHalf;
    const int s = j / kReHalf, r = j % kReHalf;
    const int e = r & 7, n = (r >> 3) % 32, kg = (r >> 3) / 32;
    const float v = wr[n * 96 + 32 * s + 8 * kg + e];
    const __nv_bfloat16 h = __float2bfloat16_rn(v);
    __nv_bfloat16* dst = blob + 6 * 2 * kProjHalf + s * 2 * kReHalf;
    dst[r] = h;
    dst[kReHalf + r] = __float2bfloat16_rn(v - __bfloat162float(h));
  }
}

size_t front_blob_bytes() { return (size_t)6 * fr::kWpStage + 3 * fr::kWrBlock; }

int run_pack_front(const SherfWeights& w, unsigned char* blob, cudaStream_t st) {
  const int total = 6 * 4 * 96 * 8 + 3 * 4 * 32 * 8;
  k_pack_front<<<ceil_div(total, 256), 256, 0, st>>>(w.proj_w, w.reproj_w, reinterpret_cast<__nv_bfloat16*>(blob));
  SHERF_LAUNCH_CHECK();
  return SHERF_OK;
}

int run_front_fused(const GatherParams& G, const SherfWeights& w, const unsigned char* blob, float* tok, cudaStream_t st) {
  if (G.np <= 0) return SHERF_OK;
  if (!G.t_vertices) { set_error("internal: the front kernel needs the seeded canonical-vertex search"); return SHERF_E_INVALID; }
  FrontArgs a;
  a.G = G; a.wblob = blob; a.bp = w.proj_b; a.br = w.reproj_b; a.tok = tok;
  { const char* e = getenv("SHERF_FRONT_KNOCK"); a.knock = e ? atoi(e) : 0; }
  static bool attr_done = false;
  static int num_sms = 148;
  if (!attr_done) {
    SHERF_CUDA_OK(cudaFuncSetAttribute(k_front_fused<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)fr::kSmemBytes));
    SHERF_CUDA_OK(cudaFuncSetAttribute(k_front_fused<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)fr::kSmemBytes));
    int dev = 0;
    SHERF_CUDA_OK(cudaGetDevice(&dev));
    SHERF_CUDA_OK(cudaDeviceGetAttribute(&num_sms, cudaDevAttrMultiProcessorCount, dev));
    attr_done = true;
  }
  const bool dbg = G.dbg_feat || G.dbg_vid3 || G.dbg_can || G.dbg_cdir || G.dbg_uv;
  const int ntiles = (G.np + 127) / 128;
  const int grid = ntiles < 2 * num_sms ? ntiles : 2 * num_sms;             // two co-resident CTAs per SM
  if (dbg) k_front_fused<true><<<grid, fr::kThreads, fr::kSmemBytes, st>>>(a);
  else k_front_fused<false><<<grid, fr::kThreads, fr::kSmemBytes, st>>>(a);
  SHERF_LAUNCH_CHECK();
  return SHERF_OK;
}

}  // namespace sherf
