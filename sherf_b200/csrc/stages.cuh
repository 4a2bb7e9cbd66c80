// Stage parameter blocks and host-side launchers shared between the .cu files.
#pragma once
#include "common.cuh"

namespace sherf {

// Survivor count known only on the device when the kernel is ENQUEUED (the first chunk of a pass is issued before the host has read
// the cull's total): np = clamp(*total - p0, 0, cap); total == NULL -> the host's np stands.
struct DevCount { const int64_t* total; int64_t p0; int cap; };
__device__ __forceinline__ int resolve_np(int np_host, const DevCount& dc) {
  if (!dc.total) return np_host;
  const int64_t r = *dc.total - dc.p0;
  return r <= 0 ? 0 : (r > dc.cap ? dc.cap : (int)r);
}

struct GatherParams {
  // rays
  const float *origins, *dirs, *nearv, *farv;
  int S;
  const float* depths;    // NULL: stratified depths from near/far; else explicit per-sample depths [N*S] (importance pass)
  // compacted points of this chunk
  const int *point_sample, *point_vid;
  int64_t p0; int np;
  DevCount dc;            // optional device-side count (front_fused.cu only)
  // frame
  const FrameConst* fc;
  const VertexWarp *T1, *T3;
  const int* g3_start; const float4* g3_verts;
  const float* t_vertices;   // [V,3] canonical vertices (seed of the knn #3 search); NULL: unseeded doubling-box search
  NnLists nl3;               // candidate lists of the canonical grid (slot == NULL: none)
  // channels-last features
  const float* planes_cl; int plane_h, plane_w;            // [3][H][W][32]
  const float* feat_cl; int feat_h, feat_w, feat_ch;       // [fh][fw][64]
  const float* img; int img_h, img_w;                      // [3][H][W] (NCHW, 3 channels only)
  const float* vol_cl[3]; int vol_ch[3]; int vol_d[3], vol_h[3], vol_w[3];
  // outputs (chunk-relative rows)
  float* comb;      // [np][288]: token k at k*96: tri_k(32) | f2d_k(32) | (f3d_k written by the projection GEMM)
  float* f3raw;     // [np][192]
  float* geo;       // [np][8]: can xyz, cdir xyz, 0, 0
  // backward only (run_point_scatter): channels-last gradient grids, same shapes as planes_cl / feat_cl / vol_cl; comb / f3raw are then inputs
  float* g_planes_cl; float* g_feat_cl; float* g_vol_cl[3];
  // optional taps (absolute point index)
  int* dbg_vid3; float *dbg_can, *dbg_cdir, *dbg_uv, *dbg_feat; int64_t dbg_max, dbg_feat_max;
};

int run_to_channels_last_multi(int n, const float* const* in, float* const* out, const int* C, const int64_t* M, cudaStream_t st);
int run_point_gather(const GatherParams& P, cudaStream_t st);
int run_point_scatter(const GatherParams& P, cudaStream_t st);
// S / depths: the sample set to cull -- (rays.n_samples, NULL) for the stratified coarse samples, (rays.n_importance, t_fine) for the fine pass
int run_cull(const SherfRays& rays, int S, const float* depths, const FrameTables& ft, int* sample_vid, int* ray_count, int* block_sums,
             int* ray_start, int64_t* total_dev, int* point_sample, int* point_vid, cudaStream_t st, int write_all = 1);

// Row-major activation buffers of one chunk of `cap` points (fp32).
struct ChunkBuffers {
  int cap;
  float *comb;   // [cap][288]   token k at k*96: tri_k | f2d_k | f3d_k
  float *f3raw;  // [cap][192]
  float *geo;    // [cap][8]
  float *tok;    // [3cap][32]   conv1d_reprojection output
  float *ln;     // [3cap][32]
  float *qkv;    // [3cap][144]
  float *att;    // [3cap][48]
  float *tok2;   // [3cap][32]
  float *ffh;    // [3cap][32]
  float *tok3;   // [3cap][32]
  float *x;      // [cap][72]    PE6(can) | tok0 | 0
  float *h1, *h2;// [cap][128]
  float *hb;     // [cap][200]   x | h (skip concat, triplane.py:299-300)
  float *fv;     // [cap][188]   feature | PE4(dir) | tok1 | 0
  float *vh;     // [cap][64]
};
size_t chunk_buffer_floats(int cap);
void carve_chunk_buffers(float* base, int cap, ChunkBuffers& cb);

// Packed (transposed, zero-padded) weights: Wt[kp][np], kp = round_up(K,16), np = round_up(N,32).
struct PackedLayer { const float* wt; const float* bias; int K, N, kp, np; };
struct PackedWeights {
  PackedLayer proj, reproj, qkv, attn_out, ff1, ff2, pts[8], feature, views;
};
size_t packed_weight_floats();
int run_pack_weights(const SherfWeights& w, float* base, PackedWeights& pw, cudaStream_t st);

// Canonical (UMMA K-major, no-swizzle) tf32 weights for the tensor-core path: hi part and error-compensation lo part.
struct CanonLayer { const float* hi; const float* lo; const float* bias; int N, K, Np, nchunks; };
struct CanonWeights { CanonLayer proj, reproj, qkv, attn_out, ff1, ff2, pts[8], feature, views; };
size_t canonical_weight_floats();
int run_pack_canonical(const SherfWeights& w, float* base, CanonWeights& cw, cudaStream_t st);
int launch_umma_linear(int prec, const CanonLayer& L, const float* A, int lda, float* Y, int ldy, int M, int act, cudaStream_t st,
                       const float* Res, int ldr, int ygroup, int ygstride, const float* ln_w = nullptr, const float* ln_b = nullptr,
                       float* Y2 = nullptr, int ldy2 = 0);
int launch_simt_linear(const PackedLayer& L, const float* A, int lda, float* Y, int ldy, int M, int act, cudaStream_t st,
                       const float* Res, int ldr, int ygroup, int ygstride);
// Backward on the tensor cores (3xTF32): weights packed transposed for dX = dY . W (mlp_umma.cu), dW = dY^T [X | 1] (backward_umma.cu)
struct CanonBwdWeights { CanonLayer views, feature, pts[8] /* [5] = the h4 half */, pts5x, ff2, ff1, attn_out, qkv, reproj, proj; };
size_t canonical_bwd_weight_floats();
int run_pack_canonical_bwd(const SherfWeights& w, float* base, CanonBwdWeights& cb, cudaStream_t st);
int launch_umma_dx(const CanonLayer& L, const float* dY, int lda, float* dX, int ldx, int M, cudaStream_t st, const float* Mask = nullptr,
                   int ldm = 0, int accum = 0, int agroup = 0, int agstride = 0);
// sparse convolutions on the tensor cores (mlp_umma.cu): the layer as a gathered linear layer with K = 27 c_in, split-K partial tiles
size_t spconv_canon_floats();
int run_pack_spconv(const float* W, int cout, int cin, int mode, float* buf, CanonLayer& L, cudaStream_t st);
int launch_umma_spconv(const CanonLayer& L, const float* X, int kin, const int* rowtab, const int* Mdev, int Mcap, float* Ypart, int nsplit,
                       cudaStream_t st);
constexpr int kGradWMaxSplits = 1024;      // capacity of the partial-sum buffer; the launcher uses one wave of CTAs (<= 444 on a B200)
// part[s][n][K + 1] = sum over the rows of split s of dY[m][n] . [X | 1][m][k];  *splits_out = number of splits written
int launch_umma_grad_w(const float* dY, int lda, int N, const float* X, int ldb, int K, int M, float* part, int* splits_out, cudaStream_t st,
                       int agroup = 0, int agstride = 0);

// Fused tensor-core decoder trunk (decoder_fused.cu)
struct FusedChunk { uint32_t w_off; uint32_t w_bytes; uint16_t src; uint16_t kg0; uint16_t nkg; uint16_t layer; uint16_t first; uint16_t last; };
struct FusedSchedule { FusedChunk ch[44]; uint16_t layer_np[10]; uint16_t pad[2]; };
// Ping-pong bf16x3 decoder (decoder_pp.cu): weight chunk offsets, packed weights / biases, packed X|V input tiles of one chunk
struct PpPlan { uint32_t w_off[23]; const unsigned char* blob; const float* bias; unsigned char* xp; unsigned char* vp; };
struct FusedPlan { FusedSchedule sch; const unsigned char* blob; const float* bias; const float* xf_blob; const float* ff_blob; const PpPlan* pp;
                   const unsigned char* xb_blob; /* bf16 transformer weights (xformer_bf16.cu) */ const unsigned char* fr_blob; /* front kernel weights (front_fused.cu) */ };
size_t pp_blob_bytes();
size_t pp_xv_bytes(int cap);
int run_pack_pp(const SherfWeights& w, unsigned char* blob, float* bias, PpPlan& plan, cudaStream_t st);
int run_pack_xv(const float* x, int ldx, const float* fv, int ldfv, int np, unsigned char* xp, unsigned char* vp, cudaStream_t st);
int run_decoder_pp(const PpPlan& plan, const SherfWeights& w, const unsigned char* xp, const unsigned char* vp, float* sigma, float* rgb, int np,
                   cudaStream_t st, DevCount dc = DevCount{nullptr, 0, 0});
size_t fused_blob_bytes();
extern long long* g_fused_trace;
int run_pack_fused_plan(const SherfWeights& w, unsigned char* blob, float* bias, FusedPlan& plan, cudaStream_t st);
int run_decoder_fused_plan(int prec, const FusedPlan& plan, const float* X, int ldx, const float* fv, int ldfv, float* sigma, float* rgb,
                           const float* rgb_w, const float* rgb_b, int np, cudaStream_t st);

// Fused tensor-core feature fusion: conv1d_projection + conv1d_reprojection + LayerNorm-1 (fusion_fused.cu)
size_t fusion_blob_floats();
int run_pack_fusion(const SherfWeights& w, float* blob, cudaStream_t st);
int run_fusion_fused(int prec, const SherfWeights& w, const float* blob, const float* f3raw, const float* comb, float* tok, float* ln,
                     int np, cudaStream_t st);

// Fused tensor-core transformer layer + decoder-input assembly (xformer_fused.cu)
size_t xformer_blob_floats();
int run_pack_xformer(const SherfWeights& w, float* blob, cudaStream_t st);
int run_xformer_fused(int prec, const SherfWeights& w, const float* blob, const float* ln1, const float* tok, const float* geo, float* x,
                      float* fv, int np, float* dbg_tok, int64_t p0, int64_t dbg_max, cudaStream_t st, unsigned char* xp, unsigned char* vp,
                      float* pe_buf /* [np][64] scratch for the positional encodings */);

// Front kernel: warp + gather + conv1d_projection / reprojection in one kernel (front_fused.cu); tok [np][3][32]
size_t front_blob_bytes();
int run_pack_front(const SherfWeights& w, unsigned char* blob, cudaStream_t st);
int run_front_fused(const GatherParams& G, const SherfWeights& w, const unsigned char* blob, float* tok, cudaStream_t st);

// bf16 split-product transformer, two CTAs per SM (xformer_bf16.cu)
size_t xformer_bf16_blob_bytes();
int run_pack_xformer_bf16(const SherfWeights& w, unsigned char* blob, cudaStream_t st);
int run_xformer_bf16(const SherfWeights& w, const unsigned char* blob, const float* tok, const float* geo, int np, float* dbg_tok, int64_t p0,
                     int64_t dbg_max, cudaStream_t st, unsigned char* xp, unsigned char* vp, float* pe_buf, DevCount dc = DevCount{nullptr, 0, 0});
int run_point_pe(const float* geo, float* pe, int np, cudaStream_t st, DevCount dc = DevCount{nullptr, 0, 0});

// The fusion / transformer / decoder stack on one chunk.  renderer.py:350,423-432; triplane.py:285-316
// prec: SHERF_MLP_FP32 (CUDA-core fp32 FMA) | SHERF_MLP_TF32 | SHERF_MLP_TF32X3 | SHERF_MLP_BF16X3 (tcgen05 tensor cores)
int run_mlp(int prec, const SherfWeights& w, const PackedWeights& pw, const CanonWeights& cw, const FusedPlan* fused, const ChunkBuffers& cb, int np,
            int64_t p0, float* sigma_out, float* rgb_out, float* dbg_tok, int64_t dbg_max, cudaStream_t st,
            void (*span_begin)(int) = nullptr, void (*span_end)() = nullptr, DevCount dc = DevCount{nullptr, 0, 0});

// Backward pass (backward.cu)
struct BwdChunk {
  int cap;
  // activations kept by the recompute pass
  float *comb, *f3raw, *geo, *tok, *ln1, *qkv, *att, *tok2, *ln2, *ffp, *ffa, *tok3, *x, *hb, *fv, *vh, *h[8];
  // gradients
  float *dvh, *dpre, *dfv, *dha, *dhb, *dx, *dtok3, *dff, *dln, *dtok2, *dtok, *datt, *dqkv, *dcomb, *df3raw;
  float *part, *ln_part;
};
size_t bwd_chunk_floats(int cap);
void carve_bwd_chunk(float* base, int cap, BwdChunk& b);
int run_composite_backward(const SherfRays& rays, const FrameConst* fc, const int* ray_start, const int* point_sample, const float* sigma,
                           const float* rgb, const float* noise, int white_back, const float* g_rgb, const float* g_depth, const float* g_acc,
                           float* dsig, float* drgb, cudaStream_t st);
int run_backward_chunk(const SherfWeights& w, const PackedWeights& pw, const CanonWeights& cw, const CanonBwdWeights& cbw, const SherfWeightGrads& gw,
                       GatherParams G, const BwdChunk& b, int np, int64_t p0, const float* rgb, const float* dsig, const float* drgb, cudaStream_t st);
int run_backward_chunk_inputs(const SherfWeights& w, const CanonBwdWeights& cbw, GatherParams G, const BwdChunk& b, int np, int64_t p0, cudaStream_t st);
int run_from_channels_last(const float* in, float* out, int C, int64_t M, cudaStream_t st);
int run_layernorm32(const float* x, const float* w, const float* b, float* y, int rows, cudaStream_t st);
int run_attention3(const float* qkv, float* att, int np, cudaStream_t st);
int run_decoder_inputs(const float* geo, const float* tok3, float* x, float* hb, float* fv, int np, cudaStream_t st);

int run_debug_linear(int prec, const float* A, int lda, const float* W, const float* bias, float* Y, int ldy, int M, int N, int K,
                     int act, float* wscratch, cudaStream_t st);

int run_composite(const SherfRays& rays, const FrameConst* fc, const int* ray_start, const int* point_sample,
                  const float* sigma, const float* rgb, const float* noise, int white_back, const SherfOut& out, cudaStream_t st);

// Dataset-side ray setup (rays.cu): get_rays + get_near_far, RenderPeople_dataset.py:14-27,68-101,129-134
int run_generate_rays(const double* K, const double* R, const double* T, int H, int W, const double* bounds, float* origins, float* dirs,
                      float* nearv, float* farv, unsigned char* mask_at_box, cudaStream_t st);

// Sparse 3-D encoder (sparse_encoder.cu): renderer.py:744-785
size_t sparse_encoder_scratch_bytes(int n, const int32_t* out_sh);
int run_sparse_encode(const SherfSparseEncoder& enc, const int* coord, const float* feat, int n, const int32_t* out_sh, float* const* vols,
                      void* scratch, size_t scratch_bytes, cudaStream_t st);

size_t sparse_encoder_train_scratch_bytes(int n, const int32_t* out_sh);
int run_sparse_encode_train(const SherfSparseEncoder& enc, const int* coord, const float* feat, int n, const int32_t* out_sh, float* const* vols,
                            float* batch_stats, int* row_counts, int use_running_stats, void* scratch, size_t scratch_bytes, cudaStream_t st);
int run_sparse_encode_backward(const SherfSparseEncoder& enc, const int* coord, int n, const int32_t* out_sh, const float* const* g_vols,
                               const SherfSparseEncoderGrads& gr, float* g_feat, int use_running_stats, void* scratch, size_t scratch_bytes, cudaStream_t st);

// Dataset-side SMPL forward (smpl_forward.cu): smpl_numpy.py:46-98
size_t smpl_forward_scratch_bytes();
int run_smpl_vertices(const SherfSmplModel& smpl, const SherfPose& pose, float* verts_smpl, float* verts_world, void* scratch, size_t scratch_bytes,
                      cudaStream_t st);

// Observation preparation (observation.cu): triplane.py:105-137
size_t observation_scratch_bytes(int V, int maxcell);
int run_prepare_observation(const SherfSmplModel& smpl, const SherfObservation& ob, float* vert_feat, int32_t* coord, uint8_t* vmask_out,
                            float* bounds_out, int32_t* out_sh_host, float* can_out, void* scratch, size_t scratch_bytes, cudaStream_t st);

int run_prepare_observation_backward(const SherfSmplModel& smpl, const SherfObservation& ob, const float* g_vert_feat, float* g_proj_w, float* g_proj_b,
                                     float* g_obs_feat, void* scratch, size_t scratch_bytes, cudaStream_t st);

// Importance (fine) pass, importance.cu (renderer.py:373-393, 446-456, 483-542)
int run_importance_sample(const SherfRays& rays, const int* ray_start, const int* point_sample, const float* sigma, const float* noise,
                          const float* w_in, const float* u, float* t_fine, int* bins_out, float* w_out, cudaStream_t st);
int run_composite_merged(const SherfRays& rays, const FrameConst* fc, const int* vid_c, const int* start_c, const float* sigma_c,
                         const float* rgb_c, const float* noise_c, const float* t_fine, const int* vid_f, const int* start_f,
                         const float* sigma_f, const float* rgb_f, const float* noise_f, int white_back, const SherfOut& out,
                         cudaStream_t st);
int run_dense_taps(const int* point_sample, const float* sg, const float* c3, int64_t P, int64_t n_dense, float* sigma, float* rgb,
                   cudaStream_t st);

}  // namespace sherf
