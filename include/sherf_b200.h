/*
 * sherf_b200 -- C ABI of the B200-native SHERF volumetric render hot path.
 *
 * The reference has no FFI for this path: it is Python calling torch ops.  The boundary a
 * maintainer binds instead is ImportanceRenderer.forward
 *   /root/reference/sherf/training/volumetric_rendering/renderer.py:286-398
 * plus NeRFDecoder.forward
 *   /root/reference/sherf/training/triplane.py:285-316
 * Every entry point below names the reference lines it replaces.  All pointers are DEVICE
 * pointers to contiguous fp32 / int32 arrays unless marked "host"; the library BORROWS them for
 * the duration of one call and owns nothing but the caller-provided scratch arena.  Batch is 1
 * per call (the reference renderer only works for per-GPU batch 1, renderer.py:320-321).
 * All functions return 0 on success or a negative SHERF_E_* code and never throw;
 * sherf_last_error() returns a thread-local description.  Kernels are enqueued on `stream`
 * (a cudaStream_t passed as void*), nothing synchronises the device except where noted.
 */
#ifndef SHERF_B200_H
#define SHERF_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SHERF_ABI_VERSION 5
#if defined(__GNUC__)
#define SHERF_API __attribute__((visibility("default")))
#else
#define SHERF_API
#endif
#define SHERF_NUM_JOINTS 24
#define SHERF_NUM_LEVELS 3

enum {
  SHERF_OK = 0,
  SHERF_E_INVALID = -1,   /* bad argument (null pointer, unsupported shape / option) */
  SHERF_E_SCRATCH = -2,   /* scratch arena too small */
  SHERF_E_CUDA = -3,      /* a CUDA runtime call failed; see sherf_last_error() */
  SHERF_E_UNSUPPORTED = -4
};

/* MLP arithmetic.  FP32 = CUDA-core fp32 FMA (parity mode, the reference disables TF32,
 * training_loop.py:169-171).  TF32 / TF32X3 = tcgen05 tensor-core paths (single-pass / error-compensated
 * 3xTF32).  BF16X3 = 3xTF32 for the fusion conv and the transformer, bf16 split products (a_hi*w_hi +
 * a_lo*w_hi + a_hi*w_lo, 16 significand bits per operand, fp32 accumulate) for the NeRF decoder. */
enum { SHERF_MLP_FP32 = 0, SHERF_MLP_TF32 = 1, SHERF_MLP_TF32X3 = 2, SHERF_MLP_BF16X3 = 3 };

/* The SMPL body model the reference loads in ImportanceRenderer.__init__ (renderer.py:282-284,
 * SMPL_to_tensor renderer.py:65-74). */
typedef struct SherfSmplModel {
  const float* v_template;   /* [V,3] */
  const float* shapedirs;    /* [V,3,10] */
  const float* posedirs;     /* [V,3,207] */
  const float* j_regressor;  /* [24,V] dense */
  const float* weights;      /* [V,24] */
  int32_t parents[SHERF_NUM_JOINTS]; /* host; kintree_table[0], parents[0] ignored */
  int32_t n_verts;           /* V (6890) */
} SherfSmplModel;

/* One `params` dict of the dataset (RenderPeople_dataset.py:195-204). */
typedef struct SherfPose {
  const float* poses;   /* [72] axis-angle */
  const float* shapes;  /* [10] */
  const float* R;       /* [3,3] row-major; smpl = (world - Th) @ R */
  const float* Th;      /* [3] */
} SherfPose;

/* Per-frame inputs = the non-ray entries of `input_data` (RenderPeople_dataset.py:362-391) and
 * obs_sp_input (triplane.py:174-217). */
typedef struct SherfFrame {
  SherfPose target;            /* input_data['params'] */
  SherfPose canonical;         /* input_data['t_params'] (R, Th unused, as in the reference) */
  SherfPose obs;               /* input_data['obs_params'] */
  const float* vertices;       /* [V,3] posed target vertices, world space */
  const float* t_vertices;     /* [V,3] canonical ("big pose") vertices */
  const float* t_world_bounds; /* [2,3] tri-plane box (renderer.py:239) */
  const float* obs_K;          /* [3,3] observation camera (renderer.py:686-699) */
  const float* obs_R;          /* [3,3] */
  const float* obs_T;          /* [3] */
  const float* sp_bounds;      /* [2,3] obs_sp_input['bounds'][0] (renderer.py:548) */
  int32_t out_sh[3];           /* host; obs_sp_input['out_sh'] (z,y,x) (renderer.py:552) */
} SherfFrame;

/* Feature tensors in the layouts the reference hands to forward() (NCHW / NCDHW, batch 1). */
typedef struct SherfScene {
  const float* planes;     /* [3,plane_ch,plane_h,plane_w]  renderer.py:234-243 */
  int32_t plane_ch, plane_h, plane_w;
  const float* obs_img;    /* [3,img_h,img_w]               renderer.py:336 */
  int32_t img_h, img_w;
  const float* obs_feat;   /* [feat_ch,feat_h,feat_w]       renderer.py:333 */
  int32_t feat_ch, feat_h, feat_w;
  const float* vol[SHERF_NUM_LEVELS];      /* dense [C,D,H,W] pyramid levels, renderer.py:762-782 */
  int32_t vol_ch[SHERF_NUM_LEVELS];
  int32_t vol_dim[SHERF_NUM_LEVELS][3];    /* D,H,W */
} SherfScene;

/* Hot-path parameters, PyTorch layouts ([out,in] row-major weights).  Names = checkpoint names
 * (SURVEY.md 8b): renderer.* from renderer.py:271-276, decoder.* from triplane.py:267-283. */
typedef struct SherfWeights {
  const float *proj_w, *proj_b;         /* renderer.conv1d_projection   [96,192(,1)], [96]  */
  const float *reproj_w, *reproj_b;     /* renderer.conv1d_reprojection [32,96(,1)],  [32]  */
  const float *ln1_w, *ln1_b;           /* transformer.layers.0.0.fn.norm               [32] */
  const float *qkv_w;                   /* ...0.0.fn.fn.to_qkv.weight  [144,32] (no bias)    */
  const float *attn_out_w, *attn_out_b; /* ...0.0.fn.fn.to_out.0       [32,48], [32]         */
  const float *ln2_w, *ln2_b;           /* ...0.1.fn.norm                               [32] */
  const float *ff1_w, *ff1_b;           /* ...0.1.fn.fn.net.0          [32,32], [32]         */
  const float *ff2_w, *ff2_b;           /* ...0.1.fn.fn.net.3          [32,32], [32]         */
  const float *pts_w[8], *pts_b[8];     /* decoder.pts_linears.{0..7}: [128,71],[128,128]x4,[128,199],[128,128]x2 */
  const float *alpha_w, *alpha_b;       /* decoder.alpha_linear   [1,128], [1]   */
  const float *feature_w, *feature_b;   /* decoder.feature_linear [128,128], [128] */
  const float *views_w, *views_b;       /* decoder.views_linear   [64,187], [64] */
  const float *rgb_w, *rgb_b;           /* decoder.rgb_linear     [3,64], [3]    */
} SherfWeights;

/* Rays of one view (RenderPeople_dataset.py:14-27,129-134). */
typedef struct SherfRays {
  const float* origins;  /* [N,3] */
  const float* dirs;     /* [N,3] un-normalised */
  const float* near_;    /* [N] */
  const float* far_;     /* [N] */
  int32_t n_rays;        /* N */
  int32_t n_samples;     /* S = rendering_options['depth_resolution'] (2..256) */
  int32_t n_importance;  /* S_f = rendering_options['depth_resolution_importance'] (0 = coarse pass only; else 1..256, needs S >= 3) */
  int32_t reserved;
} SherfRays;

/* rendering_options subset used by the path (train.py:328-351, ray_marcher.py:25-64). */
typedef struct SherfOptions {
  int32_t white_back;        /* ray_marcher.py:59 */
  int32_t mlp_precision;     /* SHERF_MLP_* */
  float depth_clamp_min;     /* used only if use_external_clamp != 0: global min/max of ALL depths of the */
  float depth_clamp_max;     /*   full (unsharded) view, ray_marcher.py:57 -- needed when rays are sharded */
  int32_t use_external_clamp;
  const float* density_noise; /* optional additive sigma noise, already scaled, ONE VALUE PER SURVIVING POINT in compacted (row-major [N,S]
                                 surviving) order, at least n_points long -- what `sigma += randn_like(sigma) * density_noise` adds at
                                 renderer.py:435-436.  The count comes from sherf_count_survivors.  NULL = none */
  const float* importance_u;  /* [N*S_f] uniform draws in [0,1) standing for torch.rand at renderer.py:526; required when
                                 n_importance > 0 (the caller owns the RNG, SURVEY.md 8b "RNG") */
  const float* density_noise_importance; /* optional [N*S_f] additive sigma noise of the fine samples, per fine SAMPLE (their survivor count
                                            depends on the coarse pass; the reference's own fine pass cannot run, SURVEY a13); NULL = none */
  uint64_t weights_version;   /* 0: the weights are re-packed into the scratch arena on every call.  Non-zero: the caller vouches
                                 that SherfWeights' contents are unchanged since the previous call THAT USED THE SAME scratch arena,
                                 mlp_precision and shapes with the same non-zero value; the packed copies made by that call are then
                                 reused (the reference keeps its nn.Parameters as they are between calls, too).  Change the value
                                 whenever a parameter is written or the arena is re-allocated. */
  uint64_t scene_version;     /* same contract for SherfScene: non-zero and unchanged since the previous call on this arena = the feature
                                 tensors (planes, 2-D map, volumes) are unchanged, so the channels-last copies the arena holds (312 MB at
                                 512x512) are reused instead of re-made -- the "prepare once per observation, render many views" split of
                                 SURVEY.md 8b (orbit views, ray shards, streamed poses).  0 = copy on every call. */
} SherfOptions;

/* Outputs of forward (renderer.py:398): rgb in (-1,1), depth, accumulated weight. */
typedef struct SherfOut {
  float* rgb;    /* [N,3] */
  float* depth;  /* [N]   */
  float* acc;    /* [N]   */
} SherfOut;

/* Optional stage-wise taps for parity tests (any pointer may be NULL).  Point-indexed arrays are
 * in compaction order = row-major order of surviving samples (renderer.py:320-321); the caller
 * sizes them for N*S points or reads n_points from a previous call. */
typedef struct SherfDebug {
  int32_t* sample_vid;   /* [N*S] nearest posed-vertex id of every sample within the cull radius, -1 otherwise */
  int32_t* point_sample; /* [P] flat sample index n*S+i of each surviving point */
  int32_t* point_vid3;   /* [P] nearest canonical vertex (renderer.py:627) */
  float* point_can;      /* [P,3] canonical position (renderer.py:615) */
  float* point_cdir;     /* [P,3] canonical view direction (renderer.py:618) */
  float* point_uv;       /* [P,2] observation-image pixel coordinates (renderer.py:699) */
  float* point_feat;     /* [P,384] tri(3x32) | f2d(96) | f3d_raw(192) (renderer.py:340, :794, :402) */
  float* point_tok;      /* [P,64] tokens 0,1 after the transformer (renderer.py:427) */
  float* point_sigma;    /* [P] (triplane.py:302) */
  float* point_rgb;      /* [P,3] (triplane.py:314) */
  int64_t max_points;    /* capacity (in points) of the point-indexed arrays except point_feat */
  int64_t max_feat_points; /* capacity (in points) of point_feat */
  /* importance (fine) pass taps, dense per sample like the reference's own arrays (renderer.py:364-371, :378): */
  float* coarse_weights;   /* [N*S]   ray-marcher weights of the coarse pass (renderer.py:376) */
  float* fine_depths;      /* [N*S_f] importance-sampled depths, in draw order (renderer.py:378) */
  int32_t* fine_bins;      /* [N*S_f] searchsorted(cdf, u, right=True) (renderer.py:529) */
  int32_t* fine_sample_vid;/* [N*S_f] nearest posed-vertex id of every fine sample within the cull radius, -1 otherwise */
  float* fine_sigma;       /* [N*S_f] density, -80 where culled */
  float* fine_rgb;         /* [N*S_f,3] colour, 0 where culled */
} SherfDebug;

/* Bytes of scratch sherf_render_forward needs for an (N rays, S coarse + S_f importance samples) call on
 * `scene` (only its shape fields are read).  The arena holds the per-frame tables, channels-last copies of
 * the feature tensors, per-sample bookkeeping and the activation buffers of one chunk of surviving points. */
SHERF_API size_t sherf_scratch_bytes(const SherfScene* scene, int32_t n_rays, int32_t n_samples, int32_t n_importance,
                                     int32_t n_verts);

/* Replaces ImportanceRenderer.forward (renderer.py:286-398) including the decoder call
 * (triplane.py:285-316) and the ray marcher (ray_marcher.py:25-64).
 * With rays->n_importance > 0 it also runs the fine pass (renderer.py:373-393: sample_importance :483-542,
 * unify_samples :446-456) in its REPAIRED form -- the reference's own call sites :376 / :383 cannot execute
 * (SURVEY.md a13): ray directions are passed to the coarse ray march, and the fine samples go through the same
 * cull / warp / gather / decoder stages as the coarse ones (oracle/port.py render_forward states the repair).
 * Synchronises `stream` once per pass internally (to size the point stage).  n_points_out (host, optional)
 * receives the number of samples (coarse + fine) that survived the 5 cm cull. */
SHERF_API int sherf_render_forward(const SherfSmplModel* smpl, const SherfFrame* frame, const SherfScene* scene,
                         const SherfWeights* weights, const SherfRays* rays, const SherfOptions* opts,
                         const SherfOut* out, const SherfDebug* debug /* may be NULL */,
                         void* scratch, size_t scratch_bytes, void* stream, int64_t* n_points_out);

/* Stage 0 + 1 alone (renderer.py:299-321): the number of samples within 5 cm of the body, i.e. the length of the compacted point list
 * the forward will process (what a caller needs to draw per-point density noise exactly like renderer.py:435-436).  Synchronises. */
SHERF_API int sherf_count_survivors(const SherfSmplModel* smpl, const SherfFrame* frame, const SherfScene* scene, const SherfRays* rays,
                                    const SherfOptions* opts, void* scratch, size_t scratch_bytes, void* stream, int64_t* n_points_out);

/* Replaces get_transform_params_torch (renderer.py:129-157) for one pose: writes the 24 rigid
 * transforms A[24,4,4] (device).  Exposed for tests and for the dataset-side SMPL forward. */
SHERF_API int sherf_lbs_transforms(const SherfSmplModel* smpl, const SherfPose* pose, float* A_out /* [24,16] device */,
                         void* scratch, size_t scratch_bytes, void* stream);

/* Dataset-side SMPL forward (SURVEY.md 8f rank 3): the posed vertices of one frame, replacing sherf/smpl/smpl_numpy.py:46-98
 * (`SMPL.__call__`) and the `xyz @ R.T + Th` of RenderPeople_dataset.py:210 on the host.  verts_smpl [V,3] (SMPL space) and / or
 * verts_world [V,3] (= input_data['vertices']); either may be NULL.  fp64 inside (as numpy), float32 out.  scratch >= 4 KB. */
SHERF_API int sherf_smpl_vertices(const SherfSmplModel* smpl, const SherfPose* pose, float* verts_smpl, float* verts_world, void* scratch,
                                  size_t scratch_bytes, void* stream);

/* ---- Backward pass (SURVEY.md 8 f2): what autograd derives through renderer.py:286-437, triplane.py:285-316 and ray_marcher.py:25-64
 * when the reference calls loss.backward() (loss.py:175).  Same inputs as sherf_render_forward plus the gradient of the loss w.r.t. its
 * three outputs; writes the gradients w.r.t. every hot-path parameter and w.r.t. the feature tensors the encoders produce.
 * Recompute-in-backward: the library renders the view again inside the call (nothing has to be kept from the forward), then walks
 * the surviving points back chunk by chunk in fp32.  Coarse pass only (n_importance must be 0: the reference's fine pass cannot
 * execute, SURVEY a13).  Coordinates (warps, projections) carry no gradient -- SMPL parameters and cameras are data upstream. */
typedef struct SherfOutGrads {   /* dL/d(out) of sherf_render_forward; NULL = zero */
  const float* rgb;    /* [N,3] */
  const float* depth;  /* [N]   (no gradient where the depth is clamped or 0/0, like torch.clamp / nan_to_num) */
  const float* acc;    /* [N]   */
} SherfOutGrads;

typedef struct SherfWeightGrads {   /* same fields, shapes and order as SherfWeights; each is OVERWRITTEN with dL/d(param); NULL = not wanted */
  float *proj_w, *proj_b;
  float *reproj_w, *reproj_b;
  float *ln1_w, *ln1_b;
  float *qkv_w;
  float *attn_out_w, *attn_out_b;
  float *ln2_w, *ln2_b;
  float *ff1_w, *ff1_b;
  float *ff2_w, *ff2_b;
  float *pts_w[8], *pts_b[8];
  float *alpha_w, *alpha_b;
  float *feature_w, *feature_b;
  float *views_w, *views_b;
  float *rgb_w, *rgb_b;
} SherfWeightGrads;

typedef struct SherfInputGrads {    /* same shapes / layouts as the SherfScene tensors; OVERWRITTEN; NULL = not wanted */
  float* planes;                    /* [3,plane_ch,plane_h,plane_w]  (F.grid_sample backward of renderer.py:243) */
  float* obs_feat;                  /* [feat_ch,feat_h,feat_w]       (renderer.py:333) */
  float* vol[SHERF_NUM_LEVELS];     /* dense [C,D,H,W]               (renderer.py:790-797) */
} SherfInputGrads;

SHERF_API size_t sherf_backward_scratch_bytes(const SherfScene* scene, int32_t n_rays, int32_t n_samples, int32_t n_verts);
/* Returns SHERF_OK or a negative code.  `scratch` must be an arena of its own (not the one a forward that is still in flight uses):
 * >= sherf_backward_scratch_bytes.  n_points_out (optional, host): surviving samples.  Weight gradients are reduced in a fixed order
 * (run-to-run identical); the grid gradients use floating-point reductions in memory like F.grid_sample's backward. */
SHERF_API int sherf_render_backward(const SherfSmplModel* smpl, const SherfFrame* frame, const SherfScene* scene, const SherfWeights* weights,
                                    const SherfRays* rays, const SherfOptions* opts, const SherfOutGrads* grad_out,
                                    const SherfWeightGrads* grad_weights, const SherfInputGrads* grad_inputs, void* scratch,
                                    size_t scratch_bytes, void* stream, int64_t* n_points_out);

/* The same backward when the caller has JUST run sherf_render_forward with the same smpl / frame / scene / weights / rays / opts on this very
 * arena (`scratch`, sized by sherf_backward_scratch_bytes, whose first part is laid out exactly like the forward's arena) and nothing has
 * touched the arena since: the compacted point list and the per-point sigma / rgb of that forward are reused instead of rendering the view a
 * second time (3.1 ms of a 512x512x64 training view).  n_points: the survivor count that forward reported. */
SHERF_API int sherf_render_backward_after_forward(const SherfSmplModel* smpl, const SherfFrame* frame, const SherfScene* scene,
                                                  const SherfWeights* weights, const SherfRays* rays, const SherfOptions* opts,
                                                  const SherfOutGrads* grad_out, const SherfWeightGrads* grad_weights,
                                                  const SherfInputGrads* grad_inputs, void* scratch, size_t scratch_bytes, void* stream,
                                                  int64_t n_points);

/* Global depth-clamp range of a full view: min/max over all rays of the first/last sample depth
 * (ray_marcher.py:57 via math_utils.py:101-118).  Host results; synchronises the stream. */
SHERF_API int sherf_depth_range(const SherfRays* rays, float* min_out /* host */, float* max_out /* host */,
                      void* scratch, size_t scratch_bytes, void* stream);

/* Dataset-side ray setup on the device (SURVEY.md 8f rank 3): get_rays (RenderPeople_dataset.py:14-27) + get_near_far
 * (:68-101) + the (0,1) near/far fill for rays that miss the box (:129-134) for an H x W pinhole view.
 * K, R, T, bounds ([2,3] = min xyz, max xyz of the SMPL vertices +-0.05, :284-289) are HOST arrays of doubles (row-major);
 * outputs are device arrays: origins/dirs [H*W,3] (dirs un-normalised, zeros replaced by 1e-8 as the dataset does in
 * place), near/far [H*W], mask_at_box [H*W] bytes (optional).  fp64 inside, float32 out, like numpy. */
SHERF_API int sherf_generate_rays(const double* K, const double* R, const double* T, int32_t H, int32_t W, const double* bounds,
                                  float* origins, float* dirs, float* near_out, float* far_out, uint8_t* mask_at_box /* may be NULL */,
                                  void* stream);

/* ---- Sparse 3-D encoder (SURVEY.md 8f rank 1): SparseConvNet.forward's convolutions + .dense() (renderer.py:744-785) ---- */
#define SHERF_SPARSE_CONVS 13   /* conv0 x2, down0, conv1 x2, down1, conv2 x3, down2, conv3 x3 (renderer.py:728-740; num_layers = 4) */
typedef struct SherfSparseConv {
  const float* weight;      /* [c_out,3,3,3,c_in] spconv 2.x layout of (SubM|Sparse)Conv3d.weight, no bias (renderer.py:820,869) */
  const float *bn_weight, *bn_bias, *bn_mean, *bn_var;   /* BatchNorm1d(eps=1e-3) in evaluation mode: running statistics */
  int32_t c_in, c_out;
  int32_t kind;             /* 0 = SubMConv3d k3, 1 = SparseConv3d k3 s2 p1 */
  int32_t reserved;
} SherfSparseConv;
typedef struct SherfSparseEncoder { SherfSparseConv conv[SHERF_SPARSE_CONVS]; } SherfSparseEncoder;

SHERF_API size_t sherf_sparse_encoder_scratch_bytes(int32_t n_voxels, const int32_t* out_sh /* host [3] = D,H,W */);
/* coord [n,3] int32 (z,y,x; obs_sp_input['coord'][:,1:], triplane.py:193-207) and feat [n,c_in] are the rows of the
 * SparseConvTensor of triplane.py:137; rows that share a voxel are merged by keeping the smallest row index (spconv leaves this
 * case unspecified).  vol1/2/3: dense [32,D/2,H/2,W/2], [64,D/4,..], [96,D/8,..] outputs = net1/2/3.dense() (renderer.py:762,771,780),
 * i.e. the `canonical_sp_conv_volume` list sherf_render_forward's SherfScene.vol takes. */
SHERF_API int sherf_sparse_encode(const SherfSparseEncoder* enc, const int32_t* coord, const float* feat, int32_t n,
                                  const int32_t* out_sh /* host [3] */, float* vol1, float* vol2, float* vol3, void* scratch,
                                  size_t scratch_bytes, void* stream);

/* Training mode of the sparse encoder (SURVEY.md 8 f1 / f2): nn.BatchNorm1d(eps=1e-3, momentum=0.01) in train() normalises with the BATCH
 * statistics of each layer's rows (renderer.py:822-871), and loss.backward() (loss.py:175) differentiates through SparseConvNet.forward.
 * sherf_sparse_encode_train = sherf_sparse_encode with batch statistics; it keeps every activation in `scratch`, which must reach
 * sherf_sparse_encode_backward unchanged (same enc / coord / n / out_sh).  batch_stats [13][2][96] (device, may be NULL): per conv the batch
 * mean | biased batch variance per channel; row_counts [13] int32 (device, may be NULL): rows under each BatchNorm (spconv keeps duplicate
 * input rows on the level-0 layers: they are counted) -- the caller updates running_mean / running_var / num_batches_tracked from them
 * exactly like torch (unbiased variance = biased * n / (n - 1)).  use_running_stats != 0: the differentiable forward of eval() -- BatchNorm
 * normalises with the running statistics (constants of the graph); nothing is written to batch_stats / row_counts. */
typedef struct SherfSparseEncoderGrads {
  float* weight[SHERF_SPARSE_CONVS];      /* [c_out,3,3,3,c_in] each, or NULL */
  float* bn_weight[SHERF_SPARSE_CONVS];   /* [c_out] or NULL */
  float* bn_bias[SHERF_SPARSE_CONVS];     /* [c_out] or NULL */
} SherfSparseEncoderGrads;
SHERF_API size_t sherf_sparse_encoder_train_scratch_bytes(int32_t n_voxels, const int32_t* out_sh /* host [3] */);
SHERF_API int sherf_sparse_encode_train(const SherfSparseEncoder* enc, const int32_t* coord, const float* feat, int32_t n,
                                        const int32_t* out_sh /* host [3] */, float* vol1, float* vol2, float* vol3, float* batch_stats,
                                        int32_t* row_counts, int32_t use_running_stats, void* scratch, size_t scratch_bytes, void* stream);
/* g_vol1/2/3: dL/d(vol1/2/3) in the layout of the outputs (any may be NULL = zero); grads: where to write dL/d(weights) (overwritten, not
 * accumulated); g_feat [n,c_in] (may be NULL): dL/d(feat) -- rows that were merged into another row of the same voxel get zero. */
SHERF_API int sherf_sparse_encode_backward(const SherfSparseEncoder* enc, const int32_t* coord, int32_t n, const int32_t* out_sh /* host [3] */,
                                           const float* g_vol1, const float* g_vol2, const float* g_vol3, const SherfSparseEncoderGrads* grads,
                                           float* g_feat, int32_t use_running_stats /* as in the forward */, void* scratch, size_t scratch_bytes,
                                           void* stream);

/* ---- Observation preparation (SURVEY.md 8f rank 1, "vertex-feature splat"): what TriPlaneGenerator.synthesis computes once per
 * observation image before calling the renderer (triplane.py:105-137) -- the rows of the SparseConvTensor of triplane.py:137. ---- */
typedef struct SherfObservation {
  SherfPose obs;               /* input_data['obs_params'] */
  SherfPose canonical;         /* input_data['t_params'] */
  const float* obs_vertices;   /* [V,3] input_data['obs_vertices'], world space */
  const float* t_vertices;     /* [V,3] input_data['t_vertices'] */
  const float* obs_K;          /* [3,3] */
  const float* obs_R;          /* [3,3] */
  const float* obs_T;          /* [3] */
  const int32_t* faces;        /* [F,3] SMPL_NEUTRAL['f'] as int32 (renderer.projection's `face`, renderer.py:692-695) */
  const int32_t* last_face;    /* [3,V]: for corner slot k, the LAST face f with faces[f][k] == v, or -1 (compute_normal's
                                  `norm[:, faces[:, k]] += n` is an index_put WITHOUT accumulation, renderer.py:58-60) */
  int32_t n_faces;
  int32_t reserved;
  const float* obs_img;        /* [3,img_h,img_w] input_data['obs_img_all'][:,0] */
  int32_t img_h, img_w;
  const float* obs_feat;       /* [feat_ch,feat_h,feat_w] encoder_2d_feature(obs_img, extract_feature=True) (triplane.py:108) */
  int32_t feat_ch, feat_h, feat_w;
  int32_t reserved2;
  const float *proj_w, *proj_b; /* TriPlaneGenerator.conv1d_projection [32,96(,1)], [32] (triplane.py:57,124) */
} SherfObservation;

SHERF_API size_t sherf_observation_scratch_bytes(int32_t n_verts);
/* Outputs (device unless noted): vert_feat [V,32] = obs_vertex_3d_feature (zero where the vertex faces away, triplane.py:126);
 * coord [V,4] int32 = obs_sp_input['coord'] (batch, z, y, x; triplane.py:193-207); vertex_mask [V] bytes = obs_smpl_vertex_mask (may be
 * NULL); bounds [2,3] = obs_sp_input['bounds'][0]; out_sh_host [3] (HOST) = obs_sp_input['out_sh']; canonical_out [V,3] (may be NULL)
 * = coarse_obs_vertex_canonical_pts.  Synchronises the stream once (out_sh sizes the caller's volumes). */
SHERF_API int sherf_prepare_observation(const SherfSmplModel* smpl, const SherfObservation* obs, float* vert_feat, int32_t* coord,
                                        uint8_t* vertex_mask, float* bounds, int32_t* out_sh_host, float* canonical_out, void* scratch,
                                        size_t scratch_bytes, void* stream);

/* Backward of the vertex features (triplane.py:115-126) for training: g_vert_feat [V,32] = dL/d(vert_feat) -> g_proj_w [32,96], g_proj_b [32]
 * (TriPlaneGenerator.conv1d_projection) and g_obs_feat [feat_ch,feat_h,feat_w] (adds the bilinear adjoint of triplane.py:115; the image
 * and the vertex pixels are data).  Outputs are overwritten; any may be NULL.  scratch >= sherf_observation_scratch_bytes. */
SHERF_API int sherf_prepare_observation_backward(const SherfSmplModel* smpl, const SherfObservation* obs, const float* g_vert_feat,
                                                 float* g_proj_w, float* g_proj_b, float* g_obs_feat, void* scratch, size_t scratch_bytes,
                                                 void* stream);

/* sample_importance + sample_pdf (renderer.py:483-542) alone, on caller-supplied ray-marcher weights [N*S]
 * and uniform draws u [N*S_f]: writes the fine depths [N*S_f] and (optional) the searchsorted bin indices. */
SHERF_API int sherf_debug_sample_importance(const SherfRays* rays, const float* weights, const float* u, float* t_fine_out,
                                            int32_t* bins_out /* may be NULL */, void* stream);

/* Diagnostic: one linear layer Y[M,N] = act(A[M,K] * W[N,K]^T + bias) on the selected arithmetic (SHERF_MLP_*), the building
 * block of the fusion / transformer / decoder stack (nn.Linear / Conv1d(k=1) call sites renderer.py:350,424 and
 * triplane.py:296-312).  act: 0 none, 1 ReLU, 2 GELU(erf).  Tensor-core modes need N % 16 == 0; N, K <= 256.
 * lda % 4 == 0, A 16-byte aligned.  scratch >= 2.5 MB. */
SHERF_API int sherf_debug_linear(int precision, const float* A, int lda, const float* W, const float* bias, float* Y, int ldy,
                                 int M, int N, int K, int act, void* scratch, size_t scratch_bytes, void* stream);

/* Diagnostic: device buffer [148*8] of int64 cycle counters filled by the fused decoder kernel (NULL disables). */
SHERF_API void sherf_debug_set_trace(long long* device_buf);

SHERF_API const char* sherf_last_error(void);
SHERF_API int sherf_abi_version(void);   /* == SHERF_ABI_VERSION (5) */
/* Number of kernels launched by the last sherf_render_forward on this thread (bench's gpu_launches). */
SHERF_API int64_t sherf_last_launch_count(void);
/* Number of FINE (importance) samples that survived the cull in the last sherf_render_forward on this thread
 * (n_points_out reports coarse + fine). */
SHERF_API int64_t sherf_last_importance_point_count(void);
/* Device time (ms) of the named stage of the last forward on this thread, measured with CUDA events when
 * sherf_set_profiling(1) was called; stages: 0 prologue, 1 cull+compact, 2 warp+gather, 3 mlp (whole stage), 4 composite,
 * 5 the fused tcgen05 decoder kernel alone, 6 the fused tcgen05 transformer kernel alone,
 * 7 the fused tcgen05 feature-fusion kernel alone (sub-spans of stage 3; 0 on the fp32 path). */
SHERF_API void sherf_set_profiling(int enabled);
SHERF_API float sherf_last_stage_ms(int stage);
/* Host wall time (microseconds) of the last forward on this thread: 0 launch issue until the survivor-count sync, 1 time blocked in
 * that sync, 2 launch issue of the point stages and the ray march, 3 whole call. */
SHERF_API float sherf_last_host_us(int part);
/* Nearest-vertex candidate lists of the last forward on this thread (synchronises the device): out[0] cull candidates of the last
 * cull, then for the cull grid (out[1..4]) and the canonical grid (out[5..8]): sub-cells with a list, mean and max list length, fraction
 * of them over the capacity; out[9] the capacity.  Returns SHERF_OK, or SHERF_E_INVALID when the last forward built no lists. */
SHERF_API int sherf_nn_list_stats(double* out);

#ifdef __cplusplus
}
#endif
#endif /* SHERF_B200_H */
