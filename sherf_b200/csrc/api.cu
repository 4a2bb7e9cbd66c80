// extern "C" boundary of libsherf_b200.so: scratch carving, stage orchestration, error reporting.
// See include/sherf_b200.h for the contract and the reference lines each entry point replaces.
#include "common.cuh"
#include "stages.cuh"
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <cstdlib>
#include <vector>
#include <chrono>

namespace sherf {

thread_local LaunchCounter g_launches;
thread_local bool g_pack_plan_only = false;
static thread_local char g_err[512] = "";
static thread_local int64_t g_last_launches = 0;
static thread_local int64_t g_last_fine_points = 0;
static thread_local int g_profiling = 0;
static thread_local float g_stage_ms[8] = {0, 0, 0, 0, 0, 0, 0, 0};
static thread_local FrameTables g_last_ft{};                // tables of the last forward (sherf_nn_list_stats)
static thread_local float g_host_us[4] = {0, 0, 0, 0};   // host wall time of the last forward: issue until the P sync, waiting in the sync, issue of the point stages, total
static inline double now_us() { return std::chrono::duration<double, std::micro>(std::chrono::steady_clock::now().time_since_epoch()).count(); }

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

constexpr int kMaxCell = 1 << 18;

bool nn_lists_enabled() {
  const char* e = getenv("SHERF_NN_LEGACY");
  return !(e && atoi(e) != 0);
}
int nn_list_cap() {
  const char* e = getenv("SHERF_NN_LIST_CAP");
  const int k = e ? atoi(e) : kNnlCap;
  return k < 1 ? 1 : (k > kNnlCap ? kNnlCap : k);
}
// points per MLP chunk (activation buffers are sized for this); SHERF_CHUNK_CAP overrides it for tuning experiments
static size_t chunk_cap_limit() {
  static size_t cap = 0;
  if (!cap) {
    const char* e = getenv("SHERF_CHUNK_CAP");
    const long v = e ? atol(e) : 0;
    cap = v >= 128 ? (size_t)(v / 128 * 128) : (size_t)(1 << 19);
  }
  return cap;
}

struct Arena {
  char* base; size_t size; size_t off; bool dry;
  template <typename T> T* take(size_t n) {
    off = (off + 255) & ~(size_t)255;
    T* p = dry ? nullptr : reinterpret_cast<T*>(base + off);
    off += n * sizeof(T);
    return p;
  }
};

struct Layout {
  FrameTables ft;
  float* planes_cl; float* feat_cl; float* vol_cl[3];
  int* sample_vid; int* ray_count; int* block_sums; int* ray_start; int64_t* total;
  int* point_sample; int* point_vid;
  float* sigma; float* rgb;
  // importance (fine) pass bookkeeping, sized N * S_f (absent when S_f == 0)
  float* fine_depths; int* sample_vid_f; int* ray_count_f; int* ray_start_f; int64_t* total_f; int* point_sample_f; int* point_vid_f;
  float* sigma_f; float* rgb_f;
  float* packed_w;
  float* canon_w;
  unsigned char* fused_blob; float* fused_bias; float* xf_blob; float* ff_blob;
  unsigned char* pp_blob; float* pp_bias; unsigned char* pp_xv;
  unsigned char* xb_blob; unsigned char* fr_blob;
  float* chunk;
  float* gather2;        // second set of gather outputs (comb | f3raw | geo) for the gather / MLP overlap
  float* lbs_joints; float* lbs_pf;
};

static int chunk_cap(int N, int S, int SF) {
  const size_t NS = (size_t)N * (S > SF ? S : SF);
  return (int)((NS < chunk_cap_limit()) ? ((NS + 127) / 128 * 128) : chunk_cap_limit());
}

static size_t carve(Arena& a, const SherfScene& sc, int N, int S, int SF, int V, Layout& L) {
  const size_t NS = (size_t)N * S, NF = (size_t)N * SF;
  FrameTables& ft = L.ft;
  ft.fc = a.take<FrameConst>(1);
  ft.A = a.take<float>(3 * kJoints * 16);
  ft.joints = a.take<float>(3 * kJoints * 3);
  ft.posefeat = a.take<float>(3 * kPoseFeat);
  ft.poff = a.take<float>((size_t)3 * V * 3);
  ft.soff = a.take<float>((size_t)2 * V * 3);
  ft.verts_smpl = a.take<float>((size_t)V * 3);
  ft.T1 = a.take<VertexWarp>(V);
  ft.T3 = a.take<VertexWarp>(V);
  ft.g1_cell_start = a.take<int>(kMaxCell + 1);
  ft.g3_cell_start = a.take<int>(kMaxCell + 1);
  ft.g_cursor = a.take<int>((size_t)2 * kMaxCell);
  ft.g_block_sums = a.take<int>((size_t)2 * (kMaxCell / 1024 + 2));
  ft.g_total = a.take<int64_t>(2);
  ft.g1_verts = a.take<float4>(V);
  ft.g3_verts = a.take<float4>(V);
  ft.g1_occ = a.take<unsigned char>(kMaxCell);
  ft.maxcell = kMaxCell;
  ft.nnl_on = nn_lists_enabled() ? 1 : 0;
  ft.nnl_cap = nn_list_cap();
  ft.nnl_count = a.take<int>(4);
  ft.nnl_cand = a.take<unsigned char>((size_t)kMaxCell * kNnlSub3);
  for (int g = 0; g < 2; ++g) {
    ft.nnl_slot[g] = a.take<int>(kMaxCell);
    ft.nnl_slot_cell[g] = a.take<int>(kNnlSlots);
    ft.nnl_len[g] = a.take<int>((size_t)kNnlSlots * kNnlSub3);
    ft.nnl_ent[g] = a.take<float4>((size_t)kNnlSlots * kNnlSub3 * kNnlCap);
  }
  L.lbs_joints = a.take<float>(kJoints * 3);
  L.lbs_pf = a.take<float>(kPoseFeat);
  L.planes_cl = a.take<float>((size_t)3 * sc.plane_ch * sc.plane_h * sc.plane_w);
  L.feat_cl = a.take<float>((size_t)sc.feat_ch * sc.feat_h * sc.feat_w);
  for (int l = 0; l < 3; ++l)
    L.vol_cl[l] = a.take<float>((size_t)sc.vol_ch[l] * sc.vol_dim[l][0] * sc.vol_dim[l][1] * sc.vol_dim[l][2]);
  L.sample_vid = a.take<int>(NS);
  L.ray_count = a.take<int>(N);
  L.block_sums = a.take<int>((size_t)N / 1024 + 2);
  L.ray_start = a.take<int>((size_t)N + 1);
  L.total = a.take<int64_t>(1);
  L.point_sample = a.take<int>(NS);
  L.point_vid = a.take<int>(NS);
  L.sigma = a.take<float>(NS);
  L.rgb = a.take<float>(NS * 3);
  L.fine_depths = nullptr; L.sample_vid_f = nullptr; L.ray_count_f = nullptr; L.ray_start_f = nullptr; L.total_f = nullptr;
  L.point_sample_f = nullptr; L.point_vid_f = nullptr; L.sigma_f = nullptr; L.rgb_f = nullptr;
  if (SF > 0) {
    L.fine_depths = a.take<float>(NF);
    L.sample_vid_f = a.take<int>(NF);
    L.ray_count_f = a.take<int>(N);
    L.ray_start_f = a.take<int>((size_t)N + 1);
    L.total_f = a.take<int64_t>(1);
    L.point_sample_f = a.take<int>(NF);
    L.point_vid_f = a.take<int>(NF);
    L.sigma_f = a.take<float>(NF);
    L.rgb_f = a.take<float>(NF * 3);
  }
  L.packed_w = a.take<float>(packed_weight_floats());
  L.canon_w = a.take<float>(canonical_weight_floats());
  L.fused_blob = a.take<unsigned char>(fused_blob_bytes());
  L.fused_bias = a.take<float>(10 * 144);
  L.xf_blob = a.take<float>(xformer_blob_floats());
  L.ff_blob = a.take<float>(fusion_blob_floats());
  const int cap = chunk_cap(N, S, SF);
  L.chunk = a.take<float>(chunk_buffer_floats(cap));
  L.pp_blob = a.take<unsigned char>(pp_blob_bytes());
  L.pp_bias = a.take<float>(10 * 128);
  L.pp_xv = a.take<unsigned char>(pp_xv_bytes(cap));
  L.gather2 = a.take<float>((size_t)cap * (288 + 192 + 8));
  L.xb_blob = a.take<unsigned char>(xformer_bf16_blob_bytes());
  L.fr_blob = a.take<unsigned char>(front_blob_bytes());
  return a.off;
}

// Device-time accounting per stage: every begin()/end() pair is a CUDA-event span on the launching stream; spans of
// the same stage are summed (the point stages run once per chunk).
struct StageTimer {
  struct Span { int stage; cudaEvent_t a, b; cudaStream_t s; };
  std::vector<Span> spans; bool on = false; cudaStream_t st = nullptr;
  std::vector<int> open_stack;
  // events are pooled per thread: creating / destroying ~60 events per forward costs more than the stages they time
  static std::vector<cudaEvent_t>& pool() { static thread_local std::vector<cudaEvent_t> p; return p; }
  size_t used = 0;
  cudaEvent_t get_event() {
    auto& p = pool();
    if (used == p.size()) { cudaEvent_t e; cudaEventCreate(&e); p.push_back(e); }
    return p[used++];
  }
  void init(bool enable, cudaStream_t s) { on = enable; st = s; used = 0; }
  void begin(int stage, cudaStream_t on_stream = nullptr) {
    if (!on) return;
    Span sp; sp.stage = stage; sp.s = on_stream ? on_stream : st;
    sp.a = get_event(); sp.b = get_event();
    cudaEventRecord(sp.a, sp.s);
    spans.push_back(sp);
    open_stack.push_back((int)spans.size() - 1);
  }
  void end() {
    if (!on || open_stack.empty()) return;
    cudaEventRecord(spans[open_stack.back()].b, spans[open_stack.back()].s);
    open_stack.pop_back();
  }
  void finish() {
    if (!on) return;
    for (int i = 0; i < 8; ++i) g_stage_ms[i] = 0.f;
    cudaStreamSynchronize(st);
    for (auto& sp : spans) {
      float ms = 0.f;
      cudaEventElapsedTime(&ms, sp.a, sp.b);
      g_stage_ms[sp.stage] += ms;
    }
    spans.clear();
  }
};

static thread_local StageTimer* g_tm = nullptr;

// Packed-weight reuse (SherfOptions.weights_version): identity of the packed blobs currently held by a scratch arena
struct PackTag { const void* base = nullptr; size_t need = 0; uint64_t version = 0; int precision = -1; int dev = -1; uint64_t scene = 0; };
static thread_local PackTag g_pack_tag;

// Pinned host words for the survivor counts: a device-to-host cudaMemcpyAsync into PAGEABLE memory blocks the calling thread until the
// copy has run, i.e. until the whole cull has finished (r1_x: 466 us of "launch issue"), which serialised the side-stream work behind it.
static int64_t* pinned_counts() {
  static thread_local int64_t* p = nullptr;
  if (!p && cudaHostAlloc((void**)&p, 4 * sizeof(int64_t), cudaHostAllocDefault) != cudaSuccess) p = nullptr;
  return p;
}

// Events recorded right after the survivor-count copies: the host waits on THEM, not on the stream, so the first chunk of the point stages
// (issued earlier with a device-side count) keeps the GPU busy while the host learns P.
static cudaEvent_t count_event(int which) {
  static thread_local cudaEvent_t ev[2] = {nullptr, nullptr};
  static thread_local int dev = -1;
  int d = 0;
  if (cudaGetDevice(&d) != cudaSuccess) return nullptr;
  if (d != dev) { ev[0] = ev[1] = nullptr; dev = d; }
  if (!ev[which] && cudaEventCreateWithFlags(&ev[which], cudaEventDisableTiming) != cudaSuccess) ev[which] = nullptr;
  return ev[which];
}

// Internal side stream (per host thread): the warp+gather kernel of chunk i+1 runs concurrently with the persistent MLP
// kernels of chunk i (they leave most issue slots idle and the gather kernel needs no shared memory).
struct SideStream {
  cudaStream_t s = nullptr; cudaEvent_t fork = nullptr, ldone = nullptr, gdone[2] = {nullptr, nullptr}, mdone[2] = {nullptr, nullptr}; int dev = -1;
  int ensure() {
    int d = 0;
    if (cudaGetDevice(&d) != cudaSuccess) return -1;
    if (s && d == dev) return 0;
    dev = d;
    // highest priority: the side stream carries chains of tiny dependent kernels (SMPL tables, grids) next to the machine-filling cull
    // kernels of the caller's stream; at default priority each of them queued behind thousands of cull blocks (r1_u: +0.3 ms)
    int lo = 0, hi = 0;
    cudaDeviceGetStreamPriorityRange(&lo, &hi);
    if (cudaStreamCreateWithPriority(&s, cudaStreamNonBlocking, hi) != cudaSuccess) return -1;
    cudaEventCreateWithFlags(&fork, cudaEventDisableTiming);
    cudaEventCreateWithFlags(&ldone, cudaEventDisableTiming);
    for (int i = 0; i < 2; ++i) { cudaEventCreateWithFlags(&gdone[i], cudaEventDisableTiming); cudaEventCreateWithFlags(&mdone[i], cudaEventDisableTiming); }
    return 0;
  }
};
static thread_local SideStream g_side;
// the per-call constants of the warp + gather kernels (forward chunks and the backward's recompute / scatter)
static void fill_gather_params(GatherParams& G, const SherfRays& rays, const SherfFrame& frame, const SherfScene& scene, const Layout& L) {
  G.origins = rays.origins; G.dirs = rays.dirs; G.nearv = rays.near_; G.farv = rays.far_; G.S = rays.n_samples; G.depths = nullptr;
  G.point_sample = L.point_sample; G.point_vid = L.point_vid; G.p0 = 0; G.np = 0; G.dc = DevCount{nullptr, 0, 0};
  G.fc = L.ft.fc; G.T1 = L.ft.T1; G.T3 = L.ft.T3; G.g3_start = L.ft.g3_cell_start; G.g3_verts = L.ft.g3_verts;
  G.t_vertices = getenv("SHERF_KNN3_UNSEEDED") ? nullptr : frame.t_vertices;
  G.nl3 = L.ft.lists(1);
  G.planes_cl = L.planes_cl; G.plane_h = scene.plane_h; G.plane_w = scene.plane_w;
  G.feat_cl = L.feat_cl; G.feat_h = scene.feat_h; G.feat_w = scene.feat_w; G.feat_ch = scene.feat_ch;
  G.img = scene.obs_img; G.img_h = scene.img_h; G.img_w = scene.img_w;
  for (int l = 0; l < 3; ++l) {
    G.vol_cl[l] = L.vol_cl[l]; G.vol_ch[l] = scene.vol_ch[l];
    G.vol_d[l] = scene.vol_dim[l][0]; G.vol_h[l] = scene.vol_dim[l][1]; G.vol_w[l] = scene.vol_dim[l][2];
  }
  G.comb = nullptr; G.f3raw = nullptr; G.geo = nullptr;
  G.g_planes_cl = nullptr; G.g_feat_cl = nullptr; G.g_vol_cl[0] = G.g_vol_cl[1] = G.g_vol_cl[2] = nullptr;
  G.dbg_vid3 = nullptr; G.dbg_can = nullptr; G.dbg_cdir = nullptr; G.dbg_uv = nullptr; G.dbg_feat = nullptr; G.dbg_max = 0; G.dbg_feat_max = 0;
}

// Backward arena = the forward arena (same carve, so the internal forward leaves its tables, layouts and per-point results where the backward
// expects them) followed by the backward's own buffers.
struct BwdLayout {
  float* out;                 // rgb | depth | acc of the internal forward (5 N)
  float* dsig; float* drgb;   // dL/d(sigma), dL/d(rgb) per surviving point
  float* g_planes_cl; float* g_feat_cl; float* g_vol_cl[3];
  float* canon_w; float* canon_bwd;   // tf32 hi / lo weights of the recompute pass and, transposed, of the dX products
  float* chunk; int bcap;
};
// points per backward chunk: 22.9 KB of kept activations / gradients per point.  Measured on B200 (512x512x64 view, 891 311 points): 2^17 -> 43.6 ms
// (then-current kernels), 2^18 -> 39.6, 2^19 -> 37.1, 2^20 -> 35.6 ms per training view (fewer, fuller launches); 2^20 = 24 GB of the 180 GB.
// SHERF_BWD_CHUNK_CAP lowers it; a view with fewer samples than the cap sizes the buffers by its own N x S.
static int bwd_chunk_cap(int N, int S) {
  const char* e = getenv("SHERF_BWD_CHUNK_CAP");                    // read per call: tests switch it between two backward passes
  const long v = e ? atol(e) : 0;
  const int cap = v >= 128 ? (int)(v / 128 * 128) : (1 << 20);
  const size_t NS = (size_t)N * S;
  return (int)(NS < (size_t)cap ? (NS + 127) / 128 * 128 : (size_t)cap);
}
static size_t carve_backward(Arena& a, const SherfScene& sc, int N, int S, int V, Layout& L, BwdLayout& B, size_t* fwd_need) {
  const size_t f = carve(a, sc, N, S, 0, V, L);
  if (fwd_need) *fwd_need = f;
  const size_t NS = (size_t)N * S;
  B.out = a.take<float>((size_t)5 * N);
  B.dsig = a.take<float>(NS);
  B.drgb = a.take<float>(NS * 3);
  B.g_planes_cl = a.take<float>((size_t)3 * sc.plane_ch * sc.plane_h * sc.plane_w);
  B.g_feat_cl = a.take<float>((size_t)sc.feat_ch * sc.feat_h * sc.feat_w);
  for (int l = 0; l < 3; ++l) B.g_vol_cl[l] = a.take<float>((size_t)sc.vol_ch[l] * sc.vol_dim[l][0] * sc.vol_dim[l][1] * sc.vol_dim[l][2]);
  B.canon_w = a.take<float>(canonical_weight_floats());
  B.canon_bwd = a.take<float>(canonical_bwd_weight_floats());
  B.bcap = bwd_chunk_cap(N, S);
  B.chunk = a.take<float>(bwd_chunk_floats(B.bcap));
  return a.off;
}

static void nested_begin(int stage) { if (g_tm) g_tm->begin(stage); }
static void nested_end() { if (g_tm) g_tm->end(); }

}  // namespace sherf

using namespace sherf;

extern "C" {

int sherf_abi_version(void) { return SHERF_ABI_VERSION; }
const char* sherf_last_error(void) { return g_err; }
int64_t sherf_last_launch_count(void) { return g_last_launches; }
int64_t sherf_last_importance_point_count(void) { return g_last_fine_points; }
void sherf_set_profiling(int enabled) { g_profiling = enabled; }
float sherf_last_stage_ms(int stage) { return (stage >= 0 && stage < 8) ? g_stage_ms[stage] : 0.f; }
float sherf_last_host_us(int part) { return (part >= 0 && part < 4) ? g_host_us[part] : 0.f; }

int sherf_nn_list_stats(double* out) {
  if (!out || !g_last_ft.nnl_on) { set_error("the last forward on this thread built no candidate lists"); return SHERF_E_INVALID; }
  const FrameTables& ft = g_last_ft;
  SHERF_CUDA_OK(cudaDeviceSynchronize());
  int cnt[4];
  SHERF_CUDA_OK(cudaMemcpy(cnt, ft.nnl_count, sizeof(cnt), cudaMemcpyDeviceToHost));
  out[0] = cnt[2];
  std::vector<int> len((size_t)kNnlSlots * kNnlSub3);
  for (int g = 0; g < 2; ++g) {
    const int nsub = (cnt[g] < kNnlSlots ? cnt[g] : kNnlSlots) * kNnlSub3;
    SHERF_CUDA_OK(cudaMemcpy(len.data(), ft.nnl_len[g], sizeof(int) * (size_t)nsub, cudaMemcpyDeviceToHost));
    double sum = 0.0, mx = 0.0, over = 0.0;
    for (int i = 0; i < nsub; ++i) {
      if (len[i] < 0) over += 1.0;
      else { sum += len[i]; mx = len[i] > mx ? len[i] : mx; }
    }
    out[1 + 4 * g] = nsub;
    out[2 + 4 * g] = nsub > over ? sum / (nsub - over) : 0.0;
    out[3 + 4 * g] = mx;
    out[4 + 4 * g] = nsub ? over / nsub : 0.0;
  }
  out[9] = ft.nnl_cap;
  return SHERF_OK;
}

size_t sherf_scratch_bytes(const SherfScene* scene, int32_t n_rays, int32_t n_samples, int32_t n_importance, int32_t n_verts) {
  if (!scene || n_rays <= 0 || n_samples < 2 || n_importance < 0 || n_verts <= 0) return 0;
  Arena a{nullptr, 0, 0, true};
  Layout L;
  return carve(a, *scene, n_rays, n_samples, n_importance, n_verts, L) + 512;   // + slack for aligning the caller's base pointer
}

static int validate(const SherfSmplModel* smpl, const SherfFrame* fr, const SherfScene* sc, const SherfWeights* w,
                    const SherfRays* rays, const SherfOptions* opts, const SherfOut* out) {
  if (!smpl || !fr || !sc || !w || !rays || !opts || !out) { set_error("null argument struct"); return SHERF_E_INVALID; }
  if (rays->n_rays <= 0 || rays->n_samples < 2 || rays->n_samples > 256) {
    set_error("n_rays must be > 0 and 2 <= n_samples <= 256 (got %d, %d)", rays->n_rays, rays->n_samples);
    return SHERF_E_INVALID;
  }
  if ((int64_t)rays->n_rays * rays->n_samples >= (1LL << 31)) { set_error("n_rays * n_samples must be < 2^31"); return SHERF_E_INVALID; }
  if (rays->n_importance < 0 || rays->n_importance > 256) { set_error("n_importance must be in 0..256 (got %d)", rays->n_importance); return SHERF_E_INVALID; }
  if (rays->n_importance > 0) {
    if (rays->n_samples < 3) { set_error("the importance pass needs n_samples >= 3 (sample_pdf bins, renderer.py:498-499)"); return SHERF_E_INVALID; }
    if (!opts->importance_u) { set_error("n_importance > 0 needs SherfOptions.importance_u (the torch.rand draws of renderer.py:526)"); return SHERF_E_INVALID; }
    const int64_t smax = rays->n_samples > rays->n_importance ? rays->n_samples : rays->n_importance;
    if ((int64_t)rays->n_rays * smax >= (1LL << 30)) { set_error("n_rays * max(n_samples, n_importance) must be < 2^30 with the importance pass"); return SHERF_E_INVALID; }
  }
  if (sc->plane_ch != 32 || sc->feat_ch != 64 || sc->vol_ch[0] != 32 || sc->vol_ch[1] != 64 || sc->vol_ch[2] != 96) {
    set_error("unsupported channel counts (planes %d, feat %d, volumes %d/%d/%d; expected 32, 64, 32/64/96)", sc->plane_ch,
              sc->feat_ch, sc->vol_ch[0], sc->vol_ch[1], sc->vol_ch[2]);
    return SHERF_E_UNSUPPORTED;
  }
  if (opts->mlp_precision < SHERF_MLP_FP32 || opts->mlp_precision > SHERF_MLP_BF16X3) { set_error("unknown mlp_precision %d", opts->mlp_precision); return SHERF_E_UNSUPPORTED; }
  if (!rays->origins || !rays->dirs || !rays->near_ || !rays->far_ || !out->rgb || !out->depth || !out->acc || !sc->planes ||
      !sc->obs_img || !sc->obs_feat || !sc->vol[0] || !sc->vol[1] || !sc->vol[2] || !smpl->weights || !smpl->posedirs) {
    set_error("null device pointer in arguments");
    return SHERF_E_INVALID;
  }
  {
    const SherfPose* poses[3] = {&fr->target, &fr->canonical, &fr->obs};
    bool ok = fr->vertices && fr->t_vertices && fr->t_world_bounds && fr->obs_K && fr->obs_R && fr->obs_T && fr->sp_bounds && smpl->v_template &&
              smpl->shapedirs && smpl->j_regressor;
    for (int i = 0; i < 3; ++i) ok = ok && poses[i]->poses && poses[i]->shapes;
    ok = ok && fr->target.R && fr->target.Th && fr->obs.R && fr->obs.Th;
    const float* const* wp = reinterpret_cast<const float* const*>(w);
    for (size_t i = 0; i < sizeof(SherfWeights) / sizeof(const float*); ++i) ok = ok && wp[i] != nullptr;
    if (!ok) { set_error("null device pointer in SherfFrame / SherfSmplModel / SherfWeights"); return SHERF_E_INVALID; }
  }
  return SHERF_OK;
}

#define RC(x) do { int _rc = (x); if (_rc) return _rc; } while (0)

int sherf_render_forward(const SherfSmplModel* smpl, const SherfFrame* frame, const SherfScene* scene,
                         const SherfWeights* weights, const SherfRays* rays, const SherfOptions* opts, const SherfOut* out,
                         const SherfDebug* dbg, void* scratch, size_t scratch_bytes, void* stream, int64_t* n_points_out) {
  g_err[0] = 0;
  const double t_enter = now_us();
  RC(validate(smpl, frame, scene, weights, rays, opts, out));
  const int N = rays->n_rays, S = rays->n_samples, SF = rays->n_importance, V = smpl->n_verts;
  cudaStream_t st = (cudaStream_t)stream;
  Arena a{(char*)scratch, scratch_bytes, 0, false};
  // align the arena base to 256 B
  const size_t mis = ((size_t)a.base) & 255;
  if (mis) { a.base += 256 - mis; a.size -= 256 - mis; }
  Layout L;
  const size_t need = carve(a, *scene, N, S, SF, V, L);
  if (!scratch || need > a.size) { set_error("scratch arena too small: need %zu bytes, have %zu", need, scratch_bytes); return SHERF_E_SCRATCH; }
  g_launches.n = 0;
  g_last_fine_points = 0;
  StageTimer tm;
  tm.init(g_profiling != 0, st);
  g_tm = &tm;
  // every exit path (the RC / SHERF_CUDA_OK early returns included) clears the thread-local timer pointer and, if the side stream was
  // forked and not yet joined, joins it into the caller's stream: the caller may free its tensors as soon as ITS stream has passed
  struct Guard {
    cudaStream_t st; bool forked = false, joined = false;
    ~Guard() {
      g_tm = nullptr;
      if (forked && !joined && g_side.s) { cudaEventRecord(g_side.ldone, g_side.s); cudaStreamWaitEvent(st, g_side.ldone, 0); }
    }
  } guard;
  guard.st = st;

  // ---- stage 0 + 1.  Per-frame work is split by consumer.  The caller's stream runs only what the cull needs (FrameConst, posed
  //      vertices in SMPL space, cull grid, depth range) and goes straight on to the cull + ordered compaction; an internal side stream
  //      runs, concurrently, what only the point stages need: SMPL chain / offsets / per-vertex warp tables / canonical grid (tiny
  //      latency-bound grids), the channels-last copies of the feature tensors (one launch) and the weight packing.  The host issues
  //      the cull BEFORE the side-stream work: these ~40 launches are host-issue bound (profiles/r1_t), and the point stages wait
  //      for both streams anyway. ----
  const bool side = !getenv("SHERF_NO_PROLOGUE_OVERLAP") && g_side.ensure() == 0;
  cudaStream_t ls = side ? g_side.s : st;
  tm.begin(0);
  RC(run_prologue_frame(*frame, L.ft, st));
  if (side) { SHERF_CUDA_OK(cudaEventRecord(g_side.fork, st)); SHERF_CUDA_OK(cudaStreamWaitEvent(ls, g_side.fork, 0)); guard.forked = true; }
  RC(run_prologue_cull(*smpl, *frame, *rays, *opts, L.ft, st));
  tm.end();
  tm.begin(1);
  int* sample_vid = (dbg && dbg->sample_vid) ? dbg->sample_vid : L.sample_vid;
  // dense per-sample ids of rays that miss the body are only needed by the debug taps and by the merged march of the fine pass
  RC(run_cull(*rays, S, nullptr, L.ft, sample_vid, L.ray_count, L.block_sums, L.ray_start, L.total, L.point_sample, L.point_vid, st,
              (dbg != nullptr || SF > 0) ? 1 : 0));
  tm.end();
  int64_t* hcount = pinned_counts();
  if (!hcount) { set_error("cudaHostAlloc failed for the survivor-count words"); return SHERF_E_CUDA; }
  SHERF_CUDA_OK(cudaMemcpyAsync(&hcount[0], L.total, sizeof(int64_t), cudaMemcpyDeviceToHost, st));
  cudaEvent_t ev_cnt0 = count_event(0), ev_cnt1 = count_event(1);
  if (!ev_cnt0 || !ev_cnt1) { set_error("cudaEventCreate failed"); return SHERF_E_CUDA; }
  SHERF_CUDA_OK(cudaEventRecord(ev_cnt0, st));

  RC(run_prologue_tables(*smpl, *frame, L.ft, ls));
  int devid0 = 0;
  SHERF_CUDA_OK(cudaGetDevice(&devid0));
  const bool scene_cached = opts->scene_version != 0 && g_pack_tag.scene == opts->scene_version && g_pack_tag.base == (const void*)a.base &&
                            g_pack_tag.need == need && g_pack_tag.dev == devid0 && !getenv("SHERF_NO_SCENE_REUSE");
  if (!scene_cached) {
    const size_t plane = (size_t)scene->plane_ch * scene->plane_h * scene->plane_w;
    const float* in[7] = {scene->planes, scene->planes + plane, scene->planes + 2 * plane, scene->obs_feat, scene->vol[0], scene->vol[1], scene->vol[2]};
    float* outp[7] = {L.planes_cl, L.planes_cl + plane, L.planes_cl + 2 * plane, L.feat_cl, L.vol_cl[0], L.vol_cl[1], L.vol_cl[2]};
    int C[7] = {scene->plane_ch, scene->plane_ch, scene->plane_ch, scene->feat_ch, scene->vol_ch[0], scene->vol_ch[1], scene->vol_ch[2]};
    int64_t M[7] = {(int64_t)scene->plane_h * scene->plane_w, (int64_t)scene->plane_h * scene->plane_w, (int64_t)scene->plane_h * scene->plane_w,
                    (int64_t)scene->feat_h * scene->feat_w, 0, 0, 0};
    for (int l = 0; l < 3; ++l) M[4 + l] = (int64_t)scene->vol_dim[l][0] * scene->vol_dim[l][1] * scene->vol_dim[l][2];
    RC(run_to_channels_last_multi(7, in, outp, C, M, ls));
    g_pack_tag.scene = 0;                       // (set below, once the arena identity of this call is recorded)
  }
  // Weight blobs: packed into the arena on this call unless the caller vouches (SherfOptions.weights_version != 0, unchanged since
  // the previous call on this arena, same arithmetic) that the parameters have not changed -- then only the host-side plans are rebuilt.
  PackedWeights pw;
  CanonWeights cw;
  FusedPlan fplan;
  PpPlan pplan;
  fplan.pp = nullptr; fplan.xf_blob = nullptr; fplan.ff_blob = nullptr; fplan.blob = nullptr; fplan.bias = nullptr; fplan.xb_blob = nullptr; fplan.fr_blob = nullptr;
  const bool use_fused = opts->mlp_precision != SHERF_MLP_FP32 && !getenv("SHERF_NO_FUSED_DECODER");
  const bool fuse_ff = use_fused && !getenv("SHERF_NO_FUSED_FUSION"), fuse_xf = use_fused && !getenv("SHERF_NO_FUSED_XFORMER");
  const bool use_pp = use_fused && opts->mlp_precision == SHERF_MLP_BF16X3;
  {
    int devid = 0;
    SHERF_CUDA_OK(cudaGetDevice(&devid));
    const bool reuse = opts->weights_version != 0 && g_pack_tag.version == opts->weights_version && g_pack_tag.base == (const void*)a.base &&
                       g_pack_tag.need == need && g_pack_tag.precision == opts->mlp_precision && g_pack_tag.dev == devid && !getenv("SHERF_NO_PACK_REUSE");
    g_pack_plan_only = reuse;
    int rc = SHERF_OK;
    if (opts->mlp_precision == SHERF_MLP_FP32) rc = run_pack_weights(*weights, L.packed_w, pw, ls);
    else if (!fuse_ff || !fuse_xf || !use_fused) rc = run_pack_canonical(*weights, L.canon_w, cw, ls);      // per-layer tensor-core kernels
    if (!rc && use_fused && !use_pp) rc = run_pack_fused_plan(*weights, L.fused_blob, L.fused_bias, fplan, ls);   // tf32 / 3xtf32 fused decoder
    if (!rc && fuse_ff) { if (!reuse) rc = run_pack_fusion(*weights, L.ff_blob, ls); fplan.ff_blob = L.ff_blob; }
    if (!rc && fuse_xf) { if (!reuse) rc = run_pack_xformer(*weights, L.xf_blob, ls); fplan.xf_blob = L.xf_blob; }
    if (!rc && use_pp) {
      rc = run_pack_pp(*weights, L.pp_blob, L.pp_bias, pplan, ls);
      const int cap = chunk_cap(N, S, SF);
      pplan.xp = L.pp_xv;
      pplan.vp = L.pp_xv + (size_t)((cap + 127) / 128) * 40960;
      fplan.pp = &pplan;
      if (!rc && fuse_xf && !getenv("SHERF_LEGACY_XFORMER")) {              // bf16 split-product transformer, two CTAs per SM
        if (!reuse) rc = run_pack_xformer_bf16(*weights, L.xb_blob, ls);
        fplan.xb_blob = L.xb_blob;
        if (!rc && fuse_ff && !getenv("SHERF_LEGACY_FRONT") && !getenv("SHERF_KNN3_UNSEEDED") && !getenv("SHERF_GATHER_V1")) {
          if (!reuse) rc = run_pack_front(*weights, L.fr_blob, ls);       // warp + gather + fusion in one kernel (front_fused.cu)
          fplan.fr_blob = L.fr_blob;
        }
      }
    }
    g_pack_plan_only = false;
    if (rc) return rc;
    g_pack_tag.base = a.base; g_pack_tag.need = need; g_pack_tag.version = opts->weights_version; g_pack_tag.precision = opts->mlp_precision;
    g_pack_tag.dev = devid;
    g_pack_tag.scene = opts->scene_version;
  }
  if (side) SHERF_CUDA_OK(cudaEventRecord(g_side.ldone, ls));

  // ---- stages 2+3 per chunk of surviving points: warp + gather (+ fusion), then transformer / decoder ----
  ChunkBuffers cb;
  carve_chunk_buffers(L.chunk, chunk_cap(N, S, SF), cb);
  ChunkBuffers cbs[2] = {cb, cb};                                   // two sets of gather outputs, everything else shared
  cbs[1].comb = L.gather2; cbs[1].f3raw = L.gather2 + (size_t)cb.cap * 288; cbs[1].geo = L.gather2 + (size_t)cb.cap * (288 + 192);
  // one chunk of a compacted point list (coarse: stratified depths; fine: importance-sampled depths): renderer.py:323-362.
  // dc.total != NULL: the chunk's point count is resolved on the device (np is then the upper bound that sizes the grids)
  auto issue_chunk = [&](const int* point_sample, const int* point_vid, int64_t p0, int np, int Sn, const float* depths, float* sigma_out,
                         float* rgb_out, const SherfDebug* d, DevCount dc, int ci, bool overlap, cudaStream_t gs) -> int {
    const int bsel = overlap ? (ci & 1) : 0;
    const ChunkBuffers& cbi = cbs[bsel];
    GatherParams G;
    fill_gather_params(G, *rays, *frame, *scene, L);
    G.S = Sn; G.depths = depths; G.point_sample = point_sample; G.point_vid = point_vid; G.p0 = p0; G.np = np; G.dc = dc;
    G.comb = cbi.comb; G.f3raw = cbi.f3raw; G.geo = cbi.geo;
    G.dbg_vid3 = d ? d->point_vid3 : nullptr; G.dbg_can = d ? d->point_can : nullptr;
    G.dbg_cdir = d ? d->point_cdir : nullptr; G.dbg_uv = d ? d->point_uv : nullptr;
    G.dbg_feat = d ? d->point_feat : nullptr; G.dbg_max = d ? d->max_points : 0;
    G.dbg_feat_max = d ? d->max_feat_points : 0;
    // gather of chunk ci (side stream): its output buffers must have been released by the MLP of chunk ci-2
    if (overlap && ci >= 2) SHERF_CUDA_OK(cudaStreamWaitEvent(gs, g_side.mdone[bsel], 0));
    tm.begin(2, gs);
    if (fplan.fr_blob) RC(run_front_fused(G, *weights, fplan.fr_blob, cbi.tok, gs));     // tokens straight from the gather lanes (no comb / f3raw)
    else RC(run_point_gather(G, gs));
    tm.end();
    if (overlap) { SHERF_CUDA_OK(cudaEventRecord(g_side.gdone[bsel], gs)); SHERF_CUDA_OK(cudaStreamWaitEvent(st, g_side.gdone[bsel], 0)); }
    tm.begin(3);
    RC(run_mlp(opts->mlp_precision, *weights, pw, cw, use_fused ? &fplan : nullptr, cbi, np, p0, sigma_out, rgb_out, d ? d->point_tok : nullptr,
               d ? d->max_points : 0, st, nested_begin, nested_end, dc));
    tm.end();
    if (overlap) SHERF_CUDA_OK(cudaEventRecord(g_side.mdone[bsel], st));
    return SHERF_OK;
  };
  // chunks [first_p0, Pn) of a pass with the host-side count
  auto run_points = [&](const int* point_sample, const int* point_vid, int64_t Pn, int64_t first_p0, int Sn, const float* depths, float* sigma_out,
                        float* rgb_out, const SherfDebug* d) -> int {
    // measured on B200 (r1): the overlap is neutral (6.98 vs 7.00 ms) -- the gather blocks delay the start of the persistent MLP CTAs
    // by as much as they hide -- so it is opt-in (SHERF_OVERLAP=1)
    const bool overlap = first_p0 == 0 && Pn > cb.cap && getenv("SHERF_OVERLAP") && g_side.ensure() == 0;
    cudaStream_t gs = overlap ? g_side.s : st;
    if (overlap) { SHERF_CUDA_OK(cudaEventRecord(g_side.fork, st)); SHERF_CUDA_OK(cudaStreamWaitEvent(gs, g_side.fork, 0)); }
    int ci = (int)(first_p0 / cb.cap);
    for (int64_t p0 = first_p0; p0 < Pn; p0 += cb.cap, ++ci) {
      const int np = (int)((Pn - p0 < cb.cap) ? (Pn - p0) : cb.cap);
      RC(issue_chunk(point_sample, point_vid, p0, np, Sn, depths, sigma_out, rgb_out, d, DevCount{nullptr, 0, 0}, ci, overlap, gs));
    }
    return SHERF_OK;
  };
  // The FIRST chunk of a pass is enqueued before the host knows the survivor count: its kernels resolve min(P, cap) from device memory
  // (front_fused / xformer_bf16 / decoder_pp, i.e. the default bf16x3 path without debug taps).  The host then waits for the COUNT EVENT
  // only -- the GPU is already working on chunk 0 -- and enqueues the remaining chunks with exact counts.
  const bool async_first = fplan.fr_blob && fplan.xb_blob && use_pp && !dbg && !getenv("SHERF_SYNC_FIRST_CHUNK");
  if (side) { SHERF_CUDA_OK(cudaStreamWaitEvent(st, g_side.ldone, 0)); guard.joined = true; }         // layouts + packed weights are ready
  if (async_first)
    RC(issue_chunk(L.point_sample, L.point_vid, 0, cb.cap, S, nullptr, L.sigma, L.rgb, nullptr, DevCount{L.total, 0, cb.cap}, 0, false, st));
  const double t_sync0 = now_us();
  SHERF_CUDA_OK(cudaEventSynchronize(ev_cnt0));              // the survivor count P (the cull is done; everything enqueued after it may still run)
  const int64_t P = hcount[0];
  const double t_sync1 = now_us();
  if (n_points_out) *n_points_out = P;
  if (dbg && dbg->point_sample && P > 0)
    SHERF_CUDA_OK(cudaMemcpyAsync(dbg->point_sample, L.point_sample, sizeof(int) * (size_t)(P < dbg->max_points ? P : dbg->max_points),
                                  cudaMemcpyDeviceToDevice, st));
  RC(run_points(L.point_sample, L.point_vid, P, async_first ? cb.cap : 0, S, nullptr, L.sigma, L.rgb, dbg));
  if (dbg && P > 0) {
    const size_t cnt = (size_t)(P < dbg->max_points ? P : dbg->max_points);
    if (dbg->point_sigma) SHERF_CUDA_OK(cudaMemcpyAsync(dbg->point_sigma, L.sigma, sizeof(float) * cnt, cudaMemcpyDeviceToDevice, st));
    if (dbg->point_rgb) SHERF_CUDA_OK(cudaMemcpyAsync(dbg->point_rgb, L.rgb, sizeof(float) * 3 * cnt, cudaMemcpyDeviceToDevice, st));
  }

  if (SF == 0) {
    // ---- stage 4: composite ----
    tm.begin(4);
    RC(run_composite(*rays, L.ft.fc, L.ray_start, L.point_sample, L.sigma, L.rgb, opts->density_noise, opts->white_back, *out, st));
    tm.end();
  } else {
    // ---- fine pass (renderer.py:373-393, repaired): coarse weights -> importance depths -> cull / gather / MLP on the fine samples ->
    //      ray march over the depth-sorted union ----
    tm.begin(4);
    RC(run_importance_sample(*rays, L.ray_start, L.point_sample, L.sigma, opts->density_noise, nullptr, opts->importance_u, L.fine_depths,
                             dbg ? dbg->fine_bins : nullptr, dbg ? dbg->coarse_weights : nullptr, st));
    tm.end();
    tm.begin(1);
    int* vid_f = (dbg && dbg->fine_sample_vid) ? dbg->fine_sample_vid : L.sample_vid_f;
    RC(run_cull(*rays, SF, L.fine_depths, L.ft, vid_f, L.ray_count_f, L.block_sums, L.ray_start_f, L.total_f, L.point_sample_f, L.point_vid_f, st));
    tm.end();
    SHERF_CUDA_OK(cudaMemcpyAsync(&hcount[1], L.total_f, sizeof(int64_t), cudaMemcpyDeviceToHost, st));
    SHERF_CUDA_OK(cudaEventRecord(ev_cnt1, st));
    if (async_first)
      RC(issue_chunk(L.point_sample_f, L.point_vid_f, 0, cb.cap, SF, L.fine_depths, L.sigma_f, L.rgb_f, nullptr, DevCount{L.total_f, 0, cb.cap}, 0, false, st));
    SHERF_CUDA_OK(cudaEventSynchronize(ev_cnt1));
    const int64_t PF = hcount[1];
    if (n_points_out) *n_points_out = P + PF;
    g_last_fine_points = PF;
    RC(run_points(L.point_sample_f, L.point_vid_f, PF, async_first ? cb.cap : 0, SF, L.fine_depths, L.sigma_f, L.rgb_f, nullptr));
    if (dbg) {
      if (dbg->fine_depths) SHERF_CUDA_OK(cudaMemcpyAsync(dbg->fine_depths, L.fine_depths, sizeof(float) * (size_t)N * SF, cudaMemcpyDeviceToDevice, st));
      RC(run_dense_taps(L.point_sample_f, L.sigma_f, L.rgb_f, PF, (int64_t)N * SF, dbg->fine_sigma, dbg->fine_rgb, st));
    }
    tm.begin(4);
    RC(run_composite_merged(*rays, L.ft.fc, sample_vid, L.ray_start, L.sigma, L.rgb, opts->density_noise, L.fine_depths, vid_f, L.ray_start_f,
                            L.sigma_f, L.rgb_f, opts->density_noise_importance, opts->white_back, *out, st));
    tm.end();
  }
  tm.finish();
  g_last_launches = g_launches.n;
  g_last_ft = L.ft;
  { const double t_exit = now_us(); g_host_us[0] = (float)(t_sync0 - t_enter); g_host_us[1] = (float)(t_sync1 - t_sync0); g_host_us[2] = (float)(t_exit - t_sync1); g_host_us[3] = (float)(t_exit - t_enter); }
  return SHERF_OK;
}

size_t sherf_backward_scratch_bytes(const SherfScene* scene, int32_t n_rays, int32_t n_samples, int32_t n_verts) {
  if (!scene || n_rays <= 0 || n_samples < 2 || n_verts <= 0) return 0;
  Arena a{nullptr, 0, 0, true};
  Layout L;
  BwdLayout B;
  return carve_backward(a, *scene, n_rays, n_samples, n_verts, L, B, nullptr) + 512;
}

static int render_backward_impl(const SherfSmplModel* smpl, const SherfFrame* frame, const SherfScene* scene, const SherfWeights* weights,
                                const SherfRays* rays, const SherfOptions* opts, const SherfOutGrads* grad_out, const SherfWeightGrads* grad_weights,
                                const SherfInputGrads* grad_inputs, void* scratch, size_t scratch_bytes, void* stream, int64_t* n_points_out,
                                int64_t forward_points /* >= 0: the forward already ran on this arena */);

int sherf_render_backward(const SherfSmplModel* smpl, const SherfFrame* frame, const SherfScene* scene, const SherfWeights* weights,
                          const SherfRays* rays, const SherfOptions* opts, const SherfOutGrads* grad_out, const SherfWeightGrads* grad_weights,
                          const SherfInputGrads* grad_inputs, void* scratch, size_t scratch_bytes, void* stream, int64_t* n_points_out) {
  return render_backward_impl(smpl, frame, scene, weights, rays, opts, grad_out, grad_weights, grad_inputs, scratch, scratch_bytes, stream, n_points_out, -1);
}

int sherf_render_backward_after_forward(const SherfSmplModel* smpl, const SherfFrame* frame, const SherfScene* scene, const SherfWeights* weights,
                                        const SherfRays* rays, const SherfOptions* opts, const SherfOutGrads* grad_out,
                                        const SherfWeightGrads* grad_weights, const SherfInputGrads* grad_inputs, void* scratch, size_t scratch_bytes,
                                        void* stream, int64_t n_points) {
  if (n_points < 0) { g_err[0] = 0; set_error("n_points must be the survivor count the forward reported"); return SHERF_E_INVALID; }
  return render_backward_impl(smpl, frame, scene, weights, rays, opts, grad_out, grad_weights, grad_inputs, scratch, scratch_bytes, stream, nullptr, n_points);
}

}  // extern "C"

static int render_backward_impl(const SherfSmplModel* smpl, const SherfFrame* frame, const SherfScene* scene, const SherfWeights* weights,
                                const SherfRays* rays, const SherfOptions* opts, const SherfOutGrads* grad_out, const SherfWeightGrads* grad_weights,
                                const SherfInputGrads* grad_inputs, void* scratch, size_t scratch_bytes, void* stream, int64_t* n_points_out,
                                int64_t forward_points) {
  g_err[0] = 0;
  if (!smpl || !frame || !scene || !weights || !rays || !opts || !grad_out || !scratch) { set_error("null argument"); return SHERF_E_INVALID; }
  if (rays->n_importance != 0) {
    set_error("sherf_render_backward covers the coarse pass only (n_importance must be 0; the reference's fine pass cannot execute, SURVEY a13)");
    return SHERF_E_UNSUPPORTED;
  }
  const int N = rays->n_rays, S = rays->n_samples, V = smpl->n_verts;
  if (N <= 0 || S < 2 || V <= 0) { set_error("bad sizes"); return SHERF_E_INVALID; }
  cudaStream_t st = (cudaStream_t)stream;
  Arena a{(char*)scratch, scratch_bytes, 0, false};
  const size_t mis = ((size_t)a.base) & 255;
  if (mis) { a.base += 256 - mis; a.size -= 256 - mis; }
  Layout L;
  BwdLayout B;
  size_t fwd_need = 0;
  const size_t need = carve_backward(a, *scene, N, S, V, L, B, &fwd_need);
  if (need > a.size) { set_error("backward scratch arena too small: need %zu bytes, have %zu", need, scratch_bytes); return SHERF_E_SCRATCH; }

  // ---- the view once more on the fast path: leaves frame tables, channels-last layouts, the compacted point list and per-point sigma / rgb
  //      in the first part of the arena ----
  SherfOut fout; fout.rgb = B.out; fout.depth = B.out + (size_t)3 * N; fout.acc = B.out + (size_t)4 * N;
  int64_t P = forward_points;
  int64_t launches = 0;
  if (forward_points < 0) {
    RC(sherf_render_forward(smpl, frame, scene, weights, rays, opts, &fout, nullptr, a.base, fwd_need + 256, stream, &P));
    launches = g_launches.n;
  } else if (forward_points > (int64_t)N * S) { set_error("n_points exceeds n_rays * n_samples"); return SHERF_E_INVALID; }
  if (n_points_out) *n_points_out = P;
  g_launches.n = 0;

  // ---- outputs start from zero ----
  SherfWeightGrads gw;
  if (grad_weights) gw = *grad_weights; else memset(&gw, 0, sizeof(gw));
  {
    float* const* gp = reinterpret_cast<float* const*>(&gw);
    const int n_out[20] = {96, 32, 32, 144, 32, 32, 32, 32, 128, 128, 128, 128, 128, 128, 128, 128, 1, 128, 64, 3};
    const int n_in[20] = {192, 96, 0, 32, 48, 0, 32, 32, 71, 128, 128, 128, 128, 199, 128, 128, 128, 128, 187, 64};
    // struct order: proj w,b | reproj w,b | ln1 w,b | qkv w | attn_out w,b | ln2 w,b | ff1 w,b | ff2 w,b | pts_w[8] | pts_b[8] | alpha.. | feature.. | views.. | rgb..
    size_t sizes[39]; int k = 0;
    auto wb = [&](int layer, bool bias) { sizes[k++] = (size_t)n_out[layer] * (n_in[layer] ? n_in[layer] : 1); if (bias) sizes[k++] = n_out[layer]; };
    wb(0, true); wb(1, true);
    sizes[k++] = 32; sizes[k++] = 32;                 // ln1 weight, bias
    wb(3, false); wb(4, true);
    sizes[k++] = 32; sizes[k++] = 32;                 // ln2
    wb(6, true); wb(7, true);
    for (int i = 0; i < 8; ++i) sizes[k++] = (size_t)128 * n_in[8 + i];
    for (int i = 0; i < 8; ++i) sizes[k++] = 128;
    wb(16, true); wb(17, true); wb(18, true); wb(19, true);
    if (k != 39 || sizeof(SherfWeightGrads) != 39 * sizeof(float*)) { set_error("internal: weight table mismatch"); return SHERF_E_INVALID; }
    for (int i = 0; i < 39; ++i)
      if (gp[i]) SHERF_CUDA_OK(cudaMemsetAsync(gp[i], 0, sizes[i] * sizeof(float), st));
  }
  const bool want_planes = grad_inputs && grad_inputs->planes, want_feat = grad_inputs && grad_inputs->obs_feat;
  bool want_vol[3];
  for (int l = 0; l < 3; ++l) want_vol[l] = grad_inputs && grad_inputs->vol[l];
  const size_t plane = (size_t)scene->plane_ch * scene->plane_h * scene->plane_w;
  if (want_planes) SHERF_CUDA_OK(cudaMemsetAsync(B.g_planes_cl, 0, 3 * plane * sizeof(float), st));
  if (want_feat) SHERF_CUDA_OK(cudaMemsetAsync(B.g_feat_cl, 0, (size_t)scene->feat_ch * scene->feat_h * scene->feat_w * sizeof(float), st));
  size_t vol_n[3];
  for (int l = 0; l < 3; ++l) {
    vol_n[l] = (size_t)scene->vol_ch[l] * scene->vol_dim[l][0] * scene->vol_dim[l][1] * scene->vol_dim[l][2];
    if (want_vol[l]) SHERF_CUDA_OK(cudaMemsetAsync(B.g_vol_cl[l], 0, vol_n[l] * sizeof(float), st));
  }

  if (P > 0) {
    PackedWeights pw;
    g_pack_plan_only = false;
    RC(run_pack_weights(*weights, L.packed_w, pw, st));
    CanonWeights cw;
    CanonBwdWeights cbw;
    RC(run_pack_canonical(*weights, B.canon_w, cw, st));
    RC(run_pack_canonical_bwd(*weights, B.canon_bwd, cbw, st));
    RC(run_composite_backward(*rays, L.ft.fc, L.ray_start, L.point_sample, L.sigma, L.rgb, opts->density_noise, opts->white_back, grad_out->rgb,
                              grad_out->depth, grad_out->acc, B.dsig, B.drgb, st));
    BwdChunk bc;
    carve_bwd_chunk(B.chunk, B.bcap, bc);
    GatherParams G;
    fill_gather_params(G, *rays, *frame, *scene, L);
    // the candidate lists in the arena are those of whichever forward ran on it last (with or without lists): the re-gather takes the
    // grid search, which picks the same vertices
    G.nl3 = NnLists{nullptr, nullptr, nullptr, nullptr};
    for (int64_t p0 = 0; p0 < P; p0 += B.bcap) {
      const int np = (int)((P - p0 < B.bcap) ? (P - p0) : B.bcap);
      RC(run_backward_chunk(*weights, pw, cw, cbw, gw, G, bc, np, p0, L.rgb, B.dsig, B.drgb, st));
      GatherParams Gs = G;
      Gs.g_planes_cl = want_planes ? B.g_planes_cl : nullptr;
      Gs.g_feat_cl = want_feat ? B.g_feat_cl : nullptr;
      for (int l = 0; l < 3; ++l) Gs.g_vol_cl[l] = want_vol[l] ? B.g_vol_cl[l] : nullptr;
      RC(run_backward_chunk_inputs(*weights, cbw, Gs, bc, np, p0, st));
    }
  }
  // ---- channels-last gradient grids -> the caller's PyTorch layouts ----
  if (want_planes)
    for (int k = 0; k < 3; ++k)
      RC(run_from_channels_last(B.g_planes_cl + k * plane, grad_inputs->planes + k * plane, scene->plane_ch, (int64_t)scene->plane_h * scene->plane_w, st));
  if (want_feat) RC(run_from_channels_last(B.g_feat_cl, grad_inputs->obs_feat, scene->feat_ch, (int64_t)scene->feat_h * scene->feat_w, st));
  for (int l = 0; l < 3; ++l)
    if (want_vol[l])
      RC(run_from_channels_last(B.g_vol_cl[l], grad_inputs->vol[l], scene->vol_ch[l], (int64_t)(vol_n[l] / scene->vol_ch[l]), st));
  g_last_launches = launches + g_launches.n;
  return SHERF_OK;
}

extern "C" {

int sherf_count_survivors(const SherfSmplModel* smpl, const SherfFrame* frame, const SherfScene* scene, const SherfRays* rays, const SherfOptions* opts,
                          void* scratch, size_t scratch_bytes, void* stream, int64_t* n_points_out) {
  g_err[0] = 0;
  if (!smpl || !frame || !scene || !rays || !opts || !scratch || !n_points_out) { set_error("null argument"); return SHERF_E_INVALID; }
  if (rays->n_rays <= 0 || rays->n_samples < 2 || rays->n_samples > 256 || !rays->origins || !rays->dirs || !rays->near_ || !rays->far_) {
    set_error("bad rays"); return SHERF_E_INVALID;
  }
  const int N = rays->n_rays, S = rays->n_samples, SF = rays->n_importance, V = smpl->n_verts;
  cudaStream_t st = (cudaStream_t)stream;
  Arena a{(char*)scratch, scratch_bytes, 0, false};
  const size_t mis = ((size_t)a.base) & 255;
  if (mis) { a.base += 256 - mis; a.size -= 256 - mis; }
  Layout L;
  const size_t need = carve(a, *scene, N, S, SF, V, L);
  if (need > a.size) { set_error("scratch arena too small: need %zu bytes, have %zu", need, scratch_bytes); return SHERF_E_SCRATCH; }
  g_launches.n = 0;
  RC(run_prologue_frame(*frame, L.ft, st));
  RC(run_prologue_cull(*smpl, *frame, *rays, *opts, L.ft, st));
  RC(run_cull(*rays, S, nullptr, L.ft, L.sample_vid, L.ray_count, L.block_sums, L.ray_start, L.total, L.point_sample, L.point_vid, st));
  int64_t* hcount = pinned_counts();
  if (!hcount) { set_error("cudaHostAlloc failed for the survivor-count words"); return SHERF_E_CUDA; }
  SHERF_CUDA_OK(cudaMemcpyAsync(&hcount[2], L.total, sizeof(int64_t), cudaMemcpyDeviceToHost, st));
  SHERF_CUDA_OK(cudaStreamSynchronize(st));
  *n_points_out = hcount[2];
  g_last_launches = g_launches.n;
  return SHERF_OK;
}

int sherf_debug_sample_importance(const SherfRays* rays, const float* weights, const float* u, float* t_fine_out, int32_t* bins_out,
                                  void* stream) {
  g_err[0] = 0;
  if (!rays || !weights || !u || !t_fine_out || !rays->near_ || !rays->far_) { set_error("null argument"); return SHERF_E_INVALID; }
  if (rays->n_rays <= 0 || rays->n_samples < 3 || rays->n_samples > 256 || rays->n_importance < 1 || rays->n_importance > 256) {
    set_error("need n_rays > 0, 3 <= n_samples <= 256, 1 <= n_importance <= 256");
    return SHERF_E_INVALID;
  }
  g_launches.n = 0;
  RC(run_importance_sample(*rays, nullptr, nullptr, nullptr, nullptr, weights, u, t_fine_out, bins_out, nullptr, (cudaStream_t)stream));
  g_last_launches = g_launches.n;
  return SHERF_OK;
}

int sherf_generate_rays(const double* K, const double* R, const double* T, int32_t H, int32_t W, const double* bounds, float* origins,
                        float* dirs, float* near_out, float* far_out, uint8_t* mask_at_box, void* stream) {
  g_err[0] = 0;
  if (!K || !R || !T || !bounds || !origins || !dirs || !near_out || !far_out) { set_error("null argument"); return SHERF_E_INVALID; }
  if (H <= 0 || W <= 0 || (int64_t)H * W >= (1LL << 31)) { set_error("bad image size %d x %d", H, W); return SHERF_E_INVALID; }
  g_launches.n = 0;
  RC(run_generate_rays(K, R, T, H, W, bounds, origins, dirs, near_out, far_out, mask_at_box, (cudaStream_t)stream));
  g_last_launches = g_launches.n;
  return SHERF_OK;
}

size_t sherf_sparse_encoder_scratch_bytes(int32_t n_voxels, const int32_t* out_sh) {
  if (n_voxels <= 0 || !out_sh || out_sh[0] <= 0 || out_sh[1] <= 0 || out_sh[2] <= 0) return 0;
  return sparse_encoder_scratch_bytes(n_voxels, out_sh);
}

int sherf_sparse_encode(const SherfSparseEncoder* enc, const int32_t* coord, const float* feat, int32_t n, const int32_t* out_sh, float* vol1,
                        float* vol2, float* vol3, void* scratch, size_t scratch_bytes, void* stream) {
  g_err[0] = 0;
  if (!enc || !coord || !feat || !out_sh || !vol1 || !vol2 || !vol3 || !scratch) { set_error("null argument"); return SHERF_E_INVALID; }
  if (n <= 0 || out_sh[0] <= 0 || out_sh[1] <= 0 || out_sh[2] <= 0 || (int64_t)out_sh[0] * out_sh[1] * out_sh[2] >= (1LL << 31)) {
    set_error("bad sparse input: n = %d, out_sh = %d x %d x %d", n, out_sh[0], out_sh[1], out_sh[2]);
    return SHERF_E_INVALID;
  }
  for (int c = 0; c < SHERF_SPARSE_CONVS; ++c)
    if (!enc->conv[c].weight || !enc->conv[c].bn_weight || !enc->conv[c].bn_bias || !enc->conv[c].bn_mean || !enc->conv[c].bn_var) {
      set_error("sparse conv %d: null parameter pointer", c);
      return SHERF_E_INVALID;
    }
  float* vols[3] = {vol1, vol2, vol3};
  g_launches.n = 0;
  RC(run_sparse_encode(*enc, coord, feat, n, out_sh, vols, scratch, scratch_bytes, (cudaStream_t)stream));
  g_last_launches = g_launches.n;
  return SHERF_OK;
}

static int check_sparse_args(const SherfSparseEncoder* enc, const int32_t* coord, int32_t n, const int32_t* out_sh) {
  if (!enc || !coord || !out_sh) { set_error("null argument"); return SHERF_E_INVALID; }
  if (n <= 0 || out_sh[0] <= 0 || out_sh[1] <= 0 || out_sh[2] <= 0 || (int64_t)out_sh[0] * out_sh[1] * out_sh[2] >= (1LL << 31)) {
    set_error("bad sparse input: n = %d, out_sh = %d x %d x %d", n, out_sh[0], out_sh[1], out_sh[2]);
    return SHERF_E_INVALID;
  }
  for (int c = 0; c < SHERF_SPARSE_CONVS; ++c)
    if (!enc->conv[c].weight || !enc->conv[c].bn_weight || !enc->conv[c].bn_bias || !enc->conv[c].bn_mean || !enc->conv[c].bn_var) {
      set_error("sparse conv %d: null parameter pointer", c);
      return SHERF_E_INVALID;
    }
  return SHERF_OK;
}

size_t sherf_sparse_encoder_train_scratch_bytes(int32_t n_voxels, const int32_t* out_sh) {
  if (n_voxels <= 0 || !out_sh || out_sh[0] <= 0 || out_sh[1] <= 0 || out_sh[2] <= 0) return 0;
  return sparse_encoder_train_scratch_bytes(n_voxels, out_sh);
}

int sherf_sparse_encode_train(const SherfSparseEncoder* enc, const int32_t* coord, const float* feat, int32_t n, const int32_t* out_sh, float* vol1,
                              float* vol2, float* vol3, float* batch_stats, int32_t* row_counts, int32_t use_running_stats, void* scratch,
                              size_t scratch_bytes, void* stream) {
  g_err[0] = 0;
  RC(check_sparse_args(enc, coord, n, out_sh));
  if (!feat || !vol1 || !vol2 || !vol3 || !scratch) { set_error("null argument"); return SHERF_E_INVALID; }
  float* vols[3] = {vol1, vol2, vol3};
  g_launches.n = 0;
  RC(run_sparse_encode_train(*enc, coord, feat, n, out_sh, vols, batch_stats, row_counts, use_running_stats, scratch, scratch_bytes, (cudaStream_t)stream));
  g_last_launches = g_launches.n;
  return SHERF_OK;
}

int sherf_sparse_encode_backward(const SherfSparseEncoder* enc, const int32_t* coord, int32_t n, const int32_t* out_sh, const float* g_vol1,
                                 const float* g_vol2, const float* g_vol3, const SherfSparseEncoderGrads* grads, float* g_feat,
                                 int32_t use_running_stats, void* scratch, size_t scratch_bytes, void* stream) {
  g_err[0] = 0;
  RC(check_sparse_args(enc, coord, n, out_sh));
  if (!grads || !scratch) { set_error("null argument"); return SHERF_E_INVALID; }
  if (!g_vol3) { set_error("the gradient of the last level (vol3) is required: nothing else reaches conv3"); return SHERF_E_INVALID; }
  const float* gv[3] = {g_vol1, g_vol2, g_vol3};
  g_launches.n = 0;
  RC(run_sparse_encode_backward(*enc, coord, n, out_sh, gv, *grads, g_feat, use_running_stats, scratch, scratch_bytes, (cudaStream_t)stream));
  g_last_launches = g_launches.n;
  return SHERF_OK;
}

int sherf_prepare_observation_backward(const SherfSmplModel* smpl, const SherfObservation* obs, const float* g_vert_feat, float* g_proj_w,
                                       float* g_proj_b, float* g_obs_feat, void* scratch, size_t scratch_bytes, void* stream) {
  g_err[0] = 0;
  if (!smpl || !obs || !g_vert_feat || !scratch) { set_error("null argument"); return SHERF_E_INVALID; }
  if (smpl->n_verts <= 0 || !obs->obs_vertices || !obs->faces || !obs->last_face || !obs->obs_img || !obs->obs_feat || !obs->proj_w || !obs->obs_K ||
      !obs->obs_R || !obs->obs_T || !obs->obs.R || !obs->obs.Th) {
    set_error("null device pointer in SherfObservation / SherfSmplModel");
    return SHERF_E_INVALID;
  }
  if (obs->feat_ch != 64 || obs->img_h <= 0 || obs->img_w <= 0 || obs->feat_h <= 0 || obs->feat_w <= 0) {
    set_error("unsupported observation shapes (feature channels %d, expected 64)", obs->feat_ch);
    return SHERF_E_UNSUPPORTED;
  }
  g_launches.n = 0;
  RC(run_prepare_observation_backward(*smpl, *obs, g_vert_feat, g_proj_w, g_proj_b, g_obs_feat, scratch, scratch_bytes, (cudaStream_t)stream));
  g_last_launches = g_launches.n;
  return SHERF_OK;
}

size_t sherf_observation_scratch_bytes(int32_t n_verts) { return n_verts > 0 ? observation_scratch_bytes(n_verts, kMaxCell) + 512 : 0; }

int sherf_prepare_observation(const SherfSmplModel* smpl, const SherfObservation* obs, float* vert_feat, int32_t* coord, uint8_t* vertex_mask,
                              float* bounds, int32_t* out_sh_host, float* canonical_out, void* scratch, size_t scratch_bytes, void* stream) {
  g_err[0] = 0;
  if (!smpl || !obs || !vert_feat || !coord || !bounds || !out_sh_host || !scratch) { set_error("null argument"); return SHERF_E_INVALID; }
  if (smpl->n_verts <= 0 || !smpl->weights || !smpl->posedirs || !obs->obs_vertices || !obs->t_vertices || !obs->faces || !obs->last_face ||
      !obs->obs_img || !obs->obs_feat || !obs->proj_w || !obs->proj_b || !obs->obs_K || !obs->obs_R || !obs->obs_T || !obs->obs.poses ||
      !obs->canonical.poses) {
    set_error("null device pointer in SherfObservation / SherfSmplModel");
    return SHERF_E_INVALID;
  }
  if (obs->feat_ch != 64 || obs->img_h <= 0 || obs->img_w <= 0 || obs->feat_h <= 0 || obs->feat_w <= 0) {
    set_error("unsupported observation shapes (feature channels %d, expected 64)", obs->feat_ch);
    return SHERF_E_UNSUPPORTED;
  }
  g_launches.n = 0;
  RC(run_prepare_observation(*smpl, *obs, vert_feat, coord, vertex_mask, bounds, out_sh_host, canonical_out, scratch, scratch_bytes,
                             (cudaStream_t)stream));
  g_last_launches = g_launches.n;
  return SHERF_OK;
}

void sherf_debug_set_trace(long long* device_buf) { g_fused_trace = device_buf; }

int sherf_debug_linear(int precision, const float* A, int lda, const float* W, const float* bias, float* Y, int ldy, int M, int N,
                       int K, int act, void* scratch, size_t scratch_bytes, void* stream) {
  g_err[0] = 0;
  if (!A || !W || !Y || !scratch || M <= 0 || N <= 0 || K <= 0 || N > 256 || K > 256) { set_error("bad argument"); return SHERF_E_INVALID; }
  const size_t need = (size_t)8 * 272 * 272 * sizeof(float) + 512;
  if (scratch_bytes < need) { set_error("scratch arena too small: need %zu bytes", need); return SHERF_E_SCRATCH; }
  char* b = (char*)scratch;
  const size_t mis = ((size_t)b) & 255;
  if (mis) b += 256 - mis;
  cudaStream_t st = (cudaStream_t)stream;
  g_launches.n = 0;
  RC(run_debug_linear(precision, A, lda, W, bias, Y, ldy, M, N, K, act, (float*)b, st));
  g_last_launches = g_launches.n;
  return SHERF_OK;
}

int sherf_lbs_transforms(const SherfSmplModel* smpl, const SherfPose* pose, float* A_out, void* scratch, size_t scratch_bytes,
                         void* stream) {
  g_err[0] = 0;
  if (!smpl || !pose || !A_out || !scratch) { set_error("null argument"); return SHERF_E_INVALID; }
  const size_t need = (kJoints * 3 + kPoseFeat) * sizeof(float) + 256;
  if (scratch_bytes < need) { set_error("scratch arena too small: need %zu bytes, have %zu", need, scratch_bytes); return SHERF_E_SCRATCH; }
  char* b = (char*)scratch;
  const size_t mis = ((size_t)b) & 255;
  if (mis) b += 256 - mis;
  float* joints = (float*)b;
  float* pf = joints + kJoints * 3;
  g_launches.n = 0;
  RC(run_lbs_only(*smpl, *pose, A_out, joints, pf, (cudaStream_t)stream));
  g_last_launches = g_launches.n;
  return SHERF_OK;
}

int sherf_smpl_vertices(const SherfSmplModel* smpl, const SherfPose* pose, float* verts_smpl, float* verts_world, void* scratch, size_t scratch_bytes,
                        void* stream) {
  g_err[0] = 0;
  if (!smpl || !pose || !scratch || (!verts_smpl && !verts_world)) { set_error("null argument"); return SHERF_E_INVALID; }
  if (!smpl->v_template || !smpl->shapedirs || !smpl->posedirs || !smpl->j_regressor || !smpl->weights || !pose->poses || !pose->shapes || smpl->n_verts <= 0) {
    set_error("null device pointer in SherfSmplModel / SherfPose"); return SHERF_E_INVALID;
  }
  if (verts_world && (!pose->R || !pose->Th)) { set_error("verts_world needs SherfPose.R and .Th"); return SHERF_E_INVALID; }
  g_launches.n = 0;
  RC(run_smpl_vertices(*smpl, *pose, verts_smpl, verts_world, scratch, scratch_bytes, (cudaStream_t)stream));
  g_last_launches = g_launches.n;
  return SHERF_OK;
}

int sherf_depth_range(const SherfRays* rays, float* min_out, float* max_out, void* scratch, size_t scratch_bytes, void* stream) {
  g_err[0] = 0;
  if (!rays || !min_out || !max_out || !scratch) { set_error("null argument"); return SHERF_E_INVALID; }
  if (scratch_bytes < sizeof(FrameConst) + 256) { set_error("scratch arena too small"); return SHERF_E_SCRATCH; }
  char* b = (char*)scratch;
  const size_t mis = ((size_t)b) & 255;
  if (mis) b += 256 - mis;
  FrameConst* fc = (FrameConst*)b;
  cudaStream_t st = (cudaStream_t)stream;
  int init[2] = {0x7fffffff, (int)0x80000000};
  SHERF_CUDA_OK(cudaMemcpyAsync(&fc->dmin_bits, init, sizeof(init), cudaMemcpyHostToDevice, st));
  g_launches.n = 0;
  RC(run_depth_range(*rays, fc, st));
  int bits[2];
  SHERF_CUDA_OK(cudaMemcpyAsync(bits, &fc->dmin_bits, sizeof(bits), cudaMemcpyDeviceToHost, st));
  SHERF_CUDA_OK(cudaStreamSynchronize(st));
  for (int i = 0; i < 2; ++i) {
    int v = bits[i] >= 0 ? bits[i] : bits[i] ^ 0x7fffffff;
    float f; memcpy(&f, &v, 4);
    (i == 0 ? *min_out : *max_out) = f;
  }
  g_last_launches = g_launches.n;
  return SHERF_OK;
}

}  // extern "C"
