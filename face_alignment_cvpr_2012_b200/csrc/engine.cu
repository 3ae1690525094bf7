// Per-GPU context, work buffers and the C ABI (include/crf_b200.h) of the CRF inference path.
// Orchestrates what FaceForest::analyzeFace does for one face (reference src/FaceForest.cpp:183-258),
// for whole batches of faces at a time.  There is no CPU fallback: every stage is a CUDA kernel.
#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <sstream>
#include <string>
#include <thread>
#include <unordered_map>
#include <vector>

#include "kernels.cuh"
#include "model.h"

struct crf_model { crf::Model m; };

namespace crf {

thread_local std::string g_last_error;
static int fail(int code, const std::string& msg) { g_last_error = msg; return code; }

#define CU(call)                                                                                          \
  do {                                                                                                    \
    cudaError_t e_ = (call);                                                                              \
    if (e_ != cudaSuccess) return fail(CRF_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_)); \
  } while (0)

struct Buf {
  void* p = nullptr;
  size_t bytes = 0;
  int reserve(size_t need) {
    if (need <= bytes) return CRF_OK;
    if (p) cudaFree(p);
    p = nullptr; bytes = 0;
    size_t want = need + need / 8;
    cudaError_t e = cudaMalloc(&p, want);
    if (e != cudaSuccess) { e = cudaMalloc(&p, need); want = need; }
    if (e != cudaSuccess) { p = nullptr; return fail(CRF_ERR_CUDA, std::string("cudaMalloc: ") + cudaGetErrorString(e)); }
    bytes = want;
    return CRF_OK;
  }
  void release() { if (p) cudaFree(p); p = nullptr; bytes = 0; }
  template <class T> T* as() const { return reinterpret_cast<T*>(p); }
};

static int patches_1d(int len, int stride) { return len > kPatch ? (len - kPatch + stride - 1) / stride : 0; }

// createKernel / initGaborKernels (include/FeatureChannelFactory.hpp:186-251; SURVEY A.4), built in f64 with libm.
static void build_gabor_bank(std::vector<float2> coef[5], int widths[5]) {
  const double sigma = 1.0 / 2.0 * M_PI, dF = std::sqrt(2.0);
  for (int nu = 0; nu <= 4; nu++) {
    const double k = (M_PI / 2) / std::pow(dF, (double)nu);
    double width = std::round((sigma / k) * 6 + 1);
    if (std::fmod(width, 2.0) == 0.0) width++;
    const int w = (int)width, off = (int)((width - 1) / 2);
    widths[nu] = w;
    coef[nu].assign((size_t)7 * w * w, make_float2(0.f, 0.f));
    for (int mu = 0; mu < 7; mu++) {
      const double phi = M_PI * mu / 8;
      for (int i = 0; i < w; i++)
        for (int j = 0; j < w; j++) {
          const int x = i - off, y = j - off;
          const double t1 = (std::pow(k, 2) / std::pow(sigma, 2)) *
                            std::exp(-(std::pow((double)x, 2) + std::pow((double)y, 2)) * std::pow(k, 2) / (2 * std::pow(sigma, 2)));
          const double t2 = std::cos(k * std::cos(phi) * x + k * std::sin(phi) * y) - std::exp(-(std::pow(sigma, 2) / 2));
          const double t3 = std::sin(k * std::cos(phi) * x + k * std::sin(phi) * y);
          coef[nu][(size_t)mu * w * w + (size_t)j * w + i] = make_float2((float)(t1 * t2), (float)(t1 * t3));
        }
    }
  }
}

// Separable factors of one scale for k_gabor_sep: float2 hx[7][K], float2 hy[7][K], float g1[K], float dc
// (same expressions, in double, as the oracle's create_gabor_kernel).
static void build_gabor_sep(int nu, int w, std::vector<float>& out) {
  const double sigma = 1.0 / 2.0 * M_PI, dF = std::sqrt(2.0);
  const double k = (M_PI / 2) / std::pow(dF, (double)nu);
  const int off = (w - 1) / 2;
  out.assign((size_t)7 * w * 4 + w + 1, 0.f);
  for (int mu = 0; mu < 7; mu++) {
    const double phi = M_PI * mu / 8;
    const double ax = k * std::cos(phi), ay = k * std::sin(phi);
    for (int i = 0; i < w; i++) {
      const double x = (double)(i - off);
      const double env = std::sqrt(k * k / (sigma * sigma)) * std::exp(-(x * x) * k * k / (2 * sigma * sigma));
      out[((size_t)mu * w + i) * 2 + 0] = (float)(env * std::cos(ax * x));
      out[((size_t)mu * w + i) * 2 + 1] = (float)(env * std::sin(ax * x));
      out[(size_t)7 * w * 2 + ((size_t)mu * w + i) * 2 + 0] = (float)(env * std::cos(ay * x));
      out[(size_t)7 * w * 2 + ((size_t)mu * w + i) * 2 + 1] = (float)(env * std::sin(ay * x));
      out[(size_t)7 * w * 4 + i] = (float)env;
    }
  }
  out[(size_t)7 * w * 4 + w] = (float)std::exp(-(sigma * sigma) / 2);
}

struct StageTimer {
  bool on = false;
  std::vector<cudaEvent_t> pool;
  struct Span { int stage; cudaEvent_t a, b; };
  std::vector<Span> spans;
  size_t next = 0;
  float ms[CRF_NUM_STAGES] = {0};
  int launches[CRF_NUM_STAGES] = {0};
  cudaEvent_t get() {
    if (next == pool.size()) { cudaEvent_t e; cudaEventCreate(&e); pool.push_back(e); }
    return pool[next++];
  }
  void collect() {
    for (auto& s : spans) { float t = 0; if (cudaEventElapsedTime(&t, s.a, s.b) == cudaSuccess) ms[s.stage] += t; }
    spans.clear(); next = 0;
  }
  void destroy() { for (auto e : pool) cudaEventDestroy(e); pool.clear(); }
};

// Planes of an ImageSample in the order extractFeatureChannels appends them: features sorted by id, FC_GRAY 1 plane,
// FC_GABOR 35, FC_SOBEL 2 (d/dy, d/dx), FC_MIN_MAX 2 (erode, dilate), FC_CANNY 1, FC_NORM 1
// (src/ImageSample.cpp:77-90, include/FeatureChannelFactory.hpp:35-183).
struct ChannelLayout {
  int nplanes = 0;
  int gabor_first = -1;   // first of the 35 Gabor planes, -1 = FC_GABOR not configured
  PlainPlanes pp{};       // the non-Gabor planes: kernel selector + output plane
  int n_plain = 0;
  bool canny = false;
};
static ChannelLayout layout_of(const std::vector<int>& sorted_features) {
  ChannelLayout L;
  auto plain = [&](int which) { L.pp.which[L.n_plain] = which; L.pp.plane[L.n_plain] = L.nplanes++; L.n_plain++; };
  for (int f : sorted_features) {
    switch (f) {
      case 0: plain(0); break;
      case 1: L.gabor_first = L.nplanes; L.nplanes += 35; break;
      case 2: plain(1); plain(2); break;
      case 3: plain(3); plain(4); break;
      case 4: plain(6); L.canny = true; break;
      case 5: plain(5); break;
      default: break;
    }
  }
  return L;
}

}  // namespace crf

using namespace crf;

struct crf_ctx {
  int device = 0;
  cudaStream_t copy_stream = nullptr;
  cudaEvent_t ev_copied[2] = {nullptr, nullptr}, ev_consumed[2] = {nullptr, nullptr};
  uint8_t* h_stage[2] = {nullptr, nullptr};   // pinned staging for ROI-mode uploads
  size_t h_stage_bytes[2] = {0, 0};
  crf_options_t opt{};
  int hp_ntrees = 0, mp_ntrees_cfg = 0, num_channels = 38;
  ChannelLayout layout;   // planes of the model's feature list
  bool full_model = true; // head-pose forest + 5 pose forests: what analyzeFace needs (a partial model serves Forest<S> alone)
  PackedForest hp, mp;  // host copies (object-id maps for the stage API)
  // device model
  Buf d_hp_slotsn, d_mp_slotsn, d_hp_nroot, d_mp_nroot, d_hp_slotsw, d_mp_slotsw, d_hp_slots16, d_mp_slots16, d_hp_slots, d_hp_roots, d_hp_m, d_mp_slots, d_mp_roots, d_mp_mask, d_mp_leaf, d_xs, d_coef[5], d_coef_sep[5];
  int gabor_width[5] = {0, 0, 0, 0, 0};
  ComposeTables ct{};
  // work buffers: two complete sets, so that consecutive chunks run on two streams and kernels bound by different
  // units (fp32 issue for the Gabor bank, L1/L2 gathers for the forests, latency for the sequential folds) overlap
  struct WorkSet {
    cudaStream_t stream = nullptr;
    Buf d_gabor_scratch, d_gabor_counters;
    Buf d_scaled, d_stacks, d_mag, d_minmax, d_hp_leaf, d_ffd_leaf, d_face_roots, d_face_ntrees, d_votes, d_vote_counts, d_vote_base, d_seg_counts, d_u8planes, d_int32;
    size_t scaled_fs = 0, stack_fs = 0, plane_stride = 0, mag_fs = 0, mag_ps = 0, hp_leaf_fs = 0, ffd_leaf_fs = 0, vote_cap = 0, u8_fs = 0;
    Buf* all[16] = {&d_gabor_scratch, &d_gabor_counters, &d_scaled, &d_stacks, &d_mag, &d_minmax, &d_hp_leaf, &d_ffd_leaf, &d_face_roots, &d_face_ntrees, &d_votes, &d_vote_counts, &d_vote_base,
                    &d_seg_counts, &d_u8planes, &d_int32};
  };
  WorkSet ws[2];
  WorkSet* w = &ws[0];   // set of the chunk being enqueued
  Buf d_imgs[2], d_fd, d_faces, d_counters, d_misc;
  crf_counters_t cnt{};
  bool counting = false;
  int traverse_variant = 0;  // 0 = pick by stride (see launch_traverse)
  int sm_count = 148;
  int win_hp = 0, win_ffd = 0;   // k_traverse_win variants (0 = default)
  bool win_smem_ok = true;       // the device grants a CTA the 231 040 bytes of dynamic shared memory the window needs
  int win_tex = 1;               // node records of k_traverse_win through the texture pipe (CRF_WIN_TEX=0: 256-bit global loads)
  cudaTextureObject_t tex_hp = 0, tex_mp = 0, tex_hp_wide = 0, tex_mp_wide = 0, tex_hp_n = 0, tex_mp_n = 0;
  int win_fmt = 2;               // 2 = k_traverse_win2 on the internal-nodes-only records (default), 1 = k_traverse_win (CRF_WIN_FMT)
  // 1 = consecutive chunks run back to back on one stream (default: measured faster — co-resident Gabor CTAs shrink the L1
  // the gathers live on, and two chunks' stacks thrash L2); 2 = alternate chunks between two streams / work sets
  int nstreams = 1;
  // CRF_GABOR_FUSED=1: the fused per-scale Gabor kernels (k_gabor_fused: rolling row pass, magnitudes in an L2-resident scratch, quantisation in
  // the same kernel).  Bit-identical and MEASURED SLOWER on B200 (30.4 vs 22.3 ms per 4096 faces: the serial phases of a CTA that owns a whole
  // plane cost more than the 27 % of multiply-adds and the 18 GB of DRAM traffic it saves), so the banded kernels stay the default.
  int gabor_fused = 0;
  int gabor_band = 32;       // rows per CTA of k_gabor_sep (CRF_GABOR_BAND = 16 | 32): 32 repeats fewer halo rows in the row pass, 21.7 -> 20.1 ms per 4096 faces
  int gabor_quant_old = 0;   // CRF_GABOR_QUANT_OLD=1: k_gabor_quant_integral (one column per thread) instead of k_gabor_quant_band
  int ms_mode = CRF_MS_FAST;   // resolved from crf_options_t::ms_mode / CRF_MS_MODE at creation
  int ms_variant = 3;   // resident MeanShift CTAs per SM the kernel is compiled for (register cap); CRF_MS_VARIANT overrides
  size_t work_budget = (size_t)64 << 30;  // bytes of work buffers a launch may use (min(64 GB, half of the free memory at creation))
  StageTimer timer;
  // face-box source (haar.cuh): device image of the last cascade used + the buffers of a group of frames
  unsigned long long haar_cached = 0;   // crf_cascade::id of the cascade in d_haar_stages / weak / feats / nodes / leaves / tilt (0 = none)
  // d_haar_weak: HaarWeak of a stump cascade or HaarTree of a tree cascade; d_haar_T: tilted integrals, for cascades with tilted features
  Buf d_haar_stages, d_haar_weak, d_haar_feats, d_haar_nodes, d_haar_leaves, d_haar_tilt, d_haar_T, d_haar_frames, d_haar_S, d_haar_Q, d_haar_flags, d_haar_list[2], d_haar_rows, d_haar_levels, d_haar_counts, d_haar_cand;
  // first stage of each cascade stage group after the first (CRF_HAAR_SPLIT="a,b,..."; measured, DESIGN §4.5)
  std::vector<int> haar_split{3, 8};
};

namespace crf {

struct Span {
  crf_ctx* c; int stage; cudaEvent_t a = nullptr;
  Span(crf_ctx* ctx, int st) : c(ctx), stage(st) {
    if (c->timer.on) { a = c->timer.get(); cudaEventRecord(a, c->w->stream); }
  }
  ~Span() {
    if (c->timer.on) { cudaEvent_t b = c->timer.get(); cudaEventRecord(b, c->w->stream); c->timer.spans.push_back({stage, a, b}); }
  }
};
static inline void count_launch(crf_ctx* c, int stage, int n = 1) { c->cnt.kernel_launches += n; c->timer.launches[stage] += n; }

#define KCHECK()                                                                                              \
  do {                                                                                                        \
    cudaError_t e_ = cudaGetLastError();                                                                      \
    if (e_ != cudaSuccess) return fail(CRF_ERR_CUDA, std::string("kernel launch: ") + cudaGetErrorString(e_)); \
  } while (0)

template <class T>
static int upload(Buf& b, const std::vector<T>& v, cudaStream_t s) {
  int rc = b.reserve(std::max<size_t>(v.size() * sizeof(T), 16));
  if (rc) return rc;
  if (!v.empty()) CU(cudaMemcpyAsync(b.p, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice, s));
  return CRF_OK;
}

// Geometry + buffer sizing for a launch over `n` faces whose tallest scaled face is Hmax.
struct Plan {
  int n = 0, Hmax = 0, nplanes = 38;
  int hp_stride = 4, ffd_stride = 3;
  int tree_cap = 20;
  int vote_factor = 3;   // vote capacity per leaf in the batched path (kParts = worst case)
  bool need_gabor = true, want_u8 = false, need_hp = true, need_ffd = true;
};

static int ensure(crf_ctx* c, const Plan& p) {
  const size_t n = (size_t)std::max(p.n, 1);
  const int H = p.Hmax;
  c->w->scaled_fs = (size_t)H * 128;
  c->w->plane_stride = (size_t)(H + 1) * kRowStride;
  c->w->stack_fs = c->w->plane_stride * p.nplanes;
  c->w->mag_ps = (size_t)H * 128;
  c->w->mag_fs = c->w->mag_ps * 35;
  const size_t np_hp = (size_t)patches_1d(125, p.hp_stride) * patches_1d(H, p.hp_stride);
  const size_t np_ffd = (size_t)patches_1d(125, p.ffd_stride) * patches_1d(H, p.ffd_stride);
  c->w->hp_leaf_fs = np_hp * std::max(c->hp_ntrees, 1);
  c->w->ffd_leaf_fs = np_ffd * p.tree_cap;
  // votes per face: worst case is kParts per leaf; the batched path budgets vote_factor per leaf and re-runs the rare
  // face that exceeds it with the worst-case capacity
  c->w->vote_cap = std::max<size_t>(c->w->ffd_leaf_fs * (size_t)std::min(p.vote_factor, kParts), 16);
  c->w->u8_fs = (size_t)p.nplanes * 125 * H;
  int rc;
  if ((rc = c->w->d_scaled.reserve(n * c->w->scaled_fs))) return rc;
  if ((rc = c->w->d_stacks.reserve(n * c->w->stack_fs * sizeof(stack_t)))) return rc;
  if (p.want_u8 && (rc = c->w->d_int32.reserve(n * c->w->stack_fs * 4))) return rc;
  if (p.need_gabor && !c->gabor_fused) {   // the fused kernels keep their magnitudes in a per-CTA scratch (launch_channels)
    if ((rc = c->w->d_mag.reserve(n * c->w->mag_fs * 4))) return rc;
    if ((rc = c->w->d_minmax.reserve(n * 35 * 2 * 4))) return rc;
  }
  if (p.need_hp && (rc = c->w->d_hp_leaf.reserve(std::max<size_t>(n * c->w->hp_leaf_fs * 4, 16)))) return rc;
  if ((rc = c->w->d_face_roots.reserve(n * kMaxList * 4))) return rc;
  if ((rc = c->w->d_face_ntrees.reserve(n * 4))) return rc;
  if (p.need_ffd) {
    if ((rc = c->w->d_ffd_leaf.reserve(std::max<size_t>(n * c->w->ffd_leaf_fs * 4, 16)))) return rc;
    if ((rc = c->w->d_votes.reserve(n * c->w->vote_cap * sizeof(DevVote)))) return rc;
    if ((rc = c->w->d_vote_counts.reserve(n * kParts * 4))) return rc;
    if ((rc = c->w->d_vote_base.reserve(n * kParts * 4))) return rc;
    if ((rc = c->w->d_seg_counts.reserve(n * kVoteSegs * kParts * 4))) return rc;
  }
  if (p.want_u8 && (rc = c->w->d_u8planes.reserve(n * c->w->u8_fs))) return rc;
  return CRF_OK;
}

// Host-side row packing of face boxes into pinned staging, split over a few threads (memcpy-bound).
template <class F>
static void parallel_for(int n, size_t bytes, F&& fn) {
  const unsigned hw = std::max(1u, std::thread::hardware_concurrency());
  const int nt = (int)std::min<size_t>(std::min<unsigned>(hw, 8u), std::max<size_t>(1, bytes >> 21));   // one thread per ~2 MB, at most 8
  if (nt <= 1 || n < 2) { for (int i = 0; i < n; i++) fn(i); return; }
  std::vector<std::thread> th;
  for (int t = 0; t < nt; t++)
    th.emplace_back([&, t] { for (int i = (int)((long long)n * t / nt), e = (int)((long long)n * (t + 1) / nt); i < e; i++) fn(i); });
  for (auto& x : th) x.join();
}

static bool is_pinned_host(const void* p) {
  cudaPointerAttributes a{};
  if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return false; }
  return a.type == cudaMemoryTypeHost;
}

// The box checks of the analysis path: nullptr if the box can be analysed, else the reason.
static const char* box_error(int rows, int cols, const crf_rect_t& b) {
  if (b.x < 0 || b.y < 0 || b.width <= 0 || b.height <= 0 || (long long)b.x + b.width > cols || (long long)b.y + b.height > rows) return "bbox outside image";
  const float scale = static_cast<float>(125) / static_cast<float>(b.width);
  const int sw = (int)(b.width * scale), sh = (int)(b.height * scale);
  if (sw <= kPatch || sh <= kPatch) return "scaled face smaller than a patch";
  if (sw > 125) return "scaled face wider than face_size";
  if (sh > CRF_MAX_SCALED_H) return "scaled face taller than CRF_MAX_SCALED_H (f32 integral exactness limit)";
  return nullptr;
}

// src/FaceForest.cpp:199-204 (scale, scaled size) + the argument checks of the path.
static int make_desc(const crf_ctx* c, int rows, int cols, size_t step, size_t img_off, const crf_rect_t& b, FaceDesc& d) {
  if (const char* e = box_error(rows, cols, b)) return fail(CRF_ERR_ARG, e);
  const float scale = static_cast<float>(125) / static_cast<float>(b.width);
  const int sw = (int)(b.width * scale), sh = (int)(b.height * scale);
  d.img_off = img_off; d.img_step = step;
  d.bx = b.x; d.by = b.y; d.bw = b.width; d.bh = b.height;
  d.W = sw; d.H = sh; d.scale = scale; d.pad = 0;
  d.scale_x = 1. / ((double)sw / b.width);
  d.scale_y = 1. / ((double)sh / b.height);
  (void)c;
  return CRF_OK;
}

// ---- stage launchers (all on c->w->stream; fd/faces point at the first face of the launch) ----------
static int launch_resize(crf_ctx* c, const FaceDesc* fd, int n, int Hmax, const uint8_t* d_imgs) {
  Span s(c, CRF_STAGE_RESIZE);
  k_gray_resize<<<dim3(Hmax, n), 128, 0, c->w->stream>>>(fd, d_imgs, c->w->d_scaled.as<uint8_t>(), c->w->scaled_fs);
  KCHECK(); count_launch(c, CRF_STAGE_RESIZE);
  return CRF_OK;
}

static int launch_channels(crf_ctx* c, const FaceDesc* fd, int n, int Hmax, const ChannelLayout& L, bool want_u8) {
  uint8_t* u8 = want_u8 ? c->w->d_u8planes.as<uint8_t>() : nullptr;
  uint32_t* dbg32 = want_u8 ? c->w->d_int32.as<uint32_t>() : nullptr;   // full 32-bit integrals, stage API only
  if (L.n_plain > 0) {
    Span s(c, CRF_STAGE_PLAIN);
    const size_t smem = L.canny ? (size_t)(Hmax + 2) * 127 * 3 : 0;   // FC_CANNY: u16 magnitudes + u8 map of the padded face
    k_plain_channels<<<dim3(L.n_plain, n), 128, smem, c->w->stream>>>(fd, c->w->d_scaled.as<uint8_t>(), c->w->scaled_fs, c->w->d_stacks.as<stack_t>(), c->w->stack_fs,
                                                                 c->w->plane_stride, u8, c->w->u8_fs, dbg32, L.pp);
    KCHECK(); count_launch(c, CRF_STAGE_PLAIN);
  }
  if (L.gabor_first < 0) return CRF_OK;
  Span s(c, CRF_STAGE_GABOR);
  const uint8_t* sc = c->w->d_scaled.as<uint8_t>();
  if (c->gabor_fused) {
    // one persistent launch per scale: (face) items from a counter, magnitudes through a per-CTA scratch slot that stays in L2
    const int grid = std::min(n, c->sm_count * 3);
    const size_t plane = (size_t)Hmax * 128;
    int rc;
    if ((rc = c->w->d_gabor_scratch.reserve((size_t)c->sm_count * 3 * 2 * plane * 4)) || (rc = c->w->d_gabor_counters.reserve(8 * 4))) return rc;
    CU(cudaMemsetAsync(c->w->d_gabor_counters.p, 0, 8 * 4, c->w->stream));
    GaborFusedArgs g{};
    g.fd = fd; g.nfaces = n; g.scaled = sc; g.scaled_face_stride = c->w->scaled_fs;
    g.scratch = c->w->d_gabor_scratch.as<float>(); g.scratch_plane_stride = plane;
    g.stacks = c->w->d_stacks.as<stack_t>(); g.stack_face_stride = c->w->stack_fs; g.plane_stride = c->w->plane_stride; g.first_plane = L.gabor_first;
    g.u8planes = u8; g.u8_face_stride = c->w->u8_fs; g.dbg32 = dbg32;
    int* cnt = c->w->d_gabor_counters.as<int>();
    g.counter = cnt + 4; k_gabor_fused<25><<<grid, 256, GaborSepSmem<25>::bytes, c->w->stream>>>(g, c->d_coef_sep[4].as<float>(), 4); KCHECK();
    g.counter = cnt + 3; k_gabor_fused<19><<<grid, 256, GaborSepSmem<19>::bytes, c->w->stream>>>(g, c->d_coef_sep[3].as<float>(), 3); KCHECK();
    g.counter = cnt + 2; k_gabor_fused<13><<<grid, 256, GaborSepSmem<13>::bytes, c->w->stream>>>(g, c->d_coef_sep[2].as<float>(), 2); KCHECK();
    g.counter = cnt + 1; k_gabor_fused<9><<<grid, 256, GaborSepSmem<9>::bytes, c->w->stream>>>(g, c->d_coef_sep[1].as<float>(), 1); KCHECK();
    g.counter = cnt + 0; k_gabor_fused7<<<std::min(n, c->sm_count * 2), 256, 0, c->w->stream>>>(g, c->d_coef[0].as<float2>()); KCHECK();
    count_launch(c, CRF_STAGE_GABOR, 5);
    return CRF_OK;
  }
  k_init_minmax<<<(n * 70 + 255) / 256, 256, 0, c->w->stream>>>(c->w->d_minmax.as<uint32_t>(), n * 70);
  KCHECK();
  const dim3 grid((Hmax + 15) / 16, 2LL * n * ((Hmax + 15) / 16) <= c->sm_count ? 7 : 1, n);   // k_gabor_mag<7>: orientations in the CTA, or one CTA each for small batches
  float* mag = c->w->d_mag.as<float>();
  uint32_t* mm = c->w->d_minmax.as<uint32_t>();
  // small batches (single faces, one video frame): one CTA per (band, face, orientation) instead of a loop over the orientations
  // 9x9 .. 25x25 in separable form (heaviest first), 7x7 as the direct raster sum that equals cv2 bit for bit
  if (c->gabor_band == 32) {
    const int nb = (Hmax + 31) / 32;
    const dim3 g32(nb, n, 2LL * n * nb <= c->sm_count ? 7 : 1);
    k_gabor_sep<25, 32><<<g32, 512, GaborSepSmem<25, 32>::bytes, c->w->stream>>>(fd, sc, c->w->scaled_fs, c->d_coef_sep[4].as<float>(), 4, mag, c->w->mag_fs, c->w->mag_ps, mm); KCHECK();
    k_gabor_sep<19, 32><<<g32, 512, GaborSepSmem<19, 32>::bytes, c->w->stream>>>(fd, sc, c->w->scaled_fs, c->d_coef_sep[3].as<float>(), 3, mag, c->w->mag_fs, c->w->mag_ps, mm); KCHECK();
    k_gabor_sep<13, 32><<<g32, 512, GaborSepSmem<13, 32>::bytes, c->w->stream>>>(fd, sc, c->w->scaled_fs, c->d_coef_sep[2].as<float>(), 2, mag, c->w->mag_fs, c->w->mag_ps, mm); KCHECK();
    k_gabor_sep<9, 32><<<g32, 512, GaborSepSmem<9, 32>::bytes, c->w->stream>>>(fd, sc, c->w->scaled_fs, c->d_coef_sep[1].as<float>(), 1, mag, c->w->mag_fs, c->w->mag_ps, mm); KCHECK();
  } else {
    const dim3 gsym((Hmax + 15) / 16, n, 2LL * n * ((Hmax + 15) / 16) <= c->sm_count ? 7 : 1);
    k_gabor_sep<25><<<gsym, 256, GaborSepSmem<25>::bytes, c->w->stream>>>(fd, sc, c->w->scaled_fs, c->d_coef_sep[4].as<float>(), 4, mag, c->w->mag_fs, c->w->mag_ps, mm); KCHECK();
    k_gabor_sep<19><<<gsym, 256, GaborSepSmem<19>::bytes, c->w->stream>>>(fd, sc, c->w->scaled_fs, c->d_coef_sep[3].as<float>(), 3, mag, c->w->mag_fs, c->w->mag_ps, mm); KCHECK();
    k_gabor_sep<13><<<gsym, 256, GaborSepSmem<13>::bytes, c->w->stream>>>(fd, sc, c->w->scaled_fs, c->d_coef_sep[2].as<float>(), 2, mag, c->w->mag_fs, c->w->mag_ps, mm); KCHECK();
    k_gabor_sep<9><<<gsym, 256, GaborSepSmem<9>::bytes, c->w->stream>>>(fd, sc, c->w->scaled_fs, c->d_coef_sep[1].as<float>(), 1, mag, c->w->mag_fs, c->w->mag_ps, mm); KCHECK();
  }
  k_gabor_mag<7><<<grid, 256, 0, c->w->stream>>>(fd, sc, c->w->scaled_fs, c->d_coef[0].as<float2>(), 0, mag, c->w->mag_fs, c->w->mag_ps, mm); KCHECK();
  {
    GaborFusedArgs g{};
    g.fd = fd; g.nfaces = n;
    g.stacks = c->w->d_stacks.as<stack_t>(); g.stack_face_stride = c->w->stack_fs; g.plane_stride = c->w->plane_stride; g.first_plane = L.gabor_first;
    g.u8planes = u8; g.u8_face_stride = c->w->u8_fs; g.dbg32 = dbg32;
    if (c->gabor_quant_old)
      k_gabor_quant_integral<<<dim3(35, n), 128, 0, c->w->stream>>>(fd, mag, c->w->mag_fs, c->w->mag_ps, mm, c->w->d_stacks.as<stack_t>(), c->w->stack_fs, c->w->plane_stride, L.gabor_first,
                                                                 u8, c->w->u8_fs, dbg32);
    else
      k_gabor_quant_band<<<dim3(35, n), 256, 0, c->w->stream>>>(g, mag, c->w->mag_fs, c->w->mag_ps, mm);
  }
  KCHECK(); count_launch(c, CRF_STAGE_GABOR, 7);
  return CRF_OK;
}

static int launch_traverse(crf_ctx* c, const FaceDesc* fd, int n, int Hmax, bool hp, int stride, const int32_t* roots, int ntrees, int smem_trees,
                           bool hp_values = false) {
  const int stage = hp ? CRF_STAGE_HP_TRAVERSE : CRF_STAGE_FFD_TRAVERSE;
  Span s(c, stage);
  TraverseArgs a{};
  a.fd = fd; a.stacks = c->w->d_stacks.as<stack_t>(); a.stack_face_stride = c->w->stack_fs; a.plane_stride = c->w->plane_stride;
  a.stride = stride;
  if (hp) {
    a.slots = c->d_hp_slots.as<DevSlot>(); a.slots16 = c->d_hp_slots16.as<DevSlot16>(); a.slotsw = c->d_hp_slotsw.as<DevSlotW>(); a.slotsw_tex = c->tex_hp; a.slots_tex = c->tex_hp_wide; a.roots = roots; a.ntrees = ntrees;
    a.slotsn_tex = c->tex_hp_n; a.nroot_of_slot = c->d_hp_nroot.as<int32_t>();
    a.leaf_out = c->w->d_hp_leaf.as<int32_t>(); a.leaf_face_stride = c->w->hp_leaf_fs;
    a.cnt_tests = CNT_HP_TESTS; a.cnt_trav = CNT_HP_TRAV;
    if (hp_values) a.leaf_value = c->d_hp_m.as<float>();
  } else {
    a.slots = c->d_mp_slots.as<DevSlot>(); a.slots16 = c->d_mp_slots16.as<DevSlot16>(); a.slotsw = c->d_mp_slotsw.as<DevSlotW>(); a.slotsw_tex = c->tex_mp; a.slots_tex = c->tex_mp_wide;
    a.slotsn_tex = c->tex_mp_n; a.nroot_of_slot = c->d_mp_nroot.as<int32_t>();
    a.face_roots = c->w->d_face_roots.as<int32_t>(); a.face_ntrees = c->w->d_face_ntrees.as<int32_t>();
    a.leaf_out = c->w->d_ffd_leaf.as<int32_t>(); a.leaf_face_stride = c->w->ffd_leaf_fs;
    a.cnt_tests = CNT_FFD_TESTS; a.cnt_trav = CNT_FFD_TRAV;
  }
  a.counters = c->counting ? c->d_counters.as<unsigned long long>() : nullptr;
  const int nx = patches_1d(125, stride), ny = patches_1d(Hmax, stride);
  if (nx <= 0 || ny <= 0) return CRF_OK;
  // Dense grids: gather from a shared-memory window instead of L1/L2 (k_traverse_win) when the model's rectangles fit the
  // window and there are enough (face, tile column) items to keep every SM's persistent CTA busy.
  // CRF_TRAVERSE_VARIANT=0x100001 forces it, any other non-zero value selects one of the global-gather variants below.
  {
    const int ncols = (patches_1d(125, 1) + kWinTile - 1) / kWinTile;
    const bool fits = stride == 1 && (hp ? c->hp.max_extent : c->mp.max_extent) <= kWinExtent && c->num_channels <= kWinMaxPlanes && c->win_smem_ok;
    const bool forced = c->traverse_variant == 0x100001;
    if (forced && !fits) return fail(CRF_ERR_ARG, "CRF_TRAVERSE_VARIANT=0x100001 needs stride 1 and rectangles inside the window");
    if (fits && (forced || (c->traverse_variant == 0 && (long long)n * ncols >= 2LL * c->sm_count))) {
      const int nitems = n * ncols, grid = std::min(nitems, c->sm_count);
      // (warps per CTA) | (walks per lane) << 8; CRF_WIN_HP / CRF_WIN_FFD override for experiments
      const bool fmt2 = c->win_fmt == 2 && (hp ? c->tex_hp_n : c->tex_mp_n) != 0;
      // defaults measured on B200 (tools/win2_variants.py): head pose 15 warps x 2 pipelined walks (30 x 1 for k_traverse_win), FFD 20 warps x 2 walks
      const int wv = hp ? (c->win_hp ? c->win_hp : (fmt2 ? (15 | 2 << 8) : (30 | 1 << 8))) : (c->win_ffd ? c->win_ffd : (20 | 2 << 8));
      bool ok = false;
#define CRF_WIN2(NW_, WK_)                                                                                                  \
      if (fmt2 && wv == (NW_ | WK_ << 8)) {                                                                                  \
        auto kf = c->counting ? k_traverse_win2<NW_, WK_, true> : k_traverse_win2<NW_, WK_, false>;                          \
        CU(cudaFuncSetAttribute(kf, cudaFuncAttributeMaxDynamicSharedMemorySize, kWinSmemBytes));                            \
        kf<<<grid, NW_ * 32, kWinSmemBytes, c->w->stream>>>(a, nitems, ncols, c->num_channels);                              \
        ok = true;                                                                                                           \
      }
      CRF_WIN2(15, 2) CRF_WIN2(20, 2) CRF_WIN2(24, 2) CRF_WIN2(30, 1) CRF_WIN2(32, 1) CRF_WIN2(20, 1)
#undef CRF_WIN2
      if (ok) { KCHECK(); count_launch(c, stage); return CRF_OK; }
#define CRF_WIN(NW_, WK_)                                                                                                   \
      if (wv == (NW_ | WK_ << 8)) {                                                                                          \
        auto kf = c->counting ? k_traverse_win<NW_, WK_, true> : c->win_tex ? k_traverse_win<NW_, WK_, false, true> : k_traverse_win<NW_, WK_, false>; \
        CU(cudaFuncSetAttribute(kf, cudaFuncAttributeMaxDynamicSharedMemorySize, kWinSmemBytes));                            \
        kf<<<grid, NW_ * 32, kWinSmemBytes, c->w->stream>>>(a, nitems, ncols, c->num_channels);                              \
        ok = true;                                                                                                           \
      }
#define CRF_WINP(NW_)                                                                                                       \
      if (wv == (NW_ | 2 << 8 | 1 << 12)) {   /* two walks per lane on horizontal neighbours, shared record fetch */        \
        auto kf = c->counting ? k_traverse_win<NW_, 2, true, false, true> : c->win_tex ? k_traverse_win<NW_, 2, false, true, true> : k_traverse_win<NW_, 2, false, false, true>; \
        CU(cudaFuncSetAttribute(kf, cudaFuncAttributeMaxDynamicSharedMemorySize, kWinSmemBytes));                            \
        kf<<<grid, NW_ * 32, kWinSmemBytes, c->w->stream>>>(a, nitems, ncols, c->num_channels);                              \
        ok = true;                                                                                                           \
      }
      CRF_WIN(15, 2) CRF_WIN(20, 2) CRF_WIN(10, 2) CRF_WIN(30, 1) CRF_WIN(32, 1) CRF_WIN(20, 1) CRF_WIN(24, 1) CRF_WIN(28, 1) CRF_WIN(16, 1)
      CRF_WINP(15) CRF_WINP(20) CRF_WINP(10) CRF_WINP(16) CRF_WINP(24)
#undef CRF_WINP
#undef CRF_WIN
      if (!ok) return fail(CRF_ERR_ARG, "unknown CRF_WIN_HP / CRF_WIN_FFD variant");
      KCHECK(); count_launch(c, stage);
      return CRF_OK;
    }
  }
  const size_t smem = (size_t)32 * smem_trees * 4;
  // variant = LW (32 or 8) | MODE << 8 | NW (5 or 10) << 16; CRF_TRAVERSE_VARIANT overrides for experiments
  // defaults from tools/traverse_variants.py on B200: one warp per tree for the 15-tree head-pose forest, 10 warps for 20 trees;
  // rows of 32 x-adjacent patches and the compact 16-byte slots at dense strides; 16 x 2 blocks and 256-bit loads of the wide
  // slots at sparse ones
  const int variant = c->traverse_variant ? c->traverse_variant
                                           : (stride >= 3 ? (16 | (2 << 8) | (15 << 16)) : (32 | (4 << 8) | ((hp ? 15 : 10) << 16)));
  const int LW = variant & 0xff, MODE = (variant >> 8) & 0xff, NW = (variant >> 16) & 0xff;
  const int tiles = ((nx + LW - 1) / LW) * ((ny + 32 / LW - 1) / (32 / LW));
  const dim3 grid(tiles, n);
#define CRF_TRAV(NW_, LW_, MODE_)                                                                          \
  if (NW == NW_ && LW == LW_ && MODE == MODE_) {                                                           \
    if (c->counting) k_traverse<NW_, true, LW_, MODE_><<<grid, NW_ * 32, smem, c->w->stream>>>(a);            \
    else k_traverse<NW_, false, LW_, MODE_><<<grid, NW_ * 32, smem, c->w->stream>>>(a);                       \
    launched = true;                                                                                       \
  }
  bool launched = false;
  if (MODE == 4 && LW == 32) {   // compact 16-byte slots
    const dim3 g16(((nx + 31) / 32) * ny, n);
    if (NW == 10) { if (c->counting) k_traverse16<10, true><<<g16, 320, smem, c->w->stream>>>(a); else k_traverse16<10, false><<<g16, 320, smem, c->w->stream>>>(a); launched = true; }
    if (NW == 15) { if (c->counting) k_traverse16<15, true><<<g16, 480, smem, c->w->stream>>>(a); else k_traverse16<15, false><<<g16, 480, smem, c->w->stream>>>(a); launched = true; }
    if (NW == 20) { if (c->counting) k_traverse16<20, true><<<g16, 640, smem, c->w->stream>>>(a); else k_traverse16<20, false><<<g16, 640, smem, c->w->stream>>>(a); launched = true; }
    if (NW == 7) { if (c->counting) k_traverse16<7, true><<<g16, 224, smem, c->w->stream>>>(a); else k_traverse16<7, false><<<g16, 224, smem, c->w->stream>>>(a); launched = true; }
  }
  CRF_TRAV(5, 32, 0) CRF_TRAV(5, 32, 1) CRF_TRAV(5, 32, 2) CRF_TRAV(5, 32, 3)
  CRF_TRAV(5, 8, 0) CRF_TRAV(5, 8, 1) CRF_TRAV(5, 8, 2) CRF_TRAV(5, 8, 3)
  CRF_TRAV(10, 32, 0) CRF_TRAV(10, 32, 2) CRF_TRAV(10, 8, 2) CRF_TRAV(10, 8, 3)
  CRF_TRAV(15, 32, 2) CRF_TRAV(20, 32, 2) CRF_TRAV(4, 32, 2) CRF_TRAV(8, 32, 2) CRF_TRAV(10, 16, 2) CRF_TRAV(15, 16, 2)
  CRF_TRAV(15, 16, 10) CRF_TRAV(10, 16, 10) CRF_TRAV(20, 16, 10) CRF_TRAV(15, 32, 10)
#undef CRF_TRAV
  if (!launched) return fail(CRF_ERR_ARG, "unknown CRF_TRAVERSE_VARIANT");
  KCHECK(); count_launch(c, stage);
  return CRF_OK;
}

static int launch_hp_reduce(crf_ctx* c, const FaceDesc* fd, int n, int stride, bool compose, int list_cap, crf_face_t* faces) {
  Span s(c, CRF_STAGE_HP_REDUCE);
  ComposeTables ct = c->ct;
  ct.list_cap = list_cap;
  k_hp_reduce_compose<<<(n + kFoldChains - 1) / kFoldChains, kFoldThreads, kHpSmem, c->w->stream>>>(fd, n, c->w->d_hp_leaf.as<float>(), c->w->hp_leaf_fs, c->hp_ntrees, stride, ct,
                                                          compose ? 1 : 0, faces, c->w->d_face_roots.as<int32_t>(), c->w->d_face_ntrees.as<int32_t>());
  KCHECK(); count_launch(c, CRF_STAGE_HP_REDUCE);
  return CRF_OK;
}

static int launch_meanshift(crf_ctx* c, const FaceDesc* fd, int nchains, crf_face_t* faces) {
  Span s(c, CRF_STAGE_MEANSHIFT);
  MeanShiftOpt mo{c->opt.ms_kernel_size, c->opt.ms_max_iterations, c->opt.ms_stopping_criteria};
  // 32 chains share a fold warp when there are enough chains to fill the GPU; small batches spread over more CTAs
  const int cpc = nchains >= 8192 ? 32 : std::max(1, std::min(8, nchains / 296));   // small batches: up to two CTAs per SM before chains share one
  const dim3 grid((nchains + cpc - 1) / cpc);
  unsigned long long* cnt = c->counting ? c->d_counters.as<unsigned long long>() : nullptr;
  if (c->ms_mode == CRF_MS_FAST) {
    // one CTA per chain; wide CTAs when the grids are dense (a stride-1 chain holds ~18 k votes, a default-stride one ~2 k)
    const bool dense = c->w->ffd_leaf_fs >= 65536 || c->w->vote_cap >= 65536;
    if (dense) k_meanshift_fast<512><<<nchains, 512, 0, c->w->stream>>>(fd, nchains, c->w->d_votes.as<DevVote>(), c->w->vote_cap, c->w->d_vote_counts.as<int32_t>(),
                                                                       c->w->d_vote_base.as<int32_t>(), mo, faces, cnt);
    else k_meanshift_fast<128><<<nchains, 128, 0, c->w->stream>>>(fd, nchains, c->w->d_votes.as<DevVote>(), c->w->vote_cap, c->w->d_vote_counts.as<int32_t>(),
                                                                 c->w->d_vote_base.as<int32_t>(), mo, faces, cnt);
    KCHECK(); count_launch(c, CRF_STAGE_MEANSHIFT);
    return CRF_OK;
  }
#define CRF_MS(MINB)                                                                                                                                    \
  k_meanshift<MINB, false><<<grid, kFoldThreads, MsGeom<false>::smem, c->w->stream>>>(fd, nchains, c->w->d_votes.as<DevVote>(), c->w->vote_cap, c->w->d_vote_counts.as<int32_t>(), \
                                                                  c->w->d_vote_base.as<int32_t>(), cpc, mo, faces, cnt)
  if (cpc < 32)
    k_meanshift<3, true><<<grid, kFoldThreads, MsGeom<true>::smem, c->w->stream>>>(fd, nchains, c->w->d_votes.as<DevVote>(), c->w->vote_cap, c->w->d_vote_counts.as<int32_t>(),
                                                                     c->w->d_vote_base.as<int32_t>(), cpc, mo, faces, cnt);
  else if (c->ms_variant == 2) CRF_MS(2); else if (c->ms_variant == 4) CRF_MS(4); else CRF_MS(3);
#undef CRF_MS
  KCHECK(); count_launch(c, CRF_STAGE_MEANSHIFT);
  return CRF_OK;
}

static int launch_votes_meanshift(crf_ctx* c, const FaceDesc* fd, int n, int stride, crf_face_t* faces) {
  {
    Span s(c, CRF_STAGE_VOTES);
    VoteArgs a{};
    a.fd = fd; a.leaf_ids = c->w->d_ffd_leaf.as<int32_t>(); a.leaf_face_stride = c->w->ffd_leaf_fs; a.face_ntrees = c->w->d_face_ntrees.as<int32_t>(); a.stride = stride;
    a.mp_mask = c->d_mp_mask.as<uint16_t>(); a.mp_leaf = c->d_mp_leaf.as<DevMpLeaf>(); a.votes = c->w->d_votes.as<DevVote>(); a.vote_cap = c->w->vote_cap;
    a.seg_counts = c->w->d_seg_counts.as<int32_t>(); a.vote_counts = c->w->d_vote_counts.as<int32_t>(); a.vote_base = c->w->d_vote_base.as<int32_t>(); a.faces = faces;
    CU(cudaMemsetAsync(a.vote_counts, 0, (size_t)n * kParts * 4, c->w->stream));
    k_votes_count<<<dim3(kVoteSegs / 8, n), 256, 0, c->w->stream>>>(a);
    KCHECK();
    k_votes_offsets<<<(n + 127) / 128, 128, 0, c->w->stream>>>(a, n);
    KCHECK();
    k_votes_emit<<<dim3(kVoteSegs / 8, n), 256, 0, c->w->stream>>>(a);
    KCHECK(); count_launch(c, CRF_STAGE_VOTES, 3);
  }
  return launch_meanshift(c, fd, n * kParts, faces);
}

// The whole path for faces [0, n) of a launch: fd, faces are device pointers to the first of them.
static int run_faces(crf_ctx* c, const FaceDesc* d_fd, int n, int Hmax, const uint8_t* d_imgs, crf_face_t* d_faces, bool headpose_only, int tree_cap,
                     cudaEvent_t imgs_consumed) {
  int rc;
  if ((rc = launch_resize(c, d_fd, n, Hmax, d_imgs))) return rc;
  if (imgs_consumed) CU(cudaEventRecord(imgs_consumed, c->w->stream));
  if ((rc = launch_channels(c, d_fd, n, Hmax, c->layout, false))) return rc;
  if ((rc = launch_traverse(c, d_fd, n, Hmax, true, c->opt.hp_stride, c->d_hp_roots.as<int32_t>(), c->hp_ntrees, c->hp_ntrees, true))) return rc;
  if ((rc = launch_hp_reduce(c, d_fd, n, c->opt.hp_stride, !headpose_only, tree_cap, d_faces))) return rc;
  if (headpose_only) return CRF_OK;
  if ((rc = launch_traverse(c, d_fd, n, Hmax, false, c->opt.ffd_stride, nullptr, 0, tree_cap))) return rc;
  if ((rc = launch_votes_meanshift(c, d_fd, n, c->opt.ffd_stride, d_faces))) return rc;
  return CRF_OK;
}

// Faces resident per launch: as many as fit a work-buffer budget (the ordered vote lists are sized for the worst
// case of every leaf voting for every part), at most 4096 unless the caller asks otherwise.  Latency-bound tails
// (sequential folds) want many faces in flight; nothing else depends on the choice (results are chunk-invariant).
static int pick_chunk(const crf_ctx* c, int Hmax, bool headpose_only) {
  const size_t np_hp = (size_t)patches_1d(125, c->opt.hp_stride) * patches_1d(Hmax, c->opt.hp_stride);
  const size_t np_ffd = headpose_only ? 0 : (size_t)patches_1d(125, c->opt.ffd_stride) * patches_1d(Hmax, c->opt.ffd_stride);
  // the same terms ensure() reserves per face
  const size_t per_face = (size_t)Hmax * 128 + (size_t)(Hmax + 1) * kRowStride * sizeof(stack_t) * c->layout.nplanes +
                          (c->layout.gabor_first >= 0 && !c->gabor_fused ? (size_t)Hmax * 128 * 4 * 35 + 35 * 2 * 4 : 0) + np_hp * c->hp_ntrees * 4 +
                          np_ffd * c->mp_ntrees_cfg * (4 + 3 * sizeof(DevVote)) + (size_t)kMaxList * 4 + 4 +
                          (headpose_only ? 0 : (size_t)kVoteSegs * kParts * 4 + 2 * kParts * 4) + sizeof(FaceDesc) + sizeof(crf_face_t);
  const size_t budget = c->work_budget / c->nstreams;
  long long chunk = (long long)(budget / per_face);
  const int cap = c->opt.max_chunk > 0 ? c->opt.max_chunk : 4096;
  return (int)std::max<long long>(1, std::min<long long>(std::min<long long>(chunk, cap), 32768));
}

static int pull_counters(crf_ctx* c) {
  if (!c->counting) return CRF_OK;
  unsigned long long h[CNT_NUM];
  CU(cudaMemcpyAsync(h, c->d_counters.p, sizeof h, cudaMemcpyDeviceToHost, c->w->stream));
  CU(cudaStreamSynchronize(c->w->stream));
  c->cnt.hp_node_tests += h[CNT_HP_TESTS]; c->cnt.ffd_node_tests += h[CNT_FFD_TESTS];
  c->cnt.hp_traversals += h[CNT_HP_TRAV]; c->cnt.ffd_traversals += h[CNT_FFD_TRAV];
  c->cnt.votes += h[CNT_VOTES]; c->cnt.vote_passes += h[CNT_VOTE_PASSES];
  CU(cudaMemsetAsync(c->d_counters.p, 0, sizeof h, c->w->stream));
  CU(cudaStreamSynchronize(c->w->stream));
  return CRF_OK;
}

// Faces whose composition asked for more trees than the batched launch holds (flags bit 1; only reachable
// when areaUnderCurve's Riemann sum overshoots, i.e. a near-zero head-pose variance) are re-run one at a
// time with the widest list, so that the result still equals the reference-shaped oracle.
static int rerun_wide(crf_ctx* c, const FaceDesc* d_fd_all, const std::vector<FaceDesc>& descs, const uint8_t* d_imgs, crf_face_t* d_faces_all,
                      const std::vector<int>& which) {
  for (int i : which) {
    Plan p; p.n = 1; p.Hmax = descs[i].H; p.nplanes = c->layout.nplanes; p.need_gabor = c->layout.gabor_first >= 0; p.hp_stride = c->opt.hp_stride; p.ffd_stride = c->opt.ffd_stride; p.tree_cap = kMaxList; p.vote_factor = kParts;
    int rc = ensure(c, p);
    if (rc) return rc;
    if ((rc = run_faces(c, d_fd_all + i, 1, p.Hmax, d_imgs, d_faces_all + i, false, kMaxList, nullptr))) return rc;
  }
  return CRF_OK;
}

static size_t image_bytes(const crf_image_t& im) { return (size_t)im.rows * im.step; }

static bool bad_geometry(const crf_image_t& im) { return im.rows < 1 || im.cols < 1 || im.step < (size_t)im.cols * 3; }

// The descriptor rule of the _mixed calls: every frame has pixels, rows, cols >= 1 and step >= cols * 3.
static int image_args(const crf_image_t* images, int n_images) {
  for (int i = 0; i < n_images; i++) {
    if (!images[i].bgr) return fail(CRF_ERR_ARG, "null frame");
    if (bad_geometry(images[i])) return fail(CRF_ERR_ARG, "bad frame descriptor (rows, cols >= 1, step >= cols * 3)");
  }
  return CRF_OK;
}

// The checks a boxes-given call makes before any work: each box names a frame in range with pixels and fits that frame's analysis path.
// (A null frame that no box names is accepted here: the equal-size calls always did.)
static int box_args(const crf_image_t* images, int n_images, const crf_rect_t* boxes, const int* image_of_box, int n) {
  for (int k = 0; k < n_images; k++)
    if (bad_geometry(images[k])) return fail(CRF_ERR_ARG, "bad frame descriptor (rows, cols >= 1, step >= cols * 3)");
  for (int i = 0; i < n; i++) {
    const int im = image_of_box ? image_of_box[i] : i;
    if (im < 0 || im >= n_images || !images[im].bgr) return fail(CRF_ERR_ARG, "image index out of range");
    if (const char* e = box_error(images[im].rows, images[im].cols, boxes[i])) return fail(CRF_ERR_ARG, e);
  }
  return CRF_OK;
}

// n_images descriptors of equal-size frames: what the calls that take one (rows, cols, step) pass to the generalised core.  NULL when
// images is (the core reports it).
static const crf_image_t* same_size(const uint8_t* const* images, int n_images, int rows, int cols, size_t step, std::vector<crf_image_t>& v) {
  if (!images) return nullptr;
  v.resize((size_t)std::max(n_images, 0));
  for (int i = 0; i < n_images; i++) v[(size_t)i] = crf_image_t{images[i], rows, cols, step};
  return v.data();
}

// Host-resident inputs.  images[k] describes frame k; faces are processed in chunks, frames of a chunk are copied on a second stream
// into one of two device buffers so the copy of chunk k+1 overlaps chunk k.
static int analyze_host(crf_ctx* c, const crf_image_t* images, int n_images, const crf_rect_t* boxes, const int* image_of_box, int n,
                        crf_face_t* out, bool headpose_only) {
  if (!c) return fail(CRF_ERR_STATE, "context is not initialised");
  if (!c->full_model) return fail(CRF_ERR_STATE, "analyzeFace needs the head-pose forest and the 5 pose forests; this context holds a single forest");
  if (n < 0 || (n > 0 && (!images || !boxes || !out))) return fail(CRF_ERR_ARG, "null argument");
  if (n == 0) return CRF_OK;
  if (int rc = box_args(images, n_images, boxes, image_of_box, n)) return rc;
  CU(cudaSetDevice(c->device));
  std::vector<FaceDesc> descs((size_t)n);
  int Hmax_first = 0;
  for (int i = 0; i < n; i++) {
    const crf_image_t& im = images[image_of_box ? image_of_box[i] : i];
    int rc = make_desc(c, im.rows, im.cols, im.step, 0, boxes[i], descs[i]);
    if (rc) return rc;
    Hmax_first = std::max(Hmax_first, descs[i].H);
  }
  // chunks of consecutive faces; a chunk's frames are the distinct frames its faces name
  int chunk = pick_chunk(c, Hmax_first, headpose_only);
  // A batch that fits one launch but moves a lot of pixels per face (faces in video frames: ~95 KB of box pixels each at 1080p) is cut in
  // two, so that packing + copying the second half overlaps the kernels of the first: C3 (64 frames x 16 faces) 24.0 -> 21.4 ms per call.
  // Three or more pieces cost more in launch tails than they hide (measured), and crops (30 KB per face) do not pay at all.
  if (c->opt.max_chunk <= 0 && n <= chunk && n >= 512) {
    size_t box_bytes = 0;
    for (int i = 0; i < n; i++) box_bytes += (size_t)boxes[i].width * boxes[i].height * 3;
    if (box_bytes / (size_t)n >= 64 * 1024) chunk = (n + 1) / 2;
  }
  // Two upload modes per chunk.  Frame mode: the distinct frames of the chunk go up whole (crops, dense boxes).  ROI mode:
  // when the boxes cover well under the frames' area (a few faces in a 1080p / 4K frame), only the box pixels travel — packed
  // row by row into a pinned staging buffer on the host while the GPU works on the previous chunk, then one H2D copy.
  // Pageable sources always go through the staging buffer (a threaded pack + pinned H2D beats the driver's pageable copy).
  // a batch is treated as pinned only if every frame it names is (one pageable frame sends the whole batch through the packed path)
  bool src_pinned = true;
  {
    int last = -1;
    for (int i = 0; i < n && src_pinned; i++) {
      const int im = image_of_box ? image_of_box[i] : i;
      if (im != last) { src_pinned = is_pinned_host(images[im].bgr); last = im; }
    }
  }
  struct Chunk { int f0, f1, Hmax; bool roi; size_t bytes; std::vector<int> frames; std::vector<size_t> slot_off; };
  std::vector<Chunk> chunks;
  std::vector<crf_rect_t> src_box((size_t)n);   // where the pixels are in the caller's frame (ROI mode rewrites the descriptor)
  for (int f0 = 0; f0 < n; f0 += chunk) {
    Chunk ch; ch.f0 = f0; ch.f1 = std::min(n, f0 + chunk); ch.Hmax = 0; ch.roi = false; ch.bytes = 0;
    std::unordered_map<int, int> slot_of;
    size_t roi_bytes = 0;
    for (int i = f0; i < ch.f1; i++) {
      const int im = image_of_box ? image_of_box[i] : i;
      auto it = slot_of.find(im);
      int slot;
      if (it == slot_of.end()) {   // frame-mode slots: the chunk's distinct frames back to back
        slot = (int)ch.frames.size(); ch.frames.push_back(im); slot_of.emplace(im, slot);
        ch.slot_off.push_back(ch.bytes); ch.bytes += image_bytes(images[im]);
      } else slot = it->second;
      descs[i].img_off = ch.slot_off[(size_t)slot];
      src_box[i] = boxes[i];
      roi_bytes += ((size_t)boxes[i].width * boxes[i].height * 3 + 15) & ~(size_t)15;
      ch.Hmax = std::max(ch.Hmax, descs[i].H);
    }
    if (roi_bytes * 10 < ch.bytes * 6 || (!src_pinned && roi_bytes <= ch.bytes + ch.bytes / 4)) {
      ch.roi = true; ch.bytes = roi_bytes;
      size_t off = 0;
      for (int i = f0; i < ch.f1; i++) {
        descs[i].img_off = off; descs[i].img_step = (size_t)boxes[i].width * 3; descs[i].bx = 0; descs[i].by = 0;
        off += ((size_t)boxes[i].width * boxes[i].height * 3 + 15) & ~(size_t)15;
      }
    }
    chunks.push_back(std::move(ch));
  }
  int rc;
  c->w = &c->ws[0];
  cudaStream_t s0 = c->ws[0].stream;
  if ((rc = c->d_fd.reserve((size_t)n * sizeof(FaceDesc)))) return rc;
  if ((rc = c->d_faces.reserve((size_t)n * sizeof(crf_face_t)))) return rc;
  CU(cudaMemcpyAsync(c->d_fd.p, descs.data(), (size_t)n * sizeof(FaceDesc), cudaMemcpyHostToDevice, s0));
  CU(cudaMemsetAsync(c->d_faces.p, 0, (size_t)n * sizeof(crf_face_t), s0));
  c->cnt.h2d_bytes += (size_t)n * sizeof(FaceDesc);
  size_t max_bytes = 0, max_roi = 0; int Hmax_all = 0, max_faces = 0;
  for (auto& ch : chunks) {
    max_bytes = std::max(max_bytes, ch.bytes); if (ch.roi) max_roi = std::max(max_roi, ch.bytes);
    Hmax_all = std::max(Hmax_all, ch.Hmax); max_faces = std::max(max_faces, ch.f1 - ch.f0);
  }
  for (int b = 0; b < 2; b++) {
    if ((rc = c->d_imgs[b].reserve(max_bytes))) return rc;
    if (max_roi > c->h_stage_bytes[b]) {
      if (c->h_stage[b]) cudaFreeHost(c->h_stage[b]);
      c->h_stage[b] = nullptr; c->h_stage_bytes[b] = 0;
      CU(cudaHostAlloc((void**)&c->h_stage[b], max_roi + max_roi / 4, cudaHostAllocDefault));
      c->h_stage_bytes[b] = max_roi + max_roi / 4;
    }
  }
  Plan p; p.n = max_faces; p.Hmax = Hmax_all; p.nplanes = c->layout.nplanes; p.need_gabor = c->layout.gabor_first >= 0; p.hp_stride = c->opt.hp_stride; p.ffd_stride = c->opt.ffd_stride; p.tree_cap = c->mp_ntrees_cfg;
  p.need_ffd = !headpose_only;
  const int nsets = chunks.size() > 1 ? c->nstreams : 1;
  for (int k = 0; k < nsets; k++) { c->w = &c->ws[k]; if ((rc = ensure(c, p))) return rc; }
  CU(cudaStreamSynchronize(s0));   // descriptors and the zeroed records are visible to both streams
  auto copy_chunk = [&](size_t k) -> int {
    const Chunk& ch = chunks[k];
    const int b = (int)(k & 1);
    if (ch.roi) {
      if (k >= 2) CU(cudaEventSynchronize(c->ev_copied[b]));   // the staging buffer's previous upload has left the host
      uint8_t* st = c->h_stage[b];
      parallel_for(ch.f1 - ch.f0, ch.bytes, [&](int k2) {
        const int i = ch.f0 + k2;
        const crf_rect_t& bx = src_box[i];
        const crf_image_t& im = images[image_of_box ? image_of_box[i] : i];
        const size_t step = im.step;
        const uint8_t* src = im.bgr + (size_t)bx.y * step + (size_t)bx.x * 3;
        uint8_t* dst = st + descs[i].img_off;
        const size_t rowb = (size_t)bx.width * 3;
        if (rowb == step) std::memcpy(dst, src, rowb * bx.height);
        else for (int r = 0; r < bx.height; r++) std::memcpy(dst + (size_t)r * rowb, src + (size_t)r * step, rowb);
      });
      CU(cudaMemcpyAsync(c->d_imgs[b].p, st, ch.bytes, cudaMemcpyHostToDevice, c->copy_stream));
      c->cnt.h2d_bytes += ch.bytes;
      CU(cudaEventRecord(c->ev_copied[b], c->copy_stream));
      return CRF_OK;
    }
    // consecutive frames that are also consecutive in host memory go in one copy
    size_t i = 0;
    while (i < ch.frames.size()) {
      size_t j = i + 1;
      while (j < ch.frames.size() && images[ch.frames[j]].bgr == images[ch.frames[j - 1]].bgr + image_bytes(images[ch.frames[j - 1]])) j++;
      const size_t end = j < ch.frames.size() ? ch.slot_off[j] : ch.bytes;
      CU(cudaMemcpyAsync(c->d_imgs[b].as<uint8_t>() + ch.slot_off[i], images[ch.frames[i]].bgr, end - ch.slot_off[i], cudaMemcpyHostToDevice, c->copy_stream));
      i = j;
    }
    c->cnt.h2d_bytes += ch.bytes;
    CU(cudaEventRecord(c->ev_copied[b], c->copy_stream));
    return CRF_OK;
  };
  // results of chunk k: D2H, pathological faces re-run with the wide capacities (needs the chunk's frames and work set)
  auto finish_chunk = [&](size_t k) -> int {
    const Chunk& ch = chunks[k];
    const int b = (int)(k & 1);
    c->w = &c->ws[k % nsets];
    const size_t m = (size_t)(ch.f1 - ch.f0);
    CU(cudaMemcpyAsync(out + ch.f0, c->d_faces.as<crf_face_t>() + ch.f0, m * sizeof(crf_face_t), cudaMemcpyDeviceToHost, c->w->stream));
    CU(cudaStreamSynchronize(c->w->stream));
    c->cnt.d2h_bytes += m * sizeof(crf_face_t);
    if (headpose_only) return CRF_OK;
    std::vector<int> wide;
    for (size_t i = 0; i < m; i++) if (out[ch.f0 + i].flags & 6) wide.push_back(ch.f0 + (int)i);
    if (wide.empty()) return CRF_OK;
    int rc2 = rerun_wide(c, c->d_fd.as<FaceDesc>(), descs, c->d_imgs[b].as<uint8_t>(), c->d_faces.as<crf_face_t>(), wide);
    if (rc2) return rc2;
    for (int i : wide) CU(cudaMemcpyAsync(out + i, c->d_faces.as<crf_face_t>() + i, sizeof(crf_face_t), cudaMemcpyDeviceToHost, c->w->stream));
    CU(cudaStreamSynchronize(c->w->stream));
    Plan q = p; q.n = (int)m; q.Hmax = ch.Hmax;
    return ensure(c, q);   // restore the batched geometry of this set
  };
  // two-deep software pipeline: chunk k runs on stream k&1 while chunk k-1 finishes on the other one
  if ((rc = copy_chunk(0))) return rc;
  for (size_t k = 0; k < chunks.size(); k++) {
    const Chunk& ch = chunks[k];
    const int b = (int)(k & 1);
    c->w = &c->ws[k % nsets];
    Plan q = p; q.n = ch.f1 - ch.f0; q.Hmax = ch.Hmax;
    if ((rc = ensure(c, q))) return rc;  // only recomputes the strides (capacity is already there)
    CU(cudaStreamWaitEvent(c->w->stream, c->ev_copied[b], 0));
    if ((rc = run_faces(c, c->d_fd.as<FaceDesc>() + ch.f0, ch.f1 - ch.f0, ch.Hmax, c->d_imgs[b].as<uint8_t>(), c->d_faces.as<crf_face_t>() + ch.f0,
                        headpose_only, c->mp_ntrees_cfg, nullptr)))
      return rc;
    if (k >= 1 && (rc = finish_chunk(k - 1))) return rc;
    if (k + 1 < chunks.size() && (rc = copy_chunk(k + 1))) return rc;   // its image buffer was chunk k-1's: free now
  }
  if ((rc = finish_chunk(chunks.size() - 1))) return rc;
  c->w = &c->ws[0];
  c->cnt.faces += n;
  c->timer.collect();
  return pull_counters(c);
}

}  // namespace crf

#include "haar.cuh"

namespace crf {
// Faces whose descriptors point into frames already in device memory (d_imgs): descriptors up, records into d_out (n x crf_face_t),
// chunked like the host path; faces flagged for the worst-case capacities are re-run wide.  Returns when d_out is complete.
static int analyze_resident(crf_ctx* c, const std::vector<FaceDesc>& descs, int Hmax, const uint8_t* d_imgs, crf_face_t* d_out, bool headpose_only) {
  const int n = (int)descs.size();
  int rc;
  c->w = &c->ws[0];
  cudaStream_t s0 = c->ws[0].stream;
  if ((rc = c->d_fd.reserve((size_t)n * sizeof(FaceDesc)))) return rc;
  CU(cudaMemcpyAsync(c->d_fd.p, descs.data(), (size_t)n * sizeof(FaceDesc), cudaMemcpyHostToDevice, s0));
  CU(cudaMemsetAsync(d_out, 0, (size_t)n * sizeof(crf_face_t), s0));
  const int chunk = pick_chunk(c, Hmax, headpose_only);
  Plan p; p.n = std::min(n, chunk); p.Hmax = Hmax; p.nplanes = c->layout.nplanes; p.need_gabor = c->layout.gabor_first >= 0; p.hp_stride = c->opt.hp_stride; p.ffd_stride = c->opt.ffd_stride; p.tree_cap = c->mp_ntrees_cfg;
  p.need_ffd = !headpose_only;
  const int nsets = n > chunk ? c->nstreams : 1;
  for (int k = 0; k < nsets; k++) { c->w = &c->ws[k]; if ((rc = ensure(c, p))) return rc; }
  CU(cudaStreamSynchronize(s0));
  // consecutive chunks alternate between the two streams / work sets
  int k = 0;
  for (int f0 = 0; f0 < n; f0 += chunk, k++) {
    const int m = std::min(chunk, n - f0);
    c->w = &c->ws[k % nsets];
    if ((rc = run_faces(c, c->d_fd.as<FaceDesc>() + f0, m, Hmax, d_imgs, d_out + f0, headpose_only, c->mp_ntrees_cfg, nullptr))) return rc;
  }
  for (int q = 0; q < nsets; q++) CU(cudaStreamSynchronize(c->ws[q].stream));
  c->w = &c->ws[0];
  if (!headpose_only) {
    // faces whose composition or vote count exceeded the batched capacities: fetch the flags, re-run those faces wide
    // (4 bytes come back, not the records: the flag is counted on the device)
    int n_wide = 0;
    CU(cudaMemsetAsync(c->d_misc.p, 0, 4, s0));
    k_count_wide<<<(n + 255) / 256, 256, 0, s0>>>(d_out, n, c->d_misc.as<int>());
    KCHECK(); count_launch(c, CRF_STAGE_MEANSHIFT);
    CU(cudaMemcpyAsync(&n_wide, c->d_misc.p, 4, cudaMemcpyDeviceToHost, s0));
    CU(cudaStreamSynchronize(s0));
    if (n_wide > 0) {
      std::vector<crf_face_t> tmp((size_t)n);
      CU(cudaMemcpyAsync(tmp.data(), d_out, (size_t)n * sizeof(crf_face_t), cudaMemcpyDeviceToHost, s0));
      CU(cudaStreamSynchronize(s0));
      std::vector<int> wide;
      for (int i = 0; i < n; i++) if (tmp[(size_t)i].flags & 6) wide.push_back(i);
      if (!wide.empty() && (rc = rerun_wide(c, c->d_fd.as<FaceDesc>(), descs, d_imgs, d_out, wide))) return rc;
      CU(cudaStreamSynchronize(s0));
    }
  }
  c->cnt.faces += n;
  c->timer.collect();
  return pull_counters(c);
}

// ---- detectMultiScale on groups of frames (haar.cuh) ------------------------------------------------------------------------
// Frames resident at once: at most this many, and no more than half the work budget holds (the analysis of a group's faces needs
// the rest), so that a long video or a batch of 4K frames is not uploaded in one piece.
constexpr int kDetectGroupFrames = 64;

// The pyramid levels of one frame: instances without their group offsets.
struct FramePlan {
  std::vector<HaarInst> levels;
  int nrows = 0;                   // window rows over all levels
  size_t nint = 0, nwin = 0;       // integral elements / windows over all levels
};

// the scales of CascadeClassifierImpl::detectMultiScale (flags 0, no maxSize); levels below min_size are not built
static FramePlan detect_plan(const Cascade& K, const crf_image_t& im, double scale_factor, int min_size) {
  FramePlan p;
  const int rows = im.rows, cols = im.cols;
  for (double factor = 1;; factor *= scale_factor) {
    HaarInst L{};
    L.factor = factor;
    L.win_w = (int)std::lrint(K.win_w * factor); L.win_h = (int)std::lrint(K.win_h * factor);
    L.sw = (int)std::lrint(cols / factor); L.sh = (int)std::lrint(rows / factor);
    if (L.win_w > cols || L.win_h > rows || L.sw < K.win_w || L.sh < K.win_h) break;
    if (L.win_w < min_size || L.win_h < min_size) continue;
    L.scale_x = 1. / ((double)L.sw / cols); L.scale_y = 1. / ((double)L.sh / rows);
    L.ystep = factor > 2. ? 1 : 2;
    L.nx = (L.sw - K.win_w + 1 + L.ystep - 1) / L.ystep; L.ny = (L.sh - K.win_h + 1 + L.ystep - 1) / L.ystep;
    L.rows = rows; L.cols = cols; L.step = im.step;
    p.nrows += L.ny;
    p.nint += (size_t)(L.sw + 1) * (L.sh + 1);
    p.nwin += (size_t)L.nx * L.ny;
    p.levels.push_back(L);
  }
  return p;
}

// Frames [f0, f0 + nf) into d_haar_frames at off[k] (prefix sums of rows x step).  Pinned frames are copied straight (frames adjacent in
// host memory in one copy); pageable ones are packed into the two pinned staging buffers (~64 MB a batch) by a few threads and copied
// from there.
static int upload_frames(crf_ctx* c, const crf_image_t* images, int f0, int nf, const std::vector<size_t>& off, cudaStream_t s) {
  auto fb = [&](int k) { return image_bytes(images[f0 + k]); };
  uint8_t* d = c->d_haar_frames.as<uint8_t>();
  std::vector<int> pageable;
  for (int k = 0; k < nf;) {
    if (!is_pinned_host(images[f0 + k].bgr)) { pageable.push_back(k++); continue; }
    int j = k + 1;
    while (j < nf && images[f0 + j].bgr == images[f0 + j - 1].bgr + fb(j - 1) && is_pinned_host(images[f0 + j].bgr)) j++;
    CU(cudaMemcpyAsync(d + off[(size_t)k], images[f0 + k].bgr, off[(size_t)j] - off[(size_t)k], cudaMemcpyHostToDevice, s));
    k = j;
  }
  const size_t batch = (size_t)64 << 20;
  for (size_t p0 = 0, b = 0; p0 < pageable.size(); b ^= 1) {
    size_t p1 = p0 + 1, bytes = fb(pageable[p0]);
    while (p1 < pageable.size() && bytes + fb(pageable[p1]) <= batch) bytes += fb(pageable[p1++]);
    CU(cudaEventSynchronize(c->ev_copied[b]));   // the buffer's previous copy has left the host
    if (c->h_stage_bytes[b] < bytes) {
      if (c->h_stage[b]) cudaFreeHost(c->h_stage[b]);
      c->h_stage[b] = nullptr; c->h_stage_bytes[b] = 0;
      CU(cudaHostAlloc((void**)&c->h_stage[b], bytes, cudaHostAllocDefault));
      c->h_stage_bytes[b] = bytes;
    }
    uint8_t* st = c->h_stage[b];
    std::vector<size_t> st_off(p1 - p0 + 1, 0);
    for (size_t i = p0; i < p1; i++) st_off[i - p0 + 1] = st_off[i - p0] + fb(pageable[i]);
    parallel_for((int)(p1 - p0), bytes, [&](int i) { std::memcpy(st + st_off[(size_t)i], images[f0 + pageable[p0 + i]].bgr, fb(pageable[p0 + i])); });
    for (size_t i = p0; i < p1;) {   // runs of consecutive frame slots in one copy
      size_t j = i + 1;
      while (j < p1 && pageable[j] == pageable[j - 1] + 1) j++;
      CU(cudaMemcpyAsync(d + off[(size_t)pageable[i]], st + st_off[i - p0], st_off[j - p0] - st_off[i - p0], cudaMemcpyHostToDevice, s));
      i = j;
    }
    CU(cudaEventRecord(c->ev_copied[b], s));
    p0 = p1;
  }
  c->cnt.h2d_bytes += off[(size_t)nf];
  return CRF_OK;
}

// detectMultiScale on n_images frames of any sizes, a group of consecutive frames at a time.  After a group's boxes are grouped,
// per_group(f0, nf, off, boxes) runs while the group's frames are still in d_haar_frames (frame f0 + k at off[k]); boxes[k] are frame
// f0 + k's.
template <class F>
static int detect_frames(crf_ctx* c, const crf_cascade* cas, const crf_image_t* images, int n_images, double scale_factor, int min_neighbors,
                         int min_size, F&& per_group) {
  const Cascade& K = cas->c;
  std::vector<FramePlan> plans((size_t)n_images);
  for (int i = 0; i < n_images; i++) {
    plans[(size_t)i] = detect_plan(K, images[i], scale_factor, min_size);
    // work lists hold 32-bit flag indices
    if (plans[(size_t)i].nwin >= ((size_t)1 << 31)) return fail(CRF_ERR_ARG, "frame too large for the detector (2^31 windows)");
  }
  CU(cudaSetDevice(c->device));
  c->w = &c->ws[0];
  cudaStream_t s = c->w->stream;
  int rc;
  // the kernel variant follows what the cascade holds: stumps or trees, upright features only or some tilted ones
  const bool tree = K.is_tree(), tilt = K.has_tilted;
  if (c->haar_cached != cas->id) {
    if ((rc = upload(c->d_haar_stages, K.stages, s)) || (rc = upload(c->d_haar_feats, K.features, s))) return rc;
    if (tree ? (rc = upload(c->d_haar_weak, K.trees, s)) || (rc = upload(c->d_haar_nodes, K.nodes, s)) || (rc = upload(c->d_haar_leaves, K.leaves, s))
             : (rc = upload(c->d_haar_weak, K.weak, s)))
      return rc;
    if (tilt && (rc = upload(c->d_haar_tilt, K.tilted, s))) return rc;
    c->haar_cached = cas->id;
  }
  const HaarDev dev{c->d_haar_stages.as<HaarStage>(), tree ? nullptr : c->d_haar_weak.as<HaarWeak>(), c->d_haar_feats.as<HaarFeature>(), (int)K.stages.size(), K.win_w, K.win_h,
                    tree ? c->d_haar_weak.as<HaarTree>() : nullptr, tree ? c->d_haar_nodes.as<HaarNode>() : nullptr, tree ? c->d_haar_leaves.as<float>() : nullptr,
                    tilt ? c->d_haar_tilt.as<uint8_t>() : nullptr};
  auto eval_first = tree ? (tilt ? k_haar_eval_first<true, true> : k_haar_eval_first<true, false>) : (tilt ? k_haar_eval_first<false, true> : k_haar_eval_first<false, false>);
  auto eval_list = tree ? (tilt ? k_haar_eval_list<true, true> : k_haar_eval_list<true, false>) : (tilt ? k_haar_eval_list<false, true> : k_haar_eval_list<false, false>);
  // stage groups: [0, split[0]), [split[0], split[1]), ..., up to the last stage
  std::vector<int> bounds;
  for (int b : c->haar_split) if (b > (bounds.empty() ? 0 : bounds.back()) && b < dev.nstages) bounds.push_back(b);
  bounds.push_back(dev.nstages);
  // integrals: S and Q, plus T for a tilted cascade
  const size_t int_bytes = tilt ? 12 : 8;
  auto footprint = [&](int i) { const FramePlan& p = plans[(size_t)i]; return image_bytes(images[i]) + p.nint * int_bytes + p.nwin * (1 + 2 * sizeof(uint2)) + (size_t)p.nrows * 4; };
  std::vector<std::vector<crf_rect_t>> boxes;
  std::vector<int> frame_count;
  for (int f0 = 0, f1; f0 < n_images; f0 = f1) {
    // a group: consecutive frames, at most kDetectGroupFrames, within half the work budget, fewer than 2^32 windows
    size_t bytes = footprint(f0), wins = plans[(size_t)f0].nwin;
    for (f1 = f0 + 1; f1 < n_images && f1 - f0 < kDetectGroupFrames; f1++) {
      if (bytes + footprint(f1) > c->work_budget / 2 || wins + plans[(size_t)f1].nwin > ((size_t)1 << 32) - 1) break;
      bytes += footprint(f1); wins += plans[(size_t)f1].nwin;
    }
    const int nf = f1 - f0;
    boxes.assign((size_t)nf, {});
    // the instance table (frame-major, then level), the frames' device offsets and their window-row ranges
    std::vector<HaarInst> inst;
    std::vector<size_t> off((size_t)nf + 1, 0);
    std::vector<int> frame_rows((size_t)nf + 1, 0);
    size_t io = 0, fo = 0;
    int nrows = 0, brows = 0, bcols = 0, beval = 0, btilt = 0;
    std::vector<int> blk_tilt;   // first block of each instance in k_haar_tilted
    for (int k = 0; k < nf; k++) {
      off[(size_t)k + 1] = off[(size_t)k] + image_bytes(images[f0 + k]);
      for (HaarInst L : plans[(size_t)(f0 + k)].levels) {
        L.img_off = off[(size_t)k]; L.frame = k;
        L.int_off = io; io += (size_t)(L.sw + 1) * (L.sh + 1);
        L.flag_off = fo; fo += (size_t)L.nx * L.ny;
        L.row_off = nrows; nrows += L.ny;
        L.blk_rows = brows; brows += (L.sh + 7) / 8;
        L.blk_cols = bcols; bcols += (L.sw + 1 + 31) / 32;
        L.blk_eval = beval; beval += (L.nx + 127) / 128 * L.ny;
        if (tilt) { blk_tilt.push_back(btilt); btilt += 2 * ((L.sw + L.sh + 31) / 32); }
        inst.push_back(L);
      }
      frame_rows[(size_t)k + 1] = nrows;
    }
    if (!inst.empty()) {
      const int ninst = (int)inst.size();
      // one upload: the instances, then the frames' row ranges, then the search keys (HaarKeys, then blk_tilt for a tilted cascade)
      const size_t tab = ((size_t)ninst * sizeof(HaarInst) + 15) & ~(size_t)15;
      std::vector<int> ints(frame_rows);
      for (int k = 0; k < 5; k++)
        for (const HaarInst& L : inst)
          ints.push_back(k == 0 ? L.blk_rows : k == 1 ? L.blk_cols : k == 2 ? L.blk_eval : k == 3 ? L.row_off : (int)(unsigned)L.flag_off);
      ints.insert(ints.end(), blk_tilt.begin(), blk_tilt.end());
      std::vector<uint8_t> table(tab + ints.size() * sizeof(int));
      std::memcpy(table.data(), inst.data(), (size_t)ninst * sizeof(HaarInst));
      std::memcpy(table.data() + tab, ints.data(), ints.size() * sizeof(int));
      if ((rc = c->d_haar_frames.reserve(off[(size_t)nf])) || (rc = c->d_haar_S.reserve(io * 4)) || (rc = c->d_haar_Q.reserve(io * 4)) ||
          (rc = c->d_haar_flags.reserve(fo)) || (rc = c->d_haar_list[0].reserve(fo * sizeof(uint2))) || (rc = c->d_haar_list[1].reserve(fo * sizeof(uint2))) ||
          (rc = c->d_haar_rows.reserve((size_t)nrows * 4)) || (rc = c->d_haar_counts.reserve((size_t)(kDetectGroupFrames + 4) * 4)) ||
          (tilt && (rc = c->d_haar_T.reserve(io * 4))))
        return rc;
      if ((rc = upload_frames(c, images, f0, nf, off, s))) return rc;
      if ((rc = upload(c->d_haar_levels, table, s))) return rc;
      const HaarInst* d_inst = c->d_haar_levels.as<HaarInst>();
      const int* d_frame_rows = reinterpret_cast<const int*>(c->d_haar_levels.as<uint8_t>() + tab);
      const int* d_key = d_frame_rows + frame_rows.size();
      const HaarKeys keys{d_key, d_key + ninst, d_key + 2 * ninst, d_key + 3 * ninst, reinterpret_cast<const unsigned*>(d_key + 4 * ninst)};
      unsigned* lists_n = c->d_haar_counts.as<unsigned>();   // [0], [1]: lengths of the two work lists; [4...]: candidates per frame
      int* fcount = c->d_haar_counts.as<int>() + 4;
      CU(cudaMemsetAsync(lists_n, 0, 4 * sizeof(unsigned), s));
      uint32_t* S = c->d_haar_S.as<uint32_t>();
      uint32_t* Q = c->d_haar_Q.as<uint32_t>();
      uint8_t* flags = c->d_haar_flags.as<uint8_t>();
      uint2* list[2] = {c->d_haar_list[0].as<uint2>(), c->d_haar_list[1].as<uint2>()};
      uint32_t* T = tilt ? c->d_haar_T.as<uint32_t>() : nullptr;
      if (tilt) {
        // the tilted integrals from the row prefixes k_haar_rows leaves in S, before k_haar_cols turns them into the integrals
        k_haar_rows<true><<<brows, 256, 0, s>>>(d_inst, keys, ninst, c->d_haar_frames.as<uint8_t>(), S, Q, T);
        k_haar_tilted<<<btilt, dim3(32, 32), 0, s>>>(d_inst, d_key + 5 * ninst, ninst, S, T);
        KCHECK(); count_launch(c, CRF_STAGE_RESIZE, 2);
      } else {
        k_haar_rows<false><<<brows, 256, 0, s>>>(d_inst, keys, ninst, c->d_haar_frames.as<uint8_t>(), S, Q, nullptr);
        KCHECK(); count_launch(c, CRF_STAGE_RESIZE);
      }
      k_haar_cols<<<bcols, dim3(32, 32), 0, s>>>(d_inst, keys, ninst, S, Q);
      eval_first<<<beval, 128, 0, s>>>(d_inst, keys, ninst, S, Q, T, dev, bounds[0], flags, list[0], lists_n);
      KCHECK(); count_launch(c, CRF_STAGE_RESIZE, 2);
      for (size_t g = 1; g < bounds.size(); g++) {
        const int in = (int)((g - 1) & 1), out = (int)(g & 1);
        if (g >= 2) CU(cudaMemsetAsync(lists_n + out, 0, sizeof(unsigned), s));
        eval_list<<<c->sm_count * 8, 128, 0, s>>>(d_inst, keys, ninst, S, T, dev, bounds[g - 1], bounds[g], list[in], lists_n + in, flags, list[out], lists_n + out);
        KCHECK(); count_launch(c, CRF_STAGE_RESIZE);
      }
      int* d_rows = c->d_haar_rows.as<int>();
      k_haar_scan<true><<<(nrows + 7) / 8, 256, 0, s>>>(d_inst, keys, ninst, nrows, flags, d_rows, nullptr, nullptr);
      k_haar_row_offsets<<<nf, 1024, 0, s>>>(d_frame_rows, d_rows, fcount);
      KCHECK(); count_launch(c, CRF_STAGE_RESIZE, 2);
      frame_count.assign((size_t)nf, 0);
      CU(cudaMemcpyAsync(frame_count.data(), fcount, (size_t)nf * 4, cudaMemcpyDeviceToHost, s));
      CU(cudaStreamSynchronize(s));
      size_t total = 0;
      for (int v : frame_count) total += (size_t)v;
      if ((rc = c->d_haar_cand.reserve(std::max<size_t>(total, 1) * sizeof(crf_rect_t)))) return rc;
      k_haar_scan<false><<<(nrows + 7) / 8, 256, 0, s>>>(d_inst, keys, ninst, nrows, flags, d_rows, fcount, c->d_haar_cand.as<crf_rect_t>());
      KCHECK(); count_launch(c, CRF_STAGE_RESIZE);
      std::vector<crf_rect_t> cand(total);
      if (total) CU(cudaMemcpyAsync(cand.data(), c->d_haar_cand.p, total * sizeof(crf_rect_t), cudaMemcpyDeviceToHost, s));
      CU(cudaStreamSynchronize(s));
      c->cnt.d2h_bytes += (size_t)nf * 4 + total * sizeof(crf_rect_t);
      for (int k = 0, o = 0; k < nf; o += frame_count[(size_t)k], k++) boxes[(size_t)k].assign(cand.begin() + o, cand.begin() + o + frame_count[(size_t)k]);
      // cv::groupRectangles per frame; quadratic in a frame's candidates, so the work estimate is their square
      size_t work = 0;
      for (int v : frame_count) work += (size_t)v * v;
      parallel_for(nf, work * 64, [&](int k) { group_rectangles(boxes[(size_t)k], min_neighbors, 0.2); });
    }
    if ((rc = per_group(f0, nf, off, boxes))) return rc;
  }
  return CRF_OK;
}

// FaceForest::detectFace's enlargement (src/FaceForest.cpp:147-157): 5 % of the width left and right, 15 % of the WIDTH added to the height
// twice, intersected with the frame (intersect() of src/face_utils.cpp:325-347 returns (0, 0, 0, 0) when they do not overlap).
static crf_rect_t enlarge_detection(const crf_rect_t& r, int rows, int cols) {
  const int ox = (int)(r.width * 0.05), oy = (int)(r.width * 0.15);
  const int x0 = std::max(r.x - ox, 0), y0 = std::max(r.y, 0), x1 = std::min(r.x - ox + r.width + 2 * ox, cols), y1 = std::min(r.y + r.height + 2 * oy, rows);
  return x1 > x0 && y1 > y0 ? crf_rect_t{x0, y0, x1 - x0, y1 - y0} : crf_rect_t{0, 0, 0, 0};
}

static int detect_args(crf_ctx* c, const crf_cascade* cas, const crf_image_t* images, int n_images, double scale_factor, int cap, const void* out) {
  if (!c) return fail(CRF_ERR_STATE, "context is not initialised");
  if (!cas || n_images < 0 || (n_images > 0 && !images) || !(scale_factor > 1.0) || cap < 0 || (cap > 0 && !out)) return fail(CRF_ERR_ARG, "bad argument");
  return image_args(images, n_images);
}

// the equal-size calls check their one geometry even without frames
static int same_size_args(const crf_ctx* c, int rows, int cols, size_t step) {
  if (c && (rows < 1 || cols < 1 || step < (size_t)cols * 3)) return fail(CRF_ERR_ARG, "bad argument");
  return CRF_OK;
}

// detectMultiScale on n_images frames: returns the total box count, the first `cap` boxes in out and, when image_of_box is given, their frames
static int detect_boxes(crf_ctx* c, const crf_cascade* cas, const crf_image_t* images, int n_images, double scale_factor, int min_neighbors, int min_size,
                        crf_rect_t* out, int* image_of_box, int cap) {
  int total = 0;
  const int rc = detect_frames(c, cas, images, n_images, scale_factor, min_neighbors, min_size,
                               [&](int f0, int nf, const std::vector<size_t>&, std::vector<std::vector<crf_rect_t>>& boxes) -> int {
    for (int k = 0; k < nf; k++)
      for (const crf_rect_t& r : boxes[(size_t)k]) {
        if (total < cap) { out[total] = r; if (image_of_box) image_of_box[total] = f0 + k; }
        total++;
      }
    return CRF_OK;
  });
  return rc ? rc : total;
}
}  // namespace crf


// =============================================================================================
// C ABI
// =============================================================================================
extern "C" {

// ---- FaceForest::detectFace's box source (src/FaceForest.cpp:136-146): cv::CascadeClassifier::load + detectMultiScale
int crf_cascade_load(const char* path, crf_cascade** out) {
  if (!path || !out) return fail(CRF_ERR_ARG, "null argument");
  *out = nullptr;
  static std::atomic<unsigned long long> next_id{1};
  std::unique_ptr<crf_cascade> c(new crf_cascade());
  c->id = next_id++;
  std::string err;
  const int rc = load_cascade(path, c->c, err);
  if (rc) return fail(rc, err);
  *out = c.release();
  return CRF_OK;
}
void crf_cascade_free(crf_cascade* c) { delete c; }

int crf_cascade_info(const crf_cascade* c, int* win_w, int* win_h, int* nstages, int* nweak) {
  if (!c) return fail(CRF_ERR_ARG, "null argument");
  if (win_w) *win_w = c->c.win_w;
  if (win_h) *win_h = c->c.win_h;
  if (nstages) *nstages = (int)c->c.stages.size();
  if (nweak) *nweak = c->c.nweak();
  return CRF_OK;
}

int crf_detect_faces_batch_mixed(crf_ctx* c, const crf_cascade* cas, const crf_image_t* images, int n_images, double scale_factor, int min_neighbors,
                                 int min_size, crf_rect_t* out, int* image_of_box, int cap) {
  if (int rc = detect_args(c, cas, images, n_images, scale_factor, cap, out)) return rc;
  if (cap > 0 && !image_of_box) return fail(CRF_ERR_ARG, "bad argument");
  return detect_boxes(c, cas, images, n_images, scale_factor, min_neighbors, min_size, out, image_of_box, cap);
}

int crf_detect_faces(crf_ctx* c, const crf_cascade* cas, const uint8_t* bgr, int rows, int cols, size_t step, double scale_factor, int min_neighbors, int min_size,
                     crf_rect_t* out, int cap) {
  const crf_image_t im{bgr, rows, cols, step};
  if (int rc = detect_args(c, cas, &im, 1, scale_factor, cap, out)) return rc;
  return detect_boxes(c, cas, &im, 1, scale_factor, min_neighbors, min_size, out, nullptr, cap);
}

int crf_detect_faces_batch(crf_ctx* c, const crf_cascade* cas, const uint8_t* const* images, int n_images, int rows, int cols, size_t step, double scale_factor,
                           int min_neighbors, int min_size, crf_rect_t* out, int* image_of_box, int cap) {
  if (int rc = same_size_args(c, rows, cols, step)) return rc;
  std::vector<crf_image_t> v;
  return crf_detect_faces_batch_mixed(c, cas, same_size(images, n_images, rows, cols, step, v), n_images, scale_factor, min_neighbors, min_size, out, image_of_box, cap);
}

int crf_analyze_images_mixed(crf_ctx* c, const crf_cascade* cas, const crf_image_t* images, int n_images, double scale_factor, int min_neighbors, int min_size,
                             crf_rect_t* boxes, int* image_of_box, crf_face_t* out, int cap) {
  if (int rc = detect_args(c, cas, images, n_images, scale_factor, cap, boxes)) return rc;
  if (cap > 0 && (!image_of_box || !out)) return fail(CRF_ERR_ARG, "bad argument");
  if (!c->full_model) return fail(CRF_ERR_STATE, "analyzeFace needs the head-pose forest and the 5 pose forests; this context holds a single forest");
  int total = 0;
  const int rc = detect_frames(c, cas, images, n_images, scale_factor, min_neighbors, min_size,
                               [&](int f0, int nf, const std::vector<size_t>& off, std::vector<std::vector<crf_rect_t>>& det) -> int {
    // FaceDescs point into the group's device frames: the analysis reads the copy made for detection
    std::vector<FaceDesc> descs;
    std::vector<int> slot;   // output index of descs[i]
    int Hmax = 0;
    for (int k = 0; k < nf; k++) {
      const crf_image_t& im = images[f0 + k];
      for (const crf_rect_t& r : det[(size_t)k]) {
        if (total < cap) {
          const crf_rect_t e = enlarge_detection(r, im.rows, im.cols);
          boxes[total] = e; image_of_box[total] = f0 + k; out[total] = crf_face_t{};
          if (box_error(im.rows, im.cols, e)) {
            out[total].flags = CRF_FACE_NOT_ANALYSED;
          } else {
            FaceDesc d;
            if (int rc2 = make_desc(c, im.rows, im.cols, im.step, off[(size_t)k], e, d)) return rc2;
            descs.push_back(d); slot.push_back(total);
            Hmax = std::max(Hmax, d.H);
          }
        }
        total++;
      }
    }
    if (descs.empty()) return CRF_OK;
    int rc2;
    if ((rc2 = c->d_faces.reserve(descs.size() * sizeof(crf_face_t)))) return rc2;
    if ((rc2 = analyze_resident(c, descs, Hmax, c->d_haar_frames.as<uint8_t>(), c->d_faces.as<crf_face_t>(), false))) return rc2;
    c->cnt.h2d_bytes += descs.size() * sizeof(FaceDesc);
    std::vector<crf_face_t> rec(descs.size());
    CU(cudaMemcpyAsync(rec.data(), c->d_faces.p, rec.size() * sizeof(crf_face_t), cudaMemcpyDeviceToHost, c->ws[0].stream));
    CU(cudaStreamSynchronize(c->ws[0].stream));
    c->cnt.d2h_bytes += rec.size() * sizeof(crf_face_t);
    for (size_t i = 0; i < rec.size(); i++) out[slot[i]] = rec[i];
    return CRF_OK;
  });
  return rc ? rc : total;
}

int crf_analyze_images(crf_ctx* c, const crf_cascade* cas, const uint8_t* const* images, int n_images, int rows, int cols, size_t step, double scale_factor,
                       int min_neighbors, int min_size, crf_rect_t* boxes, int* image_of_box, crf_face_t* out, int cap) {
  if (int rc = same_size_args(c, rows, cols, step)) return rc;
  std::vector<crf_image_t> v;
  return crf_analyze_images_mixed(c, cas, same_size(images, n_images, rows, cols, step, v), n_images, scale_factor, min_neighbors, min_size, boxes, image_of_box,
                                  out, cap);
}

const char* crf_last_error(void) { return g_last_error.c_str(); }
const char* crf_version(void) { return "crf_b200 0.1 (sm_100a)"; }

void crf_options_default(crf_options_t* o) {
  if (!o) return;
  o->hp_stride = 4; o->hp_min_foreground = 0.5f;                       // include/FaceForest.hpp:33-43
  o->ffd_stride = 3; o->ffd_min_samples = 2; o->ffd_min_foreground = 0.5f; o->ffd_min_pf = 0.25f; o->ffd_max_variance = 25.f;  // :45-58
  o->ms_kernel_size = 10; o->ms_max_iterations = 7; o->ms_stopping_criteria = 0.05f;  // include/MeanShift.hpp:16-25
  o->max_chunk = 0; o->max_scaled_h = 0; o->ms_mode = CRF_MS_DEFAULT;
}

int crf_model_load(const char* hp_dir, int hp_ntrees, const char* ffd_dir, int ffd_ntrees, crf_model** out) {
  if (!out || !hp_dir || !ffd_dir) return fail(CRF_ERR_ARG, "null argument");
  *out = nullptr;
  std::unique_ptr<crf_model> m(new crf_model());
  std::string err;
  int rc = load_model_dirs(hp_dir, hp_ntrees, ffd_dir, ffd_ntrees, m->m, err);
  if (rc) { std::fprintf(stderr, "(!) %s\n", err.c_str()); return fail(rc, err); }
  *out = m.release();
  return CRF_OK;
}

int crf_model_save_packed(const crf_model* m, const char* path) {
  if (!m || !path) return fail(CRF_ERR_ARG, "null argument");
  std::string err;
  int rc = save_model_packed(m->m, path, err);
  return rc ? fail(rc, err) : CRF_OK;
}

int crf_model_load_packed(const char* path, crf_model** out) {
  if (!out || !path) return fail(CRF_ERR_ARG, "null argument");
  *out = nullptr;
  std::unique_ptr<crf_model> m(new crf_model());
  std::string err;
  int rc = load_model_packed(path, m->m, err);
  if (rc) return fail(rc, err);
  *out = m.release();
  return CRF_OK;
}

// Forest<S>::load on its own (include/Forest.hpp:103-129): a model holding just the head-pose forest (kind 0) or just one
// facial-feature forest (kind 1, as pose forest 0).  Serves the Forest / Tree / ImageSample level of the reference interface;
// analyzeFace needs crf_model_load.
int crf_model_load_forest(const char* dir, int ntrees, int kind, crf_model** out) {
  if (!out || !dir || (kind != 0 && kind != 1)) return fail(CRF_ERR_ARG, "bad argument");
  *out = nullptr;
  std::unique_ptr<crf_model> m(new crf_model());
  std::string err;
  int rc;
  if (kind == 0) {
    rc = load_forest_dir(dir, ntrees, KIND_HEADPOSE, m->m.hp, err);
    m->m.hp_ntrees_cfg = ntrees;
  } else {
    m->m.jungle.resize(1);
    rc = load_forest_dir(dir, ntrees, KIND_MULTIPART, m->m.jungle[0], err);
    m->m.mp_ntrees_cfg = ntrees;
  }
  if (rc == CRF_OK) rc = validate_model(m->m, err);
  if (rc) { std::fprintf(stderr, "(!) %s\n", err.c_str()); return fail(rc, err); }
  *out = m.release();
  return CRF_OK;
}

// Tree<S>::load(Tree**, path) (include/Tree.hpp:193-237): a model holding the single tree of one archive file.
int crf_model_load_tree(const char* path, int kind, crf_model** out) {
  if (!out || !path || (kind != 0 && kind != 1)) return fail(CRF_ERR_ARG, "bad argument");
  *out = nullptr;
  std::unique_ptr<crf_model> m(new crf_model());
  std::string err;
  FlatForest& f = kind == 0 ? m->m.hp : (m->m.jungle.resize(1), m->m.jungle[0]);
  f.kind = kind == 0 ? KIND_HEADPOSE : KIND_MULTIPART;
  f.trees.resize(1);
  int rc = parse_tree_file(path, f.kind, f.trees[0], err);
  // Forest::load_tree rejects unfinished trees (include/Forest.hpp:142-152); Tree::load itself reloads them
  if (rc == CRF_OK) { (kind == 0 ? m->m.hp_ntrees_cfg : m->m.mp_ntrees_cfg) = 1; rc = validate_model(m->m, err); }
  if (rc) { std::fprintf(stderr, "  %s\n", err.c_str()); return fail(rc, err); }
  *out = m.release();
  return CRF_OK;
}

// ForestParam::features as the run-time configuration gives them (data/config_*.txt line 22; src/FaceForest.cpp:207 uses
// hp_forest_param.features for both forests).  Default: the list stored in the head-pose forest's archives.
int crf_model_set_features(crf_model* m, const int* features, int n) {
  if (!m) return fail(CRF_ERR_ARG, "null argument");
  std::string err;
  const int rc = set_model_features(m->m, features, n, err);
  return rc ? fail(rc, err) : CRF_OK;
}

int crf_model_get_features(const crf_model* m, int* features, int cap) {
  if (!m) return fail(CRF_ERR_ARG, "null argument");
  for (int i = 0; i < (int)m->m.features.size() && i < cap && features; i++) features[i] = m->m.features[i];
  return (int)m->m.features.size();
}

// Leaf payloads of one tree in pre-order leaf numbering, 44 floats per leaf:
//   head pose (which = -1): [object_id, hp_nsamples, hp_foreground, hp_labels[5]]                       (include/HeadPoseSample.hpp:144-162)
//   pose forest which >= 0: [object_id, mp_samples, mp_foreground, mp_parts_offset[10][2], mp_parts_variance[10], mp_prob_foreground[10]]  (include/MPSample.hpp:137-159)
int crf_model_leaf_dump(const crf_model* m, int which, int tree, float* out, int cap_leaves) {
  if (!m) return fail(CRF_ERR_ARG, "null argument");
  if (which >= (int)m->m.jungle.size()) return fail(CRF_ERR_ARG, "forest index out of range");
  const FlatForest& f = which < 0 ? m->m.hp : m->m.jungle[which];
  if (tree < 0 || tree >= (int)f.trees.size()) return fail(CRF_ERR_ARG, "tree index out of range");
  const FlatTree& t = f.trees[tree];
  const int n = which < 0 ? (int)t.hp_leaves.size() : (int)t.mp_leaves.size();
  for (int i = 0; i < n && i < cap_leaves && out; i++) {
    float* o = out + (size_t)i * 44;
    std::fill(o, o + 44, 0.f);
    if (which < 0) {
      const HpLeaf& L = t.hp_leaves[i];
      o[0] = (float)L.object_id; o[1] = (float)L.nsamples; o[2] = L.foreground;
      for (int j = 0; j < 5; j++) o[3 + j] = (float)L.labels[j];
    } else {
      const MpLeaf& L = t.mp_leaves[i];
      o[0] = (float)L.object_id; o[1] = (float)L.samples; o[2] = L.foreground;
      for (int j = 0; j < 10; j++) { o[3 + 2 * j] = (float)L.offset[j][0]; o[4 + 2 * j] = (float)L.offset[j][1]; o[23 + j] = L.variance[j]; o[33 + j] = L.prob_foreground[j]; }
    }
  }
  return n;
}

int crf_model_info(const crf_model* m, crf_model_info_t* info) {
  if (!m || !info) return fail(CRF_ERR_ARG, "null argument");
  std::memset(info, 0, sizeof *info);
  info->hp_trees = (int)m->m.hp.trees.size();
  for (auto& t : m->m.hp.trees) { info->hp_nodes += (int)t.nodes.size(); info->hp_leaves += (int)t.hp_leaves.size(); info->hp_max_depth = std::max(info->hp_max_depth, t.max_depth); }
  info->mp_forests = (int)m->m.jungle.size();
  for (auto& f : m->m.jungle)
    for (auto& t : f.trees) { info->mp_trees++; info->mp_nodes += (int)t.nodes.size(); info->mp_leaves += (int)t.mp_leaves.size(); info->mp_max_depth = std::max(info->mp_max_depth, t.max_depth); }
  info->patch_size = m->m.patch_size; info->face_size = m->m.face_size; info->num_channels = m->m.num_channels;
  info->hp_ntrees_cfg = m->m.hp_ntrees_cfg; info->mp_ntrees_cfg = m->m.mp_ntrees_cfg;
  return CRF_OK;
}

int crf_model_tree_dump(const crf_model* m, int which, int tree, int32_t* out, int cap_nodes) {
  if (!m) return fail(CRF_ERR_ARG, "null argument");
  if (which >= (int)m->m.jungle.size()) return fail(CRF_ERR_ARG, "forest index out of range");
  const FlatForest& f = which < 0 ? m->m.hp : m->m.jungle[which];
  if (tree < 0 || tree >= (int)f.trees.size()) return fail(CRF_ERR_ARG, "tree index out of range");
  const FlatTree& t = f.trees[tree];
  const int n = (int)t.nodes.size();
  for (int i = 0; i < n && i < cap_nodes && out; i++) {
    const FlatNode& nd = t.nodes[i];
    int32_t* o = out + (size_t)i * 16;
    const bool leaf = nd.leaf >= 0;
    o[0] = leaf; o[1] = nd.depth; o[2] = nd.channel;
    for (int k = 0; k < 4; k++) { o[3 + k] = nd.r1[k]; o[7 + k] = nd.r2[k]; }
    o[11] = nd.threshold_raw; o[12] = nd.left; o[13] = nd.right;
    o[14] = !leaf ? 0 : (which < 0 ? t.hp_leaves[nd.leaf].nsamples : t.mp_leaves[nd.leaf].samples);
    o[15] = i;
  }
  return n;
}

// Host-only self-check of the device image (no GPU needed): packs the forests as crf_ctx_create does and verifies that the
// three record forms of every node (wide DevSlot, compact DevSlot16, window DevSlotW) describe the same test, that children
// are adjacent, that window leaves loop onto themselves, and that max_extent is the largest rectangle extent.
// Returns the number of records checked (> 0) or a negative status; *max_extent_hp / *max_extent_ffd may be NULL.
int crf_model_check_packing(const crf_model* m, int* max_extent_hp, int* max_extent_ffd) {
  if (!m) return fail(CRF_ERR_ARG, "null argument");
  PackOptions po;
  std::string err;
  long long checked = 0;
  for (int which = 0; which < 2; which++) {
    PackedForest pf;
    std::vector<const FlatForest*> fs;
    if (which == 0) fs.push_back(&m->m.hp); else for (auto& f : m->m.jungle) fs.push_back(&f);
    const int rc = pack_forests(fs, which == 0 ? KIND_HEADPOSE : KIND_MULTIPART, po, pf, err);
    if (rc) return fail(rc, err);
    if (pf.slots.size() != pf.slots16.size() || pf.slots.size() != pf.slotsw.size()) return fail(CRF_ERR_STATE, "record arrays differ in length");
    int ext = 0;
    for (size_t i = 0; i < pf.slots.size(); i++) {
      const DevSlot& a = pf.slots[i]; const DevSlot16& b = pf.slots16[i]; const DevSlotW& w = pf.slotsw[i];
      const bool leaf16 = (b.r1 >> 26) & 1u, leafw = (w.tw >> 31) & 1u;
      if ((a.is_leaf != 0) != leaf16 || leaf16 != leafw) return fail(CRF_ERR_STATE, "leaf flags disagree");
      if (a.is_leaf) {
        if (b.child != a.child || (int32_t)w.m2 != a.child || w.child != (int32_t)i || (w.tw & 0xffffu) != 0x7fffu || w.px1 || w.px2 || w.yh1 || w.yh2 || w.m1)
          return fail(CRF_ERR_STATE, "leaf record mismatch");
      } else {
        const int x1 = a.a1 % kRowStride, y1 = a.a1 / kRowStride, x2 = a.a2 % kRowStride, y2 = a.a2 / kRowStride;
        const int h1 = ((a.ns1 - 1) * a.hs1 + a.hl1) / kRowStride, h2 = ((a.ns2 - 1) * a.hs2 + a.hl2) / kRowStride;
        const bool ok16 = (int)(b.r1 & 31) == x1 && (int)((b.r1 >> 5) & 31) == y1 && (int)((b.r1 >> 10) & 31) == a.w1 && (int)((b.r1 >> 15) & 31) == h1 &&
                          (int)((b.r1 >> 20) & 63) == a.ch && (int)(b.r2 & 31) == x2 && (int)((b.r2 >> 5) & 31) == y2 && (int)((b.r2 >> 10) & 31) == a.w2 &&
                          (int)((b.r2 >> 15) & 31) == h2 && (int)((b.r2 >> 20) & 0x3ff) - 256 == a.thr && b.child == a.child &&
                          (b.areas & 0xffff) == (uint32_t)a.w1 * h1 && (b.areas >> 16) == (uint32_t)a.w2 * h2;
        const bool okw = w.px1 == (uint32_t)a.ch * kWinPlaneBytes + x1 * 4u && w.px2 == (uint32_t)a.ch * kWinPlaneBytes + x2 * 4u &&
                         w.yh1 == ((uint32_t)y1 * kWinRowBytes | ((uint32_t)h1 * kWinRowBytes) << 16) && w.yh2 == ((uint32_t)y2 * kWinRowBytes | ((uint32_t)h2 * kWinRowBytes) << 16) &&
                         w.m1 == a.m1 && w.m2 == a.m2 && w.child == a.child && (int)(short)(w.tw & 0xffffu) == a.thr &&
                         ((w.tw >> 16) & 0xffu) == a.w1 * 4u && ((w.tw >> 24) & 0x7fu) == a.w2 * 4u &&
                         a.m1 == magic_for_area((uint32_t)a.w1 * h1) && a.m2 == magic_for_area((uint32_t)a.w2 * h2);
        if (!ok16 || !okw) return fail(CRF_ERR_STATE, "record forms disagree at slot " + std::to_string(i));
        if (a.child <= (int32_t)i || (size_t)a.child + 1 >= pf.slots.size()) return fail(CRF_ERR_STATE, "children are not laid out after their parent");
        ext = std::max(ext, std::max(std::max(x1 + a.w1, y1 + h1), std::max(x2 + a.w2, y2 + h2)));
      }
      checked++;
    }
    if (ext != pf.max_extent) return fail(CRF_ERR_STATE, "max_extent is not the largest rectangle extent");
    // internal-nodes-only form: walking it from every root must visit the same tests and end on the same leaves as the wide form
    if (!pf.nroot.empty()) {
      if (pf.nroot.size() != pf.roots.size()) return fail(CRF_ERR_STATE, "nroot and roots differ in length");
      std::vector<std::pair<int32_t, int32_t>> st;
      for (size_t t = 0; t < pf.roots.size(); t++) {
        st.assign(1, {pf.roots[t], pf.nroot[t]});
        while (!st.empty()) {
          const auto [si, ni] = st.back(); st.pop_back();
          const DevSlot& a = pf.slots[si];
          if (a.is_leaf) { if (ni != ~a.child) return fail(CRF_ERR_STATE, "DevSlotN leaf tag mismatch"); continue; }
          if (ni < 0 || (size_t)ni >= pf.slotsn.size()) return fail(CRF_ERR_STATE, "DevSlotN index out of range");
          const DevSlotN& r = pf.slotsn[ni]; const DevSlotW& w = pf.slotsw[si];
          const int32_t left = (int32_t)((uint32_t)r.left_thr << (32 - kSlotNChildBits)) >> (32 - kSlotNChildBits), thr = r.left_thr >> kSlotNChildBits;
          if ((r.pw1 & 0x3ffffu) != w.px1 || (r.pw2 & 0x3ffffu) != w.px2 || (r.pw1 >> 18) != ((w.tw >> 16) & 0xffu) || (r.pw2 >> 18) != ((w.tw >> 24) & 0x7fu) ||
              r.yh1 != w.yh1 || r.yh2 != w.yh2 || r.m1 != w.m1 || r.m2 != w.m2 || thr != std::min(255, std::max(-256, (int)a.thr)))
            return fail(CRF_ERR_STATE, "DevSlotN test mismatch at slot " + std::to_string(si));
          st.push_back({a.child, left});
          st.push_back({a.child + 1, r.right});
        }
      }
    }
    if (which == 0 && max_extent_hp) *max_extent_hp = ext;
    if (which == 1 && max_extent_ffd) *max_extent_ffd = ext;
  }
  return (int)std::min<long long>(checked, 0x7fffffff);
}

void crf_model_free(crf_model* m) { delete m; }

int crf_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
  return n;
}

void crf_ctx_destroy(crf_ctx* c) {
  if (!c) return;
  cudaSetDevice(c->device);
  for (auto& w : c->ws) if (w.stream) cudaStreamSynchronize(w.stream);
  if (c->tex_hp) cudaDestroyTextureObject(c->tex_hp);
  if (c->tex_mp) cudaDestroyTextureObject(c->tex_mp);
  if (c->tex_hp_n) cudaDestroyTextureObject(c->tex_hp_n);
  if (c->tex_mp_n) cudaDestroyTextureObject(c->tex_mp_n);
  if (c->tex_hp_wide) cudaDestroyTextureObject(c->tex_hp_wide);
  if (c->tex_mp_wide) cudaDestroyTextureObject(c->tex_mp_wide);
  Buf* all[] = {&c->d_hp_slotsn, &c->d_mp_slotsn, &c->d_hp_nroot, &c->d_mp_nroot, &c->d_hp_slotsw, &c->d_mp_slotsw, &c->d_hp_slots16, &c->d_mp_slots16, &c->d_hp_slots, &c->d_hp_roots, &c->d_hp_m, &c->d_mp_slots, &c->d_mp_roots, &c->d_mp_mask, &c->d_mp_leaf, &c->d_xs, &c->d_coef[0], &c->d_coef[1],
                &c->d_coef[2], &c->d_coef[3], &c->d_coef[4], &c->d_coef_sep[1], &c->d_coef_sep[2], &c->d_coef_sep[3], &c->d_coef_sep[4], &c->d_imgs[0], &c->d_imgs[1], &c->d_fd, &c->d_faces, &c->d_counters, &c->d_misc,
                &c->d_haar_stages, &c->d_haar_weak, &c->d_haar_feats, &c->d_haar_nodes, &c->d_haar_leaves, &c->d_haar_tilt, &c->d_haar_T, &c->d_haar_frames, &c->d_haar_S, &c->d_haar_Q, &c->d_haar_flags, &c->d_haar_list[0],
                &c->d_haar_list[1], &c->d_haar_rows, &c->d_haar_levels, &c->d_haar_counts, &c->d_haar_cand};
  for (Buf* b : all) b->release();
  for (auto& w : c->ws) {
    for (Buf* b : w.all) b->release();
    if (w.stream) cudaStreamDestroy(w.stream);
  }
  c->timer.destroy();
  for (int i = 0; i < 2; i++) { if (c->ev_copied[i]) cudaEventDestroy(c->ev_copied[i]); if (c->ev_consumed[i]) cudaEventDestroy(c->ev_consumed[i]); }
  if (c->copy_stream) cudaStreamDestroy(c->copy_stream);
  for (int i = 0; i < 2; i++) if (c->h_stage[i]) cudaFreeHost(c->h_stage[i]);
  delete c;
}

int crf_ctx_create(const crf_model* m, int device, const crf_options_t* opt, crf_ctx** out) {
  if (!out) return fail(CRF_ERR_ARG, "null argument");
  *out = nullptr;
  // m == NULL: a context without forests, for the stages that need none (feature channels, evalTest, MeanShift) —
  // ImageSample and MeanShift of the reference interface exist independently of any forest
  static const crf_model no_forests = [] { crf_model e; e.m.features = {0, 1, 2}; e.m.num_channels = 38; return e; }();
  if (!m) m = &no_forests;
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0) { cudaGetLastError(); return fail(CRF_ERR_CUDA, "no CUDA device: this library has no CPU fallback"); }
  if (device < 0 || device >= ndev) return fail(CRF_ERR_ARG, "device index out of range");
  // analyzeFace needs the head-pose forest and exactly 5 pose forests (poseT hard-codes 5 bins, src/FaceForest.cpp:216-222); a model
  // with one of the two (Forest<S>::load on its own) still gets a context for the Forest / ImageSample level of the interface
  const bool full = !m->m.hp.trees.empty() && m->m.jungle.size() == CRF_NUM_POSE_FORESTS;
  if (!m->m.hp.trees.empty() && !m->m.jungle.empty() && m->m.jungle.size() != CRF_NUM_POSE_FORESTS)
    return fail(CRF_ERR_UNSUPPORTED, "the facial-feature jungle must hold 5 pose forests (src/FaceForest.cpp:216-222)");
  CU(cudaSetDevice(device));
  crf_ctx* c = new crf_ctx();
  struct Guard { crf_ctx* c; ~Guard() { if (c) crf_ctx_destroy(c); } } guard{c};
  c->device = device;
  if (opt) c->opt = *opt; else crf_options_default(&c->opt);
  if (c->opt.hp_stride < 1 || c->opt.ffd_stride < 1) return fail(CRF_ERR_ARG, "strides must be >= 1");
  if (const char* v = std::getenv("CRF_TRAVERSE_VARIANT")) c->traverse_variant = (int)std::strtol(v, nullptr, 0);
  if (const char* v = std::getenv("CRF_WIN_TEX")) c->win_tex = (int)std::strtol(v, nullptr, 0);
  if (const char* v = std::getenv("CRF_WIN_FMT")) c->win_fmt = (int)std::strtol(v, nullptr, 0);
  if (const char* v = std::getenv("CRF_WIN_HP")) c->win_hp = (int)std::strtol(v, nullptr, 0);
  if (const char* v = std::getenv("CRF_WIN_FFD")) c->win_ffd = (int)std::strtol(v, nullptr, 0);
  if (const char* v = std::getenv("CRF_GABOR_FUSED")) c->gabor_fused = (int)std::strtol(v, nullptr, 0);
  if (const char* v = std::getenv("CRF_GABOR_QUANT_OLD")) c->gabor_quant_old = (int)std::strtol(v, nullptr, 0);
  if (const char* v = std::getenv("CRF_GABOR_BAND")) c->gabor_band = std::strtol(v, nullptr, 0) == 16 ? 16 : 32;
  if (const char* v = std::getenv("CRF_MS_VARIANT")) c->ms_variant = (int)std::strtol(v, nullptr, 0);
  c->ms_mode = c->opt.ms_mode == CRF_MS_EXACT ? CRF_MS_EXACT : CRF_MS_FAST;
  if (c->opt.ms_mode == CRF_MS_DEFAULT)
    if (const char* v = std::getenv("CRF_MS_MODE")) c->ms_mode = std::strcmp(v, "exact") == 0 ? CRF_MS_EXACT : CRF_MS_FAST;
  if (c->opt.ms_mode < CRF_MS_DEFAULT || c->opt.ms_mode > CRF_MS_FAST) return fail(CRF_ERR_ARG, "ms_mode must be CRF_MS_DEFAULT, CRF_MS_EXACT or CRF_MS_FAST");
  if (const char* v = std::getenv("CRF_STREAMS")) c->nstreams = std::strtol(v, nullptr, 0) == 2 ? 2 : 1;
  if (const char* v = std::getenv("CRF_HAAR_SPLIT")) {
    c->haar_split.clear();
    for (char* e = nullptr;; v = e + 1) {
      const long k = std::strtol(v, &e, 0);
      if (e == v) break;
      c->haar_split.push_back((int)k);
      if (*e != ',') break;
    }
  }
  for (auto& w : c->ws) CU(cudaStreamCreateWithFlags(&w.stream, cudaStreamNonBlocking));
  CU(cudaStreamCreateWithFlags(&c->copy_stream, cudaStreamNonBlocking));
  for (int i = 0; i < 2; i++) {
    CU(cudaEventCreateWithFlags(&c->ev_copied[i], cudaEventDisableTiming));
    CU(cudaEventCreateWithFlags(&c->ev_consumed[i], cudaEventDisableTiming));
  }
  PackOptions po;
  po.hp_min_foreground = c->opt.hp_min_foreground; po.ffd_min_samples = c->opt.ffd_min_samples; po.ffd_min_foreground = c->opt.ffd_min_foreground;
  po.ffd_min_pf = c->opt.ffd_min_pf; po.ffd_max_variance = c->opt.ffd_max_variance;
  std::string err;
  int rc = CRF_OK;
  if (!m->m.hp.trees.empty() && (rc = pack_forests({&m->m.hp}, KIND_HEADPOSE, po, c->hp, err))) return fail(rc, err);
  std::vector<const FlatForest*> jf;
  for (auto& f : m->m.jungle) jf.push_back(&f);
  if (!jf.empty() && (rc = pack_forests(jf, KIND_MULTIPART, po, c->mp, err))) return fail(rc, err);
  c->hp_ntrees = (int)c->hp.roots.size();
  c->mp_ntrees_cfg = std::max(m->m.mp_ntrees_cfg, 1);
  c->num_channels = m->m.num_channels;
  c->full_model = full;
  c->layout = layout_of(std::vector<int>(m->m.features.begin(), m->m.features.end()));
  if (c->layout.nplanes != c->num_channels) return fail(CRF_ERR_STATE, "feature list and plane count disagree");
  if (c->hp_ntrees > kMaxList || c->mp_ntrees_cfg > kMaxList) return fail(CRF_ERR_UNSUPPORTED, "forest size outside 1..128 trees");
  if ((rc = upload(c->d_hp_slots16, c->hp.slots16, c->w->stream)) || (rc = upload(c->d_mp_slots16, c->mp.slots16, c->w->stream))) return rc;
  if ((rc = upload(c->d_hp_slotsw, c->hp.slotsw, c->w->stream)) || (rc = upload(c->d_mp_slotsw, c->mp.slotsw, c->w->stream))) return rc;
  CU(cudaDeviceGetAttribute(&c->sm_count, cudaDevAttrMultiProcessorCount, device));
  {
    int optin = 0;
    CU(cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, device));
    c->win_smem_ok = optin >= kWinSmemBytes;   // otherwise dense grids stay on the global-gather kernels
  }
  if ((rc = upload(c->d_hp_slots, c->hp.slots, c->w->stream)) || (rc = upload(c->d_hp_roots, c->hp.roots, c->w->stream)) || (rc = upload(c->d_hp_m, c->hp.hp_m, c->w->stream)) ||
      (rc = upload(c->d_mp_slots, c->mp.slots, c->w->stream)) || (rc = upload(c->d_mp_roots, c->mp.roots, c->w->stream)) ||
      (rc = upload(c->d_mp_mask, c->mp.mp_mask, c->w->stream)) || (rc = upload(c->d_mp_leaf, c->mp.mp_leaf, c->w->stream)))
    return rc;
  // internal-nodes-only records (k_traverse_win2) + the map from a root's DevSlot index to its DevSlotN index
  for (int k = 0; k < 2; k++) {
    const PackedForest& pf = k ? c->mp : c->hp;
    if (pf.slotsn.empty() && pf.nroot.empty()) continue;
    std::vector<int32_t> map(pf.slots.size(), -1);
    for (size_t t = 0; t < pf.roots.size(); t++) map[pf.roots[t]] = pf.nroot[t];
    // a forest of one-leaf trees has no records at all: keep the texture bindable
    std::vector<DevSlotN> recs = pf.slotsn;
    if (recs.empty()) recs.emplace_back();
    if ((rc = upload(k ? c->d_mp_slotsn : c->d_hp_slotsn, recs, c->w->stream)) || (rc = upload(k ? c->d_mp_nroot : c->d_hp_nroot, map, c->w->stream))) return rc;
  }
  for (int k = 0; k < 6; k++) {   // node records as linear uint4 textures: window form (k < 2), wide form (2, 3), internal-only form (4, 5)
    cudaResourceDesc rd{}; rd.resType = cudaResourceTypeLinear;
    void* ptrs[6] = {c->d_hp_slotsw.p, c->d_mp_slotsw.p, c->d_hp_slots.p, c->d_mp_slots.p, c->d_hp_slotsn.p, c->d_mp_slotsn.p};
    const size_t counts[6] = {c->hp.slotsw.size(), c->mp.slotsw.size(), c->hp.slots.size(), c->mp.slots.size(),
                              c->d_hp_slotsn.p ? std::max<size_t>(c->hp.slotsn.size(), 1) : 0, c->d_mp_slotsn.p ? std::max<size_t>(c->mp.slotsn.size(), 1) : 0};
    cudaTextureObject_t* objs[6] = {&c->tex_hp, &c->tex_mp, &c->tex_hp_wide, &c->tex_mp_wide, &c->tex_hp_n, &c->tex_mp_n};
    if (counts[k] == 0) continue;   // a partial model has no records of the other kind
    rd.res.linear.devPtr = ptrs[k];
    rd.res.linear.desc = cudaCreateChannelDesc<uint4>();
    rd.res.linear.sizeInBytes = counts[k] * 32;
    cudaTextureDesc td{}; td.readMode = cudaReadModeElementType;
    CU(cudaCreateTextureObject(objs[k], &rd, &td, nullptr));
  }
  // Riemann abscissae of areaUnderCurve (src/face_utils.cpp:304-323) for the bins of src/FaceForest.cpp:216-222
  {
    float poseT[6];
    poseT[0] = -2.5; poseT[1] = -0.35; poseT[2] = -0.20; poseT[3] = -poseT[2]; poseT[4] = -poseT[1]; poseT[5] = -poseT[0];
    std::vector<double> xs;
    for (int j = 0; j < 5; j++) {
      c->ct.bin_begin[j] = (int)xs.size();
      const double step = 0.01;
      for (double x = poseT[j]; x < poseT[j + 1]; x += step) xs.push_back(x);
    }
    c->ct.bin_begin[5] = (int)xs.size();
    if ((rc = upload(c->d_xs, xs, c->w->stream))) return rc;
    c->ct.xs = c->d_xs.as<double>();
    c->ct.jungle_roots = c->d_mp_roots.as<int32_t>();
    for (int i = 0; i < 5 && i < (int)c->mp.forest_base.size(); i++) { c->ct.forest_base[i] = c->mp.forest_base[i]; c->ct.forest_ntrees[i] = c->mp.forest_ntrees[i]; }
    c->ct.ntrees_cfg = c->mp_ntrees_cfg;
    c->ct.list_cap = c->mp_ntrees_cfg;
  }
  {
    std::vector<float2> coef[5];
    build_gabor_bank(coef, c->gabor_width);
    const int expect[5] = {7, 9, 13, 19, 25};
    for (int i = 0; i < 5; i++) {
      if (c->gabor_width[i] != expect[i]) return fail(CRF_ERR_STATE, "unexpected Gabor kernel width");
      if ((rc = upload(c->d_coef[i], coef[i], c->w->stream))) return rc;
      if (i > 0) {
        std::vector<float> sep;
        build_gabor_sep(i, c->gabor_width[i], sep);
        if ((rc = upload(c->d_coef_sep[i], sep, c->w->stream))) return rc;
      }
    }
  }
  {
    ExpfTable t;
    for (int i = 0; i < 32; i++) {
      const double v = std::exp2((double)i / 32.0);
      unsigned long long u;
      std::memcpy(&u, &v, 8);
      t.tab[i] = u - ((unsigned long long)i << 47);
    }
    CU(cudaMemcpyToSymbolAsync(c_expf, &t, sizeof t, 0, cudaMemcpyHostToDevice, c->w->stream));
  }
  {
    size_t free_b = 0, total_b = 0;
    if (cudaMemGetInfo(&free_b, &total_b) == cudaSuccess) c->work_budget = std::min(c->work_budget, free_b / 2);
  }
  CU(cudaFuncSetAttribute(k_gabor_sep<25>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)GaborSepSmem<25>::bytes));
  CU(cudaFuncSetAttribute(k_gabor_sep<19>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)GaborSepSmem<19>::bytes));
  CU(cudaFuncSetAttribute(k_gabor_sep<13>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)GaborSepSmem<13>::bytes));
  CU(cudaFuncSetAttribute(k_gabor_sep<9>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)GaborSepSmem<9>::bytes));
  CU(cudaFuncSetAttribute(k_gabor_sep<25, 32>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)GaborSepSmem<25, 32>::bytes));
  CU(cudaFuncSetAttribute(k_gabor_sep<19, 32>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)GaborSepSmem<19, 32>::bytes));
  CU(cudaFuncSetAttribute(k_gabor_sep<13, 32>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)GaborSepSmem<13, 32>::bytes));
  CU(cudaFuncSetAttribute(k_gabor_sep<9, 32>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)GaborSepSmem<9, 32>::bytes));
  CU(cudaFuncSetAttribute(k_gabor_fused<25>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)GaborSepSmem<25>::bytes));
  CU(cudaFuncSetAttribute(k_gabor_fused<19>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)GaborSepSmem<19>::bytes));
  CU(cudaFuncSetAttribute(k_gabor_fused<13>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)GaborSepSmem<13>::bytes));
  CU(cudaFuncSetAttribute(k_gabor_fused<9>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)GaborSepSmem<9>::bytes));
  if (const char* v = std::getenv("CRF_CARVEOUT")) {   // experiment: shared-memory carveout (percent) of the traversal kernels
    const int pct = (int)std::strtol(v, nullptr, 0);
    CU(cudaFuncSetAttribute(k_traverse16<10, false>, cudaFuncAttributePreferredSharedMemoryCarveout, pct));
    CU(cudaFuncSetAttribute(k_traverse16<15, false>, cudaFuncAttributePreferredSharedMemoryCarveout, pct));
  }
  CU(cudaFuncSetAttribute(k_plain_channels, cudaFuncAttributeMaxDynamicSharedMemorySize, (CRF_MAX_SCALED_H + 2) * 127 * 3));
  CU(cudaFuncSetAttribute(k_hp_reduce_compose, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kHpSmem));
  CU(cudaFuncSetAttribute(k_meanshift<2, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)MsGeom<false>::smem));
  CU(cudaFuncSetAttribute(k_meanshift<3, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)MsGeom<false>::smem));
  CU(cudaFuncSetAttribute(k_meanshift<4, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)MsGeom<false>::smem));
  CU(cudaFuncSetAttribute(k_meanshift<3, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)MsGeom<true>::smem));
  if ((rc = c->d_counters.reserve(sizeof(unsigned long long) * CNT_NUM))) return rc;
  CU(cudaMemsetAsync(c->d_counters.p, 0, sizeof(unsigned long long) * CNT_NUM, c->w->stream));
  if ((rc = c->d_misc.reserve(4096))) return rc;
  CU(cudaStreamSynchronize(c->w->stream));
  guard.c = nullptr;
  *out = c;
  return CRF_OK;
}

int crf_ctx_set_profiling(crf_ctx* c, int on) {
  if (!c) return fail(CRF_ERR_STATE, "context is not initialised");
  c->timer.on = on & 1;
  c->counting = (on & 2) != 0;
  return CRF_OK;
}

int crf_ctx_stage_ms(crf_ctx* c, float ms[CRF_NUM_STAGES], int launches[CRF_NUM_STAGES]) {
  if (!c) return fail(CRF_ERR_STATE, "context is not initialised");
  for (int i = 0; i < CRF_NUM_STAGES; i++) { if (ms) ms[i] = c->timer.ms[i]; if (launches) launches[i] = c->timer.launches[i]; }
  return CRF_OK;
}

int crf_ctx_counters(crf_ctx* c, crf_counters_t* out) {
  if (!c || !out) return fail(CRF_ERR_ARG, "null argument");
  *out = c->cnt;
  return CRF_OK;
}

int crf_ctx_reset_counters(crf_ctx* c) {
  if (!c) return fail(CRF_ERR_STATE, "context is not initialised");
  c->cnt = crf_counters_t{};
  for (int i = 0; i < CRF_NUM_STAGES; i++) { c->timer.ms[i] = 0; c->timer.launches[i] = 0; }
  return CRF_OK;
}

void* crf_ctx_stream(crf_ctx* c) { return c ? (void*)c->ws[0].stream : nullptr; }

int crf_host_alloc(void** p, size_t bytes) {
  if (!p) return fail(CRF_ERR_ARG, "null argument");
  CU(cudaHostAlloc(p, bytes, cudaHostAllocDefault));
  return CRF_OK;
}
void crf_host_free(void* p) { if (p) cudaFreeHost(p); }

int crf_analyze_faces(crf_ctx* c, const uint8_t* bgr, int rows, int cols, size_t step, const crf_rect_t* boxes, int n, crf_face_t* out) {
  std::vector<int> zero((size_t)std::max(n, 0), 0);
  const crf_image_t im{bgr, rows, cols, step};
  return analyze_host(c, &im, 1, boxes, zero.data(), n, out, false);
}

int crf_analyze_batch_mixed(crf_ctx* c, const crf_image_t* images, int n_images, const crf_rect_t* boxes, const int* image_of_box, int n, crf_face_t* out) {
  if (!image_of_box && n > 0) return fail(CRF_ERR_ARG, "null argument");
  if (n_images > 0 && !images) return fail(CRF_ERR_ARG, "null argument");
  if (int rc = image_args(images, n_images)) return rc;
  return analyze_host(c, images, n_images, boxes, image_of_box, n, out, false);
}

int crf_analyze_batch(crf_ctx* c, const uint8_t* const* images, int n_images, int rows, int cols, size_t step, const crf_rect_t* boxes,
                      const int* image_of_box, int n, crf_face_t* out) {
  if (!image_of_box && n > 0) return fail(CRF_ERR_ARG, "null argument");
  std::vector<crf_image_t> v;
  return analyze_host(c, same_size(images, n_images, rows, cols, step, v), n_images, boxes, image_of_box, n, out, false);
}

// n crops back to back in bgr_batch, one frame per crop
static const crf_image_t* crop_frames(const uint8_t* bgr_batch, int n, int rows, int cols, std::vector<crf_image_t>& v) {
  v.resize((size_t)std::max(n, 0));
  for (int i = 0; i < n; i++) v[(size_t)i] = crf_image_t{bgr_batch + (size_t)i * rows * cols * 3, rows, cols, (size_t)cols * 3};
  return v.data();
}

static int crops_host(crf_ctx* c, const uint8_t* bgr_batch, int n, int rows, int cols, crf_face_t* out, bool hp_only) {
  if (n < 0 || (n > 0 && !bgr_batch)) return fail(CRF_ERR_ARG, "null argument");
  std::vector<crf_image_t> imgs;
  std::vector<crf_rect_t> boxes((size_t)std::max(n, 0), crf_rect_t{0, 0, cols, rows});
  return analyze_host(c, crop_frames(bgr_batch, n, rows, cols, imgs), n, boxes.data(), nullptr, n, out, hp_only);
}

int crf_analyze_crops(crf_ctx* c, const uint8_t* bgr_batch, int n, int rows, int cols, crf_face_t* out) { return crops_host(c, bgr_batch, n, rows, cols, out, false); }
int crf_headpose_crops(crf_ctx* c, const uint8_t* bgr_batch, int n, int rows, int cols, crf_face_t* out) { return crops_host(c, bgr_batch, n, rows, cols, out, true); }

int crf_analyze_crops_device(crf_ctx* c, const uint8_t* d_bgr_batch, int n, int rows, int cols, crf_face_t* d_out, int headpose_only) {
  if (!c) return fail(CRF_ERR_STATE, "context is not initialised");
  if (!c->full_model) return fail(CRF_ERR_STATE, "analyzeFace needs the head-pose forest and the 5 pose forests; this context holds a single forest");
  if (n < 0 || (n > 0 && (!d_bgr_batch || !d_out))) return fail(CRF_ERR_ARG, "null argument");
  if (n == 0) return CRF_OK;
  CU(cudaSetDevice(c->device));
  std::vector<FaceDesc> descs((size_t)n);
  const size_t img_bytes = (size_t)rows * cols * 3;
  int Hmax = 0;
  for (int i = 0; i < n; i++) {
    int rc = make_desc(c, rows, cols, (size_t)cols * 3, (size_t)i * img_bytes, crf_rect_t{0, 0, cols, rows}, descs[i]);
    if (rc) return rc;
    Hmax = std::max(Hmax, descs[i].H);
  }
  return analyze_resident(c, descs, Hmax, d_bgr_batch, d_out, headpose_only != 0);
}

// ---------------------------------------------------------------------------------------------
// Several GPUs behind one caller (SURVEY 8e): one context and one host thread per GPU, contiguous shards of the faces
// (cut at frame boundaries when the boxes are grouped by frame), a full forest replica per GPU, results written straight
// into the caller's array.  No collective: faces are independent, only the records come back.
// ---------------------------------------------------------------------------------------------
struct crf_multi {
  std::vector<crf_ctx*> ctx;
};

void crf_multi_destroy(crf_multi* m) {
  if (!m) return;
  for (crf_ctx* c : m->ctx) crf_ctx_destroy(c);
  delete m;
}

int crf_multi_create(const crf_model* model, const int* devices, int n_devices, const crf_options_t* opt, crf_multi** out) {
  if (!out || !model || n_devices < 0) return fail(CRF_ERR_ARG, "bad argument");
  *out = nullptr;
  std::vector<int> dev;
  if (!devices || n_devices == 0) {
    const int n = crf_device_count();
    if (n < 1) return fail(CRF_ERR_CUDA, "no CUDA device: this library has no CPU fallback");
    for (int i = 0; i < n; i++) dev.push_back(i);
  } else dev.assign(devices, devices + n_devices);
  std::unique_ptr<crf_multi, void (*)(crf_multi*)> m(new crf_multi(), crf_multi_destroy);
  for (int d : dev) {
    crf_ctx* c = nullptr;
    const int rc = crf_ctx_create(model, d, opt, &c);
    if (rc) return rc;
    m->ctx.push_back(c);
  }
  *out = m.release();
  return CRF_OK;
}

int crf_multi_device_count(const crf_multi* m) { return m ? (int)m->ctx.size() : 0; }
crf_ctx* crf_multi_ctx(crf_multi* m, int i) { return m && i >= 0 && i < (int)m->ctx.size() ? m->ctx[(size_t)i] : nullptr; }

static int multi_run(crf_multi* m, const crf_image_t* images, int n_images, const crf_rect_t* boxes, const int* image_of_box, int n, crf_face_t* out,
                     bool headpose_only) {
  if (!m || m->ctx.empty()) return fail(CRF_ERR_STATE, "context is not initialised");
  if (n < 0 || (n > 0 && (!images || !boxes || !out))) return fail(CRF_ERR_ARG, "null argument");
  const int G = (int)m->ctx.size();
  // shard g = faces [cut[g], cut[g + 1]): even split, moved to the nearest frame boundary when consecutive boxes share frames
  std::vector<int> cut((size_t)G + 1, n);
  cut[0] = 0;
  for (int g = 1; g < G; g++) {
    int c = (int)((long long)n * g / G);
    if (image_of_box && c > 0 && c < n) {
      int lo = c, hi = c;
      while (lo > cut[(size_t)g - 1] && image_of_box[lo] == image_of_box[lo - 1]) lo--;
      while (hi < n && image_of_box[hi] == image_of_box[hi - 1]) hi++;
      // take the closer boundary unless that would empty a shard
      c = (c - lo <= hi - c && lo > cut[(size_t)g - 1]) ? lo : (hi < n ? hi : (lo > cut[(size_t)g - 1] ? lo : c));
    }
    cut[(size_t)g] = std::max(c, cut[(size_t)g - 1]);
  }
  // all-or-nothing: every shard's boxes are checked before any shard writes into out
  for (int g = 0; g < G; g++) {
    const int f0 = cut[(size_t)g], f1 = cut[(size_t)g + 1];
    if (f1 > f0 && box_args(image_of_box ? images : images + f0, image_of_box ? n_images : f1 - f0, boxes + f0, image_of_box ? image_of_box + f0 : nullptr, f1 - f0))
      return fail(CRF_ERR_ARG, "GPU shard " + std::to_string(g) + ": " + g_last_error);
  }
  std::vector<int> rcs((size_t)G, CRF_OK);
  std::vector<std::string> errs((size_t)G);
  auto work = [&](int g) {
    const int f0 = cut[(size_t)g], f1 = cut[(size_t)g + 1];
    if (f1 <= f0) return;
    // a shard names its frames through the caller's image_of_box; crops (image_of_box == NULL) are one frame per face
    rcs[(size_t)g] = analyze_host(m->ctx[(size_t)g], image_of_box ? images : images + f0, image_of_box ? n_images : f1 - f0, boxes + f0,
                                  image_of_box ? image_of_box + f0 : nullptr, f1 - f0, out + f0, headpose_only);
    if (rcs[(size_t)g]) errs[(size_t)g] = g_last_error;   // thread-local in the worker: hand it to the caller
  };
  std::vector<std::thread> th;
  for (int g = 1; g < G; g++) th.emplace_back(work, g);
  work(0);
  for (auto& t : th) t.join();
  for (int g = 0; g < G; g++)
    if (rcs[(size_t)g]) return fail(rcs[(size_t)g], "GPU shard " + std::to_string(g) + ": " + errs[(size_t)g]);
  return CRF_OK;
}

int crf_multi_analyze_batch_mixed(crf_multi* m, const crf_image_t* images, int n_images, const crf_rect_t* boxes, const int* image_of_box, int n,
                                  crf_face_t* out) {
  if (!image_of_box && n > 0) return fail(CRF_ERR_ARG, "null argument");
  if (n_images > 0 && !images) return fail(CRF_ERR_ARG, "null argument");
  if (int rc = image_args(images, n_images)) return rc;
  return multi_run(m, images, n_images, boxes, image_of_box, n, out, false);
}

int crf_multi_analyze_batch(crf_multi* m, const uint8_t* const* images, int n_images, int rows, int cols, size_t step, const crf_rect_t* boxes,
                            const int* image_of_box, int n, crf_face_t* out) {
  if (!image_of_box && n > 0) return fail(CRF_ERR_ARG, "null argument");
  std::vector<crf_image_t> v;
  return multi_run(m, same_size(images, n_images, rows, cols, step, v), n_images, boxes, image_of_box, n, out, false);
}

int crf_multi_analyze_crops(crf_multi* m, const uint8_t* bgr_batch, int n, int rows, int cols, crf_face_t* out, int headpose_only) {
  if (n < 0 || (n > 0 && !bgr_batch)) return fail(CRF_ERR_ARG, "null argument");
  std::vector<crf_image_t> imgs;
  std::vector<crf_rect_t> boxes((size_t)std::max(n, 0), crf_rect_t{0, 0, cols, rows});
  return multi_run(m, crop_frames(bgr_batch, n, rows, cols, imgs), n, boxes.data(), nullptr, n, out, headpose_only != 0);
}

// ---------------------------------------------------------------------------------------------
// Stage-level entry points
// ---------------------------------------------------------------------------------------------
int crf_stage_gray_resize(crf_ctx* c, const uint8_t* bgr, int rows, int cols, size_t step, crf_rect_t box, uint8_t* scaled, int* W, int* H) {
  if (!c) return fail(CRF_ERR_STATE, "context is not initialised");
  if (!bgr || !scaled) return fail(CRF_ERR_ARG, "null argument");
  CU(cudaSetDevice(c->device));
  FaceDesc d;
  int rc = make_desc(c, rows, cols, step, 0, box, d);
  if (rc) return rc;
  Plan p; p.n = 1; p.Hmax = d.H; p.need_gabor = false; p.need_hp = false; p.need_ffd = false;
  if ((rc = ensure(c, p)) || (rc = c->d_fd.reserve(sizeof d)) || (rc = c->d_imgs[0].reserve((size_t)rows * step))) return rc;
  CU(cudaMemcpyAsync(c->d_fd.p, &d, sizeof d, cudaMemcpyHostToDevice, c->w->stream));
  CU(cudaMemcpyAsync(c->d_imgs[0].p, bgr, (size_t)rows * step, cudaMemcpyHostToDevice, c->w->stream));
  if ((rc = launch_resize(c, c->d_fd.as<FaceDesc>(), 1, d.H, c->d_imgs[0].as<uint8_t>()))) return rc;
  CU(cudaMemcpy2DAsync(scaled, d.W, c->w->d_scaled.p, 128, d.W, d.H, cudaMemcpyDeviceToHost, c->w->stream));
  CU(cudaStreamSynchronize(c->w->stream));
  if (W) *W = d.W;
  if (H) *H = d.H;
  return CRF_OK;
}

static int stage_upload_scaled(crf_ctx* c, const uint8_t* scaled, int W, int H, int nplanes, bool gabor, bool want_u8, bool hp, bool ffd, int tree_cap,
                               int hp_stride, int ffd_stride) {
  if (W <= kPatch || W > 125 || H <= kPatch || H > CRF_MAX_SCALED_H) return fail(CRF_ERR_ARG, "plane size outside (31,125] x (31,521]");
  FaceDesc d{};
  d.W = W; d.H = H; d.bw = W; d.bh = H; d.scale = 125.f / W; d.scale_x = d.scale_y = 1.0;
  Plan p; p.n = 1; p.Hmax = H; p.nplanes = nplanes; p.need_gabor = gabor; p.want_u8 = want_u8; p.need_hp = hp; p.need_ffd = ffd; p.tree_cap = tree_cap;
  p.vote_factor = kParts;
  p.hp_stride = hp_stride; p.ffd_stride = ffd_stride;
  int rc;
  if ((rc = ensure(c, p)) || (rc = c->d_fd.reserve(sizeof d))) return rc;
  CU(cudaMemcpyAsync(c->d_fd.p, &d, sizeof d, cudaMemcpyHostToDevice, c->w->stream));
  if (scaled) CU(cudaMemcpy2DAsync(c->w->d_scaled.p, 128, scaled, W, W, H, cudaMemcpyHostToDevice, c->w->stream));
  return CRF_OK;
}

static int stage_download_planes(crf_ctx* c, int nplanes, int W, int H, uint8_t* planes_u8, uint32_t* integrals) {
  if (planes_u8) CU(cudaMemcpyAsync(planes_u8, c->w->d_u8planes.p, (size_t)nplanes * W * H, cudaMemcpyDeviceToHost, c->w->stream));
  if (integrals)
    for (int pl = 0; pl < nplanes; pl++)
      CU(cudaMemcpy2DAsync(integrals + (size_t)pl * (H + 1) * (W + 1), (size_t)(W + 1) * 4, c->w->d_int32.as<uint32_t>() + (size_t)pl * c->w->plane_stride,
                           (size_t)kRowStride * 4, (size_t)(W + 1) * 4, H + 1, cudaMemcpyDeviceToHost, c->w->stream));
  CU(cudaStreamSynchronize(c->w->stream));
  return CRF_OK;
}

// ImageSample::extractFeatureChannels for an explicit feature list (src/ImageSample.cpp:77-90): the ids are sorted, then each
// appends its planes (include/FeatureChannelFactory.hpp:35-183).  Returns the plane count (> 0) or a negative status.
int crf_stage_feature_channels(crf_ctx* c, const uint8_t* scaled, int W, int H, const int* features, int nfeatures, uint8_t* planes_u8, uint32_t* integrals) {
  if (!c) return fail(CRF_ERR_STATE, "context is not initialised");
  if (!scaled || !features || nfeatures < 1 || nfeatures > 6) return fail(CRF_ERR_ARG, "bad argument");
  std::vector<int> f(features, features + nfeatures);
  std::sort(f.begin(), f.end());
  for (size_t i = 0; i < f.size(); i++)
    if (planes_of_feature(f[i]) == 0 || (i > 0 && f[i] == f[i - 1])) return fail(CRF_ERR_ARG, "feature ids must be distinct values of 0..5");
  const ChannelLayout L = layout_of(f);
  CU(cudaSetDevice(c->device));
  int rc = stage_upload_scaled(c, scaled, W, H, L.nplanes, L.gabor_first >= 0, true, false, false, 1, 4, 3);
  if (rc) return rc;
  if ((rc = launch_channels(c, c->d_fd.as<FaceDesc>(), 1, H, L, true))) return rc;
  if ((rc = stage_download_planes(c, L.nplanes, W, H, planes_u8, integrals))) return rc;
  return L.nplanes;
}

static int stage_fixed_features(crf_ctx* c, const uint8_t* scaled, int W, int H, std::initializer_list<int> feats, uint8_t* planes_u8, uint32_t* integrals) {
  const std::vector<int> f(feats);
  const int rc = crf_stage_feature_channels(c, scaled, W, H, f.data(), (int)f.size(), planes_u8, integrals);
  return rc < 0 ? rc : CRF_OK;
}
int crf_stage_channels(crf_ctx* c, const uint8_t* scaled, int W, int H, uint8_t* planes_u8, uint32_t* integrals) { return stage_fixed_features(c, scaled, W, H, {0, 1, 2}, planes_u8, integrals); }
int crf_stage_minmax(crf_ctx* c, const uint8_t* scaled, int W, int H, uint8_t* planes_u8, uint32_t* integrals) { return stage_fixed_features(c, scaled, W, H, {3}, planes_u8, integrals); }
int crf_stage_norm(crf_ctx* c, const uint8_t* scaled, int W, int H, uint8_t* plane_u8, uint32_t* integral) { return stage_fixed_features(c, scaled, W, H, {5}, plane_u8, integral); }
int crf_stage_canny(crf_ctx* c, const uint8_t* scaled, int W, int H, uint8_t* plane_u8, uint32_t* integral) { return stage_fixed_features(c, scaled, W, H, {4}, plane_u8, integral); }

// planes -> integral stack of one synthetic face
static int stage_planes_to_stack(crf_ctx* c, const uint8_t* planes_u8, int C, int W, int H, bool hp, bool ffd, int tree_cap, int hp_stride, int ffd_stride) {
  if (!planes_u8) return fail(CRF_ERR_ARG, "null argument");
  if (C < 1 || C > 64) return fail(CRF_ERR_ARG, "plane count outside 1..64");
  int rc = stage_upload_scaled(c, nullptr, W, H, C, false, true, hp, ffd, tree_cap, hp_stride, ffd_stride);
  if (rc) return rc;
  CU(cudaMemcpyAsync(c->w->d_u8planes.p, planes_u8, (size_t)C * W * H, cudaMemcpyHostToDevice, c->w->stream));
  k_integral_from_u8<<<dim3(C, 1), 128, 0, c->w->stream>>>(c->w->d_u8planes.as<uint8_t>(), W, H, c->w->d_stacks.as<stack_t>(), c->w->stack_fs, c->w->plane_stride);
  KCHECK(); count_launch(c, CRF_STAGE_PLAIN);
  return CRF_OK;
}

static int max_channel_used(const PackedForest& f) {
  int m = 0;
  for (const DevSlot& s : f.slots) if (!s.is_leaf) m = std::max(m, (int)s.ch);
  return m;
}

static int stage_set_list(crf_ctx* c, const int* tree_forest, const int* tree_index, int ntrees) {
  if (!tree_forest || !tree_index || ntrees < 0 || ntrees > kMaxList) return fail(CRF_ERR_ARG, "bad composed forest");
  std::vector<int32_t> list((size_t)kMaxList, 0);
  for (int i = 0; i < ntrees; i++) {
    if (tree_forest[i] < 0 || tree_forest[i] >= (int)c->mp.forest_ntrees.size() || tree_index[i] < 0 || tree_index[i] >= c->mp.forest_ntrees[tree_forest[i]])
      return fail(CRF_ERR_ARG, "bad composed forest");
    list[i] = c->mp.roots[c->mp.forest_base[tree_forest[i]] + tree_index[i]];
  }
  CU(cudaMemcpyAsync(c->w->d_face_roots.p, list.data(), kMaxList * 4, cudaMemcpyHostToDevice, c->w->stream));
  CU(cudaMemcpyAsync(c->w->d_face_ntrees.p, &ntrees, 4, cudaMemcpyHostToDevice, c->w->stream));
  CU(cudaStreamSynchronize(c->w->stream));  // `list` and `ntrees` are stack/local host memory
  return CRF_OK;
}

int crf_stage_eval_forest(crf_ctx* c, int which, const int* tree_forest, const int* tree_index, int ntrees, const uint8_t* planes_u8, int C, int W, int H,
                          int stride, int32_t* leaf_ids) {
  if (!c) return fail(CRF_ERR_STATE, "context is not initialised");
  if (!leaf_ids || stride < 1) return fail(CRF_ERR_ARG, "bad argument");
  CU(cudaSetDevice(c->device));
  const bool hp = which < 0;
  const PackedForest& pf = hp ? c->hp : c->mp;
  if (pf.slots.empty()) return fail(CRF_ERR_STATE, "the context's model does not hold that forest");
  if (max_channel_used(pf) >= C) return fail(CRF_ERR_ARG, "forest reads a channel the planes do not provide");
  const int nt = hp ? c->hp_ntrees : ntrees;
  int rc = stage_planes_to_stack(c, planes_u8, C, W, H, hp, !hp, std::max(nt, 1), stride, stride);
  if (rc) return rc;
  if (!hp && (rc = stage_set_list(c, tree_forest, tree_index, ntrees))) return rc;
  if ((rc = launch_traverse(c, c->d_fd.as<FaceDesc>(), 1, H, hp, stride, c->d_hp_roots.as<int32_t>(), c->hp_ntrees, std::max(nt, 1)))) return rc;
  const size_t n = (size_t)patches_1d(W, stride) * patches_1d(H, stride) * nt;
  std::vector<int32_t> raw(n);
  if (n) CU(cudaMemcpyAsync(raw.data(), hp ? c->w->d_hp_leaf.p : c->w->d_ffd_leaf.p, n * 4, cudaMemcpyDeviceToHost, c->w->stream));
  CU(cudaStreamSynchronize(c->w->stream));
  for (size_t i = 0; i < n; i++) leaf_ids[i] = pf.leaf_oid[(size_t)raw[i]];
  c->timer.collect();
  return pull_counters(c);
}

// Forest<S>::evaluateMT for explicit patch origins (the per-sample level: one call of the reference per patch).
// patch_xy: npatches x (x, y); leaf_ids: [patch][tree] Boost object ids.
int crf_stage_eval_patches(crf_ctx* c, int which, const int* tree_forest, const int* tree_index, int ntrees, const uint8_t* planes_u8, int C, int W, int H,
                           const int* patch_xy, int npatches, int32_t* leaf_ids) {
  if (!c) return fail(CRF_ERR_STATE, "context is not initialised");
  if (!leaf_ids || !patch_xy || npatches < 0) return fail(CRF_ERR_ARG, "bad argument");
  CU(cudaSetDevice(c->device));
  const bool hp = which < 0;
  const PackedForest& pf = hp ? c->hp : c->mp;
  if (pf.slots.empty()) return fail(CRF_ERR_STATE, "the context's model does not hold that forest");
  if (max_channel_used(pf) >= C) return fail(CRF_ERR_ARG, "forest reads a channel the planes do not provide");
  for (int i = 0; i < npatches; i++)
    if (patch_xy[2 * i] < 0 || patch_xy[2 * i + 1] < 0 || patch_xy[2 * i] + kPatch > W || patch_xy[2 * i + 1] + kPatch > H) return fail(CRF_ERR_ARG, "patch outside the face");
  const int nt = hp ? c->hp_ntrees : ntrees;
  if (npatches == 0 || nt == 0) return CRF_OK;
  int rc = stage_planes_to_stack(c, planes_u8, C, W, H, false, false, std::max(nt, 1), 1, 1);
  if (rc) return rc;
  if (!hp && (rc = stage_set_list(c, tree_forest, tree_index, ntrees))) return rc;
  Buf d_p, d_leaf;
  struct Free { Buf* b[2]; ~Free() { for (Buf* x : b) x->release(); } } fr{{&d_p, &d_leaf}};
  if ((rc = d_p.reserve((size_t)npatches * 8)) || (rc = d_leaf.reserve((size_t)npatches * nt * 4))) return rc;
  CU(cudaMemcpyAsync(d_p.p, patch_xy, (size_t)npatches * 8, cudaMemcpyHostToDevice, c->w->stream));
  TraverseArgs a{};
  a.stacks = c->w->d_stacks.as<stack_t>(); a.stack_face_stride = c->w->stack_fs; a.plane_stride = c->w->plane_stride;
  a.slots = hp ? c->d_hp_slots.as<DevSlot>() : c->d_mp_slots.as<DevSlot>();
  if (hp) { a.roots = c->d_hp_roots.as<int32_t>(); a.ntrees = c->hp_ntrees; }
  else { a.face_roots = c->w->d_face_roots.as<int32_t>(); a.face_ntrees = c->w->d_face_ntrees.as<int32_t>(); }
  a.leaf_out = d_leaf.as<int32_t>();
  k_traverse_patches<<<(npatches * nt + 127) / 128, 128, 0, c->w->stream>>>(a, d_p.as<int2>(), npatches);
  KCHECK(); count_launch(c, hp ? CRF_STAGE_HP_TRAVERSE : CRF_STAGE_FFD_TRAVERSE);
  std::vector<int32_t> raw((size_t)npatches * nt);
  CU(cudaMemcpyAsync(raw.data(), d_leaf.p, raw.size() * 4, cudaMemcpyDeviceToHost, c->w->stream));
  CU(cudaStreamSynchronize(c->w->stream));
  for (size_t i = 0; i < raw.size(); i++) leaf_ids[i] = pf.leaf_oid[(size_t)raw[i]];
  return CRF_OK;
}

// ImageSample::evalTest(SimplePatchFeature, Rect) (src/ImageSample.cpp:30-64) for n tests on caller-supplied planes:
// tests = n x {channel, x1, y1, w1, h1, x2, y2, w2, h2, patch_x, patch_y}; out[i] = mean(rect1) - mean(rect2).
int crf_stage_eval_tests(crf_ctx* c, const uint8_t* planes_u8, int C, int W, int H, const int* tests, int n, int* out) {
  if (!c) return fail(CRF_ERR_STATE, "context is not initialised");
  if (n < 0 || (n > 0 && (!tests || !out))) return fail(CRF_ERR_ARG, "bad argument");
  if (n == 0) return CRF_OK;
  for (int i = 0; i < n; i++) {
    const int* t = tests + (size_t)i * 11;
    if (t[0] < 0 || t[0] >= C) return fail(CRF_ERR_ARG, "test reads a channel the planes do not provide");
    for (int k = 0; k < 2; k++) {
      const int x = t[9] + t[1 + 4 * k], y = t[10] + t[2 + 4 * k], w = t[3 + 4 * k], h = t[4 + 4 * k];
      if (w < 1 || h < 1 || x < 0 || y < 0 || x + w > W || y + h > H) return fail(CRF_ERR_ARG, "test rectangle outside the face");
    }
  }
  CU(cudaSetDevice(c->device));
  int rc = stage_planes_to_stack(c, planes_u8, C, W, H, false, false, 1, 1, 1);
  if (rc) return rc;
  Buf d_t, d_o;
  struct Free { Buf* b[2]; ~Free() { for (Buf* x : b) x->release(); } } fr{{&d_t, &d_o}};
  if ((rc = d_t.reserve((size_t)n * 44)) || (rc = d_o.reserve((size_t)n * 4))) return rc;
  CU(cudaMemcpyAsync(d_t.p, tests, (size_t)n * 44, cudaMemcpyHostToDevice, c->w->stream));
  k_eval_tests<<<(n + 127) / 128, 128, 0, c->w->stream>>>(c->w->d_stacks.as<stack_t>(), c->w->plane_stride, d_t.as<int>(), n, d_o.as<int>());
  KCHECK(); count_launch(c, CRF_STAGE_PLAIN);
  CU(cudaMemcpyAsync(out, d_o.p, (size_t)n * 4, cudaMemcpyDeviceToHost, c->w->stream));
  CU(cudaStreamSynchronize(c->w->stream));
  return CRF_OK;
}

int crf_stage_eval_tests_sum(crf_ctx* c, const uint8_t* planes_u8, int C, int W, int H, const int* tests, int n, int* out) {
  if (!c) return fail(CRF_ERR_STATE, "context is not initialised");
  if (n < 0 || C < 1 || W < 1 || H < 1 || !planes_u8 || (n > 0 && (!tests || !out))) return fail(CRF_ERR_ARG, "bad argument");
  if (n == 0) return CRF_OK;
  for (int i = 0; i < n; i++) {
    const int* t = tests + (size_t)i * 11;
    if (t[0] < 0 || t[0] >= C) return fail(CRF_ERR_ARG, "test reads a channel the planes do not provide");
    for (int k = 0; k < 2; k++) {
      const int x = t[9] + t[1 + 4 * k], y = t[10] + t[2 + 4 * k], w = t[3 + 4 * k], h = t[4 + 4 * k];
      if (w < 1 || h < 1 || x < 0 || y < 0 || x + w > W || y + h > H) return fail(CRF_ERR_ARG, "test rectangle outside the face");
    }
  }
  CU(cudaSetDevice(c->device));
  Buf d_p, d_t, d_o;
  struct Free { Buf* b[3]; ~Free() { for (Buf* x : b) x->release(); } } fr{{&d_p, &d_t, &d_o}};
  int rc;
  const size_t pbytes = (size_t)C * W * H;
  if ((rc = d_p.reserve(pbytes)) || (rc = d_t.reserve((size_t)n * 44)) || (rc = d_o.reserve((size_t)n * 4))) return rc;
  CU(cudaMemcpyAsync(d_p.p, planes_u8, pbytes, cudaMemcpyHostToDevice, c->w->stream));
  CU(cudaMemcpyAsync(d_t.p, tests, (size_t)n * 44, cudaMemcpyHostToDevice, c->w->stream));
  k_eval_tests_sum<<<(n + 127) / 128, 128, 0, c->w->stream>>>(d_p.as<uint8_t>(), W, H, d_t.as<int>(), n, d_o.as<int>());
  KCHECK(); count_launch(c, CRF_STAGE_PLAIN);
  CU(cudaMemcpyAsync(out, d_o.p, (size_t)n * 4, cudaMemcpyDeviceToHost, c->w->stream));
  CU(cudaStreamSynchronize(c->w->stream));
  return CRF_OK;
}

static void fill_list_out(crf_ctx* c, const std::vector<int32_t>& list, int n, int* tree_forest, int* tree_index) {
  for (int i = 0; i < n; i++) {
    const auto it = std::upper_bound(c->mp.roots.begin(), c->mp.roots.end(), list[i]);  // roots ascend with the tree number
    const int t = (int)(it - c->mp.roots.begin()) - 1;
    int f = 0;
    while (f + 1 < (int)c->mp.forest_base.size() && c->mp.forest_base[f + 1] <= t) f++;
    if (tree_forest) tree_forest[i] = f;
    if (tree_index) tree_index[i] = t - c->mp.forest_base[f];
  }
}

static int stage_fetch_compose(crf_ctx* c, float* headpose, float* variance, int* tree_counts, int* dominant, int* tree_forest, int* tree_index, int* ntrees, int* flags) {
  crf_face_t face;
  std::vector<int32_t> list((size_t)kMaxList);
  int nt = 0;
  CU(cudaMemcpyAsync(&face, c->d_faces.p, sizeof face, cudaMemcpyDeviceToHost, c->w->stream));
  CU(cudaMemcpyAsync(list.data(), c->w->d_face_roots.p, kMaxList * 4, cudaMemcpyDeviceToHost, c->w->stream));
  CU(cudaMemcpyAsync(&nt, c->w->d_face_ntrees.p, 4, cudaMemcpyDeviceToHost, c->w->stream));
  CU(cudaStreamSynchronize(c->w->stream));
  if (headpose) *headpose = face.headpose;
  if (variance) *variance = face.variance;
  if (tree_counts) std::memcpy(tree_counts, face.tree_counts, sizeof face.tree_counts);
  if (dominant) *dominant = face.dominant;
  if (flags) *flags = face.flags & 1;
  if (ntrees) *ntrees = nt;
  fill_list_out(c, list, nt, tree_forest, tree_index);
  return CRF_OK;
}

int crf_stage_headpose(crf_ctx* c, const uint8_t* planes_u8, int C, int W, int H, int stride, float* headpose, float* variance,
                       int tree_counts[CRF_NUM_POSE_FORESTS], int* dominant, int* tree_forest, int* tree_index, int* ntrees, int* flags) {
  if (!c) return fail(CRF_ERR_STATE, "context is not initialised");
  if (stride < 1) return fail(CRF_ERR_ARG, "bad argument");
  CU(cudaSetDevice(c->device));
  if (c->hp.slots.empty()) return fail(CRF_ERR_STATE, "the context's model does not hold the head-pose forest");
  if (max_channel_used(c->hp) >= C) return fail(CRF_ERR_ARG, "forest reads a channel the planes do not provide");
  int rc = stage_planes_to_stack(c, planes_u8, C, W, H, true, false, 1, stride, stride);
  if (rc) return rc;
  if ((rc = c->d_faces.reserve(sizeof(crf_face_t)))) return rc;
  CU(cudaMemsetAsync(c->d_faces.p, 0, sizeof(crf_face_t), c->w->stream));
  if ((rc = launch_traverse(c, c->d_fd.as<FaceDesc>(), 1, H, true, stride, c->d_hp_roots.as<int32_t>(), c->hp_ntrees, c->hp_ntrees, true))) return rc;
  // the composition needs the 5 pose forests; a head-pose-only model (Forest<HeadPoseSample>::load on its own) gets mean and variance
  if ((rc = launch_hp_reduce(c, c->d_fd.as<FaceDesc>(), 1, stride, c->full_model, kMaxList, c->d_faces.as<crf_face_t>()))) return rc;
  if (!c->full_model) CU(cudaMemsetAsync(c->w->d_face_ntrees.p, 0, 4, c->w->stream));
  rc = stage_fetch_compose(c, headpose, variance, tree_counts, dominant, tree_forest, tree_index, ntrees, flags);
  c->timer.collect();
  return rc ? rc : pull_counters(c);
}

int crf_stage_compose(crf_ctx* c, float headpose, float variance, int tree_counts[CRF_NUM_POSE_FORESTS], int* dominant, int* tree_forest, int* tree_index,
                      int* ntrees, int* flags) {
  if (!c) return fail(CRF_ERR_STATE, "context is not initialised");
  if (!c->full_model) return fail(CRF_ERR_STATE, "the forest composition needs the 5 pose forests");
  CU(cudaSetDevice(c->device));
  int rc;
  if ((rc = c->d_faces.reserve(sizeof(crf_face_t))) || (rc = c->w->d_face_roots.reserve(kMaxList * 4)) || (rc = c->w->d_face_ntrees.reserve(4))) return rc;
  CU(cudaMemsetAsync(c->d_faces.p, 0, sizeof(crf_face_t), c->w->stream));
  ComposeTables ct = c->ct;
  ct.list_cap = kMaxList;
  k_compose_only<<<1, 32, 0, c->w->stream>>>(headpose, variance, ct, c->d_faces.as<crf_face_t>(), c->w->d_face_roots.as<int32_t>(), c->w->d_face_ntrees.as<int32_t>());
  KCHECK(); count_launch(c, CRF_STAGE_HP_REDUCE);
  return stage_fetch_compose(c, nullptr, nullptr, tree_counts, dominant, tree_forest, tree_index, ntrees, flags);
}

int crf_stage_compose_batch(crf_ctx* c, const float* headpose, const float* variance, int n, int* tree_counts, int* dominant, int* ntrees, int* flags,
                            int* tree_forest, int* tree_index, int list_cap) {
  if (!c) return fail(CRF_ERR_STATE, "context is not initialised");
  if (n < 0 || (n > 0 && (!headpose || !variance)) || list_cap < 0 || list_cap > kMaxList) return fail(CRF_ERR_ARG, "bad argument");
  if (!c->full_model) return fail(CRF_ERR_STATE, "the forest composition needs the 5 pose forests");
  if (n == 0) return CRF_OK;
  CU(cudaSetDevice(c->device));
  int rc;
  Buf d_in, d_lists, d_nt, d_faces;
  struct Free { Buf* b[4]; ~Free() { for (Buf* x : b) x->release(); } } fr{{&d_in, &d_lists, &d_nt, &d_faces}};
  if ((rc = d_in.reserve((size_t)n * 8)) || (rc = d_lists.reserve((size_t)n * kMaxList * 4)) || (rc = d_nt.reserve((size_t)n * 4)) ||
      (rc = d_faces.reserve((size_t)n * sizeof(crf_face_t))))
    return rc;
  cudaStream_t s = c->w->stream;
  CU(cudaMemcpyAsync(d_in.p, headpose, (size_t)n * 4, cudaMemcpyHostToDevice, s));
  CU(cudaMemcpyAsync(d_in.as<float>() + n, variance, (size_t)n * 4, cudaMemcpyHostToDevice, s));
  CU(cudaMemsetAsync(d_faces.p, 0, (size_t)n * sizeof(crf_face_t), s));
  ComposeTables ct = c->ct;
  ct.list_cap = kMaxList;
  k_compose_batch<<<(n + 8) / 9, 288, 0, s>>>(d_in.as<float>(), d_in.as<float>() + n, n, ct, d_faces.as<crf_face_t>(), d_lists.as<int32_t>(), d_nt.as<int32_t>());
  KCHECK(); count_launch(c, CRF_STAGE_HP_REDUCE);
  std::vector<crf_face_t> faces((size_t)n);
  std::vector<int32_t> lists((size_t)n * kMaxList), nt((size_t)n);
  CU(cudaMemcpyAsync(faces.data(), d_faces.p, (size_t)n * sizeof(crf_face_t), cudaMemcpyDeviceToHost, s));
  CU(cudaMemcpyAsync(lists.data(), d_lists.p, (size_t)n * kMaxList * 4, cudaMemcpyDeviceToHost, s));
  CU(cudaMemcpyAsync(nt.data(), d_nt.p, (size_t)n * 4, cudaMemcpyDeviceToHost, s));
  CU(cudaStreamSynchronize(s));
  std::vector<int32_t> one((size_t)kMaxList);
  std::vector<int> tf((size_t)kMaxList), ti((size_t)kMaxList);
  for (int i = 0; i < n; i++) {
    if (tree_counts) std::memcpy(tree_counts + (size_t)i * CRF_NUM_POSE_FORESTS, faces[(size_t)i].tree_counts, sizeof(int) * CRF_NUM_POSE_FORESTS);
    if (dominant) dominant[i] = faces[(size_t)i].dominant;
    if (flags) flags[i] = faces[(size_t)i].flags & 1;
    if (ntrees) ntrees[i] = nt[(size_t)i];
    if (list_cap > 0 && (tree_forest || tree_index)) {
      const int m = std::min(nt[(size_t)i], list_cap);
      std::copy(lists.begin() + (size_t)i * kMaxList, lists.begin() + (size_t)i * kMaxList + m, one.begin());
      fill_list_out(c, one, m, tf.data(), ti.data());
      for (int k = 0; k < list_cap; k++) {
        if (tree_forest) tree_forest[(size_t)i * list_cap + k] = k < m ? tf[(size_t)k] : -1;
        if (tree_index) tree_index[(size_t)i * list_cap + k] = k < m ? ti[(size_t)k] : -1;
      }
    }
  }
  return CRF_OK;
}

int crf_stage_votes_meanshift(crf_ctx* c, const int* tree_forest, const int* tree_index, int ntrees, const uint8_t* planes_u8, int C, int W, int H, int stride,
                              int n_votes[CRF_NUM_PARTS], float* votes_xyw, int vote_cap, float mean_xy[CRF_NUM_PARTS][2], int rounded_xy[CRF_NUM_PARTS][2],
                              int iters[CRF_NUM_PARTS]) {
  if (!c) return fail(CRF_ERR_STATE, "context is not initialised");
  if (stride < 1) return fail(CRF_ERR_ARG, "bad argument");
  CU(cudaSetDevice(c->device));
  if (c->mp.slots.empty()) return fail(CRF_ERR_STATE, "the context's model does not hold a facial-feature forest");
  if (max_channel_used(c->mp) >= C) return fail(CRF_ERR_ARG, "forest reads a channel the planes do not provide");
  int rc = stage_planes_to_stack(c, planes_u8, C, W, H, false, true, std::max(ntrees, 1), stride, stride);
  if (rc) return rc;
  if ((rc = stage_set_list(c, tree_forest, tree_index, ntrees))) return rc;
  if ((rc = c->d_faces.reserve(sizeof(crf_face_t)))) return rc;
  CU(cudaMemsetAsync(c->d_faces.p, 0, sizeof(crf_face_t), c->w->stream));
  if ((rc = launch_traverse(c, c->d_fd.as<FaceDesc>(), 1, H, false, stride, nullptr, 0, std::max(ntrees, 1)))) return rc;
  const int saved = c->opt.ffd_stride;
  if ((rc = launch_votes_meanshift(c, c->d_fd.as<FaceDesc>(), 1, stride, c->d_faces.as<crf_face_t>()))) return rc;
  (void)saved;
  crf_face_t face;
  int32_t vbase[kParts];
  CU(cudaMemcpyAsync(&face, c->d_faces.p, sizeof face, cudaMemcpyDeviceToHost, c->w->stream));
  CU(cudaMemcpyAsync(vbase, c->w->d_vote_base.p, sizeof vbase, cudaMemcpyDeviceToHost, c->w->stream));
  CU(cudaStreamSynchronize(c->w->stream));
  for (int p = 0; p < kParts; p++) {
    if (n_votes) n_votes[p] = face.n_votes[p];
    if (mean_xy) { mean_xy[p][0] = face.ffd_f[p][0]; mean_xy[p][1] = face.ffd_f[p][1]; }
    if (rounded_xy) { rounded_xy[p][0] = face.ffd_scaled[p][0]; rounded_xy[p][1] = face.ffd_scaled[p][1]; }
    if (iters) iters[p] = face.ms_iters[p];
    if (votes_xyw && vote_cap > 0) {
      const int n = std::min(face.n_votes[p], vote_cap);
      std::vector<DevVote> v((size_t)n);
      if (n) CU(cudaMemcpy(v.data(), c->w->d_votes.as<DevVote>() + vbase[p], (size_t)n * sizeof(DevVote), cudaMemcpyDeviceToHost));
      for (int k = 0; k < n; k++) {
        float* o = votes_xyw + ((size_t)p * vote_cap + k) * 3;
        o[0] = v[k].x; o[1] = v[k].y; o[2] = v[k].w;
      }
    }
  }
  c->timer.collect();
  return pull_counters(c);
}

int crf_stage_area_under_curve(crf_ctx* c, float x1, float x2, double mean, double std_, float* area) {
  if (!c) return fail(CRF_ERR_STATE, "context is not initialised");
  if (!area) return fail(CRF_ERR_ARG, "null argument");
  if (!(x2 - x1 <= 1000.f)) return fail(CRF_ERR_ARG, "integration range too wide");   // 1e5 serial steps at most
  CU(cudaSetDevice(c->device));
  k_area_under_curve<<<1, 1, 0, c->w->stream>>>(x1, x2, mean, std_, c->d_misc.as<float>());
  KCHECK(); count_launch(c, CRF_STAGE_HP_REDUCE);
  CU(cudaMemcpyAsync(area, c->d_misc.p, 4, cudaMemcpyDeviceToHost, c->w->stream));
  CU(cudaStreamSynchronize(c->w->stream));
  return CRF_OK;
}

// MeanShift::shift(votes, result, num_iterations, kernel, stopping_criteria) (include/MeanShift.hpp:52-76) with per-call options.
int crf_stage_meanshift_opt(crf_ctx* c, const float* votes_xyw, int n, int kernel, int max_iterations, float stopping, float mean_xy[2], int rounded_xy[2], int* iters) {
  if (!c) return fail(CRF_ERR_STATE, "context is not initialised");
  const crf_options_t saved = c->opt;
  c->opt.ms_kernel_size = kernel; c->opt.ms_max_iterations = max_iterations; c->opt.ms_stopping_criteria = stopping;
  const int rc = crf_stage_meanshift(c, votes_xyw, n, mean_xy, rounded_xy, iters);
  c->opt = saved;
  return rc;
}

int crf_stage_meanshift(crf_ctx* c, const float* votes_xyw, int n, float mean_xy[2], int rounded_xy[2], int* iters) {
  if (!c) return fail(CRF_ERR_STATE, "context is not initialised");
  if (n < 0 || (n > 0 && !votes_xyw)) return fail(CRF_ERR_ARG, "bad argument");
  CU(cudaSetDevice(c->device));
  std::vector<DevVote> v((size_t)n);
  for (int i = 0; i < n; i++) { v[i].x = (short)votes_xyw[3 * i]; v[i].y = (short)votes_xyw[3 * i + 1]; v[i].w = votes_xyw[3 * i + 2]; }
  int rc;
  if ((rc = c->w->d_votes.reserve(std::max<size_t>((size_t)n * sizeof(DevVote), 16))) || (rc = c->w->d_vote_counts.reserve(kParts * 4)) ||
      (rc = c->d_faces.reserve(sizeof(crf_face_t))) || (rc = c->d_fd.reserve(sizeof(FaceDesc))))
    return rc;
  FaceDesc d{};
  d.scale = 1.f;
  CU(cudaMemcpyAsync(c->d_fd.p, &d, sizeof d, cudaMemcpyHostToDevice, c->w->stream));
  if (n) CU(cudaMemcpyAsync(c->w->d_votes.p, v.data(), (size_t)n * sizeof(DevVote), cudaMemcpyHostToDevice, c->w->stream));
  if ((rc = c->w->d_vote_base.reserve(kParts * 4))) return rc;
  CU(cudaMemsetAsync(c->w->d_vote_base.p, 0, kParts * 4, c->w->stream));
  CU(cudaMemcpyAsync(c->w->d_vote_counts.p, &n, 4, cudaMemcpyHostToDevice, c->w->stream));
  c->w->vote_cap = (size_t)std::max(n, 1);
  if ((rc = launch_meanshift(c, c->d_fd.as<FaceDesc>(), 1, c->d_faces.as<crf_face_t>()))) return rc;
  crf_face_t face;
  CU(cudaMemcpyAsync(&face, c->d_faces.p, sizeof face, cudaMemcpyDeviceToHost, c->w->stream));
  CU(cudaStreamSynchronize(c->w->stream));
  if (mean_xy) { mean_xy[0] = face.ffd_f[0][0]; mean_xy[1] = face.ffd_f[0][1]; }
  if (rounded_xy) { rounded_xy[0] = face.ffd_scaled[0][0]; rounded_xy[1] = face.ffd_scaled[0][1]; }
  if (iters) *iters = face.ms_iters[0];
  c->timer.collect();
  return CRF_OK;
}

}  // extern "C"
