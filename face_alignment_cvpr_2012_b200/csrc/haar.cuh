// Face-box source of FaceForest::detectFace (reference src/FaceForest.cpp:136-159, SURVEY 8 f2):
// cv::CascadeClassifier::detectMultiScale for the stump-based HAAR cascade the reference ships
// (data/haarcascade_frontalface_alt.xml, new-format XML), evaluated on the GPU; and for every other HAAR cascade cv::CascadeClassifier
// loads: tree weak classifiers, 45-degree tilted features (from a tilted integral built only for such cascades), the old XML format.
//
// The algorithm is OpenCV's (objdetect/cascadedetect.cpp; not under /root/reference): per scale factor = 1.3^k a bilinear
// pyramid level of the gray frame, integral images of values and squares, then every window position of the level's
// ystep grid walks the 22 stages / 2135 stumps until a stage sum falls below its threshold; surviving windows are grouped
// by cv::groupRectangles.  Here a group of frames of any sizes goes through each step in one launch over all its (frame, level)
// instances: pyramid + row scan, column scan, the first stage group over every window (one thread per window position, adjacent threads = adjacent windows, so
// the corner loads of a stump coalesce; the cascade tables are broadcast loads), later stage groups on compacted work lists
// of the survivors, then OpenCV's "skip one more step after a stage-0 reject" scan rule and the candidate compaction on the
// device.  Only the candidate rectangles come back; grouping (cv::groupRectangles) runs on the host, a frame per thread.
// Arithmetic follows oracle/haar.py, which is pinned against cv2 4.13 on the shipped images (IoU of the boxes >= 0.9:
// cv2 builds its pyramid with INTER_LINEAR_EXACT, this path with the INTER_LINEAR arithmetic of k_gray_resize).
#pragma once

namespace crf {

struct HaarStage { int first, count; float threshold; };
struct HaarWeak { int feature; float threshold, left, right; };
struct HaarRect { int x, y, w, h; float weight; };
struct HaarFeature { HaarRect r[3]; };
// Tree weak classifiers (OpenCV's predictOrdered): a tree's nodes are nodes[node, node + n), its n + 1 leaves leaves[leaf, leaf + n + 1).
// A child > 0 is a node of the same tree, a child <= 0 the leaf -child.  The walk starts at node 0 and goes left when value * inv <
// threshold.  The loader checks that every child index is greater than its parent's, so a walk ends within n steps.
struct HaarNode { int feature; float threshold; int left, right; };
struct HaarTree { int node, leaf; };
constexpr int kHaarMaxTreeNodes = 16;   // nodes per tree accepted by the loader; OpenCV's shipped cascades use at most 3

// A stump cascade (every weak classifier a single node) keeps its weak classifiers in `weak`; a tree cascade keeps them in `trees`,
// `nodes` and `leaves`, with single-node trees among them.  Stages index whichever is used.
struct Cascade {
  int win_w = 0, win_h = 0;
  std::vector<HaarStage> stages;
  std::vector<HaarWeak> weak;
  std::vector<HaarTree> trees;
  std::vector<HaarNode> nodes;
  std::vector<float> leaves;
  std::vector<HaarFeature> features;
  std::vector<uint8_t> tilted;   // per feature: 1 = 45-degree feature, its rects summed from the tilted integral
  bool has_tilted = false;
  bool is_tree() const { return !trees.empty(); }
  int nweak() const { return (int)(is_tree() ? trees.size() : weak.size()); }
};

// ---- minimal XML reader for OpenCV's FileStorage cascade files: elements with text, the attributes kept as written -------------
struct XmlNode {
  std::string name, attrs, text;
  std::vector<XmlNode> kids;
  const XmlNode* child(const char* n) const { for (auto& k : kids) if (k.name == n) return &k; return nullptr; }
};
static bool xml_parse(const std::string& s, size_t& i, XmlNode& out) {
  // precondition: s[i] == '<' of an opening tag
  size_t e = s.find('>', i);
  if (e == std::string::npos) return false;
  std::string tag = s.substr(i + 1, e - i - 1);
  const bool self_closing = !tag.empty() && tag.back() == '/';
  if (self_closing) tag.pop_back();
  const size_t sp = tag.find_first_of(" \t\r\n");
  out.name = tag.substr(0, sp);
  if (sp != std::string::npos) out.attrs = tag.substr(sp);
  i = e + 1;
  if (self_closing) return true;
  for (;;) {
    const size_t lt = s.find('<', i);
    if (lt == std::string::npos) return false;
    out.text.append(s, i, lt - i);
    if (s.compare(lt, 4, "<!--") == 0) { const size_t c = s.find("-->", lt); if (c == std::string::npos) return false; i = c + 3; continue; }
    if (s[lt + 1] == '/') { const size_t c = s.find('>', lt); if (c == std::string::npos) return false; i = c + 1; return true; }
    out.kids.emplace_back();
    i = lt;
    if (!xml_parse(s, i, out.kids.back())) return false;
  }
}

// A feature element of either format (<rects> of 2 or 3 "x y w h weight", optional <tilted>) appended to c.features / c.tilted.
// An upright rect lies in the window; a tilted one (corners (x, y), (x + w, y + w), (x - h, y + h), (x + w - h, y + w + h)) too.
static int parse_feature(const XmlNode& ft, Cascade& c, std::string& err) {
  HaarFeature hf{};
  const bool tilt = ft.child("tilted") && std::atoi(ft.child("tilted")->text.c_str()) != 0;
  const XmlNode* rects = ft.child("rects");
  if (!rects || rects->kids.empty() || rects->kids.size() > 3) { err = "feature with an unsupported rectangle count"; return CRF_ERR_FORMAT; }
  for (size_t k = 0; k < rects->kids.size(); k++) {
    double v[5] = {0, 0, 0, 0, 0};
    if (std::sscanf(rects->kids[k].text.c_str(), "%lf %lf %lf %lf %lf", &v[0], &v[1], &v[2], &v[3], &v[4]) != 5) { err = "bad feature rectangle"; return CRF_ERR_FORMAT; }
    const HaarRect r{(int)v[0], (int)v[1], (int)v[2], (int)v[3], (float)v[4]};
    const bool inside = tilt ? r.x - r.h >= 0 && r.y >= 0 && r.w >= 1 && r.h >= 1 && r.x + r.w <= c.win_w && r.y + r.w + r.h <= c.win_h
                             : r.x >= 0 && r.y >= 0 && r.w >= 1 && r.h >= 1 && r.x + r.w <= c.win_w && r.y + r.h <= c.win_h;
    if (!inside) { err = "feature rectangle outside the window"; return CRF_ERR_FORMAT; }
    hf.r[k] = r;
  }
  c.features.push_back(hf);
  c.tilted.push_back(tilt ? 1 : 0);
  c.has_tilted |= tilt;
  return CRF_OK;
}

// One weak classifier as read, before it is stored as a stump or a tree.
struct HaarWeakIn { std::vector<HaarNode> nodes; std::vector<float> leaves; };

// Checks every tree (so that no malformed tree reaches a kernel: the device walk trusts these rules) and stores the cascade: as stumps
// when every weak classifier has one node, else as trees.
static int finish_cascade(Cascade& c, const std::vector<float>& stage_thr, const std::vector<std::vector<HaarWeakIn>>& stage_weak, std::string& err) {
  bool stumps = true;
  for (const auto& ws : stage_weak)
    for (const HaarWeakIn& w : ws) {
      const int n = (int)w.nodes.size();
      if (n < 1 || n > kHaarMaxTreeNodes) { err = "tree with an unsupported node count (1 to " + std::to_string(kHaarMaxTreeNodes) + ")"; return CRF_ERR_FORMAT; }
      if ((int)w.leaves.size() != n + 1) { err = "tree without nodes + 1 leaves"; return CRF_ERR_FORMAT; }
      std::vector<uint8_t> reached((size_t)n, 0);
      reached[0] = 1;
      for (int k = 0; k < n; k++) {
        const HaarNode& nd = w.nodes[(size_t)k];
        if (nd.feature < 0 || nd.feature >= (int)c.features.size()) { err = "weak classifier names a missing feature"; return CRF_ERR_FORMAT; }
        for (const int ch : {nd.left, nd.right}) {
          if (ch > 0) {
            if (ch <= k || ch >= n) { err = "tree node whose child does not follow it"; return CRF_ERR_FORMAT; }
            reached[(size_t)ch] = 1;
          } else if (-ch > n) { err = "tree leaf index out of range"; return CRF_ERR_FORMAT; }
        }
      }
      for (int k = 1; k < n; k++)
        if (!reached[(size_t)k]) { err = "tree with an unreachable node"; return CRF_ERR_FORMAT; }
      stumps &= n == 1;
    }
  for (size_t si = 0; si < stage_weak.size(); si++) {
    HaarStage hs{stumps ? (int)c.weak.size() : (int)c.trees.size(), (int)stage_weak[si].size(), stage_thr[si]};
    for (const HaarWeakIn& w : stage_weak[si]) {
      if (stumps) {
        const HaarNode& nd = w.nodes[0];
        c.weak.push_back(HaarWeak{nd.feature, nd.threshold, w.leaves[(size_t)-nd.left], w.leaves[(size_t)-nd.right]});
      } else {
        c.trees.push_back(HaarTree{(int)c.nodes.size(), (int)c.leaves.size()});
        c.nodes.insert(c.nodes.end(), w.nodes.begin(), w.nodes.end());
        c.leaves.insert(c.leaves.end(), w.leaves.begin(), w.leaves.end());
      }
    }
    c.stages.push_back(hs);
  }
  if (c.stages.empty() || c.win_w < 3 || c.win_h < 3) { err = "empty cascade"; return CRF_ERR_FORMAT; }
  return CRF_OK;
}

// New format (<cascade type_id="opencv-cascade-classifier">): features in one list, weak classifiers as <internalNodes> (left right
// featureIdx threshold per node) and <leafValues>.
static int load_new_format(const XmlNode& cas, Cascade& c, std::string& err) {
  if (cas.child("featureType") && cas.child("featureType")->text.find("HAAR") == std::string::npos) { err = "only HAAR cascades are supported"; return CRF_ERR_UNSUPPORTED; }
  const XmlNode* fp = cas.child("featureParams");
  if (fp && fp->child("maxCatCount") && std::atoi(fp->child("maxCatCount")->text.c_str()) > 0) { err = "categorical (maxCatCount > 0) cascades are not supported"; return CRF_ERR_UNSUPPORTED; }
  c.win_w = std::atoi(cas.child("width")->text.c_str());
  c.win_h = std::atoi(cas.child("height")->text.c_str());
  int rc;
  for (const XmlNode& ft : cas.child("features")->kids)
    if ((rc = parse_feature(ft, c, err))) return rc;
  std::vector<float> thr;
  std::vector<std::vector<HaarWeakIn>> weak;
  for (const XmlNode& st : cas.child("stages")->kids) {
    const XmlNode* t = st.child("stageThreshold");
    const XmlNode* wcs = st.child("weakClassifiers");
    if (!t || !wcs) { err = "stage without threshold / classifiers"; return CRF_ERR_FORMAT; }
    thr.push_back((float)std::atof(t->text.c_str()));
    weak.emplace_back();
    for (const XmlNode& wc : wcs->kids) {
      const XmlNode* in = wc.child("internalNodes");
      const XmlNode* lv = wc.child("leafValues");
      if (!in || !lv) { err = "bad weak classifier"; return CRF_ERR_FORMAT; }
      HaarWeakIn w;
      std::istringstream ns(in->text), ls(lv->text);
      std::vector<double> v;
      for (double x; ns >> x;) v.push_back(x);
      if (!ns.eof() || v.empty() || v.size() % 4) { err = "bad weak classifier"; return CRF_ERR_FORMAT; }
      for (size_t k = 0; k < v.size(); k += 4) {
        if (v[k] != std::floor(v[k]) || v[k + 1] != std::floor(v[k + 1]) || v[k + 2] != std::floor(v[k + 2]) || std::fabs(v[k]) > 1e6 || std::fabs(v[k + 1]) > 1e6 ||
            std::fabs(v[k + 2]) > 1e9) { err = "bad weak classifier"; return CRF_ERR_FORMAT; }
        w.nodes.push_back(HaarNode{(int)v[k + 2], (float)v[k + 3], (int)v[k], (int)v[k + 1]});
      }
      for (double x; ls >> x;) w.leaves.push_back((float)x);
      if (!ls.eof()) { err = "bad weak classifier"; return CRF_ERR_FORMAT; }
      weak.back().push_back(std::move(w));
    }
  }
  return finish_cascade(c, thr, weak, err);
}

// Old format (<name type_id="opencv-haar-classifier">): <size>, stages of <trees> (nodes with an inline <feature>, <threshold> and
// left_val | left_node, right_val | right_node), <stage_threshold>, <parent>, <next>.  Converted the way OpenCV converts it: one feature
// per node, a tree's leaves numbered in node order, left before right.  Only a chain of stages (parent = previous, no next) is accepted.
static int load_old_format(const XmlNode& cas, Cascade& c, std::string& err) {
  const XmlNode* size = cas.child("size");
  const XmlNode* stages = cas.child("stages");
  if (!size || !stages || std::sscanf(size->text.c_str(), "%d %d", &c.win_w, &c.win_h) != 2) { err = "old-format cascade without <size> / <stages>"; return CRF_ERR_FORMAT; }
  std::vector<float> thr;
  std::vector<std::vector<HaarWeakIn>> weak;
  int rc;
  for (const XmlNode& st : stages->kids) {
    const int si = (int)thr.size();
    const XmlNode* trees = st.child("trees");
    const XmlNode* t = st.child("stage_threshold");
    if (!trees || !t) { err = "stage without threshold / trees"; return CRF_ERR_FORMAT; }
    const XmlNode* parent = st.child("parent");
    const XmlNode* next = st.child("next");
    if ((parent && std::atoi(parent->text.c_str()) != si - 1) || (next && std::atoi(next->text.c_str()) != -1)) {
      err = "old-format cascade whose stages do not form a chain"; return CRF_ERR_UNSUPPORTED;
    }
    thr.push_back((float)std::atof(t->text.c_str()));
    weak.emplace_back();
    for (const XmlNode& tree : trees->kids) {
      HaarWeakIn w;
      for (const XmlNode& node : tree.kids) {
        const XmlNode* ft = node.child("feature");
        const XmlNode* th = node.child("threshold");
        if (!ft || !th) { err = "tree node without feature / threshold"; return CRF_ERR_FORMAT; }
        if ((rc = parse_feature(*ft, c, err))) return rc;
        HaarNode nd{(int)c.features.size() - 1, (float)std::atof(th->text.c_str()), 0, 0};
        for (int side = 0; side < 2; side++) {
          const XmlNode* val = node.child(side ? "right_val" : "left_val");
          const XmlNode* idx = node.child(side ? "right_node" : "left_node");
          int ch;
          if (val) { ch = -(int)w.leaves.size(); w.leaves.push_back((float)std::atof(val->text.c_str())); }
          else if (idx) ch = std::atoi(idx->text.c_str());
          else { err = "tree node without a left / right child"; return CRF_ERR_FORMAT; }
          (side ? nd.right : nd.left) = ch;
        }
        w.nodes.push_back(nd);
      }
      weak.back().push_back(std::move(w));
    }
  }
  return finish_cascade(c, thr, weak, err);
}

// OpenCV's HAAR cascades as cv::CascadeClassifier::load reads them: the new format with stump or tree weak classifiers, upright and
// tilted features, and the old opencv-haar-classifier format.  LBP / HOG features, categorical splits and stage trees are rejected.
static int load_cascade(const std::string& path, Cascade& c, std::string& err) {
  FILE* f = std::fopen(path.c_str(), "rb");
  if (!f) { err = "File not found: " + path; return CRF_ERR_IO; }
  std::string s;
  char buf[1 << 16];
  size_t n;
  while ((n = std::fread(buf, 1, sizeof buf, f)) > 0) s.append(buf, n);
  std::fclose(f);
  size_t i = s.find("<opencv_storage");
  XmlNode root;
  if (i == std::string::npos || !xml_parse(s, i, root)) { err = "not an OpenCV cascade file: " + path; return CRF_ERR_FORMAT; }
  const XmlNode* cas = root.child("cascade");
  if (cas && cas->child("stages") && cas->child("features") && cas->child("width") && cas->child("height")) return load_new_format(*cas, c, err);
  for (const XmlNode& k : root.kids)
    if (k.attrs.find("opencv-haar-classifier") != std::string::npos) return load_old_format(k, c, err);
  err = "unsupported cascade layout (expected opencv-cascade-classifier or opencv-haar-classifier): " + path;
  return CRF_ERR_FORMAT;
}

// ---- kernels ---------------------------------------------------------------------------------------------------------------
// The frames of a group (any sizes) are detected together.  The group is a table of (frame, level) instances, frame-major then level;
// every buffer holds all instances of the group in that order:
//   frames [frame] BGR rows of frame f at its img_off (prefix sums of rows x step, no padding)
//   S, Q   [instance][(sh + 1) x (sw + 1)] u32 integrals of values and squares (pitch sw + 1)
//   flags  [instance][ny][nx] u8 per window of the level's ystep grid: bit 0 = passed every stage, bit 1 = rejected by stage 0
//   rows   [instance][iy] candidates per window row, then their offsets within the frame (a frame's rows are contiguous)
//   T      [instance][(sh + 1) x (sw + 1)] u32 tilted integral, same layout as S (cascades with tilted features only)
// Each pyramid pass is one launch over every instance of the group; a block finds its instance by binary search on the instance's first
// block of that launch.  Launches per group: 3 for the pyramid passes (4 with tilted features: k_haar_tilted), 1 per later stage group, 3
// for the scan rule and the candidate compaction, whatever the number, sizes and levels of the frames.  Tree weak classifiers add none:
// the evaluation kernels are instantiated for stumps or trees and upright-only or tilted features, picked from the cascade.
struct HaarInst {
  double factor, scale_x, scale_y;
  int sw, sh, nx, ny, ystep, win_w, win_h;
  int rows, cols;             // the instance's frame
  size_t img_off, step;       // the frame's BGR rows in the group's device copy
  size_t int_off;             // S / Q of the instance
  size_t flag_off;            // flags of the instance
  int frame;                  // frame index within the group
  int row_off;                // first window row of the instance among the group's rows
  int blk_rows, blk_cols, blk_eval;   // first block of the instance in k_haar_rows / k_haar_cols / k_haar_eval_first
};

// weak: the stumps of a stump cascade; trees / nodes / leaves: those of a tree cascade; tilt: per feature, for a cascade with tilted features
struct HaarDev {
  const HaarStage* stages; const HaarWeak* weak; const HaarFeature* feats; int nstages, win_w, win_h;
  const HaarTree* trees; const HaarNode* nodes; const float* leaves; const uint8_t* tilt;
};

// The search keys of the instance table, one compact array per key (a few KB, so the searches stay in L1): key[i] is the instance's
// blk_rows / blk_cols / blk_eval / row_off / flag_off.  Each array is sorted, as the table is ordered by every offset.
struct HaarKeys { const int *blk_rows, *blk_cols, *blk_eval, *row_off; const unsigned* flag_off; };

// index of the last instance whose key is <= v
template <class T>
__device__ __forceinline__ int haar_inst_of(const T* __restrict__ key, int ninst, T v) {
  int lo = 0, hi = ninst - 1;
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (key[mid] <= v) lo = mid; else hi = mid - 1;
  }
  return lo;
}

// pyramid pixel: BGR2GRAY of the source pixels, then INTER_LINEAR (k_gray_resize's arithmetic) to sw x sh
__device__ __forceinline__ int haar_level_px(const uint8_t* __restrict__ bgr, const HaarInst& L, int dx, int dy) {
  const int rows = L.rows, cols = L.cols;
  const size_t step = L.step;
  if (L.sw == cols && L.sh == rows) return gray_at(bgr, step, dy, dx);
  float fx = (float)((dx + 0.5) * L.scale_x - 0.5);
  int sx = (int)floorf(fx);
  fx -= sx;
  if (sx < 0) { fx = 0; sx = 0; }
  if (sx >= cols - 1) { fx = 0; sx = cols - 1; }
  const int a0 = __float2int_rn((1.f - fx) * 2048.f), a1 = __float2int_rn(fx * 2048.f);
  float fy = (float)((dy + 0.5) * L.scale_y - 0.5);
  int sy = (int)floorf(fy);
  fy -= sy;
  const int b0 = __float2int_rn((1.f - fy) * 2048.f), b1 = __float2int_rn(fy * 2048.f);
  const int sy0 = min(max(sy, 0), rows - 1), sy1 = min(max(sy + 1, 0), rows - 1), sx1 = min(sx + 1, cols - 1);
  const int row0 = gray_at(bgr, step, sy0, sx) * a0 + gray_at(bgr, step, sy0, sx1) * a1;
  const int row1 = gray_at(bgr, step, sy1, sx) * a0 + gray_at(bgr, step, sy1, sx1) * a1;
  const int v = (((b0 * (row0 >> 4)) >> 16) + ((b1 * (row1 >> 4)) >> 16) + 2) >> 2;
  return min(max(v, 0), 255);
}

// Pyramid level fused with the row pass of its integrals: one warp per level row builds the row's pixels and scans them along x.  TILT:
// also zeroes the level's tilted integral T, which k_haar_tilted accumulates into.  ceil(sh / 8) blocks per instance, 256 threads.
template <bool TILT>
__global__ void __launch_bounds__(256) k_haar_rows(const HaarInst* __restrict__ inst, HaarKeys keys, int ninst, const uint8_t* __restrict__ frames,
                                                   uint32_t* __restrict__ S, uint32_t* __restrict__ Q, uint32_t* __restrict__ T) {
  const int b = (int)blockIdx.x;
  const HaarInst L = inst[haar_inst_of(keys.blk_rows, ninst, b)];
  const int y = (b - L.blk_rows) * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (y >= L.sh) return;
  const uint8_t* __restrict__ bgr = frames + L.img_off;
  const size_t P = (size_t)L.sw + 1;
  uint32_t* __restrict__ s = S + L.int_off;
  uint32_t* __restrict__ q = Q + L.int_off;
  if (y == 0) for (size_t x = lane; x < P; x += 32) { s[x] = 0; q[x] = 0; }
  if (lane == 0) { s[(size_t)(y + 1) * P] = 0; q[(size_t)(y + 1) * P] = 0; }
  if constexpr (TILT) {
    uint32_t* __restrict__ t = T + L.int_off;
    if (y == 0) for (size_t x = lane; x < P; x += 32) t[x] = 0;
    for (size_t x = lane; x < P; x += 32) t[(size_t)(y + 1) * P + x] = 0;
  }
  uint32_t cs = 0, cq = 0;
  for (int x0 = 0; x0 < L.sw; x0 += 32) {
    const int x = x0 + lane;
    uint32_t v = x < L.sw ? (uint32_t)haar_level_px(bgr, L, x, y) : 0u, sq = v * v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const uint32_t nv = __shfl_up_sync(0xffffffffu, v, o), nq = __shfl_up_sync(0xffffffffu, sq, o);
      if (lane >= o) { v += nv; sq += nq; }
    }
    if (x < L.sw) { s[(size_t)(y + 1) * P + x + 1] = cs + v; q[(size_t)(y + 1) * P + x + 1] = cq + sq; }
    cs += __shfl_sync(0xffffffffu, v, 31);
    cq += __shfl_sync(0xffffffffu, sq, 31);
  }
}

// Column pass: a CTA owns 32 columns, its 32 warps 32 consecutive chunks of rows.  Each thread sums its chunk of one column, the chunk
// totals of a column are scanned in shared memory, then every chunk is walked again with its carry.  S and Q are u32 sums modulo 2^32
// (OpenCV keeps the square sums in 32 bits too) and integer addition is associative, so any summation order gives the bits of a serial
// walk down the column.  ceil((sw + 1) / 32) blocks per instance, block (32, 32).
__global__ void __launch_bounds__(1024) k_haar_cols(const HaarInst* __restrict__ inst, HaarKeys keys, int ninst, uint32_t* __restrict__ S, uint32_t* __restrict__ Q) {
  __shared__ uint32_t ts[32][32], tq[32][32];
  const int b = (int)blockIdx.x;
  const HaarInst& L = inst[haar_inst_of(keys.blk_cols, ninst, b)];
  const int sw = L.sw, sh = L.sh;
  const int tx = threadIdx.x, ty = threadIdx.y, x = (b - L.blk_cols) * 32 + tx;
  const size_t P = (size_t)sw + 1;
  const int R = (sh + 31) / 32, y0 = 1 + ty * R, y1 = min(sh + 1, y0 + R);
  const bool col = x < (int)P;
  uint32_t* __restrict__ s = S + L.int_off + x;
  uint32_t* __restrict__ q = Q + L.int_off + x;
  uint32_t as = 0, aq = 0;
  if (col)
    for (int y = y0; y < y1; y++) { as += s[(size_t)y * P]; aq += q[(size_t)y * P]; }
  ts[ty][tx] = as; tq[ty][tx] = aq;
  __syncthreads();
  uint32_t cs = 0, cq = 0;
  for (int k = 0; k < ty; k++) { cs += ts[k][tx]; cq += tq[k][tx]; }
  if (col)
    for (int y = y0; y < y1; y++) {
      cs += s[(size_t)y * P]; cq += q[(size_t)y * P];
      s[(size_t)y * P] = cs; q[(size_t)y * P] = cq;
    }
}

// Tilted integral (cv::integral's third output, OpenCV's CV_TILTED_OFS table) of every instance, between k_haar_rows and k_haar_cols,
// while S still holds the row prefixes R(y, x) = sum_{x' < x} I(y, x') (x in [0, sw]).  With R clamped in x,
//   T(Y, X) = sum_{y < Y} R(y, clamp(X + Y - 1 - y)) - R(y, clamp(X - Y + y)),
// a prefix sum down each anti-diagonal d = X + Y - 1 minus one down each diagonal e = X - Y.  A CTA owns 32 (anti-)diagonals, its 32
// warps 32 chunks of rows; a warp reads adjacent x of one row.  As in k_haar_cols the chunk totals are scanned in shared memory and each
// chunk walked again with its carry; the two families meet in T (zeroed by k_haar_rows) through u32 atomic adds, which are exact
// modulo 2^32 in any order, so T has the bits of a serial evaluation.  2 x ceil((sw + sh) / 32) blocks per instance from blk_tilt[],
// the first half anti-diagonals, block (32, 32).
__global__ void __launch_bounds__(1024) k_haar_tilted(const HaarInst* __restrict__ inst, const int* __restrict__ blk_tilt, int ninst, const uint32_t* __restrict__ S,
                                                      uint32_t* __restrict__ T) {
  __shared__ uint32_t ts[32][32];
  const int b = (int)blockIdx.x;
  const int li = haar_inst_of(blk_tilt, ninst, b);
  const HaarInst& L = inst[li];
  const int W = L.sw, H = L.sh, nb = (W + H + 31) / 32, lb = b - blk_tilt[li];
  const bool anti = lb < nb;
  const int tx = threadIdx.x, ty = threadIdx.y, t = (anti ? lb : lb - nb) * 32 + tx;
  const bool on = t < W + H;
  const int c0 = anti ? t : t - H;          // d, or e
  const size_t P = (size_t)W + 1;
  const uint32_t* __restrict__ r = S + L.int_off + P;   // R(y, x) = r[y * P + x]
  uint32_t* __restrict__ out = T + L.int_off + P;       // T(y + 1, X) = out[y * P + X]
  const int R = (H + 31) / 32, y0 = ty * R, y1 = min(H, y0 + R);
  uint32_t a = 0;
  if (on)
    for (int y = y0; y < y1; y++) a += r[(size_t)y * P + min(max(anti ? c0 - y : c0 + y, 0), W)];
  ts[ty][tx] = a;
  __syncthreads();
  uint32_t acc = 0;
  for (int k = 0; k < ty; k++) acc += ts[k][tx];
  if (on)
    for (int y = y0; y < y1; y++) {
      acc += r[(size_t)y * P + min(max(anti ? c0 - y : c0 + y, 0), W)];
      const int X = anti ? c0 - y : c0 + y + 1;
      if (X >= 0 && X <= W) atomicAdd(out + (size_t)y * P + X, anti ? acc : 0u - acc);
    }
}

__device__ __forceinline__ uint32_t haar_rectsum(const uint32_t* __restrict__ p, size_t P, int rx, int ry, int rw, int rh) {
  return p[(size_t)(ry + rh) * P + rx + rw] - p[(size_t)ry * P + rx + rw] - p[(size_t)(ry + rh) * P + rx] + p[(size_t)ry * P + rx];
}

// CV_TILTED_OFS: the 45-degree rect with corners (x, y), (x + w, y + w), (x - h, y + h), (x + w - h, y + w + h) from the tilted integral
__device__ __forceinline__ uint32_t haar_tiltsum(const uint32_t* __restrict__ t, size_t P, int rx, int ry, int rw, int rh) {
  return t[(size_t)ry * P + rx] - t[(size_t)(ry + rh) * P + rx - rh] - t[(size_t)(ry + rw) * P + rx + rw] + t[(size_t)(ry + rw + rh) * P + rx + rw - rh];
}

// feature value: v = v + weight * rectsum over the feature's rects; TILT: a tilted feature's rects come from t0
template <bool TILT>
__device__ __forceinline__ float haar_feature(const uint32_t* __restrict__ s0, const uint32_t* __restrict__ t0, size_t P, const HaarDev& K, int fi) {
  const HaarFeature& f = K.feats[fi];
  float v = 0.f;
  if constexpr (TILT) {
    if (K.tilt[fi]) {
#pragma unroll
      for (int r = 0; r < 3; r++) {
        const HaarRect hr = f.r[r];
        if (hr.weight != 0.f) v = v + hr.weight * (float)haar_tiltsum(t0, P, hr.x, hr.y, hr.w, hr.h);
      }
      return v;
    }
  }
#pragma unroll
  for (int r = 0; r < 3; r++) {
    const HaarRect hr = f.r[r];
    if (hr.weight != 0.f) v = v + hr.weight * (float)haar_rectsum(s0, P, hr.x, hr.y, hr.w, hr.h);
  }
  return v;
}

// Stages [s_begin, s_end) of the window at s0 (t0 in the tilted integral), one thread per window, in the cascade's order: the feature
// values, sum = sum + leaf over the weak classifiers (f32, unfused under -fmad=false).  A stump picks its leaf by value * inv <
// threshold; TREE walks the tree (OpenCV's predictOrdered) with the same comparison at every node, of which a stump is the one-node
// case.  A window's sums are never split across lanes: a reordered f32 sum could flip a stump or a stage near its threshold.  Returns
// the first stage whose sum falls below its threshold, or -1.
template <bool TREE, bool TILT>
__device__ __forceinline__ int haar_stages(const uint32_t* __restrict__ s0, const uint32_t* __restrict__ t0, size_t P, float inv, const HaarDev& K,
                                           int s_begin, int s_end) {
  for (int si = s_begin; si < s_end; si++) {
    const HaarStage st = K.stages[si];
    float sum = 0.f;
    for (int k = st.first; k < st.first + st.count; k++) {
      if constexpr (TREE) {
        const HaarTree tr = K.trees[k];
        int idx = 0;
        do {   // child indices grow along a walk (checked at load), so this ends within the tree's node count
          const HaarNode nd = K.nodes[tr.node + idx];
          const float v = haar_feature<TILT>(s0, t0, P, K, nd.feature);
          idx = (v * inv < nd.threshold) ? nd.left : nd.right;
        } while (idx > 0);
        sum = sum + K.leaves[tr.leaf - idx];
      } else {
        const HaarWeak wk = K.weak[k];
        const float v = haar_feature<TILT>(s0, t0, P, K, wk.feature);
        sum = sum + ((v * inv < wk.threshold) ? wk.left : wk.right);
      }
    }
    if (!(sum >= st.threshold)) return si;
  }
  return -1;
}

// warp-aggregated append of the lanes' items to a work list (every lane of the warp calls it)
__device__ __forceinline__ void haar_append(bool keep, uint2 item, uint2* __restrict__ list, unsigned* __restrict__ count) {
  const unsigned m = __ballot_sync(0xffffffffu, keep);
  if (!m) return;
  const int lane = threadIdx.x & 31, leader = __ffs(m) - 1;
  unsigned base = 0;
  if (lane == leader) base = atomicAdd(count, (unsigned)__popc(m));
  base = __shfl_sync(0xffffffffu, base, leader);
  if (keep) list[base + __popc(m & ((1u << lane) - 1u))] = item;
}

// First stage group, every window of every instance of the group: HaarEvaluator::setWindow's variance normalisation over the inner
// (w - 2) x (h - 2) rect, stages [0, s_end); writes the window's flag byte and appends the survivors (flag index, 1 / nf) to the work list
// of the next stage group.  T: the tilted integrals (TILT only).  ceil(nx / 128) x ny blocks per instance, 128 threads.
template <bool TREE, bool TILT>
__global__ void __launch_bounds__(128) k_haar_eval_first(const HaarInst* __restrict__ inst, HaarKeys keys, int ninst, const uint32_t* __restrict__ S, const uint32_t* __restrict__ Q,
                                                         const uint32_t* __restrict__ T, HaarDev K, int s_end, uint8_t* __restrict__ flags, uint2* __restrict__ list, unsigned* __restrict__ count) {
  const int b = (int)blockIdx.x;
  const HaarInst& L = inst[haar_inst_of(keys.blk_eval, ninst, b)];
  const int nx = L.nx, ystep = L.ystep, bx = (nx + 127) / 128, lb = b - L.blk_eval, iy = lb / bx;
  const int ix = (lb - iy * bx) * 128 + threadIdx.x;
  bool keep = false;
  uint2 item = make_uint2(0u, 0u);
  if (ix < nx) {
    const size_t P = (size_t)L.sw + 1;
    const size_t o = L.int_off + (size_t)(iy * ystep) * P + (size_t)ix * ystep;
    const uint32_t* __restrict__ s0 = S + o;
    const uint32_t* __restrict__ q0 = Q + o;
    const double area = (double)((K.win_w - 2) * (K.win_h - 2));
    const double vs = (double)haar_rectsum(s0, P, 1, 1, K.win_w - 2, K.win_h - 2), vq = (double)haar_rectsum(q0, P, 1, 1, K.win_w - 2, K.win_h - 2);
    const double nf = area * vq - vs * vs;
    uint8_t out = 0;
    float inv = 0.f;
    if (nf > 0.) {
      inv = (float)(1.0 / sqrt(nf));
      if ((float)area * inv < 0.1f) {
        const int r = haar_stages<TREE, TILT>(s0, TILT ? T + o : nullptr, P, inv, K, 0, s_end);
        if (r < 0) { if (s_end >= K.nstages) out = 1; else keep = true; }
        else if (r == 0) out = 2;
      }
    }
    const size_t idx = L.flag_off + (size_t)iy * nx + ix;
    flags[idx] = out;
    item = make_uint2((unsigned)idx, __float_as_uint(inv));
  }
  haar_append(keep, item, list, count);
}

// A later stage group [s_begin, s_end) on the previous group's survivors, grid-stride over the list (its length is on the device, so the
// launch does not wait for the host).  Compaction changes which thread handles a window, never the order of its arithmetic.  Survivors of
// the last group get bit 0 of their flag; the others are appended to the next list.
template <bool TREE, bool TILT>
__global__ void __launch_bounds__(128) k_haar_eval_list(const HaarInst* __restrict__ inst, HaarKeys keys, int ninst, const uint32_t* __restrict__ S,
                                                        const uint32_t* __restrict__ T, HaarDev K,
                                                        int s_begin, int s_end, const uint2* __restrict__ list_in, const unsigned* __restrict__ count_in,
                                                        uint8_t* __restrict__ flags, uint2* __restrict__ list_out, unsigned* __restrict__ count_out) {
  const unsigned n = *count_in;
  const bool last = s_end >= K.nstages;
  for (unsigned base = blockIdx.x * blockDim.x; base < n; base += gridDim.x * blockDim.x) {
    const unsigned i = base + threadIdx.x;
    bool keep = false;
    uint2 it = make_uint2(0u, 0u);
    if (i < n) {
      it = list_in[i];
      const HaarInst& L = inst[haar_inst_of(keys.flag_off, ninst, it.x)];
      const size_t w = it.x - L.flag_off;
      const int iy = (int)(w / L.nx), ix = (int)(w - (size_t)iy * L.nx);
      const size_t P = (size_t)L.sw + 1;
      const size_t o = L.int_off + (size_t)(iy * L.ystep) * P + (size_t)ix * L.ystep;
      if (haar_stages<TREE, TILT>(S + o, TILT ? T + o : nullptr, P, __uint_as_float(it.y), K, s_begin, s_end) < 0) {
        if (last) flags[it.x] = 1; else keep = true;
      }
    }
    if (!last) haar_append(keep, it, list_out, count_out);
  }
}

// OpenCV's scan (CascadeClassifierInvoker) visits the windows of a row in x order and takes one extra step after a window rejected by
// stage 0: visited(0) = 1, visited(ix) = !(visited(ix - 1) && rej0(ix - 1)).  32 windows at a time from the ballot of their rej0 bits.
__device__ __forceinline__ unsigned haar_visited(unsigned rej0, bool& carry) {
  unsigned vis = 0;
  bool v = carry;
#pragma unroll
  for (int b = 0; b < 32; b++) {
    if (v) vis |= 1u << b;
    v = !(v && ((rej0 >> b) & 1u));
  }
  carry = v;
  return vis;
}

// One warp per window row of the group (instance by instance, then iy): candidates = visited windows that passed every stage.  COUNT: the
// row's candidate count into rows[].  Otherwise: the candidate rectangles, in (level, iy, ix) order per frame and frame after frame, at the
// row's offset (rows[] after k_haar_row_offsets) plus the counts of the frames before.  grid ceil(nrows / 8), 256 threads.
template <bool COUNT>
__global__ void __launch_bounds__(256) k_haar_scan(const HaarInst* __restrict__ inst, HaarKeys keys, int ninst, int nrows, const uint8_t* __restrict__ flags,
                                                   int* __restrict__ rows, const int* __restrict__ frame_count, crf_rect_t* __restrict__ cand) {
  const int rid = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (rid >= nrows) return;
  const HaarInst& L = inst[haar_inst_of(keys.row_off, ninst, rid)];
  const int iy = rid - L.row_off, nx = L.nx;
  const uint8_t* __restrict__ fl = flags + L.flag_off + (size_t)iy * nx;
  int base = 0;
  if (!COUNT) {
    base = rows[rid];
    for (int k = 0; k < L.frame; k++) base += frame_count[k];
  }
  bool carry = true;
  int n = 0;
  for (int x0 = 0; x0 < nx; x0 += 32) {
    const int ix = x0 + lane;
    const uint8_t v = ix < nx ? fl[ix] : 0;
    const unsigned rej0 = __ballot_sync(0xffffffffu, v & 2), pass = __ballot_sync(0xffffffffu, v & 1);
    const unsigned c = haar_visited(rej0, carry) & pass;
    if (!COUNT && ((c >> lane) & 1u))
      cand[base + n + __popc(c & ((1u << lane) - 1u))] = crf_rect_t{(int)rint(ix * L.ystep * L.factor), (int)rint(iy * L.ystep * L.factor), L.win_w, L.win_h};
    n += __popc(c);
  }
  if (COUNT && lane == 0) rows[rid] = n;
}

// Exclusive scan of one frame's row counts in place (row offsets within the frame) and the frame's candidate count.  Frame f owns the rows
// [frame_rows[f], frame_rows[f + 1]).  grid frames, 1024 threads.
__global__ void __launch_bounds__(1024) k_haar_row_offsets(const int* __restrict__ frame_rows, int* __restrict__ rows, int* __restrict__ frame_count) {
  __shared__ int wsum[32];
  const int r0 = frame_rows[blockIdx.x], nr = frame_rows[blockIdx.x + 1] - r0;
  int* __restrict__ r = rows + r0;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  int carry = 0;
  for (int b = 0; b < nr; b += 1024) {
    const int i = b + threadIdx.x;
    const int v = i < nr ? r[i] : 0;
    int x = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const int y = __shfl_up_sync(0xffffffffu, x, o); if (lane >= o) x += y; }
    if (lane == 31) wsum[warp] = x;
    __syncthreads();
    if (warp == 0) {
      int t = wsum[lane];
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) { const int y = __shfl_up_sync(0xffffffffu, t, o); if (lane >= o) t += y; }
      wsum[lane] = t;
    }
    __syncthreads();
    if (i < nr) r[i] = carry + (warp ? wsum[warp - 1] : 0) + x - v;
    carry += wsum[31];
    __syncthreads();
  }
  if (threadIdx.x == 0) frame_count[blockIdx.x] = carry;
}

// ---- host: scales, scan rule, cv::groupRectangles ----------------------------------------------------------------------------
static void group_rectangles(std::vector<crf_rect_t>& rects, int group_threshold, double eps) {
  const int n = (int)rects.size();
  if (group_threshold <= 0 || n == 0) return;
  std::vector<int> parent((size_t)n);
  for (int i = 0; i < n; i++) parent[(size_t)i] = i;
  auto find = [&](int i) { while (parent[(size_t)i] != i) { parent[(size_t)i] = parent[(size_t)parent[(size_t)i]]; i = parent[(size_t)i]; } return i; };
  auto similar = [&](const crf_rect_t& a, const crf_rect_t& b) {
    const double d = eps * (std::min(a.width, b.width) + std::min(a.height, b.height)) * 0.5;
    return std::abs(a.x - b.x) <= d && std::abs(a.y - b.y) <= d && std::abs(a.x + a.width - b.x - b.width) <= d && std::abs(a.y + a.height - b.y - b.height) <= d;
  };
  for (int i = 0; i < n; i++)
    for (int j = i + 1; j < n; j++)
      if (similar(rects[(size_t)i], rects[(size_t)j])) { const int a = find(i), b = find(j); if (a != b) parent[(size_t)b] = a; }
  std::vector<int> label((size_t)n, -1), root_label((size_t)n, -1);
  int nc = 0;
  for (int i = 0; i < n; i++) { const int r = find(i); if (root_label[(size_t)r] < 0) root_label[(size_t)r] = nc++; label[(size_t)i] = root_label[(size_t)r]; }
  std::vector<long long> acc((size_t)nc * 4, 0);
  std::vector<int> cnt((size_t)nc, 0);
  for (int i = 0; i < n; i++) {
    long long* a = &acc[(size_t)label[(size_t)i] * 4];
    a[0] += rects[(size_t)i].x; a[1] += rects[(size_t)i].y; a[2] += rects[(size_t)i].width; a[3] += rects[(size_t)i].height;
    cnt[(size_t)label[(size_t)i]]++;
  }
  std::vector<crf_rect_t> rr((size_t)nc);
  for (int l = 0; l < nc; l++) {
    const float s = 1.f / (float)cnt[(size_t)l];
    rr[(size_t)l] = crf_rect_t{(int)std::lrintf((float)acc[(size_t)l * 4] * s), (int)std::lrintf((float)acc[(size_t)l * 4 + 1] * s),
                              (int)std::lrintf((float)acc[(size_t)l * 4 + 2] * s), (int)std::lrintf((float)acc[(size_t)l * 4 + 3] * s)};
  }
  std::vector<crf_rect_t> keep;
  for (int i = 0; i < nc; i++) {
    if (cnt[(size_t)i] <= group_threshold) continue;
    const crf_rect_t r1 = rr[(size_t)i];
    const int n1 = cnt[(size_t)i];
    int j = 0;
    for (; j < nc; j++) {
      const int n2 = cnt[(size_t)j];
      if (j == i || n2 <= group_threshold) continue;
      const crf_rect_t r2 = rr[(size_t)j];
      const int dx = (int)std::lrint(r2.width * eps), dy = (int)std::lrint(r2.height * eps);
      if (r1.x >= r2.x - dx && r1.y >= r2.y - dy && r1.x + r1.width <= r2.x + r2.width + dx && r1.y + r1.height <= r2.y + r2.height + dy && (n2 > std::max(3, n1) || n1 < 3)) break;
    }
    if (j == nc) keep.push_back(r1);
  }
  rects.swap(keep);
}

}  // namespace crf

// id: unique per load, so that a context's device copy of a freed cascade is never taken for a new one at the same address
struct crf_cascade { crf::Cascade c; unsigned long long id = 0; };
