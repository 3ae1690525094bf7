// crf_b200_compat.hpp — the reference's C++ interface for the inference path, re-exposed on top of the C ABI
// (include/crf_b200.h).  Header-only; link with -lcrf_b200.
//
// Same class and member names, signatures, argument meaning and error behaviour as MatrixPlayer/face_alignment_cvpr_2012
// (citations are file:line under the reference tree): ForestParam, the option structs, Vote, Face, SimplePatchFeature,
// ThresholdSplit, HeadPoseLeaf / MPLeaf, ImageSample, HeadPoseSample / MPSample, TreeNode, Tree, Forest, FaceForest, MeanShift,
// getHeadPoseVotesMT, getFacialFeaturesVotesMT, areaUnderCurve, intersect.  Every computation is a call into libcrf_b200.so,
// i.e. a CUDA kernel: there is no host arithmetic of the path in this header and no CPU fallback.  The batch entry points
// (FaceForest::analyzeImage / analyzeFace, estimateHeadPose, estimateFacialFeatures, get*VotesMT) are the fast ones; the
// per-sample calls (Forest::evaluateMT, Tree::evaluateMT, ImageSample::evalTest) cost one small launch each, as the reference's
// cost one thread-pool task each.
//
// OpenCV types: with CRF_B200_WITH_OPENCV the real cv::Mat / cv::Rect / cv::Point are used (namespace cvlite = cv);
// otherwise layout-compatible stand-ins in namespace cvlite (the image this was built in has no OpenCV C++; tests/cpp compiles the
// OpenCV branch against a stub <opencv2/core/core.hpp> so that it cannot rot).
//
// Deviations:
//   * FaceForest's constructor loads the face cascade only if fd_option.path_face_cascade is set (the reference requires it,
//     src/FaceForest.cpp:23-28); without it analyzeImage(img, bboxes, faces) takes the boxes from the caller.  Either way all
//     faces of a frame are analysed in one launch.
//   * crf_b200::CascadeClassifier stands for cv::CascadeClassifier (load + detectMultiScale, evaluated on the GPU); it reads every
//     HAAR cascade cv::CascadeClassifier reads (stumps or trees, tilted features, old or new XML format), not LBP / HOG ones.
//   * FaceForestOptions carries three extra members at its end (device, ms_mode, mean_shift_option).
#ifndef CRF_B200_COMPAT_HPP
#define CRF_B200_COMPAT_HPP

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <dirent.h>
#include <memory>
#include <stdexcept>
#include <string>
#include <sys/stat.h>
#include <vector>

#include "crf_b200.h"

#ifdef CRF_B200_WITH_OPENCV
#include <opencv2/core/core.hpp>
namespace cvlite = cv;
#else
namespace cvlite {
#ifndef CV_8UC1
#define CV_8UC1 0
#define CV_8UC3 16
#define CV_32FC1 5
#define CV_32F 5
#endif
template <typename T> struct Rect_ { T x, y, width, height; Rect_() : x(0), y(0), width(0), height(0) {} Rect_(T x_, T y_, T w_, T h_) : x(x_), y(y_), width(w_), height(h_) {} };
template <typename T> struct Point_ { T x, y; Point_() : x(0), y(0) {} Point_(T x_, T y_) : x(x_), y(y_) {} };
typedef Rect_<int> Rect;
typedef Point_<int> Point;
// cv::Mat stand-in: 8-bit 1- or 3-channel, or 32-bit float single-channel; a view of caller memory or an owner of its own
class Mat {
 public:
  unsigned char* data; int rows, cols; size_t step;
  Mat() : data(nullptr), rows(0), cols(0), step(0), type_(CV_8UC1) {}
  Mat(int r, int c, int type) : data(nullptr), rows(0), cols(0), step(0), type_(type) { create(r, c, type); }
  Mat(int r, int c, int type, void* ext, size_t step_ = 0) : data((unsigned char*)ext), rows(r), cols(c), step(step_ ? step_ : (size_t)c * esz(type)), type_(type) {}
  void create(int r, int c, int type) { type_ = type; rows = r; cols = c; step = (size_t)c * esz(type); buf_ = std::make_shared<std::vector<unsigned char> >((size_t)r * step + 16); data = buf_->data(); }
  int type() const { return type_; }
  int channels() const { return (type_ >> 3) + 1; }
  bool empty() const { return !data || rows == 0 || cols == 0; }
  template <typename T> T& at(int y, int x) { return *reinterpret_cast<T*>(data + (size_t)y * step + (size_t)x * sizeof(T)); }
  template <typename T> const T& at(int y, int x) const { return *reinterpret_cast<const T*>(data + (size_t)y * step + (size_t)x * sizeof(T)); }
 private:
  static size_t esz(int type) { return ((type & 7) == 5 ? 4 : 1) * (size_t)((type >> 3) + 1); }
  int type_;
  std::shared_ptr<std::vector<unsigned char> > buf_;
};
}  // namespace cvlite
#endif

namespace crf_b200 {

inline void check(int rc) { if (rc < 0) throw std::runtime_error(crf_last_error()); }

// ------------------------------------------------------------------------------------------------ parameters
// include/Constants.hpp:24-60
struct ForestParam {
  int getPatchSize() { return static_cast<int>(std::round(face_size * patch_size_ratio)); }
  int max_depth = 0, min_patches = 0, ntests = 0, ntrees = 0, nimages = 0, npatches = 0, face_size = 125;
  float patch_size_ratio = 0.25f;
  std::string tree_path, image_path;
  std::vector<int> features;
};
static const int NUM_HEADPOSE_CLASSES = 5;                      // include/Constants.hpp:65-68
static const float NORM_HEADPOSE_VARIANCE_FACTOR = 0.05f;

// include/FaceForest.hpp:21-58, include/MeanShift.hpp:16-25
struct FaceDetectionOption { int min_feature_size = 30; int min_neighbors = 1; float search_scale_factor = 1.3f; std::string path_face_cascade; };
struct HeadPoseEstimatorOption { int num_head_pose_labels = NUM_HEADPOSE_CLASSES; int step_size = 4; float min_foreground_probability = 0.5f; };
struct MultiPartEstimatorOption { int num_parts = 10; int step_size = 3; int min_samples = 2; float min_forground = 0.5f; float min_pf = 0.25f; float max_variance = 25.f; };
struct MeanShiftOption { int kernel_size = 10; int max_iterations = 7; float stopping_criteria = 0.05f; };

// include/FaceForest.hpp:60-68 (same member names), then the three extensions
struct FaceForestOptions {
  ForestParam hp_forest_param, mp_forest_param;
  FaceDetectionOption fd_option;
  HeadPoseEstimatorOption hp_option;
  MultiPartEstimatorOption mp_option;
  std::vector<std::string> mp_forest_paths;
  int device = 0;                         // CUDA device of the context; -1 = all visible GPUs, the faces of a call sharded over them
  int ms_mode = CRF_MS_DEFAULT;           // crf_b200.h: MeanShift evaluation mode
  MeanShiftOption mean_shift_option;      // the reference default-constructs this inside estimateFacialFeatures (src/FaceForest.cpp:89)
};

struct Face { float headpose = 0.f; cvlite::Rect bbox; std::vector<cvlite::Point> ffd_cordinates; };   // include/FaceForest.hpp:70-75
struct Vote { Vote() : weight(0.0f), check(false) {} cvlite::Point pos; float weight; bool check; };    // include/face_utils.hpp:34-42

// include/ImageSample.hpp:22-91, include/ThresholdSplit.hpp:22-67
struct SimplePatchFeature { int feature_channel = 0; cvlite::Rect_<int> rect1, rect2; };
template <typename Feature> class ThresholdSplit {
 public:
  ThresholdSplit() : info(0), oob(0), threshold(0), margin(0), depth(0), num_thresholds(0), split_mode(0) {}
  Feature feature; double info, oob; int threshold, margin, depth, num_thresholds; float split_mode;
};
// include/HeadPoseSample.hpp:144-162, include/MPSample.hpp:137-159
class HeadPoseLeaf { public: int hp_nsamples = 0; float hp_foreground = 0.f; std::vector<int> hp_labels; };
class MPLeaf {
 public:
  int mp_samples = 0; std::vector<cvlite::Point_<int> > mp_parts_offset; std::vector<float> mp_parts_variance, mp_prob_foreground; float mp_foreground = 0.f;
};

// ------------------------------------------------------------------------------------------------ contexts
namespace detail {
inline crf_options_t make_options(const HeadPoseEstimatorOption& h, const MultiPartEstimatorOption& m, const MeanShiftOption& s, int ms_mode) {
  crf_options_t co;
  crf_options_default(&co);
  co.hp_stride = h.step_size; co.hp_min_foreground = h.min_foreground_probability;
  co.ffd_stride = m.step_size; co.ffd_min_samples = m.min_samples; co.ffd_min_foreground = m.min_forground; co.ffd_min_pf = m.min_pf; co.ffd_max_variance = m.max_variance;
  co.ms_kernel_size = s.kernel_size; co.ms_max_iterations = s.max_iterations; co.ms_stopping_criteria = s.stopping_criteria;
  co.ms_mode = ms_mode;
  return co;
}
inline int& default_device() { static int d = 0; return d; }
// A loaded model and the GPU context made for it.  The leaf-vote predicate (src/face_utils.cpp:285-290) is folded into the device
// image when a context is created, so a call with other thresholds re-creates the context (the last one is kept).
struct Loaded {
  crf_model* model = nullptr; crf_ctx* ctx = nullptr; crf_multi* multi = nullptr; crf_options_t opt; int device = 0;
  ~Loaded() { if (multi) crf_multi_destroy(multi); if (ctx) crf_ctx_destroy(ctx); if (model) crf_model_free(model); }
  // device < 0: every visible GPU behind this one caller (crf_multi_*: one context + host thread per GPU, faces sharded)
  crf_multi* all_gpus(const crf_options_t& want) {
    if (!multi) check(crf_multi_create(model, nullptr, 0, &want, &multi));
    return multi;
  }
  crf_ctx* context(const crf_options_t& want) {
    if (!ctx || std::memcmp(&want, &opt, sizeof opt) != 0) {
      if (ctx) { crf_ctx_destroy(ctx); ctx = nullptr; }
      check(crf_ctx_create(model, device < 0 ? 0 : device, &want, &ctx));
      opt = want;
    }
    return ctx;
  }
  crf_ctx* context() { if (!ctx) { crf_options_t o; crf_options_default(&o); return context(o); } return ctx; }
};
// forest-less context for ImageSample / MeanShift / areaUnderCurve, which exist independently of any forest in the reference
inline crf_ctx* plain_context() {
  static Loaded L;
  if (!L.ctx) { L.device = default_device(); check(crf_ctx_create(nullptr, L.device, nullptr, &L.ctx)); }
  return L.ctx;
}
}  // namespace detail

// CUDA device used by the objects that carry no options (ImageSample, Forest, Tree, MeanShift); set before first use.
inline void setDevice(int device) { detail::default_device() = device; }

// ------------------------------------------------------------------------------------------------ ImageSample
// include/ImageSample.hpp:146-199, src/ImageSample.cpp:11-90.  `img` is the scaled 8-bit gray face (cols <= 125, rows <= 521).
class ImageSample {
 public:
  ImageSample(const cvlite::Mat img, std::vector<int> features, bool use_integral = false) : m_use_integral(use_integral) {
    if (img.empty() || img.channels() != 1) throw std::invalid_argument("ImageSample expects an 8-bit single-channel image");
    W_ = img.cols; H_ = img.rows;
    std::vector<unsigned char> gray((size_t)W_ * H_);
    for (int y = 0; y < H_; y++) std::memcpy(&gray[(size_t)y * W_], img.data + (size_t)y * img.step, (size_t)W_);
    int n = 0;
    for (size_t i = 0; i < features.size(); i++) n += features[i] == 1 ? 35 : (features[i] == 2 || features[i] == 3) ? 2 : 1;
    planes_.resize((size_t)std::max(n, 1) * W_ * H_);
    std::vector<uint32_t> integ(use_integral ? (size_t)std::max(n, 1) * (W_ + 1) * (H_ + 1) : 0);
    C_ = 0;
    if (!features.empty()) {
      // extractFeatureChannels: the ids are sorted, then FeatureChannelFactory::extractChannel appends each one's planes
      C_ = crf_stage_feature_channels(detail::plain_context(), gray.data(), W_, H_, features.data(), (int)features.size(), planes_.data(),
                                      use_integral ? integ.data() : nullptr);
      check(C_);
    }
    for (int c = 0; c < C_; c++) {   // m_feature_channels as the reference holds them: CV_32F integrals, or the 8-bit planes
      cvlite::Mat m;
      if (use_integral) {
        m.create(H_ + 1, W_ + 1, CV_32FC1);
        for (int y = 0; y <= H_; y++) for (int x = 0; x <= W_; x++) m.at<float>(y, x) = (float)integ[((size_t)c * (H_ + 1) + y) * (W_ + 1) + x];
      } else {
        m.create(H_, W_, CV_8UC1);
        for (int y = 0; y < H_; y++) std::memcpy(m.data + (size_t)y * m.step, &planes_[((size_t)c * H_ + y) * W_], (size_t)W_);
      }
      m_feature_channels.push_back(m);
    }
  }
  virtual ~ImageSample() {}

  // src/ImageSample.cpp:30-64 (both branches give the same integers: SURVEY Appendix E.10)
  int evalTest(const SimplePatchFeature& test, const cvlite::Rect rect) const {
    const int t[11] = {test.feature_channel, test.rect1.x, test.rect1.y, test.rect1.width, test.rect1.height,
                       test.rect2.x, test.rect2.y, test.rect2.width, test.rect2.height, rect.x, rect.y};
    int out = 0;
    // the branch the reference takes follows m_use_integral: integral corners, or cv::sum over the 8-bit rectangles
    check(m_use_integral ? crf_stage_eval_tests(detail::plain_context(), planes_.data(), C_, W_, H_, t, 1, &out)
                         : crf_stage_eval_tests_sum(detail::plain_context(), planes_.data(), C_, W_, H_, t, 1, &out));
    return out;
  }

  std::vector<cvlite::Mat> m_feature_channels;
  // the 8-bit planes [C][H][W] behind m_feature_channels: what the library's stage calls take
  const unsigned char* planes() const { return planes_.data(); }
  int numChannels() const { return C_; }
  int cols() const { return W_; }
  int rows() const { return H_; }

 private:
  bool m_use_integral;
  int W_ = 0, H_ = 0, C_ = 0;
  std::vector<unsigned char> planes_;
};

// ------------------------------------------------------------------------------------------------ samples
// include/HeadPoseSample.hpp:26-141, src/HeadPoseSample.cpp:30-46 (testing constructor, evalTest, eval)
class HeadPoseSample {
 public:
  typedef ThresholdSplit<SimplePatchFeature> Split;
  typedef HeadPoseLeaf Leaf;
  HeadPoseSample(const ImageSample* sample, cvlite::Rect patch_bbox) : m_image(sample), m_patch_bbox(patch_bbox) {}
  virtual ~HeadPoseSample() {}
  int evalTest(const Split& test) const { return m_image->evalTest(test.feature, m_patch_bbox); }
  bool eval(const Split& test) const { return evalTest(test) <= test.threshold; }
  cvlite::Rect getPatch() const { return m_patch_bbox; }
  const ImageSample* image() const { return m_image; }
  static const int kind = 0;
 private:
  const ImageSample* m_image;
  cvlite::Rect m_patch_bbox;
};
// include/MPSample.hpp:27-134, src/MPSample.cpp:68-84
class MPSample {
 public:
  typedef ThresholdSplit<SimplePatchFeature> Split;
  typedef MPLeaf Leaf;
  MPSample(const ImageSample* sample, cvlite::Rect patch_bbox) : m_image(sample), m_patch_bbox(patch_bbox) {}
  virtual ~MPSample() {}
  int evalTest(const Split& test) const { return m_image->evalTest(test.feature, m_patch_bbox); }
  bool eval(const Split& test) const { return evalTest(test) <= test.threshold; }
  cvlite::Rect getPatch() { return m_patch_bbox; }
  const ImageSample* image() const { return m_image; }
  static const int kind = 1;
 private:
  const ImageSample* m_image;
  cvlite::Rect m_patch_bbox;
};

// ------------------------------------------------------------------------------------------------ TreeNode / Tree / Forest
// include/TreeNode.hpp:22-165 (the members inference touches)
template <typename Sample> class TreeNode {
 public:
  typedef typename Sample::Split Split;
  typedef typename Sample::Leaf Leaf;
  TreeNode() : right(nullptr), left(nullptr), depth(-1), is_leaf(false), has_split(false) {}
  ~TreeNode() { delete left; delete right; }
  int getDepth() { return depth; }
  bool isLeaf() const { return is_leaf; }
  Leaf* getLeaf() { return &leaf; }
  bool hasSplit() const { return has_split; }
  Split getSplit() { return split; }
  bool eval(const Sample* s) const { return s->eval(split); }   // one evalTest launch
  Leaf leaf; Split split; TreeNode<Sample>* right; TreeNode<Sample>* left;
  int depth; bool is_leaf, has_split;
  int object_id = -1;   // Boost object id == pre-order index: what the library reports as the leaf id
};

namespace detail {
inline void fill_leaf(HeadPoseLeaf& L, const float* o) { L.hp_nsamples = (int)o[1]; L.hp_foreground = o[2]; L.hp_labels.resize(5); for (int j = 0; j < 5; j++) L.hp_labels[j] = (int)o[3 + j]; }
inline void fill_leaf(MPLeaf& L, const float* o) {
  L.mp_samples = (int)o[1]; L.mp_foreground = o[2];
  L.mp_parts_offset.resize(10); L.mp_parts_variance.resize(10); L.mp_prob_foreground.resize(10);
  for (int j = 0; j < 10; j++) { L.mp_parts_offset[j] = cvlite::Point_<int>((int)o[3 + 2 * j], (int)o[4 + 2 * j]); L.mp_parts_variance[j] = o[23 + j]; L.mp_prob_foreground[j] = o[33 + j]; }
}
}  // namespace detail

// include/Tree.hpp:33-346.  A Tree is one tree of a loaded model: `root` is the host mirror of its nodes (what user code walks),
// evaluation runs on the GPU image of the same tree.
template <typename Sample> class Tree {
 public:
  typedef typename Sample::Split Split;
  typedef typename Sample::Leaf Leaf;
  Tree() : root(nullptr), m_num_nodes(0), i_node(0), which_(0), index_(0) {}
  virtual ~Tree() { delete root; }
  bool isFinished() { return m_num_nodes != 0 && i_node == m_num_nodes; }   // include/Tree.hpp:72-79

  // include/Tree.hpp:174-191.  From a root the walk is one traversal launch; from an inner node it follows TreeNode::eval.
  static void evaluateMT(const Sample* sample, TreeNode<Sample>* node, Leaf** leaf) {
    if (node->isLeaf()) { *leaf = node->getLeaf(); return; }
    Tree* t = node->object_id == 0 ? owner_of(node) : nullptr;
    if (t) { *leaf = t->leaf_of(t->evaluate_root(sample)); return; }
    if (node->eval(sample)) evaluateMT(sample, node->left, leaf);
    else evaluateMT(sample, node->right, leaf);
  }
  // include/Tree.hpp:193-237
  static bool load(Tree** tree, std::string path) {
    std::shared_ptr<detail::Loaded> L(new detail::Loaded());
    L->device = detail::default_device();
    if (crf_model_load_tree(path.c_str(), Sample::kind, &L->model) != CRF_OK) { std::printf("  File not found or unreadable: %s\n", path.c_str()); return false; }
    Tree* t = new Tree();
    t->bind(L, Sample::kind == 0 ? -1 : 0, 0);
    *tree = t;
    return true;
  }

  TreeNode<Sample>* root;

  // ---- binding to the loaded model (used by Forest / FaceForest)
  void bind(std::shared_ptr<detail::Loaded> L, int which, int index) {
    owner_ = L; which_ = which; index_ = index;
    const int n = crf_model_tree_dump(L->model, which, index, nullptr, 0);
    check(n);
    std::vector<int32_t> nodes((size_t)n * 16);
    check(crf_model_tree_dump(L->model, which, index, nodes.data(), n));
    const int nl = crf_model_leaf_dump(L->model, which, index, nullptr, 0);
    check(nl);
    std::vector<float> leaves((size_t)nl * 44);
    check(crf_model_leaf_dump(L->model, which, index, leaves.data(), nl));
    by_oid_.assign((size_t)n, nullptr);
    int next_leaf = 0;
    root = build(nodes, leaves, 0, next_leaf);
    m_num_nodes = i_node = (1 << (max_depth_ + 1)) - 1;   // a loaded tree is a finished one (Forest::load_tree rejects the others)
    registry().push_back(this);
  }
  std::shared_ptr<detail::Loaded> owner() const { return owner_; }
  int which() const { return which_; }
  int index() const { return index_; }
  Leaf* leaf_of(int object_id) { return by_oid_[(size_t)object_id]->getLeaf(); }

 private:
  TreeNode<Sample>* build(const std::vector<int32_t>& nodes, const std::vector<float>& leaves, int i, int& next_leaf) {
    const int32_t* o = &nodes[(size_t)i * 16];
    TreeNode<Sample>* nd = new TreeNode<Sample>();
    nd->depth = o[1]; nd->object_id = i; by_oid_[(size_t)i] = nd;
    max_depth_ = std::max(max_depth_, nd->depth);
    if (o[0]) { nd->is_leaf = true; detail::fill_leaf(nd->leaf, &leaves[(size_t)(next_leaf++) * 44]); return nd; }
    nd->has_split = true;
    nd->split.feature.feature_channel = o[2];
    nd->split.feature.rect1 = cvlite::Rect_<int>(o[3], o[4], o[5], o[6]);
    nd->split.feature.rect2 = cvlite::Rect_<int>(o[7], o[8], o[9], o[10]);
    nd->split.threshold = o[11];
    nd->left = build(nodes, leaves, o[12], next_leaf);     // pre-order: the left subtree's leaves come first
    nd->right = build(nodes, leaves, o[13], next_leaf);
    return nd;
  }
  int evaluate_root(const Sample* s) {
    const ImageSample* im = s->image();
    const cvlite::Rect r = const_cast<Sample*>(s)->getPatch();
    const int xy[2] = {r.x, r.y};
    const int zero = 0;
    if (which_ < 0) {   // the head-pose stage evaluates every tree of its forest: take this tree's column
      crf_model_info_t info;
      check(crf_model_info(owner_->model, &info));
      std::vector<int32_t> ids((size_t)info.hp_trees);
      check(crf_stage_eval_patches(owner_->context(), -1, nullptr, nullptr, 0, im->planes(), im->numChannels(), im->cols(), im->rows(), xy, 1, ids.data()));
      return ids[(size_t)index_];
    }
    int32_t id = 0;
    (void)zero;
    check(crf_stage_eval_patches(owner_->context(), 0, &which_, &index_, 1, im->planes(), im->numChannels(), im->cols(), im->rows(), xy, 1, &id));
    return id;
  }
  static std::vector<Tree*>& registry() { static std::vector<Tree*> r; return r; }
  static Tree* owner_of(TreeNode<Sample>* root_node) {
    for (Tree* t : registry()) if (t->root == root_node) return t;
    return nullptr;
  }
  int m_num_nodes, i_node;
  std::shared_ptr<detail::Loaded> owner_;
  int which_, index_;
  int max_depth_ = 0;
  std::vector<TreeNode<Sample>*> by_oid_;
};

// include/Forest.hpp:22-194.  Holds NON-OWNING Tree pointers, shared between a jungle and a composed forest, never freed
// (include/Forest.hpp:183, src/FaceForest.cpp:245,250; SURVEY Appendix E.12).
template <typename Sample> class Forest {
 public:
  typedef typename Sample::Split Split;
  typedef typename Sample::Leaf Leaf;
  Forest() {}
  void addTree(Tree<Sample>* tree) { m_trees.push_back(tree); }
  Tree<Sample>* getTree(int idx) { return m_trees[idx]; }
  int numberOfTrees() const { return static_cast<int>(m_trees.size()); }
  void cleanForest() { m_trees.clear(); }
  void setParam(ForestParam fp) { m_forest_param = fp; }
  ForestParam getParam() const { return m_forest_param; }

  // include/Forest.hpp:81-90: leafs[i] = leaf of tree i for this sample.  Trees of one loaded model go in one launch.
  void evaluateMT(const Sample* sample, Leaf** leafs) const {
    const ImageSample* im = sample->image();
    const cvlite::Rect r = const_cast<Sample*>(sample)->getPatch();
    const int xy[2] = {r.x, r.y};
    size_t i = 0;
    while (i < m_trees.size()) {
      size_t j = i;
      std::vector<int> fi, ti;
      while (j < m_trees.size() && m_trees[j]->owner() == m_trees[i]->owner()) { fi.push_back(std::max(m_trees[j]->which(), 0)); ti.push_back(m_trees[j]->index()); j++; }
      detail::Loaded& L = *m_trees[i]->owner();
      if (Sample::kind == 0) {
        crf_model_info_t info;
        check(crf_model_info(L.model, &info));
        std::vector<int32_t> ids((size_t)info.hp_trees);
        check(crf_stage_eval_patches(L.context(), -1, nullptr, nullptr, 0, im->planes(), im->numChannels(), im->cols(), im->rows(), xy, 1, ids.data()));
        for (size_t k = i; k < j; k++) leafs[k] = m_trees[k]->leaf_of(ids[(size_t)m_trees[k]->index()]);
      } else {
        std::vector<int32_t> ids(j - i);
        check(crf_stage_eval_patches(L.context(), 0, fi.data(), ti.data(), (int)(j - i), im->planes(), im->numChannels(), im->cols(), im->rows(), xy, 1, ids.data()));
        for (size_t k = i; k < j; k++) leafs[k] = m_trees[k]->leaf_of(ids[k - i]);
      }
      i = j;
    }
  }

  // include/Forest.hpp:103-129: tree_000 .. tree_{ntrees-1}; any missing or unfinished tree fails the whole load
  bool load(std::string path, ForestParam fp, int max_trees = -1) {
    setParam(fp);
    (void)max_trees;   // the reference's guard (numberOfTrees() > max_trees) never triggers with the default (SURVEY Appendix E.11)
    std::printf("> Trees to load: %d\n", fp.ntrees);
    std::shared_ptr<detail::Loaded> L(new detail::Loaded());
    L->device = detail::default_device();
    if (crf_model_load_forest(path.c_str(), fp.ntrees, Sample::kind, &L->model) != CRF_OK) return false;
    if (!fp.features.empty() && crf_model_set_features(L->model, fp.features.data(), (int)fp.features.size()) != CRF_OK) {
      std::fprintf(stderr, "(!) %s\n", crf_last_error());
      return false;
    }
    adopt(L, Sample::kind == 0 ? -1 : 0, fp.ntrees);
    return true;
  }
  // include/Forest.hpp:131-153
  static bool load_tree(std::string url, std::vector<Tree<Sample>*>& trees) {
    Tree<Sample>* tree;
    if (!Tree<Sample>::load(&tree, url)) return false;
    if (tree->isFinished()) { trees.push_back(tree); return true; }
    std::puts("  Tree is not finished successfully");
    delete tree;
    return false;
  }
  // trees [0, n) of forest `which` of an already loaded model (FaceForest's jungle)
  void adopt(std::shared_ptr<detail::Loaded> L, int which, int n) {
    for (int i = 0; i < n; i++) { Tree<Sample>* t = new Tree<Sample>(); t->bind(L, which, i); m_trees.push_back(t); }
  }
  // when every tree belongs to one loaded model: that model and the (forest, tree) list; else nullptr
  detail::Loaded* single_owner(std::vector<int>& fi, std::vector<int>& ti) const {
    fi.clear(); ti.clear();
    for (Tree<Sample>* t : m_trees) {
      if (t->owner() != m_trees[0]->owner()) return nullptr;
      fi.push_back(std::max(t->which(), 0)); ti.push_back(t->index());
    }
    return m_trees.empty() ? nullptr : m_trees[0]->owner().get();
  }

 private:
  std::vector<Tree<Sample>*> m_trees;
  ForestParam m_forest_param;
};

// ------------------------------------------------------------------------------------------------ face_utils
// src/face_utils.cpp:325-347
inline cvlite::Rect intersect(const cvlite::Rect r1, const cvlite::Rect r2) {
  cvlite::Rect in;
  in.x = (r1.x < r2.x) ? r2.x : r1.x;
  in.y = (r1.y < r2.y) ? r2.y : r1.y;
  in.width = ((r1.x + r1.width < r2.x + r2.width) ? r1.x + r1.width : r2.x + r2.width) - in.x;
  in.height = ((r1.y + r1.height < r2.y + r2.height) ? r1.y + r1.height : r2.y + r2.height) - in.y;
  if (in.width <= 0 || in.height <= 0) in = cvlite::Rect(0, 0, 0, 0);
  return in;
}

namespace detail {
inline void require_whole_sample(const ImageSample& s, const cvlite::Rect& b) {
  if (b.x != 0 || b.y != 0 || b.width != s.cols() || b.height != s.rows())
    throw std::invalid_argument("the face box must cover the whole ImageSample, as in FaceForest::analyzeFace (src/FaceForest.cpp:211,253)");
}
}  // namespace detail

// src/face_utils.cpp:183-242 (include/face_utils.hpp:78-88)
inline void getHeadPoseVotesMT(const ImageSample& sample, const Forest<HeadPoseSample>& forest, cvlite::Rect face_bbox, float* headpose, float* variance,
                               HeadPoseEstimatorOption options = HeadPoseEstimatorOption()) {
  detail::require_whole_sample(sample, face_bbox);
  std::vector<int> fi, ti;
  detail::Loaded* L = forest.single_owner(fi, ti);
  crf_model_info_t info;
  if (L) check(crf_model_info(L->model, &info));
  if (!L || (int)ti.size() != info.hp_trees) throw std::invalid_argument("getHeadPoseVotesMT expects a forest as Forest::load or FaceForest made it");
  crf_options_t co = detail::make_options(options, MultiPartEstimatorOption(), MeanShiftOption(), CRF_MS_DEFAULT);
  check(crf_stage_headpose(L->context(co), sample.planes(), sample.numChannels(), sample.cols(), sample.rows(), options.step_size, headpose, variance, nullptr, nullptr,
                           nullptr, nullptr, nullptr, nullptr));
}

// src/face_utils.cpp:244-302 (include/face_utils.hpp:90-99): votes[i] is appended to, in the reference's order
inline void getFacialFeaturesVotesMT(const ImageSample& sample, const Forest<MPSample>& forest, cvlite::Rect face_bbox, std::vector<std::vector<Vote> >& votes,
                                     MultiPartEstimatorOption options = MultiPartEstimatorOption()) {
  detail::require_whole_sample(sample, face_bbox);
  std::vector<int> fi, ti;
  detail::Loaded* L = forest.single_owner(fi, ti);
  if (!L) throw std::invalid_argument("getFacialFeaturesVotesMT expects trees of one loaded model");
  crf_options_t co = detail::make_options(HeadPoseEstimatorOption(), options, MeanShiftOption(), CRF_MS_DEFAULT);
  crf_ctx* ctx = L->context(co);
  int n_votes[CRF_NUM_PARTS];
  check(crf_stage_votes_meanshift(ctx, fi.data(), ti.data(), (int)ti.size(), sample.planes(), sample.numChannels(), sample.cols(), sample.rows(), options.step_size, n_votes,
                                  nullptr, 0, nullptr, nullptr, nullptr));
  int cap = 1;
  for (int p = 0; p < CRF_NUM_PARTS; p++) cap = std::max(cap, n_votes[p]);
  std::vector<float> xyw((size_t)CRF_NUM_PARTS * cap * 3);
  check(crf_stage_votes_meanshift(ctx, fi.data(), ti.data(), (int)ti.size(), sample.planes(), sample.numChannels(), sample.cols(), sample.rows(), options.step_size, n_votes,
                                  xyw.data(), cap, nullptr, nullptr, nullptr));
  for (size_t p = 0; p < votes.size() && p < (size_t)CRF_NUM_PARTS; p++)
    for (int k = 0; k < n_votes[p]; k++) {
      Vote v;
      const float* o = &xyw[((size_t)p * cap + k) * 3];
      v.pos.x = (int)o[0]; v.pos.y = (int)o[1]; v.weight = o[2]; v.check = true;
      votes[p].push_back(v);
    }
}

// src/face_utils.cpp:304-323 (include/face_utils.hpp:101-108)
inline float areaUnderCurve(float x1, float x2, double mean, double std_) {
  float a = 0.f;
  check(crf_stage_area_under_curve(detail::plain_context(), x1, x2, mean, std_, &a));
  return a;
}

// ------------------------------------------------------------------------------------------------ MeanShift
// include/MeanShift.hpp:27-136
class MeanShift {
 public:
  MeanShift() {}
  virtual ~MeanShift() {}
  static void shift(const std::vector<Vote>& votes, cvlite::Point_<int>& result, MeanShiftOption& option) {
    shift(votes, result, option.max_iterations, option.kernel_size, option.stopping_criteria);
  }
  static void shift(const std::vector<Vote>& votes, cvlite::Point_<int>& result, int num_iterations, int kernel, float stopping_criteria) {
    std::vector<float> v;
    v.reserve(votes.size() * 3);
    for (const Vote& q : votes)
      if (q.check) { v.push_back((float)q.pos.x); v.push_back((float)q.pos.y); v.push_back(q.weight); }
    int r[2] = {0, 0};
    check(crf_stage_meanshift_opt(detail::plain_context(), v.data(), (int)(v.size() / 3), kernel, num_iterations, stopping_criteria, nullptr, r, nullptr));
    result = cvlite::Point_<int>(r[0], r[1]);
  }
};

// ------------------------------------------------------------------------------------------------ CascadeClassifier
// cv::CascadeClassifier as FaceForest uses it (src/FaceForest.cpp:23, :145): load() + detectMultiScale(), the cascade evaluated on the GPU
class CascadeClassifier {
 public:
  CascadeClassifier() {}
  explicit CascadeClassifier(const std::string& filename) { load(filename); }
  ~CascadeClassifier() { if (c_) crf_cascade_free(c_); }
  CascadeClassifier(const CascadeClassifier&) = delete;
  CascadeClassifier& operator=(const CascadeClassifier&) = delete;
  bool empty() const { return c_ == nullptr; }
  bool load(const std::string& filename) {
    crf_cascade* n = nullptr;
    if (crf_cascade_load(filename.c_str(), &n) != CRF_OK) return false;
    if (c_) crf_cascade_free(c_);
    c_ = n;
    return true;
  }
  // min_size: cv::Size(min, min) of the reference's call
  void detectMultiScale(const cvlite::Mat& image, std::vector<cvlite::Rect>& objects, double scaleFactor = 1.1, int minNeighbors = 3, int flags = 0, int min_size = 0) {
    (void)flags;
    if (!c_) throw std::logic_error("CascadeClassifier::detectMultiScale on an empty classifier");
    if (image.channels() != 3) throw std::invalid_argument("detectMultiScale expects an 8-bit BGR image");
    std::vector<crf_rect_t> r(256);
    int n = crf_detect_faces(detail::plain_context(), c_, image.data, image.rows, image.cols, image.step, scaleFactor, minNeighbors, min_size, r.data(), (int)r.size());
    check(n);
    if (n > (int)r.size()) { r.resize((size_t)n); n = crf_detect_faces(detail::plain_context(), c_, image.data, image.rows, image.cols, image.step, scaleFactor, minNeighbors, min_size, r.data(), n); check(n); }
    objects.clear();
    for (int i = 0; i < n; i++) objects.push_back(cvlite::Rect(r[(size_t)i].x, r[(size_t)i].y, r[(size_t)i].width, r[(size_t)i].height));
  }
 private:
  crf_cascade* c_ = nullptr;
};

// ------------------------------------------------------------------------------------------------ FaceForest
// include/FaceForest.hpp:81-157, src/FaceForest.cpp
class FaceForest {
 public:
  FaceForest() : is_inizialized(false) {}
  explicit FaceForest(FaceForestOptions option) : is_inizialized(false) { load(option); }   // include/FaceForest.hpp:88-91
  virtual ~FaceForest() {}
  FaceForest(const FaceForest&) = delete;
  FaceForest& operator=(const FaceForest&) = delete;

  // src/FaceForest.cpp:15-58: on failure prints the error and leaves the object un-initialised.  A tree path that names a pre-packed
  // image (*.crfb200, written by crf_model_save_packed) holds both forests.
  bool load(const FaceForestOptions& o) {
    is_inizialized = false;
    m_options = o;
    if (!o.fd_option.path_face_cascade.empty()) {   // src/FaceForest.cpp:21-28
      std::puts("Loading face cascade classifier");
      if (!m_face_cascade.load(o.fd_option.path_face_cascade)) { std::fprintf(stderr, "(!) Error loading cascade classifier\n"); return false; }
    }
    loaded_.reset(new detail::Loaded());
    loaded_->device = o.device;
    m_hp_forest = Forest<HeadPoseSample>(); m_mp_forest = Forest<MPSample>(); m_mp_jungle.clear();
    const std::string& tp = o.mp_forest_param.tree_path;
    const bool packed = tp.size() > 8 && tp.compare(tp.size() - 8, 8, ".crfb200") == 0;
    int rc = packed ? crf_model_load_packed(tp.c_str(), &loaded_->model)
                    : crf_model_load(o.hp_forest_param.tree_path.c_str(), o.hp_forest_param.ntrees, tp.c_str(), o.mp_forest_param.ntrees, &loaded_->model);
    if (rc != CRF_OK) { std::fprintf(stderr, "(!) Error loading forest: %s\n", crf_last_error()); return false; }
    // the one ImageSample of a face is built from hp_forest_param.features (src/FaceForest.cpp:207)
    if (!o.hp_forest_param.features.empty() && crf_model_set_features(loaded_->model, o.hp_forest_param.features.data(), (int)o.hp_forest_param.features.size()) != CRF_OK) {
      std::fprintf(stderr, "(!) Error loading forest: %s\n", crf_last_error());
      return false;
    }
    crf_model_info_t info;
    check(crf_model_info(loaded_->model, &info));
    if (!packed) {   // src/FaceForest.cpp:39-44: the sorted sub-directories of the FFD tree path
      if (DIR* d = ::opendir(tp.c_str())) {
        while (dirent* e = ::readdir(d)) {
          const std::string n = e->d_name, p = tp + "/" + n;
          struct stat st;
          if (n != "." && n != ".." && ::stat(p.c_str(), &st) == 0 && S_ISDIR(st.st_mode)) m_options.mp_forest_paths.push_back(p);
        }
        ::closedir(d);
      }
      std::sort(m_options.mp_forest_paths.begin(), m_options.mp_forest_paths.end());
    }
    try {
      loaded_->context(options());
    } catch (const std::exception& e) {
      std::fprintf(stderr, "(!) Error creating the GPU context: %s\n", e.what());
      return false;
    }
    m_hp_forest.setParam(o.hp_forest_param);
    m_hp_forest.adopt(loaded_, -1, info.hp_trees);
    m_mp_jungle.resize((size_t)info.mp_forests);
    for (int f = 0; f < info.mp_forests; f++) { m_mp_jungle[(size_t)f].setParam(o.mp_forest_param); m_mp_jungle[(size_t)f].adopt(loaded_, f, info.mp_trees / std::max(info.mp_forests, 1)); }
    is_inizialized = true;
    return true;
  }

  // include/FaceForest.hpp:97-106, src/FaceForest.cpp:60-72
  static void estimateHeadPose(const ImageSample& sample, const cvlite::Rect& face_bbox, const Forest<HeadPoseSample>& forest, HeadPoseEstimatorOption options,
                               float* headpose, float* variance) {
    getHeadPoseVotesMT(sample, forest, face_bbox, headpose, variance, options);
  }

  // include/FaceForest.hpp:108-116, src/FaceForest.cpp:74-95: votes + MeanShift::shift x num_parts with a default MeanShiftOption
  static void estimateFacialFeatures(const ImageSample& sample, const cvlite::Rect face_bbox, const Forest<MPSample>& forest, MultiPartEstimatorOption options,
                                     std::vector<cvlite::Point>& ffd_cordinates) {
    detail::require_whole_sample(sample, face_bbox);
    std::vector<int> fi, ti;
    detail::Loaded* L = forest.single_owner(fi, ti);
    if (!L) throw std::invalid_argument("estimateFacialFeatures expects trees of one loaded model");
    crf_options_t co = detail::make_options(HeadPoseEstimatorOption(), options, MeanShiftOption(), CRF_MS_DEFAULT);
    int rounded[CRF_NUM_PARTS][2];
    check(crf_stage_votes_meanshift(L->context(co), fi.data(), ti.data(), (int)ti.size(), sample.planes(), sample.numChannels(), sample.cols(), sample.rows(),
                                    options.step_size, nullptr, nullptr, 0, nullptr, rounded, nullptr));
    ffd_cordinates.clear();
    ffd_cordinates.resize((size_t)options.num_parts);
    for (int i = 0; i < options.num_parts && i < CRF_NUM_PARTS; i++) ffd_cordinates[(size_t)i] = cvlite::Point(rounded[i][0], rounded[i][1]);
  }

  // src/FaceForest.cpp:136-159: the box enlargement of detectFace applied to given detections (5 % of the width left and right, 15 % of
  // the WIDTH added to the height twice, clipped to the image)
  static void enlargeDetections(const cvlite::Mat& img, std::vector<cvlite::Rect>& faces_bboxes) {
    for (unsigned int i = 0; i < faces_bboxes.size(); i++) {
      int offset_x = faces_bboxes[i].width * 0.05;
      int offset_y = faces_bboxes[i].width * 0.15;
      cvlite::Rect r1 = cvlite::Rect(faces_bboxes[i].x - offset_x, faces_bboxes[i].y, faces_bboxes[i].width + (offset_x * 2), faces_bboxes[i].height + (offset_y * 2));
      faces_bboxes[i] = intersect(r1, cvlite::Rect(0, 0, img.cols, img.rows));
    }
  }

  // include/FaceForest.hpp:118-126, src/FaceForest.cpp:136-159
  static void detectFace(const cvlite::Mat& img, CascadeClassifier& face_cascade, FaceDetectionOption fd_option, std::vector<cvlite::Rect>& faces_bboxes) {
    face_cascade.detectMultiScale(img, faces_bboxes, fd_option.search_scale_factor, fd_option.min_neighbors, 0, fd_option.min_feature_size);
    enlargeDetections(img, faces_bboxes);   // the face detection boxes are too tight for us
  }

  // include/FaceForest.hpp:128-133, src/FaceForest.cpp:161-181: detect, then analyse every face (appended to `faces`)
  void analyzeImage(cvlite::Mat img, std::vector<Face>& faces) {
    require_init();
    if (m_face_cascade.empty()) throw std::logic_error("analyzeImage(img, faces) needs fd_option.path_face_cascade; pass the boxes otherwise");
    std::vector<cvlite::Rect> faces_bboxes;
    detectFace(img, m_face_cascade, m_options.fd_option, faces_bboxes);
    analyze(img, faces_bboxes, faces, true);
  }

  // the same with the face boxes supplied by the caller: one launch for all faces of the frame
  void analyzeImage(cvlite::Mat img, const std::vector<cvlite::Rect>& faces_bboxes, std::vector<Face>& faces) {
    require_init();
    analyze(img, faces_bboxes, faces, true);
  }

  // src/FaceForest.cpp:183-258
  void analyzeFace(const cvlite::Mat img, cvlite::Rect face_bbox, Face& face) {
    require_init();
    std::vector<Face> faces;
    analyze(img, std::vector<cvlite::Rect>(1, face_bbox), faces, false);
    face = faces[0];
  }

  bool is_inizialized;   // sic (include/FaceForest.hpp:153)
  crf_ctx* context() { return loaded_ ? loaded_->context(options()) : nullptr; }
  // the loaded forests, as the reference's private members hold them
  Forest<HeadPoseSample>& headPoseForest() { return m_hp_forest; }
  std::vector<Forest<MPSample> >& jungle() { return m_mp_jungle; }
  Forest<MPSample>& composedForest() { return m_mp_forest; }   // m_mp_forest after the last analyzeFace (src/FaceForest.cpp:239-250)

 private:
  crf_options_t options() const { return detail::make_options(m_options.hp_option, m_options.mp_option, m_options.mean_shift_option, m_options.ms_mode); }
  void require_init() const {
    if (!is_inizialized) throw std::logic_error("CV_Assert(is_inizialized) failed (src/FaceForest.cpp:167,191)");
  }
  void analyze(const cvlite::Mat& img, const std::vector<cvlite::Rect>& boxes, std::vector<Face>& faces, bool append) {
    if (img.channels() != 3) throw std::invalid_argument("analyzeFace expects an 8-bit BGR image");
    std::vector<crf_rect_t> r(boxes.size());
    for (size_t i = 0; i < boxes.size(); i++) r[i] = crf_rect_t{boxes[i].x, boxes[i].y, boxes[i].width, boxes[i].height};
    std::vector<crf_face_t> out(boxes.size());
    if (m_options.device < 0) {
      const uint8_t* frames[1] = {img.data};
      const std::vector<int> zero(boxes.size(), 0);
      check(crf_multi_analyze_batch(loaded_->all_gpus(options()), frames, 1, img.rows, img.cols, img.step, r.data(), zero.data(), (int)r.size(), out.data()));
    } else {
      check(crf_analyze_faces(context(), img.data, img.rows, img.cols, img.step, r.data(), (int)r.size(), out.data()));
    }
    if (!append) faces.clear();
    for (size_t i = 0; i < boxes.size(); i++) {
      Face f;
      f.headpose = out[i].headpose;
      f.bbox = boxes[i];
      f.ffd_cordinates.resize(CRF_NUM_PARTS);
      for (int p = 0; p < CRF_NUM_PARTS; p++) f.ffd_cordinates[(size_t)p] = cvlite::Point(out[i].ffd[p][0], out[i].ffd[p][1]);
      faces.push_back(f);
    }
    if (!boxes.empty()) {   // m_mp_forest as analyzeFace leaves it: floor(pose_freq * ntrees) trees per pose forest, topped up from the dominant one
      const crf_face_t& last = out.back();
      m_mp_forest.setParam(m_options.mp_forest_param);
      m_mp_forest.cleanForest();
      for (size_t f = 0; f < m_mp_jungle.size() && f < (size_t)CRF_NUM_POSE_FORESTS; f++)
        for (int j = 0; j < last.tree_counts[f]; j++) m_mp_forest.addTree(m_mp_jungle[f].getTree(j));
      for (int i = m_mp_forest.numberOfTrees(); i < m_options.mp_forest_param.ntrees && i < m_mp_jungle[(size_t)last.dominant].numberOfTrees(); i++)
        m_mp_forest.addTree(m_mp_jungle[(size_t)last.dominant].getTree(i));
    }
  }
  FaceForestOptions m_options;
  CascadeClassifier m_face_cascade;
  std::shared_ptr<detail::Loaded> loaded_;
  Forest<HeadPoseSample> m_hp_forest;
  Forest<MPSample> m_mp_forest;
  std::vector<Forest<MPSample> > m_mp_jungle;
};

}  // namespace crf_b200
#endif  // CRF_B200_COMPAT_HPP
