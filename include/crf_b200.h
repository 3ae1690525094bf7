/* =============================================================================
 * crf_b200.h — C ABI of the B200-native Conditional Regression Forest inference path.
 *
 * Drop-in boundary for the hot path of MatrixPlayer/face_alignment_cvpr_2012
 * (citations are file:line under the reference tree).  The reference has no FFI layer; its
 * boundary is the C++ class API called by its mains (src/eval_ffd.cpp:89,
 * src/eval_headpose.cpp:66, src/demo.cpp:154, src/test_cvpr_2012.cpp:44).  The entry points
 * below are what a binding of that API needs; include/crf_b200_compat.hpp re-exposes the
 * reference's class names/signatures on top of them.
 *
 * Conventions: plain pointers and sizes; opaque handles; every function returns 0 on success and
 * a negative crf_status on error (crf_last_error() gives the message, mirroring the reference's
 * bool + ERROR(...) print); the caller owns all in/out buffers; the library owns device memory
 * behind a crf_ctx; one crf_ctx belongs to one GPU and is used by one host thread at a time (the
 * reference's FaceForest is not re-entrant either: src/FaceForest.cpp:239-250).
 * There is NO CPU fallback: without a CUDA device crf_ctx_create fails.
 * ============================================================================= */
#ifndef CRF_B200_H
#define CRF_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CRF_NUM_PARTS 10          /* MultiPartEstimatorOption::num_parts   include/FaceForest.hpp:49 */
#define CRF_NUM_POSE_FORESTS 5    /* poseT hard-codes 5 bins               src/FaceForest.cpp:216-222 */
#define CRF_NUM_HEADPOSE_CLASSES 5/* NUM_HEADPOSE_CLASSES                  include/Constants.hpp:66   */
#define CRF_MAX_SCALED_H 521      /* f32 integral exactness limit (sums < 2^24), SURVEY H7           */
#define CRF_ROW_STRIDE 128        /* elements per integral row on the device                          */

typedef enum {
  CRF_OK = 0,
  CRF_ERR_ARG = -1,        /* bad argument / box outside image / face too small or too tall        */
  CRF_ERR_IO = -2,         /* file not found / unreadable          (Tree::load, include/Tree.hpp:202) */
  CRF_ERR_FORMAT = -3,     /* archive does not parse / unfinished tree (Forest::load_tree :142-152)  */
  CRF_ERR_CUDA = -4,       /* CUDA runtime error or no device                                        */
  CRF_ERR_STATE = -5,      /* use before init                       (CV_Assert, src/FaceForest.cpp:167) */
  CRF_ERR_UNSUPPORTED = -6 /* model outside the packed-format limits (channel > 63, rect > 31, ...)  */
} crf_status;

typedef struct crf_model crf_model; /* host-side forests: what FaceForest's ctor loads (src/FaceForest.cpp:15-58) */
typedef struct crf_ctx crf_ctx;     /* per-GPU context: packed forests + work buffers                */

typedef struct { int x, y, width, height; } crf_rect_t; /* cv::Rect  include/opencv_serialization.hpp:65-72 */
/* one BGR frame (cv::Mat CV_8UC3) of any size: rows x cols pixels, step bytes from one row to the next (step >= cols * 3) */
typedef struct { const uint8_t* bgr; int rows, cols; size_t step; } crf_image_t;

/* HeadPoseEstimatorOption + MultiPartEstimatorOption (include/FaceForest.hpp:33-58) and
 * MeanShiftOption (include/MeanShift.hpp:16-25); crf_options_default() fills the reference defaults. */
typedef struct {
  int   hp_stride;             /* step_size = 4 */
  float hp_min_foreground;     /* min_foreground_probability = 0.5 */
  int   ffd_stride;            /* step_size = 3 */
  int   ffd_min_samples;       /* 2 */
  float ffd_min_foreground;    /* min_forground = 0.5 */
  float ffd_min_pf;            /* 0.25 (x1.5 for parts 0 and 7, src/face_utils.cpp:286-287) */
  float ffd_max_variance;      /* 25 */
  int   ms_kernel_size;        /* 10 */
  int   ms_max_iterations;     /* 7 */
  float ms_stopping_criteria;  /* 0.05 */
  int   max_chunk;             /* faces per launch; 0 = as many as fit min(64 GB, half the free memory), at most 4096 */
  int   max_scaled_h;          /* ignored: work buffers grow on demand (kept for ABI stability) */
  int   ms_mode;               /* CRF_MS_DEFAULT / CRF_MS_EXACT / CRF_MS_FAST, see below */
} crf_options_t;

/* How MeanShift::shift's sums (include/MeanShift.hpp:79-135) are evaluated.
 * CRF_MS_EXACT: the reference's sequential f32 order, double-precision norm and glibc-identical expf: iteration counts identical,
 *               means within 1e-3 px of the CPU reference (observed 0.0 on every campaign face).
 * CRF_MS_FAST:  the same iteration with tree-reduced f32 sums and a hardware exp2: deterministic, within the 0.5 px landmark
 *               tolerance of the north star (observed <= 0.024 px on 3543 campaign faces), ~8x faster.  Head pose, forest composition, leaf ids and the
 *               vote lists are bit-exact in both modes.
 * CRF_MS_DEFAULT = CRF_MS_FAST unless the environment says CRF_MS_MODE=exact. */
enum { CRF_MS_DEFAULT = 0, CRF_MS_EXACT = 1, CRF_MS_FAST = 2 };

/* Face (include/FaceForest.hpp:70-75) plus the intermediate results the parity tests need. */
typedef struct {
  float headpose, variance;          /* src/face_utils.cpp:236-241 */
  int   tree_counts[CRF_NUM_POSE_FORESTS]; /* trees taken from each pose forest (src/FaceForest.cpp:241-246) */
  int   dominant;                    /* dominant_headpose (:231-235) */
  int   scaled_w, scaled_h;          /* size after cv::resize (:204) */
  float scale;                       /* face_size / bbox.width (:202) */
  float ffd_f[CRF_NUM_PARTS][2];     /* MeanShift mean before rounding, scaled-face pixels */
  int   ffd_scaled[CRF_NUM_PARTS][2];/* Point_<int> = Point_<float> (include/MeanShift.hpp:75) */
  int   ffd[CRF_NUM_PARTS][2];       /* ffd_cordinates after *= 1/scale (src/FaceForest.cpp:256-257): bbox-relative original pixels */
  int   ms_iters[CRF_NUM_PARTS];     /* MeanShift iterations executed */
  int   n_votes[CRF_NUM_PARTS];      /* votes per part (src/face_utils.cpp:289-298) */
  int   flags;                       /* bit0: composition clamped (reference would index out of bounds); bits 1-2 are internal
                                        (face re-run with worst-case capacities) and never set in returned records;
                                        bit3: CRF_FACE_NOT_ANALYSED (crf_analyze_images only) */
} crf_face_t;

/* crf_face_t::flags of a detected box that the analysis path cannot take (record otherwise zero) */
#define CRF_FACE_NOT_ANALYSED 8

typedef struct {
  int hp_trees, hp_nodes, hp_leaves, hp_max_depth;
  int mp_forests, mp_trees, mp_nodes, mp_leaves, mp_max_depth;
  int patch_size, face_size, num_channels;
  int hp_ntrees_cfg, mp_ntrees_cfg;
} crf_model_info_t;

/* Work counters of the calls since the last reset (exact, counted on the device). */
typedef struct {
  unsigned long long faces;
  unsigned long long hp_node_tests, ffd_node_tests; /* internal-node tests (one 16-B record + 8 integral samples each) */
  unsigned long long hp_traversals, ffd_traversals; /* (patch, tree) pairs */
  unsigned long long votes;                         /* votes emitted */
  unsigned long long vote_passes;                   /* sum over (face, part) of votes x (1 + MeanShift iterations) */
  unsigned long long kernel_launches;               /* CUDA kernels launched by this library */
  unsigned long long h2d_bytes, d2h_bytes;
} crf_counters_t;

enum { CRF_STAGE_RESIZE = 0, CRF_STAGE_PLAIN, CRF_STAGE_GABOR, CRF_STAGE_HP_TRAVERSE, CRF_STAGE_HP_REDUCE,
       CRF_STAGE_FFD_TRAVERSE, CRF_STAGE_VOTES, CRF_STAGE_MEANSHIFT, CRF_NUM_STAGES };

const char* crf_last_error(void);
const char* crf_version(void);
void crf_options_default(crf_options_t* opt);

/* ---- model: Forest<S>::load / Tree<S>::load (include/Forest.hpp:103-153, include/Tree.hpp:193-237) and the
 * jungle enumeration of FaceForest::FaceForest (src/FaceForest.cpp:39-55: sub-directories of ffd_dir, sorted). */
int crf_model_load(const char* hp_dir, int hp_ntrees, const char* ffd_dir, int ffd_ntrees, crf_model** out);
/* "next" row f1: pre-packed binary image of the same forests (versioned, checksummed). */
int crf_model_save_packed(const crf_model* m, const char* path);
int crf_model_load_packed(const char* path, crf_model** out);
/* Forest<S>::load on its own (include/Forest.hpp:103-129): a model with only the head-pose forest (kind 0) or only one
 * facial-feature forest (kind 1).  Enough for the Forest / Tree / ImageSample level of the interface (crf_stage_eval_forest,
 * crf_stage_eval_patches, crf_stage_headpose's mean / variance); crf_analyze_* need crf_model_load. */
int crf_model_load_forest(const char* dir, int ntrees, int kind, crf_model** out);
/* Tree<S>::load(Tree**, path) (include/Tree.hpp:193-237): a model holding the single tree of one archive file (kind 0 / 1). */
int crf_model_load_tree(const char* path, int kind, crf_model** out);
/* ForestParam::features as the run-time configuration gives them (data/config_*.txt; src/FaceForest.cpp:207 builds the one
 * ImageSample of a face from hp_forest_param.features): any subset of {0 GRAY, 1 GABOR, 2 SOBEL, 3 MIN_MAX, 4 CANNY, 5 NORM}
 * (include/FeatureChannelFactory.hpp:18-23), sorted by the library as src/ImageSample.cpp:86 does.  Default: the list stored in the
 * archives.  Fails with CRF_ERR_UNSUPPORTED if a split of the model reads a plane the list does not provide. */
int crf_model_set_features(crf_model* m, const int* features, int n);
int crf_model_get_features(const crf_model* m, int* features, int cap);   /* returns the count */
int crf_model_info(const crf_model* m, crf_model_info_t* info);
/* Leaf payloads of one tree (which = -1 head pose, 0..4 pose forest) in pre-order leaf numbering, 44 floats per leaf:
 * head pose: [object_id, hp_nsamples, hp_foreground, hp_labels[5]]  (include/HeadPoseSample.hpp:144-162);
 * pose forest: [object_id, mp_samples, mp_foreground, mp_parts_offset[10][2], mp_parts_variance[10], mp_prob_foreground[10]]
 * (include/MPSample.hpp:137-159).  Returns the leaf count. */
int crf_model_leaf_dump(const crf_model* m, int which, int tree, float* out, int cap_leaves);
/* Pre-order dump of one tree (which = -1 head pose, 0..4 pose forest), 16 ints per node:
 * [is_leaf, depth, ch, r1x,r1y,r1w,r1h, r2x,r2y,r2w,r2h, thr, left_oid, right_oid, nsamples, object_id] */
int crf_model_tree_dump(const crf_model* m, int which, int tree, int32_t* out, int cap_nodes);
/* Host-only self-check of the device image of the forests (the node-record forms the kernels read agree: wide, compact, window, and
 * the internal-nodes-only form walked from every root; children are adjacent, window leaves self-loop); returns the number of records
 * checked or a negative status. */
int crf_model_check_packing(const crf_model* m, int* max_extent_hp, int* max_extent_ffd);
void crf_model_free(crf_model* m);

/* ---- context */
int crf_device_count(void);
/* m may be NULL: a context without forests, for the stages that need none (feature channels, evalTest, MeanShift). */
int crf_ctx_create(const crf_model* m, int device, const crf_options_t* opt, crf_ctx** out);
void crf_ctx_destroy(crf_ctx* ctx);
int crf_ctx_set_profiling(crf_ctx* ctx, int on);                  /* CUDA events around every stage */
int crf_ctx_stage_ms(crf_ctx* ctx, float ms[CRF_NUM_STAGES], int launches[CRF_NUM_STAGES]); /* accumulated since reset */
int crf_ctx_counters(crf_ctx* ctx, crf_counters_t* c);
int crf_ctx_reset_counters(crf_ctx* ctx);
void* crf_ctx_stream(crf_ctx* ctx);                               /* cudaStream_t the kernels run on */
/* pinned host memory for callers that want the fast H2D path */
int crf_host_alloc(void** p, size_t bytes);
void crf_host_free(void* p);

/* ---- FaceForest::analyzeFace (src/FaceForest.cpp:183-258) for n boxes of one BGR frame
 * (analyzeImage with the Haar boxes given, :161-181).
 * Argument checking is all-or-nothing: every box is validated before any work starts (inside the image; scaled face larger than a
 * 31-px patch, at most 125 wide and CRF_MAX_SCALED_H tall) and ONE bad box fails the whole call with CRF_ERR_ARG, leaving `out`
 * untouched — the reference would throw out of cv::Mat::operator() for that face in the middle of its loop.  Callers that take boxes
 * from a detector should clip them first (crf_b200::FaceForest::detectFace does, as src/FaceForest.cpp:152-157). */
int crf_analyze_faces(crf_ctx* ctx, const uint8_t* bgr, int rows, int cols, size_t step,
                      const crf_rect_t* boxes, int n, crf_face_t* out);
/* n boxes spread over n_images equal-size frames; image_of_box[i] selects the frame of box i. */
int crf_analyze_batch(crf_ctx* ctx, const uint8_t* const* images, int n_images, int rows, int cols, size_t step,
                      const crf_rect_t* boxes, const int* image_of_box, int n, crf_face_t* out);
/* crf_analyze_batch on frames of any sizes: images[k] describes frame k, and each box is validated against its own frame.  Argument
 * checking is all-or-nothing as above; every descriptor needs a non-null bgr, rows, cols >= 1 and step >= cols * 3.
 * Pinned and pageable frames may be mixed.  crf_analyze_faces, crf_analyze_batch and the crops calls are this call on equal-size frames. */
int crf_analyze_batch_mixed(crf_ctx* ctx, const crf_image_t* images, int n_images, const crf_rect_t* boxes, const int* image_of_box, int n,
                            crf_face_t* out);
/* n equal-size crops stored back to back (n x rows x cols x 3), box = whole crop. */
int crf_analyze_crops(crf_ctx* ctx, const uint8_t* bgr_batch, int n, int rows, int cols, crf_face_t* out);
/* stop after getHeadPoseVotesMT (src/face_utils.cpp:183-242): fills headpose, variance, scaled_*, scale. */
int crf_headpose_crops(crf_ctx* ctx, const uint8_t* bgr_batch, int n, int rows, int cols, crf_face_t* out);
/* same two, inputs and outputs already resident in device memory (d_out: n x crf_face_t); asynchronous
 * on crf_ctx_stream(); used to measure the kernel path without PCIe. */
int crf_analyze_crops_device(crf_ctx* ctx, const uint8_t* d_bgr_batch, int n, int rows, int cols, crf_face_t* d_out, int headpose_only);

/* ---- FaceForest::detectFace's box source (src/FaceForest.cpp:136-146): cv::CascadeClassifier::load on the reference's
 * data/haarcascade_frontalface_alt.xml and detectMultiScale(img, boxes, search_scale_factor, min_neighbors, 0, Size(min_feature_size,
 * min_feature_size)) with the cascade evaluated on the GPU.  The boxes are the RAW detections: the enlargement of
 * src/FaceForest.cpp:147-157 is the caller's (crf_b200::FaceForest::detectFace does both).
 * Returns the number of boxes (the first `cap` are written) or a negative status.
 * crf_cascade_load reads OpenCV's HAAR cascades as cv::CascadeClassifier::load does: the new format (opencv-cascade-classifier) with stump
 * or tree weak classifiers (up to 16 nodes a tree) and upright or 45-degree tilted features, and the old opencv-haar-classifier format
 * with its stages in a chain.  It fails with CRF_ERR_IO (no file), CRF_ERR_FORMAT (not a cascade; a tree whose child does not follow
 * its parent, with an unreachable node or a leaf index out of range; a rect outside the window) or CRF_ERR_UNSUPPORTED (LBP / HOG
 * features, categorical splits (maxCatCount > 0), old-format stage trees).  crf_cascade_info's nweak counts weak classifiers, not nodes. */
typedef struct crf_cascade crf_cascade;
int crf_cascade_load(const char* path, crf_cascade** out);
void crf_cascade_free(crf_cascade* c);
int crf_cascade_info(const crf_cascade* c, int* win_w, int* win_h, int* nstages, int* nweak);
int crf_detect_faces(crf_ctx* ctx, const crf_cascade* c, const uint8_t* bgr, int rows, int cols, size_t step, double scale_factor,
                     int min_neighbors, int min_size, crf_rect_t* out, int cap);
/* detectMultiScale on n_images equal-size frames in one call.  Boxes are grouped by frame in frame order; within a frame they are
 * exactly what crf_detect_faces returns for that frame, in the same order.  image_of_box[i] = frame of box i.
 * Each frame crosses PCIe once.  Frames are processed in groups of consecutive frames: at most 64, no more than half the context's work
 * budget (min(64 GB, half the free memory)) holds, and fewer than 2^32 windows.  A group is a table of (frame, pyramid level)
 * instances; each pyramid pass, cascade stage group and scan step of a group is one launch over all of them.
 * cap smaller than the box count: every frame is still searched, the true count is returned and the first `cap` boxes are written
 * (cap = 0 sizes a buffer).  Returns the total box count or a negative status. */
int crf_detect_faces_batch(crf_ctx* ctx, const crf_cascade* c, const uint8_t* const* images, int n_images, int rows, int cols,
                           size_t step, double scale_factor, int min_neighbors, int min_size,
                           crf_rect_t* out, int* image_of_box, int cap);
/* crf_detect_faces_batch on frames of any sizes (photo collections, mixed camera feeds), in one call.  Every descriptor needs a non-null
 * bgr, rows, cols >= 1 and step >= cols * 3.  A frame smaller than every window returns no boxes.  crf_detect_faces and
 * crf_detect_faces_batch are this call on equal-size frames. */
int crf_detect_faces_batch_mixed(crf_ctx* ctx, const crf_cascade* c, const crf_image_t* images, int n_images, double scale_factor,
                                 int min_neighbors, int min_size, crf_rect_t* out, int* image_of_box, int cap);
/* FaceForest::analyzeImage(img, faces) for n_images frames: detection as above, detectFace's enlargement + clipping
 * (src/FaceForest.cpp:147-157), then analyzeFace for every box, reading the frames from the device copy made for detection (no second
 * upload).  boxes (the enlarged boxes) / image_of_box / out: cap entries, in the order of crf_detect_faces_batch.
 * Unlike crf_analyze_faces, a box the analysis path rejects (typically a detection at the bottom border whose clipped box scales to a face
 * shorter than a 31-px patch) does not fail the call: its record is zero except flags = CRF_FACE_NOT_ANALYSED, and every other face is
 * analysed normally.  cap smaller than the face count: everything is detected, the true count is returned, and only the first `cap`
 * boxes are written and analysed.  Returns the face count or a negative status. */
int crf_analyze_images(crf_ctx* ctx, const crf_cascade* c, const uint8_t* const* images, int n_images, int rows, int cols,
                       size_t step, double scale_factor, int min_neighbors, int min_size,
                       crf_rect_t* boxes, int* image_of_box, crf_face_t* out, int cap);
/* crf_analyze_images on frames of any sizes (descriptors as in crf_detect_faces_batch_mixed): each detection is enlarged, clipped and
 * checked against its own frame.  crf_analyze_images is this call on equal-size frames. */
int crf_analyze_images_mixed(crf_ctx* ctx, const crf_cascade* c, const crf_image_t* images, int n_images, double scale_factor,
                             int min_neighbors, int min_size, crf_rect_t* boxes, int* image_of_box, crf_face_t* out, int cap);

/* ---- several GPUs behind one caller (SURVEY 8e): one context + one host thread per GPU, contiguous shards of the faces (cut at frame
 * boundaries when the boxes are grouped by frame), a forest replica per GPU, records written straight into `out`.  No collective:
 * faces are independent (FaceForest::analyzeImage's loop over faces, src/FaceForest.cpp:174-180).  devices NULL / n_devices 0 = every
 * visible GPU; a device may be listed more than once. */
typedef struct crf_multi crf_multi;
int crf_multi_create(const crf_model* m, const int* devices, int n_devices, const crf_options_t* opt, crf_multi** out);
void crf_multi_destroy(crf_multi* mg);
int crf_multi_device_count(const crf_multi* mg);
crf_ctx* crf_multi_ctx(crf_multi* mg, int i);   /* shard i's context (counters, profiling) */
int crf_multi_analyze_batch(crf_multi* mg, const uint8_t* const* images, int n_images, int rows, int cols, size_t step,
                            const crf_rect_t* boxes, const int* image_of_box, int n, crf_face_t* out);
/* crf_multi_analyze_batch on frames of any sizes (descriptors as in crf_analyze_batch_mixed) */
int crf_multi_analyze_batch_mixed(crf_multi* mg, const crf_image_t* images, int n_images, const crf_rect_t* boxes, const int* image_of_box,
                                  int n, crf_face_t* out);
int crf_multi_analyze_crops(crf_multi* mg, const uint8_t* bgr_batch, int n, int rows, int cols, crf_face_t* out, int headpose_only);

/* ---- stage-level entry points (device results copied back) used by the parity tests and by the
 * reference-shaped classes in crf_b200_compat.hpp. */
/* src/FaceForest.cpp:196-204: cvtColor + ROI + resize.  scaled: caller buffer of at least max_h x 125 bytes, dense rows of *W. */
int crf_stage_gray_resize(crf_ctx* ctx, const uint8_t* bgr, int rows, int cols, size_t step, crf_rect_t box,
                          uint8_t* scaled, int* W, int* H);
/* ImageSample::extractFeatureChannels (src/ImageSample.cpp:77-90) with features {0,1,2}:
 * planes_u8 [38][H][W] (may be NULL), integrals [38][H+1][W+1] u32 (may be NULL). */
int crf_stage_channels(crf_ctx* ctx, const uint8_t* scaled, int W, int H, uint8_t* planes_u8, uint32_t* integrals);
/* The same for an explicit feature list (any subset of 0..5, sorted by the library): planes in the order
 * FeatureChannelFactory::extractChannel appends them.  Returns the plane count (> 0) or a negative status. */
int crf_stage_feature_channels(crf_ctx* ctx, const uint8_t* scaled, int W, int H, const int* features, int nfeatures,
                               uint8_t* planes_u8, uint32_t* integrals);
/* FC_MIN_MAX (include/FeatureChannelFactory.hpp:142-165): planes [2][H][W], integrals [2][H+1][W+1]. */
int crf_stage_minmax(crf_ctx* ctx, const uint8_t* scaled, int W, int H, uint8_t* planes_u8, uint32_t* integrals);
/* FC_NORM (include/FeatureChannelFactory.hpp:58-70): cv::equalizeHist; plane [H][W], integral [H+1][W+1]. */
int crf_stage_norm(crf_ctx* ctx, const uint8_t* scaled, int W, int H, uint8_t* plane_u8, uint32_t* integral);
/* FC_CANNY (include/FeatureChannelFactory.hpp:166-179): cv::Canny(img, out, -1, 5); plane [H][W] (0 / 255), integral [H+1][W+1]. */
int crf_stage_canny(crf_ctx* ctx, const uint8_t* scaled, int W, int H, uint8_t* plane_u8, uint32_t* integral);
/* Forest<S>::evaluateMT over the dense grid of getHeadPoseVotesMT / getFacialFeaturesVotesMT.
 * Channel data comes from caller-supplied u8 planes [C][H][W] (C <= 64) so that synthetic
 * channels can be used.  which = -1: head-pose forest (tree_forest/tree_index ignored);
 * which = 0: explicit list of ntrees (forest, tree) pairs of the FFD jungle.
 * leaf_ids: [patch][tree] in the reference's order (x outer, y inner), value = Boost object id. */
int crf_stage_eval_forest(crf_ctx* ctx, int which, const int* tree_forest, const int* tree_index, int ntrees,
                          const uint8_t* planes_u8, int C, int W, int H, int stride, int32_t* leaf_ids);
/* Forest<S>::evaluateMT(sample, leafs) (include/Forest.hpp:81-90) for explicit patch origins — the per-sample level of the
 * interface.  patch_xy: npatches x (x, y) top-left corners in the scaled face; leaf_ids: [patch][tree] Boost object ids. */
int crf_stage_eval_patches(crf_ctx* ctx, int which, const int* tree_forest, const int* tree_index, int ntrees,
                           const uint8_t* planes_u8, int C, int W, int H, const int* patch_xy, int npatches, int32_t* leaf_ids);
/* ImageSample::evalTest(SimplePatchFeature, Rect) (src/ImageSample.cpp:30-64) for n tests:
 * tests = n x {channel, x1, y1, w1, h1, x2, y2, w2, h2, patch_x, patch_y}; out[i] = mean(rect1) - mean(rect2). */
int crf_stage_eval_tests(crf_ctx* ctx, const uint8_t* planes_u8, int C, int W, int H, const int* tests, int n, int* out);
/* The same tests by the branch the reference takes when ImageSample was built with use_integral = false (src/ImageSample.cpp:40-47):
 * cv::sum over the two rectangles of the 8-bit plane itself.  Same arguments, same results (both branches truncate exact sums). */
int crf_stage_eval_tests_sum(crf_ctx* ctx, const uint8_t* planes_u8, int C, int W, int H, const int* tests, int n, int* out);
/* getHeadPoseVotesMT reduce + areaUnderCurve + composition (src/face_utils.cpp:219-241, :304-323;
 * src/FaceForest.cpp:215-250) from planes: returns headpose, variance, counts, dominant and the composed list. */
int crf_stage_headpose(crf_ctx* ctx, const uint8_t* planes_u8, int C, int W, int H, int stride,
                       float* headpose, float* variance, int tree_counts[CRF_NUM_POSE_FORESTS], int* dominant,
                       int* tree_forest, int* tree_index, int* ntrees, int* flags);
/* composition alone from (headpose, variance) */
int crf_stage_compose(crf_ctx* ctx, float headpose, float variance, int tree_counts[CRF_NUM_POSE_FORESTS], int* dominant,
                      int* tree_forest, int* tree_index, int* ntrees, int* flags);
/* the same for n pairs in one launch (knife-edge sweeps of floor(area * ntrees), src/FaceForest.cpp:243): tree_counts [n][5],
 * dominant / ntrees / flags [n], tree_forest / tree_index [n][list_cap] (first list_cap entries, -1 padded); any output may be NULL. */
int crf_stage_compose_batch(crf_ctx* ctx, const float* headpose, const float* variance, int n, int* tree_counts, int* dominant,
                            int* ntrees, int* flags, int* tree_forest, int* tree_index, int list_cap);
/* getFacialFeaturesVotesMT vote emission + MeanShift::shift x10 (src/face_utils.cpp:277-301,
 * include/MeanShift.hpp:52-135) for an explicit composed forest.  votes_xyw (optional): [10][vote_cap][3]. */
int crf_stage_votes_meanshift(crf_ctx* ctx, const int* tree_forest, const int* tree_index, int ntrees,
                              const uint8_t* planes_u8, int C, int W, int H, int stride,
                              int n_votes[CRF_NUM_PARTS], float* votes_xyw, int vote_cap,
                              float mean_xy[CRF_NUM_PARTS][2], int rounded_xy[CRF_NUM_PARTS][2], int iters[CRF_NUM_PARTS]);
/* MeanShift::shift on a caller-supplied vote list (x, y, weight triples), with the context's MeanShiftOption ... */
int crf_stage_meanshift(crf_ctx* ctx, const float* votes_xyw, int n, float mean_xy[2], int rounded_xy[2], int* iters);
/* ... or with per-call options: shift(votes, result, num_iterations, kernel, stopping_criteria) (include/MeanShift.hpp:52-76). */
int crf_stage_meanshift_opt(crf_ctx* ctx, const float* votes_xyw, int n, int kernel, int max_iterations, float stopping,
                            float mean_xy[2], int rounded_xy[2], int* iters);
/* areaUnderCurve(x1, x2, mean, std) (src/face_utils.cpp:304-323; include/face_utils.hpp:103-108). */
int crf_stage_area_under_curve(crf_ctx* ctx, float x1, float x2, double mean, double std_, float* area);

/* One (frame, pyramid level) instance of the detector: the scale, the level's size sw x sh, its window grid (nx x ny windows, ystep
 * level pixels apart), the window in frame pixels, and tilted = 1 when the cascade has tilted features (T is built). */
typedef struct { double factor; int frame, sw, sh, ystep, nx, ny, win_w, win_h, tilted; } crf_haar_level_t;
/* The device passes of crf_detect_faces_batch_mixed(ctx, c, images, n_images, scale_factor, ., min_size, ...), copied back after the
 * last cascade stage group (the same launches, groups of frames and CRF_HAAR_SPLIT stage groups as detection).  Returns the instance
 * count (frame-major, then level); levels[0 .. cap) get the instances.  With cap at least the count and any of S / Q / T / flags
 * non-null, the passes run and each given buffer receives every instance's data back to back in instance order:
 *   S, Q   (sh + 1) x (sw + 1) u32 integrals of the level's pixels and of their squares, modulo 2^32 (cv::integral's layout)
 *   T      the same layout for the tilted integral (cv::integral's third output); written only when the cascade has tilted features
 *   flags  ny x nx bytes, one per window: 1 passed every stage, 2 rejected by stage 0, 0 otherwise (rejected by a later stage, or
 *          skipped by the variance test: area * sqsum - sum^2 <= 0, or area / sqrt(that) >= 0.1) */
int crf_stage_haar_levels(crf_ctx* ctx, const crf_cascade* c, const crf_image_t* images, int n_images, double scale_factor, int min_size,
                          crf_haar_level_t* levels, int cap, uint32_t* S, uint32_t* Q, uint32_t* T, uint8_t* flags);

#ifdef __cplusplus
}
#endif
#endif /* CRF_B200_H */
