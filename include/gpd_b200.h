/*
 * gpd_b200.h — C-ABI of libgpd_b200.so: the B200-native grasp-candidate hot path.
 *
 * This is the drop-in boundary for the ONE path of atenpas/gpd that this repo
 * accelerates (GraspDetector::detectGrasps steps 1-4, reference
 * src/gpd/grasp_detector.cpp:192-273):
 *
 *   sample index -> FrameEstimator local frame -> HandSearch/HandSet/FingerHand
 *   rotation sweep -> workspace/aperture filter -> ImageGenerator 60x60xC grasp
 *   image -> LeNet score.
 *
 * Conventions follow the reference's only C-ABI precedent,
 * src/detect_grasps_python.cpp:49-65,431-447,598-601: plain C structs and
 * pointers, return value = count (>= 0) or negative error code, no exceptions
 * cross the boundary, errors are also printed to stderr, the callee allocates
 * result arrays and the caller releases them with a library free function,
 * inputs are borrowed for the duration of the call only.
 *
 * Every entry point cites the reference interface it replaces. INTEGRATION.md
 * shows the reference-side bindings (a `CudaClassifier : net::Classifier`,
 * `HandSearch::searchHands`, `ImageGenerator::createImages`,
 * `GraspDetector::detectGrasps` shims) a maintainer would add.
 *
 * There is NO CPU fallback behind these symbols: every compute entry point
 * returns GPDB_ERR_CUDA when no sm_100 device is usable.
 */
#ifndef GPD_B200_H_
#define GPD_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GPDB_VERSION 1

/* error codes (all negative; >= 0 is success / a count) */
#define GPDB_OK 0
#define GPDB_ERR_INVALID (-1)   /* bad argument / parameter                      */
#define GPDB_ERR_CUDA (-2)      /* CUDA runtime error or no usable device        */
#define GPDB_ERR_STATE (-3)     /* call order: cloud or weights not set          */
#define GPDB_ERR_IO (-4)        /* weight file missing or of the wrong size      */
#define GPDB_ERR_CAPACITY (-5)  /* a neighbourhood exceeded the on-chip tile     */

#define GPDB_MAX_CAMERAS 8
#define GPDB_MAX_HAND_AXES 3

/* pose_flags bits (one byte per (sample, axis, angle) pose) */
#define GPDB_POSE_VALID 1u     /* HandSet::is_valid_ after evalHands (hand_set.cpp:111)        */
#define GPDB_POSE_FILTERED 2u  /* survives filterGraspsWorkspace [+ filterGraspsDirection]     */
#define GPDB_POSE_HALF 4u      /* Hand::isHalfAntipodal (hand_set.cpp:255-261)                 */
#define GPDB_POSE_FULL 8u      /* Hand::isFullAntipodal                                        */

/* shadow_mode for the 15-channel occlusion channels (SURVEY.md 9.4, DESIGN.md) */
#define GPDB_SHADOW_DETERMINISTIC 0 /* counter-based draws; defined in include/gpd_b200_shadow.h */

/*
 * All parameters of the path. Field names are the reference's cfg keys; the
 * defaults are the reference's defaults (grasp_detector.cpp:48-86,130-185,
 * hand_geometry.cpp:25-30, image_geometry.cpp:24-28). gpdb_params_default()
 * fills them.
 */
typedef struct gpdb_params {
  /* candidate::HandGeometry (cfg/hand_geometry.cfg:8-12) */
  double finger_width;
  double hand_outer_diameter;
  double hand_depth;
  double hand_height;
  double init_bite;
  /* descriptor::ImageGeometry (cfg/image_geometry_15channels.cfg:8-12) */
  double volume_width;  /* ImageGeometry::outer_diameter_ */
  double volume_depth;
  double volume_height;
  int32_t image_size;
  int32_t image_num_channels; /* 1, 3, 12 or 15 */
  /* candidate::HandSearch::Parameters (grasp_detector.cpp:67-86) */
  double nn_radius; /* nn_radius_frames_ */
  int32_t num_orientations;
  int32_t num_finger_placements;
  int32_t num_hand_axes;
  int32_t hand_axes[GPDB_MAX_HAND_AXES];
  int32_t deepen_hand;
  double friction_coeff;
  int32_t min_viable;
  /* GraspDetector filters (grasp_detector.cpp:158-174) */
  double min_aperture;
  double max_aperture;
  double workspace_grasps[6];
  int32_t filter_approach_direction;
  double direction[3];
  double thresh_rad;
  /* net::Classifier (grasp_detector.cpp:130-138) */
  int32_t batch_size;       /* images per LeNet launch; 0 = library default          */
  int32_t relu_after_conv;  /* 0: Caffe/Eigen LeNet (no ReLU after conv, A14);        */
                            /* 1: the PyTorch/OpenVINO 12-channel net (pytorch/network.py:32-47) */
  /* library */
  int32_t shadow_mode;      /* GPDB_SHADOW_DETERMINISTIC                              */
  int32_t device;           /* CUDA device ordinal                                    */
  int32_t chunk_samples;    /* samples per device pass; 0 = library default           */
  int32_t keep_images;      /* gpdb_detect also returns the grasp images              */
  int32_t lenet_impl;       /* 0 = default (tcgen05 when built), 1 = force SIMT fp32  */
} gpdb_params;

/* One grasp candidate = candidate::Hand (include/gpd/candidate/hand.h:267-276). */
typedef struct gpdb_pose {
  double sample[3];   /* Hand::sample_                                             */
  double frame[9];    /* Hand::orientation_, column-major: approach|binormal|axis  */
  double position[3]; /* Hand::position_ (hand.cpp:41-45)                          */
  double top;         /* BoundingBox::top_                                         */
  double bottom;
  double center;
  double width;       /* Hand::grasp_width_                                        */
  float score;        /* Label::score_ = logits[1] - logits[0] (eigen_classifier.cpp:74) */
  int32_t sample_index; /* index of the sample in the cloud                        */
  int32_t sample_slot;  /* position in the sample_idx array passed to the call     */
  int16_t pose_slot;    /* axis_i * num_orientations + angle_i                     */
  int16_t finger_idx;   /* Hand::finger_placement_index_                           */
  uint8_t half_antipodal;
  uint8_t full_antipodal;
  uint8_t pad_[6];    /* explicit tail padding (zero): sizeof(gpdb_pose) = 176 with no implicit bytes */
} gpdb_pose;

/* Result of gpdb_detect / gpdb_hand_search: callee-allocated, release with gpdb_free_result. */
typedef struct gpdb_result {
  int32_t n_samples;
  int32_t poses_per_sample; /* num_hand_axes * num_orientations                     */
  uint8_t *frame_valid;     /* [n_samples] 0 where calculateFrame found no neighbour */
  double *frames;           /* [n_samples*9] LocalFrame: normal|binormal|curvature_axis */
  uint8_t *pose_flags;      /* [n_samples*P] GPDB_POSE_* bits                        */
  float *pose_scores;       /* [n_samples*P] score, NaN where no image was classified */
  int32_t n_candidates;     /* poses with VALID and FILTERED set                     */
  gpdb_pose *candidates;    /* [n_candidates] in (sample slot, pose slot) order =    */
                            /* hands_out order of image_generator.cpp:91-98          */
  uint8_t *images;          /* [n_candidates*S*S*C] HWC uint8 (cv::Mat CV_8UC(C)) or NULL */
  double ms_candidates;     /* device time of "1. Candidate generation"  (grasp_detector.cpp:313) */
  double ms_images;         /*                "2. Descriptor extraction"                     */
  double ms_classify;       /*                "3. Classification"                            */
  int64_t kernel_launches;  /* CUDA kernels launched by this call                     */
  int32_t n_total_candidates; /* all poses with VALID and FILTERED set (= n_candidates except after gpdb_detect_select) */
  void *owner_;             /* library-private: the pinned host arena the arrays above live in (gpdb_free_result) */
} gpdb_result;

typedef struct gpdb_ctx gpdb_ctx;

/* Fill *p with the reference defaults (15-channel images, hand_axes = {2}). */
void gpdb_params_default(gpdb_params *p);

/* Replaces: GraspDetector::GraspDetector(cfg) (grasp_detector.cpp:5-190). One context = one
 * CUDA device + stream; calls on one context are serialised by the caller. */
int gpdb_create(const gpdb_params *params, gpdb_ctx **ctx_out);
void gpdb_destroy(gpdb_ctx *ctx);

/* Message of the last error on this context (or of the last failed gpdb_create when ctx==NULL). */
const char *gpdb_last_error(const gpdb_ctx *ctx);

/* Replaces: EigenClassifier::EigenClassifier weight loading (eigen_classifier.cpp:24-47).
 * `dir` is the `weights_file` cfg value: a directory (with trailing '/') holding
 * {conv1,conv2,ip1,ip2}_{weights,biases}.bin in the reference's raw float32 layout. */
int gpdb_load_weights_dir(gpdb_ctx *ctx, const char *dir);

/* Replaces: Classifier::create(model_file, weights_file, ...) weight loading for the reference's other backends
 * (classifier.cpp:33-61): `weights_file` may be a .bin parameter directory (trailing '/', as above), a Caffe
 * `.caffemodel` (layers conv1, conv2, ip1, ip2; caffe_classifier.cpp) or an OpenVINO IR `.bin` whose `.xml` is
 * `model_file` (or lies next to it; openvino_classifier.cpp:20-57). The blobs are converted to the .bin layout on the
 * host. An IR with ReLU after the convolutions needs a context created with relu_after_conv = 1. */
int gpdb_load_weights_file(gpdb_ctx *ctx, const char *model_file, const char *weights_file);
/* The host-side conversion alone (no device): fills eight caller-allocated arrays (sizes as gpdb_set_weights) in the
 * .bin layout; relu_layers_out = number of ReLU layers of an IR, -1 for a caffemodel; err_out receives the message. */
int gpdb_read_weights_file(const char *model_file, const char *weights_file, int32_t channels, float *const out[8],
                           int32_t *relu_layers_out, char *err_out, int32_t err_len);

/* Same, from memory, in the layout of the .bin files (A14): conv = OIHW row-major,
 * ip = column-major (out, in). Sizes: conv1 20*C*25, conv2 50*20*25, ip1 500*7200, ip2 2*500. */
int gpdb_set_weights(gpdb_ctx *ctx, const float *conv1_w, const float *conv1_b,
                     const float *conv2_w, const float *conv2_b, const float *ip1_w,
                     const float *ip1_b, const float *ip2_w, const float *ip2_b);

/* Replaces: the util::Cloud accessors the path reads (include/gpd/util/cloud.h:300-366):
 *   xyz          getCloudProcessed() points, packed float32 x,y,z (3*N)
 *   normals      getNormals(), 3 x N float64 column-major
 *   cam_source   getCameraSource(), k x N int32 column-major (may be NULL: all ones)
 *   view_points  getViewPoints(), 3 x k float64 column-major
 * Builds the device neighbour grid (replaces the two KdTreeFLANN builds,
 * hand_search.cpp:29-31, image_generator.cpp:37-38). */
int gpdb_set_cloud(gpdb_ctx *ctx, const float *xyz, const double *normals,
                   const int32_t *cam_source, int32_t n_points, const double *view_points,
                   int32_t n_cams);

/* Replaces: Cloud::setSamples (cloud.cpp:662; used by SequentialImportanceSampling, sequential_importance_sampling.cpp:
 * 130-131,166-168): n arbitrary float64 sample positions (3 x n column-major) next to the installed cloud. Returns N, the
 * first sample index that addresses them: gpdb_detect / gpdb_frames / gpdb_hand_search / gpdb_detect_select accept sample
 * indices N .. N + n - 1 for these positions (indices < N keep addressing cloud points, Cloud::getSampleIndices). The
 * local frame and the radius searches use the float32 image of the position, the hand-frame transforms the float64
 * position, as the reference does; the shadow draws are seeded by the sample index as for cloud points. A new cloud
 * (gpdb_set_cloud / gpdb_preprocess) drops the positions. */
int gpdb_set_samples(gpdb_ctx *ctx, const double *samples_xyz, int32_t n_samples);

/* Replaces: GraspDetector::detectGrasps steps 1-4 (grasp_detector.cpp:222-273) for the
 * samples cloud.getSampleIndices() (cloud.h:345). Returns n_candidates or a negative error. */
int gpdb_detect(gpdb_ctx *ctx, const int32_t *sample_idx, int32_t n_samples, gpdb_result *out);

/* Replaces: GraspDetector::detectGrasps steps 1-4 followed by selectGrasps (grasp_detector.cpp:222-283,405-420): the
 * `num_selected` highest-scoring candidates, sorted by descending score (ties: (sample slot, pose slot) order), selected
 * ON THE DEVICE — only those pose records cross PCIe. out->candidates holds n_candidates = min(num_selected, total)
 * records, out->n_total_candidates the number of classified candidates; the per-sample / per-pose arrays
 * (frame_valid, frames, pose_flags, pose_scores, images) are NULL. Returns n_candidates or a negative error. */
int gpdb_detect_select(gpdb_ctx *ctx, const int32_t *sample_idx, int32_t n_samples, int32_t num_selected,
                       gpdb_result *out);

/* Device-resident variant of gpdb_detect: d_sample_idx [n], d_flags_out [n*P] and d_scores_out [n*P]
 * are DEVICE pointers on the context's device; no input or result crosses PCIe (only the per-chunk
 * candidate count is read back to size the image / classifier launches). `stats` receives
 * n_candidates, stage timings and the launch count; its array members stay NULL. The caller
 * guarantees 0 <= sample index < N. Used to measure the path with inputs resident in HBM. */
int gpdb_detect_resident(gpdb_ctx *ctx, const int32_t *d_sample_idx, int32_t n_samples, uint8_t *d_flags_out,
                         float *d_scores_out, gpdb_result *stats);

/* Run all work of this context on an existing CUDA stream (cudaStream_t passed as void*), e.g. the
 * host framework's current stream, instead of the context's own stream. */
int gpdb_set_stream(gpdb_ctx *ctx, void *cuda_stream);

/* The chunk pipeline runs the hand search of the chunks ahead on a second stream, concurrently with the image stage and
 * the classifier of the current chunk (default: on; environment GPD_B200_OVERLAP=0 turns the default off). With
 * enable = 0 every kernel of a call runs on the context's stream, one after the other: the stage timers of
 * gpdb_last_timings are then exclusive per stage (bench.py takes its per-kernel times from such a pass). Results are
 * identical either way. */
int gpdb_set_overlap(gpdb_ctx *ctx, int32_t enable);

/* Stage-level entry points (used by the parity tests and by partial drop-ins). */

/* Replaces: FrameEstimator::calculateLocalFrames (frame_estimator.cpp:6-35).
 * frames_out [n*9] normal|binormal|curvature_axis, valid_out [n]. */
int gpdb_frames(gpdb_ctx *ctx, const int32_t *sample_idx, int32_t n_samples, double *frames_out,
                uint8_t *valid_out);

/* Replaces: HandSearch::searchHands (hand_search.cpp:24-64) + filterGraspsWorkspace /
 * filterGraspsDirection (grasp_detector.cpp:334-398,422-456). No images, no scores. */
int gpdb_hand_search(gpdb_ctx *ctx, const int32_t *sample_idx, int32_t n_samples,
                     gpdb_result *out);

/* Replaces: ImageGenerator::createImages (image_generator.cpp:17-70) for given hands.
 * images_out [n_poses * S*S*C] HWC uint8. */
int gpdb_images(gpdb_ctx *ctx, const gpdb_pose *poses, int32_t n_poses, uint8_t *images_out);

/* Replaces: Classifier::classifyImages (classifier.h:72-73; eigen_classifier.cpp:59-79).
 * images_hwc [n * S*S*C] continuous cv::Mat data; scores_out [n]; logits_out [n*2] or NULL. */
int gpdb_classify(gpdb_ctx *ctx, const uint8_t *images_hwc, int32_t n_images, float *scores_out,
                  float *logits_out);

/* --- cloud preprocessing (SURVEY.md 8(f).1: the step immediately before the path) -------------- */

/* Parameters of CandidatesGenerator::preprocessPointCloud (candidates_generator.cpp:14-37); field names are
 * the reference's cfg keys (grasp_detector.cpp:50-66, cfg/eigen_params.cfg:16-21). */
typedef struct gpdb_preprocess_params {
  double workspace[6];      /* cfg `workspace`: min_x max_x min_y max_y min_z max_z, strict inequalities   */
  double voxel_size;        /* cfg `voxel_size`; Cloud::voxelizeCloud(float cell_size) rounds it to float  */
  double normals_radius;    /* cfg `normals_radius`                                                        */
  int32_t voxelize;         /* cfg `voxelize`                                                              */
  int32_t estimate_normals; /* 1: Cloud::calculateNormalsOMP + reverseNormals (cloud.cpp:497-535,573-604); */
                            /* 0: keep the caller's normals (voxel-averaged, cloud.cpp:307-311,331-333)    */
} gpdb_preprocess_params;

/* Reference defaults: workspace -1..1, voxelize, voxel_size 0.003, normals_radius 0.03, estimate normals. */
void gpdb_preprocess_params_default(gpdb_preprocess_params *p);

/* Replaces: CandidatesGenerator::preprocessPointCloud steps removeNans -> filterWorkspace -> voxelizeCloud ->
 * calculateNormals (candidates_generator.cpp:18-26; cloud.cpp:154-164,207-266,286-348,458-484,497-535,573-604)
 * on the device, and installs the processed cloud in the context exactly as gpdb_set_cloud would (the neighbour
 * grid is built from the device copy). Inputs as gpdb_set_cloud (raw cloud, n_points may be millions); `normals`
 * may be NULL when estimate_normals = 1. Returns the number of processed points N' (>= 0) or a negative error.
 * Not covered: refine_normals_k, remove_outliers (PCL filters outside the default cfg), sample_above_plane (a separate
 * call on the installed cloud: gpdb_sample_above_plane) and Cloud::subsample (host-side RNG; the sample indices are an
 * input of gpdb_detect).
 * Semantics that differ from the reference by specification (DESIGN.md "preprocessing"): the voxel set is an
 * exact set (the reference's std::set comparator is not a strict weak order), output order = descending index
 * of each voxel's first point (the reference's iteration order whenever its de-duplication succeeds). */
int gpdb_preprocess(gpdb_ctx *ctx, const float *xyz, const double *normals, const int32_t *cam_source,
                    int32_t n_points, const double *view_points, int32_t n_cams,
                    const gpdb_preprocess_params *pp);

/* Reads back the cloud currently installed in the context (after gpdb_preprocess or gpdb_set_cloud):
 * xyz_out [3*N] float32, normals_out [3*N] float64 (3 x N column-major), cam_source_out [k*N] int32 (k x N
 * column-major); any output may be NULL. Returns N. These are the util::Cloud members the reference's
 * preprocessing leaves behind (cloud_processed_, normals_, camera_source_; cloud.h:300-333). */
int gpdb_get_cloud(gpdb_ctx *ctx, float *xyz_out, double *normals_out, int32_t *cam_source_out);

/* After gpdb_preprocess: src_out [N] = index into the RAW cloud of the point that represents each processed point
 * (the first point of its voxel, cloud.cpp:304-310 `(*res.first)(3)`). Returns N. */
int gpdb_get_cloud_source_index(gpdb_ctx *ctx, int32_t *src_out);

/* Device time (ms, CUDA events) of the stages of the last gpdb_preprocess call:
 * ms[0] upload, ms[1] NaN/workspace filter, ms[2] voxelise, ms[3] grid build, ms[4] normals, ms[5] whole call. */
int gpdb_preprocess_timings(const gpdb_ctx *ctx, double ms_out[6]);

/* Parameters of the support-plane fit (include/gpd_b200_plane.h). */
typedef struct gpdb_plane_params {
  double distance_threshold; /* inlier distance (cloud.cpp:418: 0.01)                                          */
  int32_t num_hypotheses;    /* RANSAC triples evaluated, 1 .. GPDB_PLANE_MAX_HYPOTHESES (default 1024)         */
  uint64_t seed;             /* seed of the counter-based draw of the triples                                    */
} gpdb_plane_params;

/* Defaults: threshold 0.01, 1024 hypotheses, seed 1. */
void gpdb_plane_params_default(gpdb_plane_params *pp);

/* What the fit found (all zero and hypothesis = -1 when no triple was valid). */
typedef struct gpdb_plane_info {
  float coefficients[4];            /* final plane a, b, c, d: refined, or the winner's when not refined           */
  float hypothesis_coefficients[4]; /* plane of the winning triple                                                 */
  int32_t hypothesis;               /* winning hypothesis h, -1 when none is valid                                  */
  int32_t hypothesis_inliers;       /* its inlier count                                                            */
  int32_t inliers;                  /* inliers of the final plane                                                  */
  int32_t refined;                  /* 1 when the coefficients were refined (the winner has >= 4 inliers)          */
} gpdb_plane_info;

/* Replaces: Cloud::sampleAbovePlane (cloud.cpp:407-435; cfg key sample_above_plane, candidates_generator.cpp:32-34):
 * PCL SACSegmentation (RANSAC plane, optimizeCoefficients) + ExtractIndices(negative) on the device, over the cloud
 * installed by gpdb_preprocess or gpdb_set_cloud, as the deterministic variant specified in include/gpd_b200_plane.h.
 * off_plane_idx_out (room for N) receives the indices of the points off the fitted plane in ascending order; these are
 * the cloud's sample indices that Cloud::subsample then draws from. Returns their number; 0 = the plane fit failed (fewer
 * than 3 points, every triple degenerate, or no point / every point on the plane: the caller keeps the whole cloud);
 * negative = error (no cloud, bad parameters). info_out may be NULL. */
int gpdb_sample_above_plane(gpdb_ctx *ctx, const gpdb_plane_params *pp, int32_t *off_plane_idx_out,
                            gpdb_plane_info *info_out);

/* Replaces: HandSearch::reevaluateHypotheses (hand_search.cpp:66-134; GraspDetector::evalGroundTruth,
 * grasp_detector.cpp:523-527): the given hands (sample, frame, top, finger_idx are read) are re-labelled against the cloud
 * installed in the context — radius search around the hand's sample, its own frame, evaluateFingers at its own depth and
 * finger placement, closing region, Antipodal::evaluateGrasp. labels_out[i] = 1 for a full antipodal grasp, else 0; the
 * half_antipodal / full_antipodal fields of the records are updated in place. Returns n. */
int gpdb_reevaluate(gpdb_ctx *ctx, gpdb_pose *hands, int32_t n_hands, int32_t *labels_out);

/* Replaces: Clustering::findClusters(hand_list, remove_inliers = false) (clustering.cpp:5-105; GraspDetector::detectGrasps
 * step 6, grasp_detector.cpp:283-301; SequentialImportanceSampling step 4) on the device: one warp per hand over the n
 * hands (n <= num_selected in detectGrasps), inliers folded in index order so that the running mean / variance are the
 * reference's. hands [n] are host records (score, position, frame read); clusters_out has room for n records and receives
 * the clusters in the order of their seed hands (position = mean inlier position, score = lower 99 % confidence bound).
 * Returns the number of clusters. */
int gpdb_find_clusters(gpdb_ctx *ctx, const gpdb_pose *hands, int32_t n_hands, int32_t min_inliers, gpdb_pose *clusters_out);

/* Replaces: freeMemoryGrasps (detect_grasps_python.cpp:598-601). The arrays of a result live in page-locked host memory
 * owned by the library (the device writes them directly, overlapped with compute); gpdb_free_result hands that memory
 * back for the next call. A result may outlive its context. */
void gpdb_free_result(gpdb_result *r);

/* --- multi-GPU (SURVEY.md 8(e)): one context per GPU, one process or thread per context ------------------------------
 * The path shards by sample: every rank runs steps 1-4 on the contiguous slice [r*n/R, (r+1)*n/R) of the sample-index
 * array over its own copy of the cloud (reference parallel loops: hand_search.cpp:168-182, image_generator.cpp:83-89,
 * eigen_classifier.cpp:67-76); the only exchange is ONE ncclAllGather of fixed-stride {score f32, flags u8} slots.
 * NCCL is loaded at run time (libnccl.so.2; the copy already in the process, e.g. PyTorch's, is reused). */
#define GPDB_COMM_ID_BYTES 128
/* ncclGetUniqueId: call on one rank, distribute the 128 bytes to the others by any means (MPI, torch.distributed, a pipe). */
int gpdb_comm_unique_id(char id_out[GPDB_COMM_ID_BYTES]);
/* ncclCommInitRank on the context's device and stream (collective: every rank calls it). nranks == 1 is allowed. */
int gpdb_comm_init(gpdb_ctx *ctx, const char id[GPDB_COMM_ID_BYTES], int32_t rank, int32_t nranks);
int gpdb_comm_destroy(gpdb_ctx *ctx);
/* Slice of rank `rank` of `nranks` over n samples and the fixed slot size (largest slice) of the all-gather. */
void gpdb_shard_bounds(int32_t n, int32_t rank, int32_t nranks, int32_t *lo, int32_t *hi, int32_t *slot_samples);
/* gpdb_set_cloud on every rank from rank `root`'s host arrays (ncclBroadcast of the device copies over NVLink; the other
 * ranks pass NULL arrays and any sizes). Every rank then builds its own neighbour grid. Returns N. */
int gpdb_set_cloud_bcast(gpdb_ctx *ctx, int32_t root, const float *xyz, const double *normals, const int32_t *cam_source,
                         int32_t n_points, const double *view_points, int32_t n_cams);
/* gpdb_detect over sharded samples: every rank passes the SAME sample_idx[n]; on return out->pose_flags / out->pose_scores
 * [n*P] hold the gathered results of ALL ranks (identical everywhere), out->candidates the pose records of this rank's
 * slice (sample_slot = position in the full array), out->n_total_candidates the global count; frames / frame_valid
 * are NULL. Returns this rank's candidate count. */
int gpdb_detect_sharded(gpdb_ctx *ctx, const int32_t *sample_idx, int32_t n_samples, gpdb_result *out);
/* Device-resident variant (measurement with inputs in HBM): d_sample_idx_local [n_local] = this rank's slice,
 * d_gathered = nranks slots of gpdb_slot_bytes(slot_samples, P) bytes each: [scores f32 slot_samples*P][flags u8
 * slot_samples*P, padded to 16 B]; this rank's results are written into slot `rank` and all-gathered in place. */
int gpdb_detect_sharded_resident(gpdb_ctx *ctx, const int32_t *d_sample_idx_local, int32_t n_local, int32_t slot_samples,
                                 uint8_t *d_gathered, gpdb_result *stats);
int64_t gpdb_slot_bytes(int32_t slot_samples, int32_t poses_per_sample);

/* --- introspection ------------------------------------------------------------------------- */
/* Device-side stage timings of the last gpdb_detect call, CUDA events on the context stream:
 * ms[0] frames, ms[1] hand search + compaction, ms[2] images, ms[3] LeNet, ms[4] whole call,
 * ms[5] conv1+pool, ms[6] conv2+pool, ms[7] ip1+ip2. */
int gpdb_last_timings(const gpdb_ctx *ctx, double ms_out[8]);
/* Development aid: per-phase SM-cycle counters of the image kernel (thread 0 of every CTA, summed over CTAs).
 * enable != 0 allocates / clears the counters, enable == 0 frees them; cycles_out (may be NULL) receives the
 * counters accumulated so far: [2] ball scan, [3] point channels, [4] shadow setup, [5] shadow casting,
 * [6] shadow bitmap pass, [7] shadow channels, [8] output flush. */
int gpdb_debug_phase_cycles(gpdb_ctx *ctx, int enable, uint64_t cycles_out[16]);

/* Version / build info string (arch, lenet implementation). */
const char *gpdb_build_info(void);

#ifdef __cplusplus
}
#endif
#endif /* GPD_B200_H_ */
