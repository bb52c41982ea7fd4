// gpd.h — C++ host shims that keep the reference's class names, namespaces and call signatures for the hot path
// and forward to the C-ABI of libgpd_b200.so (include/gpd_b200.h). Dependency-free (no PCL / Eigen / OpenCV): where
// the reference passes Eigen / PCL / cv types these shims use plain std containers with the same memory layout
// (3 x N column-major doubles, HWC uint8 images). See INTEGRATION.md for the drop-in bindings into upstream GPD.
//
// reference interfaces mirrored (paths relative to /root/reference):
//   util::ConfigFile        include/gpd/util/config_file.h:60-140, src/gpd/util/config_file.cpp
//   util::Cloud (subset)    include/gpd/util/cloud.h:300-366 (accessors the path reads), cloud.cpp:643-660 (file loading)
//   candidate::HandGeometry include/gpd/candidate/hand_geometry.h, hand_geometry.cpp:25-30
//   candidate::Hand         include/gpd/candidate/hand.h
//   candidate::HandSet      include/gpd/candidate/hand_set.h (getHands / getIsValid / getSample / getFrame)
//   candidate::HandSearch   include/gpd/candidate/hand_search.h:107-108
//   descriptor::ImageGeometry / ImageGenerator   include/gpd/descriptor/image_generator.h:92-96
//   net::Classifier         include/gpd/net/classifier.h:52-81
//   GraspDetector           include/gpd/grasp_detector.h:66-226
#ifndef GPD_B200_HOST_GPD_H_
#define GPD_B200_HOST_GPD_H_

#include <array>
#include <iostream>
#include <map>
#include <memory>
#include <sstream>
#include <string>
#include <vector>

#include "gpd_b200.h"

namespace gpd {

namespace util {

// `key = value` per line, '#' comments, first occurrence of a key wins (config_file.cpp:6-61)
class ConfigFile {
 public:
  explicit ConfigFile(const std::string &fName);
  bool ExtractKeys();
  bool keyExists(const std::string &key) const;
  template <typename ValueType>
  ValueType getValueOfKey(const std::string &key, ValueType const &defaultValue) const {
    if (!keyExists(key)) return defaultValue;
    // string_to_T (config_file.h:132-142): a value that does not parse is reported and yields the zero that a failed
    // stream extraction leaves behind, NOT the default (pinned against the reference's parser, oracle/_ref)
    std::istringstream istr(contents.find(key)->second);
    ValueType v{};
    if (!(istr >> v)) std::cout << "CFG: Not a valid value received for key " << key << "!\n";
    return v;
  }
  std::string getValueOfKeyAsString(const std::string &key, const std::string &defaultValue) const;
  std::vector<double> getValueOfKeyAsStdVectorDouble(const std::string &key, const std::string &defaultValue) const;
  std::vector<int> getValueOfKeyAsStdVectorInt(const std::string &key, const std::string &defaultValue) const;

 private:
  std::map<std::string, std::string> contents;
  std::string fName;
};

// The part of util::Cloud the hot path reads. A cloud loaded without normals is RAW: GraspDetector::preprocessPointCloud
// filters, voxelises and estimates normals on the device (gpdb_preprocess) and stores the processed cloud back here.
class Cloud {
 public:
  Cloud() {}
  // .pcd / .ply with fields x y z [normal_x normal_y normal_z | nx ny nz]; view_points 3 x k column-major
  Cloud(const std::string &filename, const std::vector<double> &view_points);
  Cloud(const std::vector<float> &xyz, const std::vector<double> &normals, const std::vector<int> &camera_source,
        const std::vector<double> &view_points);
  bool loadPointCloudFromFile(const std::string &filename);  // .pcd (ascii | binary | binary_compressed) or .ply
  bool loadPcd(const std::string &filename);
  bool loadPly(const std::string &filename);
  void setNormalsFromFile(const std::string &filename);  // CSV, one normal per row or 3 x N (cloud.cpp:607-641)
  void setNormals(const std::vector<double> &normals) { normals_ = normals; touch(); }
  void setSampleIndices(const std::vector<int> &idx) { sample_indices_ = idx; }
  // Cloud::setSamples (cloud.cpp:662): arbitrary sample positions, 3 x n column-major float64; they take precedence over the
  // sample indices in searchHands / detectGrasps (hand_search.cpp:33-47)
  void setSamples(const std::vector<double> &samples) { samples_ = samples; }
  const std::vector<double> &getSamples() const { return samples_; }
  // replaces cloud_processed_ / normals_ / camera_source_ (what Cloud::filterWorkspace / voxelizeCloud /
  // calculateNormals leave behind, cloud.cpp:207-348,458-535); sample indices are invalidated
  void setProcessed(std::vector<float> points, std::vector<double> normals, std::vector<int> camera_source);
  bool hasNormals() const { return normals_.size() == points_.size() && !points_.empty(); }
  unsigned revision() const { return revision_; }  // process-unique, renewed by every mutation of points / normals
  // draw of sample indices (cloud.cpp:350-405) with fixed-seed generators: without plane indices a uniform draw without
  // replacement over all points (subsampleUniformly); with them subsampleSampleIndices (cloud.cpp:395-405): num_samples
  // draws with replacement from the plane indices, all of them when num_samples is 0 or >= their count
  void subsample(int num_samples);
  // Cloud::sampleAbovePlane (cloud.cpp:407-435): the off-plane points the sample draws are restricted to (empty: none)
  void setPlaneIndices(const std::vector<int> &idx) { plane_indices_ = idx; }
  const std::vector<int> &getPlaneIndices() const { return plane_indices_; }
  const std::vector<float> &getPoints() const { return points_; }       // packed x,y,z
  const std::vector<double> &getNormals() const { return normals_; }    // 3 x N column-major
  const std::vector<int> &getCameraSource() const { return camera_source_; }  // k x N column-major
  const std::vector<double> &getViewPoints() const { return view_points_; }   // 3 x k column-major
  const std::vector<int> &getSampleIndices() const { return sample_indices_; }
  size_t size() const { return points_.size() / 3; }
  int numCameras() const { return (int)(view_points_.size() / 3); }

 private:
  std::vector<float> points_;
  std::vector<double> normals_;
  std::vector<int> camera_source_;
  std::vector<double> view_points_;
  std::vector<int> sample_indices_;
  std::vector<int> plane_indices_;
  std::vector<double> samples_;
  unsigned revision_{0};
  void touch();
};

}  // namespace util

namespace candidate {

struct HandGeometry {
  double finger_width_{0.01}, outer_diameter_{0.12}, depth_{0.06}, height_{0.02}, init_bite_{0.01};
  HandGeometry() {}
  explicit HandGeometry(const std::string &filepath);  // hand_geometry.cpp:20-31
};

class Hand {
 public:
  Hand() {}
  explicit Hand(const gpdb_pose &p) : p_(p) {}
  std::array<double, 3> getApproach() const { return {p_.frame[0], p_.frame[1], p_.frame[2]}; }
  std::array<double, 3> getBinormal() const { return {p_.frame[3], p_.frame[4], p_.frame[5]}; }
  std::array<double, 3> getAxis() const { return {p_.frame[6], p_.frame[7], p_.frame[8]}; }
  std::array<double, 3> getPosition() const { return {p_.position[0], p_.position[1], p_.position[2]}; }
  std::array<double, 3> getSample() const { return {p_.sample[0], p_.sample[1], p_.sample[2]}; }
  const double *getFrame() const { return p_.frame; }  // 3 x 3 column-major (Hand::orientation_)
  double getGraspWidth() const { return p_.width; }
  double getScore() const { return p_.score; }
  void setScore(double s) { p_.score = (float)s; }
  void setPosition(const std::array<double, 3> &p) { for (int i = 0; i < 3; i++) p_.position[i] = p[i]; }
  void setFullAntipodal(bool b) { p_.full_antipodal = b ? 1 : 0; }
  void setHalfAntipodal(bool b) { p_.half_antipodal = b ? 1 : 0; }
  bool isFullAntipodal() const { return p_.full_antipodal != 0; }
  bool isHalfAntipodal() const { return p_.half_antipodal != 0; }
  double getTop() const { return p_.top; }
  double getBottom() const { return p_.bottom; }
  double getCenter() const { return p_.center; }
  int getFingerPlacementIndex() const { return p_.finger_idx; }
  const gpdb_pose &raw() const { return p_; }
  void print() const;

 private:
  gpdb_pose p_{};
};

class HandSet {
 public:
  const std::vector<std::unique_ptr<Hand>> &getHands() const { return hands_; }
  std::vector<std::unique_ptr<Hand>> &getHands() { return hands_; }
  const std::vector<bool> &getIsValid() const { return is_valid_; }
  void setIsValid(const std::vector<bool> &v) { is_valid_ = v; }
  std::array<double, 3> getSample() const { return sample_; }
  const std::array<double, 9> &getFrame() const { return frame_; }  // normal | binormal | curvature axis
  std::vector<std::unique_ptr<Hand>> hands_;
  std::vector<bool> is_valid_;
  std::array<double, 3> sample_{};
  std::array<double, 9> frame_{};
};

class HandSearch {
 public:
  struct Parameters {  // hand_search.h:60-80
    double nn_radius_frames_{0.01};
    int num_orientations_{8}, num_samples_{1000}, num_threads_{1}, num_finger_placements_{10};
    std::vector<int> hand_axes_{2};
    bool deepen_hand_{true};
    double friction_coeff_{20.0};
    int min_viable_{6};
    HandGeometry hand_geometry_;
  };
  explicit HandSearch(Parameters params);
  ~HandSearch();
  // HandSearch::searchHands (hand_search.cpp:24-64): one HandSet per sample with a local frame
  std::vector<std::unique_ptr<HandSet>> searchHands(const util::Cloud &cloud_cam) const;
  const Parameters &getParams() const { return params_; }

 private:
  Parameters params_;
  gpdb_ctx *ctx_{nullptr};
};

}  // namespace candidate

namespace descriptor {

struct ImageGeometry {
  double outer_diameter_{0.10}, depth_{0.06}, height_{0.02};
  int size_{60}, num_channels_{15};
  ImageGeometry() {}
  explicit ImageGeometry(const std::string &filepath);  // image_geometry.cpp:19-29
};

// stand-in for cv::Mat(size, size, CV_8UC(channels)): continuous HWC uint8
struct Image {
  int rows{0}, cols{0}, channels{0};
  std::vector<uint8_t> data;
  bool isContinuous() const { return true; }
};

class ImageGenerator {
 public:
  ImageGenerator(const ImageGeometry &image_geometry, int num_threads, int num_orientations, bool is_plotting,
                 bool remove_plane);
  ~ImageGenerator();
  // image_generator.cpp:17-70: images of the valid hands, in (hand set, hand) order; the hands are moved to hands_out
  void createImages(const util::Cloud &cloud_cam, const std::vector<std::unique_ptr<candidate::HandSet>> &hand_set_list,
                    std::vector<std::unique_ptr<Image>> &images_out,
                    std::vector<std::unique_ptr<candidate::Hand>> &hands_out) const;

 private:
  ImageGeometry image_params_;
  gpdb_ctx *ctx_{nullptr};
};

}  // namespace descriptor

namespace net {

class Classifier {
 public:
  enum class Device : uint8_t { eCPU = 0, eGPU = 1, eVPU = 2, eFPGA = 3 };
  // classifier.cpp:46-62; `weights_file` is the .bin parameter directory EigenClassifier reads
  static std::shared_ptr<Classifier> create(const std::string &model_file, const std::string &weights_file,
                                            Device device = Device::eGPU, int batch_size = 1, int num_channels = 15);
  virtual ~Classifier() {}
  virtual std::vector<float> classifyImages(const std::vector<std::unique_ptr<descriptor::Image>> &image_list) = 0;
  virtual int getBatchSize() const = 0;
};

}  // namespace net

// Clustering::findClusters (include/gpd/clustering.h:50-80, src/gpd/clustering.cpp:5-105): a grasp whose axis, position
// and axis-orthogonal offset agree with at least min_inliers other grasps becomes a cluster: position = mean inlier
// position, score = lower bound of the 99 % confidence interval of the inlier scores. O(n^2) over the SELECTED grasps
// (n <= num_selected). This class is the host-side restatement (also remove_inliers = true); GraspDetector and
// SequentialImportanceSampling run the default remove_inliers = false form on the device (gpdb_find_clusters).
class Clustering {
 public:
  explicit Clustering(int min_inliers) : min_inliers_(min_inliers) {}
  std::vector<std::unique_ptr<candidate::Hand>> findClusters(const std::vector<std::unique_ptr<candidate::Hand>> &hand_list,
                                                             bool remove_inliers = false) const;
  int getMinInliers() const { return min_inliers_; }

 private:
  int min_inliers_;
};

class GraspDetector {
 public:
  explicit GraspDetector(const std::string &config_filename);
  ~GraspDetector();
  // grasp_detector.cpp:192-328: candidates -> filter -> images -> classify (one gpdb_detect) -> select -> sort
  std::vector<std::unique_ptr<candidate::Hand>> detectGrasps(const util::Cloud &cloud);
  // CandidatesGenerator::preprocessPointCloud (candidates_generator.cpp:14-37) on the device: removeNans,
  // filterWorkspace, voxelizeCloud, calculateNormals (skipped when the cloud brings normals), sampleAbovePlane when the
  // cfg sets sample_above_plane (gpdb_sample_above_plane), then subsample
  void preprocessPointCloud(util::Cloud &cloud);
  const gpdb_preprocess_params &getPreprocessParams() const { return pre_params_; }
  std::vector<std::unique_ptr<candidate::Hand>> selectGrasps(std::vector<std::unique_ptr<candidate::Hand>> &hands) const;
  // GraspDetector::generateGraspCandidates + filterGraspsWorkspace / filterGraspsDirection (grasp_detector.cpp:330-398,
  // 422-456, 458-470): positions (3 x m, column-major) of the samples of `cloud` (its setSamples positions, else its sample
  // indices) at which at least one hand survives — what SequentialImportanceSampling keeps of a hand-set list between rounds
  std::vector<double> candidateSamplePositions(const util::Cloud &cloud);
  // GraspDetector::pruneGraspCandidates (grasp_detector.cpp:530-552) for hand sets given by their sample positions: images
  // + classifier on the device, hands with score > min_score, in (sample, pose) order
  std::vector<std::unique_ptr<candidate::Hand>> classifyAtPositions(const util::Cloud &cloud, const std::vector<double> &positions,
                                                                    double min_score);
  // GraspDetector::createGraspImages (grasp_detector.cpp:458-521): candidates -> workspace / direction filters -> grasp images,
  // no classification. images_out[i] = the cv::Mat bytes (image_size x image_size x channels, HWC) of hands_out[i]
  bool createGraspImages(util::Cloud &cloud, std::vector<std::unique_ptr<candidate::Hand>> &hands_out,
                         std::vector<std::vector<uint8_t>> &images_out);
  // GraspDetector::generateGraspCandidates (grasp_detector.cpp:330-332) flattened to its valid hands, as
  // detect_grasps_python.cpp:310-329 does. The device path returns the hands that ALSO pass filterGraspsWorkspace /
  // filterGraspsDirection (the only pose records that leave the GPU); with the shipped cfgs the filters are wide open
  std::vector<std::unique_ptr<candidate::Hand>> generateGraspCandidates(const util::Cloud &cloud);
  // GraspDetector::evalGroundTruth (grasp_detector.cpp:523-527) -> HandSearch::reevaluateHypotheses: re-labels the hands
  // against `cloud_gt` (e.g. a ground-truth mesh cloud) on the device; returns 1 per full-antipodal hand, updates the flags
  std::vector<int> evalGroundTruth(const util::Cloud &cloud_gt, std::vector<std::unique_ptr<candidate::Hand>> &hands);
  // Clustering::findClusters(hands, remove_inliers = false) on the device (gpdb_find_clusters); the host class Clustering
  // below stays for remove_inliers = true and for callers without a detector
  std::vector<std::unique_ptr<candidate::Hand>> findClustersOnDevice(const std::vector<std::unique_ptr<candidate::Hand>> &hands,
                                                                     int min_inliers);
  // multi-GPU detectGrasps (the reference's OpenMP loop over samples, sharded over GPUs instead of CPU threads): one thread
  // and one context per device, cloud broadcast + sample slices + one all-gather inside libgpd_b200 (gpdb_comm_init,
  // gpdb_set_cloud_bcast, gpdb_detect_sharded); returns the num_selected best hands over all devices, sorted by score
  std::vector<std::unique_ptr<candidate::Hand>> detectGraspsMultiGpu(const util::Cloud &cloud, int num_gpus);
  const gpdb_params &getParams() const { return params_; }
  const candidate::HandSearch::Parameters &getHandSearchParameters() const { return hand_search_params_; }
  int getNumSamples() const { return num_samples_; }
  double last_ms_candidates{0}, last_ms_images{0}, last_ms_classify{0};

 private:
  gpdb_params params_{};
  gpdb_preprocess_params pre_params_{};
  gpdb_ctx *ctx_{nullptr};
  const util::Cloud *installed_cloud_{nullptr};  // cloud whose processed arrays are resident on the device
  unsigned installed_revision_{0};
  candidate::HandSearch::Parameters hand_search_params_;
  int num_selected_{100}, num_samples_{1000};
  bool cluster_grasps_{false};
  bool sample_above_plane_{false};
  int min_inliers_{1};
  bool has_classifier_{false};
  std::string model_file_, weights_file_;
  bool ensureCloud(const util::Cloud &cloud);
};

// SequentialImportanceSampling (include/gpd/sequential_importance_sampling.h, src/gpd/sequential_importance_sampling.cpp:
// 10-185): the cross-entropy outer loop over the same path — hand search at num_init_samples cloud points, then
// num_iterations rounds of num_samples_per_iteration ARBITRARY positions (Cloud::setSamples -> gpdb_set_samples): Gaussians
// around the samples of the hand sets found so far (sum- or max-of-Gaussians) mixed with prob_rand_samples uniform draws
// inside the workspace; every round runs the hand search + filters on the device; at the end all surviving hand sets are
// classified (pruneGraspCandidates) and clustered. The reference draws from rand() / std::random_device; here the
// generator is seeded (setSeed) so that a run can be reproduced and checked.
class SequentialImportanceSampling {
 public:
  explicit SequentialImportanceSampling(const std::string &config_filename);
  std::vector<std::unique_ptr<candidate::Hand>> detectGrasps(util::Cloud &cloud);
  void setSeed(unsigned seed) { seed_ = seed; }
  // 3 x m positions of every sample that was evaluated / that carried a hand set, over all rounds (for the parity tests)
  const std::vector<double> &evaluatedPositions() const { return evaluated_; }
  const std::vector<double> &handSetPositions() const { return kept_; }
  GraspDetector &detector() { return *grasp_detector_; }

 private:
  int num_init_samples_{50}, num_iterations_{5}, num_samples_{50}, sampling_method_{0};
  double prob_rand_samples_{0.3}, radius_{0.02}, min_score_{0};
  std::vector<double> workspace_;
  std::unique_ptr<GraspDetector> grasp_detector_;
  std::unique_ptr<Clustering> clustering_;
  unsigned seed_{1};
  std::vector<double> evaluated_, kept_;
};

// fills gpdb_params from the reference's cfg keys (grasp_detector.cpp:22-185); returns false if the file is missing
bool paramsFromConfig(const std::string &config_filename, gpdb_params &p, std::string &weights_file, int &num_selected,
                      int &num_samples, int &min_inliers);
// cfg keys voxelize, voxel_size, workspace, normals_radius (grasp_detector.cpp:56-66); keys of steps that are not
// implemented (remove_outliers, refine_normals_k) are reported and ignored. sample_above_plane is read by GraspDetector.
bool preprocessParamsFromConfig(const std::string &config_filename, gpdb_preprocess_params &pp);

}  // namespace gpd

// ---- the reference's own C interface for Python callers (src/detect_grasps_python.cpp:49-65,431-549,598-607; the two
// calcGraspDescriptors* entry points write HDF5 through cv::hdf and are not provided),
// same names, argument order and struct layout, over the B200 path (exported by libgpd_host.so) -----------------
extern "C" {
struct Grasp {       // detect_grasps_python.cpp:49-56
  double *pos;       // Hand position (3)
  double *orient;    // Eigen::Quaterniond(hand frame) coefficients x, y, z, w (4)
  double *sample;    // the sample the hand was found at (3); the reference allocates it and never fills it
  double score;
  bool label;        // Hand::isFullAntipodal
  int *image;        // {-1}: no descriptor attached (the reference writes -1 into a zero-length array)
};
// points: packed x,y,z (3 * size); camera_index: num_view_points x size, column-major; view_points: 3 x
// num_view_points. Preprocesses (GraspDetector::preprocessPointCloud) and detects. Returns the number of grasps
// (>= 0) or -1; *grasps_out is allocated by the callee and released with freeMemoryGrasps.
int detectGraspsInCloud(char *config_filename, float *points, int *camera_index, float *view_points, int size,
                        int num_view_points, struct Grasp **grasps_out);
int detectGraspsInCloudNormals(char *config_filename, float *points, float *normals, int *camera_index,
                               float *view_points, int size, int num_view_points, struct Grasp **grasps_out);
int freeMemoryGrasps(struct Grasp *in);  // unlike the reference (`delete[] in` only) this also frees the members
// detect_grasps_python.cpp:468-488: cloud from a .pcd / .ply file (+ optional normals file, "" = none); returns 0 when the
// file is missing or empty
int detectGraspsInFile(char *config_filename, char *pcd_filename, char *normals_filename, float *view_points, int num_view_points,
                       struct Grasp **grasps_out);
// :530-549: preprocessing + hand search + filters, no classification (score 0)
int generateGraspCandidatesInFile(char *config_filename, char *pcd_filename, char *normals_filename, float *view_points,
                                  int num_view_points, struct Grasp **grasps_out);
// :490-528: candidates + images in the camera cloud, `label` from HandSearch::reevaluateHypotheses against the ground-truth mesh
// cloud (points_gt / normals_gt: 3 x size_gt, packed per point); Grasp.image = the hand's image as image_size^2 x channels ints
int detectAndEvalGrasps(char *config_filename, float *points, int *camera_index, float *view_points, int size, int num_view_points,
                        float *points_gt, float *normals_gt, int size_gt, struct Grasp **grasps_out);
int CopyAndFree(float *in, float *out, int n);  // :603-607 (`in` must come from new float[])
// Eigen::Quaterniond(Matrix3d) (Eigen/src/Geometry/Quaternion.h, quaternionbase_assign_impl<Other,3,3>):
// m column-major 3x3 -> q = x, y, z, w
void gpdQuaternionFromMatrix(const double *m, double *q);
// Clustering::findClusters over plain pose records (testing aid): out has room for n records; returns the cluster count
int gpdFindClusters(const gpdb_pose *hands, int n, int min_inliers, int remove_inliers, gpdb_pose *out);
// util::ConfigFile of the shim over plain C types (testing aid: pinned against the reference's own parser, oracle/_ref)
int gpdConfigGet(const char *file, const char *key, const char *def, char *out, int out_len);
double gpdConfigGetDouble(const char *file, const char *key, double def);
int gpdConfigGetInt(const char *file, const char *key, int def);
int gpdConfigGetBool(const char *file, const char *key, int def);
int gpdConfigGetDoubles(const char *file, const char *key, const char *def, double *out, int cap);
void gpdHandGeometry(const char *file, double out[5]);                  // candidate::HandGeometry(filepath)
void gpdImageGeometry(const char *file, double out[3], int out2[2]);   // descriptor::ImageGeometry(filepath)
// util::Cloud::subsample over n_points points whose plane indices are plane_idx[n_plane] (n_plane = 0: none); out has
// room for max(num_samples, n_points) indices; returns the number of sample indices (testing aid)
int gpdSubsample(int n_points, const int *plane_idx, int n_plane, int num_samples, int *out);
}

#endif  // GPD_B200_HOST_GPD_H_
