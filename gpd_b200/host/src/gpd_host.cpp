// gpd_host.cpp — implementation of the C++ host shims (include/gpd/gpd.h) over the C-ABI of libgpd_b200.so.
#include <atomic>
#include <random>
#include <thread>

#include "gpd/gpd.h"

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <iostream>

namespace gpd {

// ------------------------------------------------------------------------------------------------ util::ConfigFile
namespace util {

ConfigFile::ConfigFile(const std::string &fName) : fName(fName) {}

// Follows the reference's parser statement by statement, corner cases included (config_file.cpp:6-101; pinned against
// the reference's own object code, oracle/_ref): only '#' starts a comment; a line counts as blank only if it consists of
// SPACES; a line without '=' or with nothing after it is reported but STILL stored (key = first token, value = the
// rest of the line resp. ""); the first occurrence of a key wins; '\r' is not stripped.
bool ConfigFile::ExtractKeys() {
  std::ifstream file(fName.c_str());
  if (!file) {
    std::cout << "Config file " + fName + " could not be found!\n";
    return false;
  }
  std::string line;
  size_t lineNo = 0;
  while (std::getline(file, line)) {
    lineNo++;
    if (line.empty()) continue;
    if (line.find('#') != line.npos) line.erase(line.find('#'));   // removeComment
    if (line.find_first_not_of(' ') == line.npos) continue;        // onlyWhitespace
    if (line.find('=') == line.npos) std::cout << "CFG: Couldn't find separator on line: " << lineNo << "\n";
    {  // validLine: only reported
      std::string t = line;
      t.erase(0, t.find_first_not_of("\t "));
      bool valid = false;
      if (!(t.size() > 0 && t[0] == '='))
        for (size_t i = t.find('=') + 1; i < t.length(); i++)
          if (t[i] != ' ') { valid = true; break; }
      if (!valid) std::cout << "CFG: Bad format for line: " << lineNo << "\n";
    }
    // extractContents
    std::string temp = line;
    temp.erase(0, temp.find_first_not_of("\t "));
    const size_t sepPos = temp.find('=');
    std::string key = temp.substr(0, sepPos);
    if (key.find('\t') != temp.npos || key.find(' ') != temp.npos) key.erase(key.find_first_of("\t "));
    std::string value = temp.substr(sepPos + 1);  // sepPos == npos: the whole line (npos + 1 wraps to 0), as upstream
    value.erase(0, value.find_first_not_of("\t "));
    value.erase(value.find_last_not_of("\t ") + 1);
    if (!keyExists(key)) contents.insert(std::make_pair(key, value));
    else std::cout << "CFG: Can only have unique key names!\n";
  }
  return true;
}

bool ConfigFile::keyExists(const std::string &key) const { return contents.find(key) != contents.end(); }

std::string ConfigFile::getValueOfKeyAsString(const std::string &key, const std::string &defaultValue) const {
  if (!keyExists(key)) return defaultValue;
  return contents.find(key)->second;
}

std::vector<double> ConfigFile::getValueOfKeyAsStdVectorDouble(const std::string &key, const std::string &defaultValue) const {
  std::stringstream ss(getValueOfKeyAsString(key, defaultValue));  // stringToDouble (config_file.cpp:139-152)
  std::vector<double> v;
  double x;
  while (ss >> x) {
    v.push_back(x);
    if (ss.peek() == ' ') ss.ignore();
  }
  return v;
}

std::vector<int> ConfigFile::getValueOfKeyAsStdVectorInt(const std::string &key, const std::string &defaultValue) const {
  std::stringstream ss(getValueOfKeyAsString(key, defaultValue));  // stringToInt reads doubles and truncates (:154-167)
  std::vector<int> v;
  double x;
  while (ss >> x) {
    v.push_back((int)x);
    if (ss.peek() == ' ') ss.ignore();
  }
  return v;
}

// ------------------------------------------------------------------------------------------------ util::Cloud
Cloud::Cloud(const std::string &filename, const std::vector<double> &view_points) : view_points_(view_points) {
  if (view_points_.empty()) view_points_ = {0.0, 0.0, 0.0};
  loadPointCloudFromFile(filename);
  camera_source_.assign((size_t)numCameras() * size(), 0);
  for (size_t i = 0; i < size(); i++) camera_source_[i * numCameras()] = 1;  // single view: all points seen by camera 0
  if (numCameras() > 1) std::fill(camera_source_.begin(), camera_source_.end(), 1);
  touch();
}

Cloud::Cloud(const std::vector<float> &xyz, const std::vector<double> &normals, const std::vector<int> &camera_source,
             const std::vector<double> &view_points)
    : points_(xyz), normals_(normals), camera_source_(camera_source), view_points_(view_points) {
  touch();
}

// File readers (replace pcl::io::loadPCDFile / loadPLYFile in cloud.cpp:643-660); NaN points are dropped (Cloud::removeNans).
// LZF decompression (Marc Lehmann's liblzf format, used by PCD "DATA binary_compressed"): control byte < 32 = literal run
// of ctrl + 1 bytes; otherwise a back reference of length (ctrl >> 5) + 2 (7 = extended by the next byte) at distance
// ((ctrl & 31) << 8 | next) + 1.
static bool lzf_decompress(const unsigned char *in, size_t in_len, unsigned char *out, size_t out_len) {
  size_t ip = 0, op = 0;
  while (ip < in_len) {
    unsigned ctrl = in[ip++];
    if (ctrl < 32) {
      size_t n = ctrl + 1;
      if (ip + n > in_len || op + n > out_len) return false;
      std::memcpy(out + op, in + ip, n);
      ip += n;
      op += n;
    } else {
      size_t len = ctrl >> 5;
      if (len == 7) {
        if (ip >= in_len) return false;
        len += in[ip++];
      }
      if (ip >= in_len) return false;
      size_t dist = ((size_t)(ctrl & 31) << 8) + in[ip++] + 1;
      len += 2;
      if (dist > op || op + len > out_len) return false;
      for (size_t k = 0; k < len; k++, op++) out[op] = out[op - dist];  // may overlap: byte by byte
    }
  }
  return op == out_len;
}

static double read_scalar(const char *src, const std::string &type, int size) {
  if (type == "F" && size == 4) { float v; std::memcpy(&v, src, 4); return v; }
  if (type == "F" && size == 8) { double v; std::memcpy(&v, src, 8); return v; }
  if (size == 4) { int32_t v; std::memcpy(&v, src, 4); return type == "U" ? (double)(uint32_t)v : (double)v; }
  if (size == 2) { int16_t v; std::memcpy(&v, src, 2); return type == "U" ? (double)(uint16_t)v : (double)v; }
  return type == "I" ? (double)(signed char)src[0] : (double)(unsigned char)src[0];
}

// Cloud::loadPointCloudFromFile (cloud.cpp:643-660): .pcd (pcl::io::loadPCDFile) or .ply (pcl::io::loadPLYFile) by extension
bool Cloud::loadPointCloudFromFile(const std::string &filename) {
  const std::string extension = filename.size() >= 3 ? filename.substr(filename.size() - 3) : "";
  if (extension == "ply") return loadPly(filename);
  return loadPcd(filename);
}

// .ply reader: "format ascii 1.0" or "binary_little_endian 1.0", element vertex with properties x y z [nx ny nz] (any
// scalar types; other properties and elements after the vertices are ignored; list properties inside the vertex element
// are not supported). NaN points are dropped.
bool Cloud::loadPly(const std::string &filename) {
  std::ifstream f(filename.c_str(), std::ios::binary);
  if (!f) {
    std::cout << "Couldn't read PLY file: " << filename << "\n";
    return false;
  }
  std::string line, format;
  struct Prop { std::string name, type; int size; };
  std::vector<Prop> props;
  size_t nvert = 0;
  bool in_vertex = false, vertex_first = true, seen_element = false;
  auto type_size = [](const std::string &t) {
    if (t == "char" || t == "uchar" || t == "int8" || t == "uint8") return 1;
    if (t == "short" || t == "ushort" || t == "int16" || t == "uint16") return 2;
    if (t == "int" || t == "uint" || t == "float" || t == "int32" || t == "uint32" || t == "float32") return 4;
    if (t == "double" || t == "float64") return 8;
    return 0;
  };
  if (!std::getline(f, line) || line.substr(0, 3) != "ply") {
    std::cout << "Not a PLY file: " << filename << "\n";
    return false;
  }
  while (std::getline(f, line)) {
    if (!line.empty() && line.back() == '\r') line.pop_back();
    std::istringstream ss(line);
    std::string tag;
    ss >> tag;
    if (tag == "format") ss >> format;
    else if (tag == "element") {
      std::string name;
      size_t n;
      ss >> name >> n;
      in_vertex = name == "vertex";
      if (in_vertex) { nvert = n; vertex_first = !seen_element; }
      seen_element = true;
    } else if (tag == "property" && in_vertex) {
      std::string t, name;
      ss >> t;
      if (t == "list") { std::cout << "PLY: list property inside the vertex element is not supported\n"; return false; }
      ss >> name;
      props.push_back({name, t, type_size(t)});
      if (props.back().size == 0) { std::cout << "PLY: unknown property type " << t << "\n"; return false; }
    } else if (tag == "end_header") break;
  }
  auto idx_of = [&](const char *a, const char *b) { for (size_t i = 0; i < props.size(); i++) if (props[i].name == a || props[i].name == b) return (int)i; return -1; };
  const int ix = idx_of("x", "x"), iy = idx_of("y", "y"), iz = idx_of("z", "z");
  const int inx = idx_of("nx", "normal_x"), iny = idx_of("ny", "normal_y"), inz = idx_of("nz", "normal_z");
  if (ix < 0 || iy < 0 || iz < 0 || !vertex_first) {
    std::cout << "PLY: need a leading vertex element with x y z: " << filename << "\n";
    return false;
  }
  points_.clear();
  normals_.clear();
  std::vector<double> row(props.size());
  auto push = [&]() {
    if (!std::isfinite(row[ix]) || !std::isfinite(row[iy]) || !std::isfinite(row[iz])) return;
    points_.push_back((float)row[ix]); points_.push_back((float)row[iy]); points_.push_back((float)row[iz]);
    if (inx >= 0 && iny >= 0 && inz >= 0) {
      normals_.push_back((double)(float)row[inx]); normals_.push_back((double)(float)row[iny]); normals_.push_back((double)(float)row[inz]);
    }
  };
  if (format == "ascii") {
    for (size_t v = 0; v < nvert && std::getline(f, line); v++) {
      std::istringstream ss(line);
      bool ok = true;
      for (size_t i = 0; i < props.size() && ok; i++) {
        std::string tok;
        if (!(ss >> tok)) ok = false;
        else row[i] = (tok == "nan" || tok == "NaN") ? NAN : std::atof(tok.c_str());
      }
      if (ok) push();
    }
  } else if (format == "binary_little_endian") {
    size_t stride = 0;
    std::vector<size_t> off(props.size());
    for (size_t i = 0; i < props.size(); i++) { off[i] = stride; stride += (size_t)props[i].size; }
    std::vector<char> buf(stride);
    for (size_t v = 0; v < nvert && f.read(buf.data(), stride); v++) {
      for (size_t i = 0; i < props.size(); i++) {
        const std::string &t = props[i].type;
        const bool is_f = t[0] == 'f' || t[0] == 'd';
        const bool is_u = t[0] == 'u';
        row[i] = read_scalar(buf.data() + off[i], is_f ? "F" : (is_u ? "U" : "I"), props[i].size);
      }
      push();
    }
  } else {
    std::cout << "Unsupported PLY format '" << format << "' (ascii and binary_little_endian are supported)\n";
    return false;
  }
  printf("Loaded point cloud with %zu points\n", size());
  return true;
}

// .pcd reader: header fields FIELDS/SIZE/TYPE/COUNT/POINTS/DATA (ascii | binary | binary_compressed)
bool Cloud::loadPcd(const std::string &filename) {
  std::ifstream f(filename.c_str(), std::ios::binary);
  if (!f) {
    std::cout << "Couldn't read PCD file: " << filename << "\n";
    return false;
  }
  std::vector<std::string> fields, types;
  std::vector<int> sizes, counts;
  size_t npoints = 0;
  std::string data_kind, line;
  while (std::getline(f, line)) {
    if (!line.empty() && line.back() == '\r') line.pop_back();
    std::istringstream ss(line);
    std::string tag;
    ss >> tag;
    std::string tok;
    if (tag == "FIELDS") while (ss >> tok) fields.push_back(tok);
    else if (tag == "SIZE") while (ss >> tok) sizes.push_back(std::atoi(tok.c_str()));
    else if (tag == "TYPE") while (ss >> tok) types.push_back(tok);
    else if (tag == "COUNT") while (ss >> tok) counts.push_back(std::atoi(tok.c_str()));
    else if (tag == "POINTS") ss >> npoints;
    else if (tag == "DATA") { ss >> data_kind; break; }
  }
  if (counts.empty()) counts.assign(fields.size(), 1);
  bool header_ok = !fields.empty() && sizes.size() == fields.size() && types.size() == fields.size() && counts.size() == fields.size();
  for (size_t i = 0; header_ok && i < fields.size(); i++)  // the readers below index buffers with these: trust nothing
    header_ok = (sizes[i] == 1 || sizes[i] == 2 || sizes[i] == 4 || sizes[i] == 8) && counts[i] >= 1 && counts[i] <= 4096 &&
                (types[i] == "F" || types[i] == "I" || types[i] == "U") && !(types[i] == "F" && sizes[i] < 4);
  if (!header_ok) {
    std::cout << "Bad .pcd header: " << filename << "\n";
    return false;
  }
  auto idx_of = [&](const char *n) { for (size_t i = 0; i < fields.size(); i++) if (fields[i] == n) return (int)i; return -1; };
  const int ix = idx_of("x"), iy = idx_of("y"), iz = idx_of("z");
  const int inx = idx_of("normal_x"), iny = idx_of("normal_y"), inz = idx_of("normal_z");
  if (ix < 0 || iy < 0 || iz < 0) {
    std::cout << "No x/y/z fields in: " << filename << "\n";
    return false;
  }
  points_.clear();
  normals_.clear();
  std::vector<double> row(fields.size());
  auto push = [&]() {
    if (!std::isfinite(row[ix]) || !std::isfinite(row[iy]) || !std::isfinite(row[iz])) return;
    points_.push_back((float)row[ix]); points_.push_back((float)row[iy]); points_.push_back((float)row[iz]);
    if (inx >= 0 && iny >= 0 && inz >= 0) {  // PCL normals are float32
      normals_.push_back((double)(float)row[inx]); normals_.push_back((double)(float)row[iny]); normals_.push_back((double)(float)row[inz]);
    }
  };
  if (data_kind == "ascii") {
    while (std::getline(f, line)) {
      std::istringstream ss(line);
      bool ok = true;
      for (size_t i = 0; i < fields.size() && ok; i++) {
        std::string tok;
        for (int c = 0; c < counts[i]; c++) {
          if (!(ss >> tok)) { ok = false; break; }
          if (c == 0) row[i] = (tok == "nan" || tok == "NaN") ? NAN : std::atof(tok.c_str());
        }
      }
      if (ok) push();
    }
  } else if (data_kind == "binary") {
    size_t stride = 0;
    std::vector<size_t> off(fields.size());
    for (size_t i = 0; i < fields.size(); i++) { off[i] = stride; stride += (size_t)sizes[i] * counts[i]; }
    std::vector<char> buf(stride);
    for (size_t p = 0; p < npoints && f.read(buf.data(), stride); p++) {
      for (size_t i = 0; i < fields.size(); i++) row[i] = read_scalar(buf.data() + off[i], types[i], sizes[i]);
      push();
    }
  } else if (data_kind == "binary_compressed") {
    // uint32 compressed size, uint32 uncompressed size, LZF stream; the payload is stored field by field (SoA):
    // all values of field 0, then all of field 1, ... (pcl/io/pcd_io.cpp)
    uint32_t csize = 0, usize = 0;
    f.read(reinterpret_cast<char *>(&csize), 4);
    f.read(reinterpret_cast<char *>(&usize), 4);
    size_t stride = 0;
    std::vector<size_t> foff(fields.size());
    for (size_t i = 0; i < fields.size(); i++) { foff[i] = stride * npoints; stride += (size_t)sizes[i] * counts[i]; }
    std::vector<unsigned char> comp(csize), raw(usize);
    if (!f.read(reinterpret_cast<char *>(comp.data()), csize) || (size_t)usize != stride * npoints ||
        !lzf_decompress(comp.data(), csize, raw.data(), usize)) {
      std::cout << "Bad binary_compressed payload in: " << filename << "\n";
      return false;
    }
    for (size_t p = 0; p < npoints; p++) {
      for (size_t i = 0; i < fields.size(); i++)
        row[i] = read_scalar(reinterpret_cast<const char *>(raw.data()) + foff[i] + p * (size_t)sizes[i] * counts[i], types[i], sizes[i]);
      push();
    }
  } else {
    std::cout << "Unsupported .pcd DATA kind '" << data_kind << "' (ascii, binary and binary_compressed are supported)\n";
    return false;
  }
  printf("Loaded point cloud with %zu points\n", size());
  return true;
}

void Cloud::setNormalsFromFile(const std::string &filename) {
  std::ifstream f(filename.c_str());
  std::vector<std::vector<double>> rows;
  std::string line;
  while (std::getline(f, line)) {
    for (char &c : line) if (c == ',') c = ' ';
    std::istringstream ss(line);
    std::vector<double> r;
    double v;
    while (ss >> v) r.push_back(v);
    if (!r.empty()) rows.push_back(r);
  }
  const size_t n = size();
  normals_.assign(3 * n, 0.0);
  if (rows.size() == 3 && rows[0].size() == n) {  // 3 x N
    for (size_t i = 0; i < n; i++) for (int r = 0; r < 3; r++) normals_[3 * i + r] = rows[r][i];
  } else if (rows.size() == n && rows[0].size() >= 3) {  // N x 3
    for (size_t i = 0; i < n; i++) for (int r = 0; r < 3; r++) normals_[3 * i + r] = rows[i][r];
  } else {
    std::cout << "ERROR: normals file does not match the cloud (" << rows.size() << " rows for " << n << " points)\n";
    normals_.clear();
  }
  touch();
}

void Cloud::touch() {
  static std::atomic<unsigned> counter{0};  // clouds may be built on several threads
  revision_ = ++counter;
}

void Cloud::setProcessed(std::vector<float> points, std::vector<double> normals, std::vector<int> camera_source) {
  points_ = std::move(points);
  normals_ = std::move(normals);
  camera_source_ = std::move(camera_source);
  sample_indices_.clear();
  plane_indices_.clear();
  touch();
}

void Cloud::subsample(int num_samples) {
  const int n = (int)size();
  if (!plane_indices_.empty()) {  // subsampleSampleIndices (cloud.cpp:350-361,395-405), rand() -> a fixed-seed LCG
    const unsigned m = (unsigned)plane_indices_.size();
    if (num_samples <= 0 || (unsigned)num_samples >= m) {
      sample_indices_ = plane_indices_;
      return;
    }
    sample_indices_.resize(num_samples);
    unsigned s = 42u;
    for (int i = 0; i < num_samples; i++) {
      s = s * 1664525u + 1013904223u;
      sample_indices_[i] = plane_indices_[s % m];
    }
    return;
  }
  sample_indices_.clear();
  if (num_samples <= 0 || n == 0) return;
  if (num_samples >= n) {  // pcl::RandomSample returns every index (cloud.cpp:364-370)
    for (int i = 0; i < n; i++) sample_indices_.push_back(i);
    return;
  }
  std::vector<int> perm(n);
  for (int i = 0; i < n; i++) perm[i] = i;
  unsigned s = 42u;
  for (int i = 0; i < num_samples; i++) {  // partial Fisher-Yates with a fixed-seed LCG
    s = s * 1664525u + 1013904223u;
    int j = i + (int)(s % (unsigned)(n - i));
    std::swap(perm[i], perm[j]);
  }
  sample_indices_.assign(perm.begin(), perm.begin() + num_samples);
}

}  // namespace util

// ------------------------------------------------------------------------------------------------ geometry cfg
namespace candidate {
HandGeometry::HandGeometry(const std::string &filepath) {
  util::ConfigFile c(filepath);
  c.ExtractKeys();
  finger_width_ = c.getValueOfKey<double>("finger_width", 0.01);
  outer_diameter_ = c.getValueOfKey<double>("hand_outer_diameter", 0.12);
  depth_ = c.getValueOfKey<double>("hand_depth", 0.06);
  height_ = c.getValueOfKey<double>("hand_height", 0.02);
  init_bite_ = c.getValueOfKey<double>("init_bite", 0.01);
}
void Hand::print() const {
  auto v = [](const std::array<double, 3> &a) { printf("%g %g %g\n", a[0], a[1], a[2]); };
  printf("position: "); v(getPosition());
  printf("approach: "); v(getApproach());
  printf("binormal: "); v(getBinormal());
  printf("axis: "); v(getAxis());
  printf("score: %g\nfull-antipodal: %d\nhalf-antipodal: %d\nclosing box:\n bottom: %g\n top: %g\n center: %g\n", getScore(),
         (int)isFullAntipodal(), (int)isHalfAntipodal(), getBottom(), getTop(), getCenter());
}
}  // namespace candidate
namespace descriptor {
ImageGeometry::ImageGeometry(const std::string &filepath) {
  util::ConfigFile c(filepath);
  c.ExtractKeys();
  outer_diameter_ = c.getValueOfKey<double>("volume_width", 0.10);
  depth_ = c.getValueOfKey<double>("volume_depth", 0.06);
  height_ = c.getValueOfKey<double>("volume_height", 0.02);
  size_ = c.getValueOfKey<int>("image_size", 60);
  num_channels_ = c.getValueOfKey<int>("image_num_channels", 15);
}
}  // namespace descriptor

// ------------------------------------------------------------------------------------------------ helpers
static void fill_hand_search(gpdb_params &p, const candidate::HandSearch::Parameters &hs) {
  p.finger_width = hs.hand_geometry_.finger_width_;
  p.hand_outer_diameter = hs.hand_geometry_.outer_diameter_;
  p.hand_depth = hs.hand_geometry_.depth_;
  p.hand_height = hs.hand_geometry_.height_;
  p.init_bite = hs.hand_geometry_.init_bite_;
  p.nn_radius = hs.nn_radius_frames_;
  p.num_orientations = hs.num_orientations_;
  p.num_finger_placements = hs.num_finger_placements_;
  p.num_hand_axes = (int32_t)std::min<size_t>(hs.hand_axes_.size(), GPDB_MAX_HAND_AXES);
  for (int i = 0; i < p.num_hand_axes; i++) p.hand_axes[i] = hs.hand_axes_[i];
  p.deepen_hand = hs.deepen_hand_;
  p.friction_coeff = hs.friction_coeff_;
  p.min_viable = hs.min_viable_;
}
static void fill_image_geometry(gpdb_params &p, const descriptor::ImageGeometry &g) {
  p.volume_width = g.outer_diameter_;
  p.volume_depth = g.depth_;
  p.volume_height = g.height_;
  p.image_size = g.size_;
  p.image_num_channels = g.num_channels_;
}
static gpdb_ctx *make_ctx(const gpdb_params &p) {
  gpdb_ctx *ctx = nullptr;
  if (gpdb_create(&p, &ctx) != GPDB_OK) {
    printf("ERROR: %s\n", gpdb_last_error(nullptr));
    return nullptr;
  }
  return ctx;
}
static int upload_cloud(gpdb_ctx *ctx, const util::Cloud &cloud) {
  if (cloud.getNormals().size() != 3 * cloud.size()) {
    printf("ERROR: the cloud has no surface normals: call GraspDetector::preprocessPointCloud first (gpdb_preprocess)\n");
    return GPDB_ERR_INVALID;
  }
  return gpdb_set_cloud(ctx, cloud.getPoints().data(), cloud.getNormals().data(),
                        cloud.getCameraSource().empty() ? nullptr : cloud.getCameraSource().data(), (int)cloud.size(),
                        cloud.getViewPoints().data(), cloud.numCameras());
}

bool paramsFromConfig(const std::string &config_filename, gpdb_params &p, std::string &weights_file, int &num_selected,
                      int &num_samples, int &min_inliers) {
  util::ConfigFile config_file(config_filename);
  if (!config_file.ExtractKeys()) return false;
  gpdb_params_default(&p);
  std::string hand_geometry_filename = config_file.getValueOfKeyAsString("hand_geometry_filename", "");
  if (hand_geometry_filename == "0" || hand_geometry_filename.empty()) hand_geometry_filename = config_filename;
  std::string image_geometry_filename = config_file.getValueOfKeyAsString("image_geometry_filename", "");
  if (image_geometry_filename == "0" || image_geometry_filename.empty()) image_geometry_filename = config_filename;
  candidate::HandSearch::Parameters hs;
  hs.hand_geometry_ = candidate::HandGeometry(hand_geometry_filename);
  hs.nn_radius_frames_ = config_file.getValueOfKey<double>("nn_radius", 0.01);
  hs.num_samples_ = config_file.getValueOfKey<int>("num_samples", 1000);
  hs.num_threads_ = config_file.getValueOfKey<int>("num_threads", 1);
  hs.num_orientations_ = config_file.getValueOfKey<int>("num_orientations", 8);
  hs.num_finger_placements_ = config_file.getValueOfKey<int>("num_finger_placements", 10);
  hs.deepen_hand_ = config_file.getValueOfKey<bool>("deepen_hand", true);
  hs.hand_axes_ = config_file.getValueOfKeyAsStdVectorInt("hand_axes", "2");
  hs.friction_coeff_ = config_file.getValueOfKey<double>("friction_coeff", 20.0);
  hs.min_viable_ = config_file.getValueOfKey<int>("min_viable", 6);
  fill_hand_search(p, hs);
  fill_image_geometry(p, descriptor::ImageGeometry(image_geometry_filename));
  weights_file = config_file.getValueOfKeyAsString("weights_file", "");
  p.device = 0;  // the cfg `device` key selects the reference's CPU/GPU/VPU backend; here: CUDA device 0
  p.batch_size = 0;
  std::vector<double> ws = config_file.getValueOfKeyAsStdVectorDouble("workspace_grasps", "-1 1 -1 1 -1 1");
  for (size_t i = 0; i < 6 && i < ws.size(); i++) p.workspace_grasps[i] = ws[i];
  p.min_aperture = config_file.getValueOfKey<double>("min_aperture", 0.0);
  p.max_aperture = config_file.getValueOfKey<double>("max_aperture", 0.085);
  p.filter_approach_direction = config_file.getValueOfKey<bool>("filter_approach_direction", false);
  std::vector<double> dir = config_file.getValueOfKeyAsStdVectorDouble("direction", "1 0 0");
  for (size_t i = 0; i < 3 && i < dir.size(); i++) p.direction[i] = dir[i];
  p.thresh_rad = config_file.getValueOfKey<double>("thresh_rad", 2.3);
  min_inliers = config_file.getValueOfKey<int>("min_inliers", 1);
  num_selected = config_file.getValueOfKey<int>("num_selected", 100);
  num_samples = hs.num_samples_;
  return true;
}

// ------------------------------------------------------------------------------------------------ HandSearch
namespace candidate {
HandSearch::HandSearch(Parameters params) : params_(params) {
  gpdb_params p;
  gpdb_params_default(&p);
  fill_hand_search(p, params_);
  // HandSearch::searchHands does not filter (the workspace / aperture filters belong to GraspDetector): open them
  p.min_aperture = -1e300;
  p.max_aperture = 1e300;
  for (int i = 0; i < 3; i++) {
    p.workspace_grasps[2 * i] = -1e300;
    p.workspace_grasps[2 * i + 1] = 1e300;
  }
  ctx_ = make_ctx(p);
}
HandSearch::~HandSearch() { gpdb_destroy(ctx_); }

std::vector<std::unique_ptr<HandSet>> HandSearch::searchHands(const util::Cloud &cloud_cam) const {
  std::vector<std::unique_ptr<HandSet>> out;
  const std::vector<int> &idx = cloud_cam.getSampleIndices();
  if (!ctx_ || idx.empty()) {
    std::cout << "Error: No samples or no indices!\n";
    return out;
  }
  if (upload_cloud(ctx_, cloud_cam) != GPDB_OK) return out;
  gpdb_result r;
  if (gpdb_hand_search(ctx_, idx.data(), (int)idx.size(), &r) < 0) {
    printf("ERROR: %s\n", gpdb_last_error(ctx_));
    return out;
  }
  const int P = r.poses_per_sample;
  int c = 0;
  for (int i = 0; i < r.n_samples; i++) {
    if (!r.frame_valid[i]) continue;  // frames without neighbours are dropped (frame_estimator.cpp:24-29)
    auto hs = std::make_unique<HandSet>();
    if (idx[i] < (int)cloud_cam.size())  // evalHandSet always sets sample_ (hand_set.cpp:36), also for sets without a hand
      for (int k = 0; k < 3; k++) hs->sample_[k] = (double)cloud_cam.getPoints()[3 * (size_t)idx[i] + k];
    for (int k = 0; k < 9; k++) hs->frame_[k] = r.frames[9 * (size_t)i + k];
    hs->hands_.resize(P);
    hs->is_valid_.assign(P, false);
    for (int j = 0; j < P; j++) {
      const uint8_t fl = r.pose_flags[(size_t)i * P + j];
      // a hand is handed on only when it is valid AND survives the filters (its record exists): a VALID pose that a filter
      // removed must not reach ImageGenerator::createImages with an empty Hand
      hs->is_valid_[j] = (fl & 3) == 3;
      if ((fl & 3) == 3) {
        hs->hands_[j] = std::make_unique<Hand>(r.candidates[c]);
        for (int k = 0; k < 3; k++) hs->sample_[k] = r.candidates[c].sample[k];
        c++;
      } else {
        hs->hands_[j] = std::make_unique<Hand>();  // invalid pose: no record (the reference keeps a stale pre-deepen box)
      }
    }
    out.push_back(std::move(hs));
  }
  gpdb_free_result(&r);
  printf("Found %d hand sets\n", (int)out.size());
  return out;
}
}  // namespace candidate

// ------------------------------------------------------------------------------------------------ ImageGenerator
namespace descriptor {
ImageGenerator::ImageGenerator(const ImageGeometry &image_geometry, int, int, bool, bool) : image_params_(image_geometry) {
  gpdb_params p;
  gpdb_params_default(&p);
  fill_image_geometry(p, image_params_);
  ctx_ = make_ctx(p);
}
ImageGenerator::~ImageGenerator() { gpdb_destroy(ctx_); }

void ImageGenerator::createImages(const util::Cloud &cloud_cam,
                                  const std::vector<std::unique_ptr<candidate::HandSet>> &hand_set_list,
                                  std::vector<std::unique_ptr<Image>> &images_out,
                                  std::vector<std::unique_ptr<candidate::Hand>> &hands_out) const {
  if (!ctx_ || upload_cloud(ctx_, cloud_cam) != GPDB_OK) return;
  std::vector<gpdb_pose> poses;
  for (const auto &hs : hand_set_list)
    for (size_t j = 0; j < hs->getHands().size(); j++)
      if (hs->getIsValid()[j]) poses.push_back(hs->getHands()[j]->raw());
  const size_t isz = (size_t)image_params_.size_ * image_params_.size_ * image_params_.num_channels_;
  std::vector<uint8_t> buf(isz * poses.size());
  if (gpdb_images(ctx_, poses.data(), (int)poses.size(), buf.data()) < 0) {
    printf("ERROR: %s\n", gpdb_last_error(ctx_));
    return;
  }
  size_t k = 0;
  for (const auto &hs : hand_set_list)
    for (size_t j = 0; j < hs->getHands().size(); j++)
      if (hs->getIsValid()[j]) {
        auto im = std::make_unique<Image>();
        im->rows = im->cols = image_params_.size_;
        im->channels = image_params_.num_channels_;
        im->data.assign(buf.begin() + isz * k, buf.begin() + isz * (k + 1));
        images_out.push_back(std::move(im));
        hands_out.push_back(std::move(const_cast<std::unique_ptr<candidate::Hand> &>(hs->getHands()[j])));
        k++;
      }
  printf("Created %zu images\n", images_out.size());
}
}  // namespace descriptor

// ------------------------------------------------------------------------------------------------ Classifier
// An OpenVINO IR (weights_file *.bin / *.xml, not a directory) may carry ReLU layers after the convolutions
// (models/openvino/two_views_12_channels_curv_axis.xml): the context must be created with relu_after_conv = 1 then.
static int relu_after_conv_of(const std::string &model_file, const std::string &weights_file, int num_channels) {
  if (weights_file.empty() || weights_file.back() == '/') return 0;
  const bool ir = weights_file.size() > 4 && (weights_file.compare(weights_file.size() - 4, 4, ".bin") == 0 ||
                                               weights_file.compare(weights_file.size() - 4, 4, ".xml") == 0);
  if (!ir) return 0;
  const size_t sizes[8] = {(size_t)20 * num_channels * 25, 20, 50 * 20 * 25, 50, (size_t)500 * 7200, 500, 1000, 2};
  std::vector<std::vector<float>> bufs(8);
  float *ptrs[8];
  for (int i = 0; i < 8; i++) {
    bufs[i].resize(sizes[i]);
    ptrs[i] = bufs[i].data();
  }
  int relu = -1;
  char err[512];
  if (gpdb_read_weights_file(model_file.empty() ? nullptr : model_file.c_str(), weights_file.c_str(), num_channels, ptrs, &relu, err,
                             sizeof(err)) != GPDB_OK)
    return 0;
  return relu >= 3 ? 1 : 0;
}

namespace net {
namespace {
class CudaClassifier : public Classifier {
 public:
  CudaClassifier(const std::string &model_file, const std::string &weights_file, int batch_size, int num_channels)
      : batch_size_(batch_size) {
    gpdb_params p;
    gpdb_params_default(&p);
    p.image_num_channels = num_channels;
    p.batch_size = batch_size > 1 ? batch_size : 0;
    p.relu_after_conv = relu_after_conv_of(model_file, weights_file, num_channels);
    ctx_ = make_ctx(p);
    if (ctx_ && gpdb_load_weights_file(ctx_, model_file.empty() ? nullptr : model_file.c_str(), weights_file.c_str()) != GPDB_OK)
      printf("ERROR: %s\n", gpdb_last_error(ctx_));
    isz_ = (size_t)p.image_size * p.image_size * num_channels;
  }
  ~CudaClassifier() override { gpdb_destroy(ctx_); }
  std::vector<float> classifyImages(const std::vector<std::unique_ptr<descriptor::Image>> &image_list) override {
    std::vector<float> predictions(image_list.size(), 0.0f);
    if (!ctx_ || image_list.empty()) return predictions;
    std::vector<uint8_t> packed(isz_ * image_list.size(), 0);
    for (size_t i = 0; i < image_list.size(); i++)
      if (image_list[i]->isContinuous() && image_list[i]->data.size() == isz_)
        std::memcpy(&packed[i * isz_], image_list[i]->data.data(), isz_);
    if (gpdb_classify(ctx_, packed.data(), (int)image_list.size(), predictions.data(), nullptr) < 0)
      printf("ERROR: %s\n", gpdb_last_error(ctx_));
    return predictions;
  }
  int getBatchSize() const override { return batch_size_; }

 private:
  gpdb_ctx *ctx_{nullptr};
  int batch_size_;
  size_t isz_{0};
};
}  // namespace
std::shared_ptr<Classifier> Classifier::create(const std::string &model_file, const std::string &weights_file, Device,
                                               int batch_size, int num_channels) {
  return std::make_shared<CudaClassifier>(model_file, weights_file, batch_size, num_channels);
}
}  // namespace net

// ------------------------------------------------------------------------------------------------ Clustering
std::vector<std::unique_ptr<candidate::Hand>> Clustering::findClusters(
    const std::vector<std::unique_ptr<candidate::Hand>> &hand_list, bool remove_inliers) const {
  const double AXIS_ALIGN_ANGLE_THRESH = 12.0 * M_PI / 180.0;  // clustering.cpp:9-13
  const double AXIS_ALIGN_DIST_THRESH = 0.005;
  const double MAX_DIST_THRESH = 0.05;
  std::vector<std::unique_ptr<candidate::Hand>> hands_out;
  const int n = (int)hand_list.size();
  std::vector<bool> has_used(n, false);
  for (int i = 0; i < n; i++) {
    int num_inliers = 0;
    double position_delta[3] = {0, 0, 0};
    const std::array<double, 3> ai = hand_list[i]->getAxis(), pi = hand_list[i]->getPosition();
    double outer[3][3];  // axis * axis^T
    for (int r = 0; r < 3; r++)
      for (int c = 0; c < 3; c++) outer[r][c] = ai[r] * ai[c];
    double mean = 0.0, standard_deviation = 0.0;
    for (int j = 0; j < n; j++) {
      if (i == j || (remove_inliers && has_used[j])) continue;
      const std::array<double, 3> aj = hand_list[j]->getAxis(), pj = hand_list[j]->getPosition();
      const double axis_aligned = ai[0] * aj[0] + ai[1] * aj[1] + ai[2] * aj[2];
      const bool axis_aligned_binary = std::fabs(axis_aligned) > std::cos(AXIS_ALIGN_ANGLE_THRESH);
      const double d[3] = {pi[0] - pj[0], pi[1] - pj[1], pi[2] - pj[2]};
      const bool delta_pos_mag_binary = std::sqrt(d[0] * d[0] + d[1] * d[1] + d[2] * d[2]) <= MAX_DIST_THRESH;
      double proj[3];  // (I - axis axis^T) * delta_pos
      for (int r = 0; r < 3; r++)
        proj[r] = ((r == 0 ? 1.0 : 0.0) - outer[r][0]) * d[0] + ((r == 1 ? 1.0 : 0.0) - outer[r][1]) * d[1] +
                  ((r == 2 ? 1.0 : 0.0) - outer[r][2]) * d[2];
      const bool delta_pos_proj_mag_binary =
          std::sqrt(proj[0] * proj[0] + proj[1] * proj[1] + proj[2] * proj[2]) <= AXIS_ALIGN_DIST_THRESH;
      if (axis_aligned_binary && delta_pos_mag_binary && delta_pos_proj_mag_binary) {
        num_inliers++;
        for (int r = 0; r < 3; r++) position_delta[r] += pj[r];
        const double old_mean = mean, sj = hand_list[j]->getScore();
        mean += (sj - mean) / (double)num_inliers;             // Welford update (clustering.cpp:66-70)
        standard_deviation += (sj - mean) * (sj - old_mean);
        if (remove_inliers) has_used[j] = true;
      }
    }
    if (num_inliers >= min_inliers_) {
      const double dn = (double)num_inliers;
      for (int r = 0; r < 3; r++) position_delta[r] = position_delta[r] / dn - pi[r];
      standard_deviation /= dn;
      if (standard_deviation != 0) standard_deviation = std::sqrt(standard_deviation);
      const double conf_lb = mean - 2.576 * standard_deviation / std::sqrt((double)num_inliers);
      auto hand = std::make_unique<candidate::Hand>(*hand_list[i]);
      hand->setPosition({pi[0] + position_delta[0], pi[1] + position_delta[1], pi[2] + position_delta[2]});
      hand->setScore(conf_lb);
      hand->setFullAntipodal(hand_list[i]->isFullAntipodal());
      hands_out.push_back(std::move(hand));
    }
  }
  return hands_out;
}

// ------------------------------------------------------------------------------------------------ GraspDetector
GraspDetector::GraspDetector(const std::string &config_filename) {
  std::string weights_file;
  int min_inliers = 0;
  if (!paramsFromConfig(config_filename, params_, weights_file, num_selected_, num_samples_, min_inliers)) return;
  cluster_grasps_ = min_inliers > 0;
  min_inliers_ = min_inliers;
  preprocessParamsFromConfig(config_filename, pre_params_);
  std::string model_file;
  {
    util::ConfigFile config_file(config_filename);
    if (config_file.ExtractKeys()) {
      model_file = config_file.getValueOfKeyAsString("model_file", "");  // grasp_detector.cpp:130
      sample_above_plane_ = config_file.getValueOfKey<bool>("sample_above_plane", false);  // grasp_detector.cpp:54-55
    }
  }
  if (relu_after_conv_of(model_file, weights_file, params_.image_num_channels)) params_.relu_after_conv = 1;
  model_file_ = model_file;
  weights_file_ = weights_file;
  ctx_ = make_ctx(params_);
  if (ctx_ && !weights_file.empty()) {
    // .bin parameter directory (EigenClassifier), .caffemodel (Caffe backend) or OpenVINO IR (classifier.cpp:33-61)
    if (gpdb_load_weights_file(ctx_, model_file.empty() ? nullptr : model_file.c_str(), weights_file.c_str()) == GPDB_OK)
      has_classifier_ = true;
    else printf("ERROR: %s\n", gpdb_last_error(ctx_));
  }
  printf("============ CLASSIFIER ======================\nweights_file: %s\n==============================================\n",
         weights_file.c_str());
}
GraspDetector::~GraspDetector() { gpdb_destroy(ctx_); }

bool preprocessParamsFromConfig(const std::string &config_filename, gpdb_preprocess_params &pp) {
  util::ConfigFile config_file(config_filename);
  gpdb_preprocess_params_default(&pp);
  if (!config_file.ExtractKeys()) return false;
  pp.voxelize = config_file.getValueOfKey<bool>("voxelize", true) ? 1 : 0;
  pp.voxel_size = config_file.getValueOfKey<double>("voxel_size", 0.003);
  pp.normals_radius = config_file.getValueOfKey<double>("normals_radius", 0.03);
  std::vector<double> ws = config_file.getValueOfKeyAsStdVectorDouble("workspace", "-1 1 -1 1 -1 1");
  for (size_t i = 0; i < 6 && i < ws.size(); i++) pp.workspace[i] = ws[i];
  if (config_file.getValueOfKey<bool>("remove_outliers", false) || config_file.getValueOfKey<int>("refine_normals_k", 0) > 0)
    printf("NOTE: remove_outliers / refine_normals_k are not part of the accelerated preprocessing: ignored\n");
  return true;
}

void GraspDetector::preprocessPointCloud(util::Cloud &cloud) {
  printf("Processing cloud with %zu points.\n", cloud.size());
  if (!ctx_ || cloud.size() == 0) return;
  gpdb_preprocess_params pp = pre_params_;
  // the reference recomputes the normals unconditionally (cloud.cpp:458-484), which discards a NORMALS_FILE the
  // caller supplied; here supplied normals are kept (voxel-averaged, cloud.cpp:307-311,331-333)
  pp.estimate_normals = cloud.hasNormals() ? 0 : 1;
  const int n = gpdb_preprocess(ctx_, cloud.getPoints().data(), cloud.hasNormals() ? cloud.getNormals().data() : nullptr,
                                cloud.getCameraSource().empty() ? nullptr : cloud.getCameraSource().data(), (int)cloud.size(),
                                cloud.getViewPoints().data(), cloud.numCameras(), &pp);
  if (n < 0) {
    printf("ERROR: %s\n", gpdb_last_error(ctx_));
    return;
  }
  double ms[6];
  gpdb_preprocess_timings(ctx_, ms);
  if (pp.voxelize) printf("Voxelized cloud: %d\n", n);
  if (pp.estimate_normals) printf("Calculated %d surface normals in %3.4fs (mode: B200).\n", n, ms[4] * 1e-3);
  std::vector<float> xyz(3 * (size_t)n);
  std::vector<double> nrm(3 * (size_t)n);
  std::vector<int> cam((size_t)n * cloud.numCameras());
  if (n > 0 && gpdb_get_cloud(ctx_, xyz.data(), nrm.data(), cam.data()) < 0) {
    printf("ERROR: %s\n", gpdb_last_error(ctx_));
    return;
  }
  cloud.setProcessed(std::move(xyz), std::move(nrm), std::move(cam));
  installed_cloud_ = n > 0 ? &cloud : nullptr;  // the processed cloud is already resident: detectGrasps skips the upload
  installed_revision_ = cloud.revision();
  if (sample_above_plane_ && n > 0) {  // Cloud::sampleAbovePlane (candidates_generator.cpp:32-34, cloud.cpp:407-435)
    printf("Sampling above plane ...\n");
    gpdb_plane_params plp;
    gpdb_plane_params_default(&plp);
    std::vector<int> off((size_t)n);
    const int m = gpdb_sample_above_plane(ctx_, &plp, off.data(), nullptr);
    if (m < 0) {
      printf("ERROR: %s\n", gpdb_last_error(ctx_));
    } else if (m > 0) {
      off.resize(m);
      cloud.setPlaneIndices(off);
      printf(" Plane fit succeeded. %zu samples above plane.\n", off.size());
    } else {
      printf(" Plane fit failed. Using entire point cloud ...\n");
    }
  }
  cloud.subsample(num_samples_);
}

std::vector<std::unique_ptr<candidate::Hand>> GraspDetector::selectGrasps(
    std::vector<std::unique_ptr<candidate::Hand>> &hands) const {
  printf("Selecting the %d highest scoring grasps ...\n", num_selected_);
  int middle = std::min((int)hands.size(), num_selected_);
  std::partial_sort(hands.begin(), hands.begin() + middle, hands.end(),
                    [](const std::unique_ptr<candidate::Hand> &a, const std::unique_ptr<candidate::Hand> &b) {
                      return a->getScore() > b->getScore();
                    });
  std::vector<std::unique_ptr<candidate::Hand>> out;
  for (int i = 0; i < middle; i++) out.push_back(std::move(hands[i]));
  return out;
}

bool GraspDetector::ensureCloud(const util::Cloud &cloud) {
  if (installed_cloud_ == &cloud && installed_revision_ == cloud.revision()) return true;
  if (upload_cloud(ctx_, cloud) != GPDB_OK) {
    printf("ERROR: %s\n", gpdb_last_error(ctx_));
    return false;
  }
  installed_cloud_ = &cloud;
  installed_revision_ = cloud.revision();
  return true;
}

// sample indices of a cloud for the C-ABI: its setSamples positions (installed with gpdb_set_samples) take precedence over
// its sample indices (hand_search.cpp:33-47)
static bool sample_indices_of(gpdb_ctx *ctx, const util::Cloud &cloud, std::vector<int> &idx) {
  idx = cloud.getSampleIndices();
  if (!cloud.getSamples().empty()) {
    const int ns = (int)(cloud.getSamples().size() / 3);
    const int first = gpdb_set_samples(ctx, cloud.getSamples().data(), ns);
    if (first < 0) {
      printf("ERROR: %s\n", gpdb_last_error(ctx));
      return false;
    }
    idx.resize(ns);
    for (int i = 0; i < ns; i++) idx[i] = first + i;
  }
  return true;
}

std::vector<std::unique_ptr<candidate::Hand>> GraspDetector::generateGraspCandidates(const util::Cloud &cloud) {
  std::vector<std::unique_ptr<candidate::Hand>> hands;
  if (!ctx_ || !ensureCloud(cloud)) return hands;
  std::vector<int> idx;
  if (!sample_indices_of(ctx_, cloud, idx) || idx.empty()) return hands;
  gpdb_result r;
  if (gpdb_hand_search(ctx_, idx.data(), (int)idx.size(), &r) < 0) {
    printf("ERROR: %s\n", gpdb_last_error(ctx_));
    return hands;
  }
  for (int i = 0; i < r.n_candidates; i++) hands.push_back(std::make_unique<candidate::Hand>(r.candidates[i]));
  gpdb_free_result(&r);
  return hands;
}

bool GraspDetector::createGraspImages(util::Cloud &cloud, std::vector<std::unique_ptr<candidate::Hand>> &hands_out,
                                      std::vector<std::vector<uint8_t>> &images_out) {
  hands_out.clear();
  images_out.clear();
  if (cloud.size() == 0) {
    printf("ERROR: Point cloud is empty!");
    return false;
  }
  hands_out = generateGraspCandidates(cloud);  // 1. candidates, 2. filters (fused in the hand-search kernel)
  printf("Generated %zu filtered grasp candidates.\n", hands_out.size());
  if (hands_out.empty()) return false;
  // 3. grasp descriptors (ImageGenerator::createImages) for exactly these hands
  const size_t isz = (size_t)params_.image_size * params_.image_size * params_.image_num_channels;
  std::vector<gpdb_pose> rec(hands_out.size());
  for (size_t i = 0; i < rec.size(); i++) rec[i] = hands_out[i]->raw();
  std::vector<uint8_t> all(isz * rec.size());
  if (gpdb_images(ctx_, rec.data(), (int)rec.size(), all.data()) < 0) {
    printf("ERROR: %s\n", gpdb_last_error(ctx_));
    hands_out.clear();
    return false;
  }
  images_out.resize(rec.size());
  for (size_t i = 0; i < rec.size(); i++) images_out[i].assign(all.begin() + isz * i, all.begin() + isz * (i + 1));
  return true;
}

std::vector<int> GraspDetector::evalGroundTruth(const util::Cloud &cloud_gt, std::vector<std::unique_ptr<candidate::Hand>> &hands) {
  std::vector<int> labels(hands.size(), 0);
  if (!ctx_ || hands.empty() || !ensureCloud(cloud_gt)) return labels;
  std::vector<gpdb_pose> rec(hands.size());
  for (size_t i = 0; i < hands.size(); i++) rec[i] = hands[i]->raw();
  if (gpdb_reevaluate(ctx_, rec.data(), (int)rec.size(), labels.data()) < 0) {
    printf("ERROR: %s\n", gpdb_last_error(ctx_));
    return std::vector<int>(hands.size(), 0);
  }
  for (size_t i = 0; i < hands.size(); i++) {
    hands[i]->setHalfAntipodal(rec[i].half_antipodal != 0);
    hands[i]->setFullAntipodal(rec[i].full_antipodal != 0);
  }
  return labels;
}

// Clustering::findClusters (remove_inliers = false) on the device: gpdb_find_clusters
std::vector<std::unique_ptr<candidate::Hand>> GraspDetector::findClustersOnDevice(
    const std::vector<std::unique_ptr<candidate::Hand>> &hands, int min_inliers) {
  std::vector<std::unique_ptr<candidate::Hand>> out;
  if (!ctx_ || hands.empty()) return out;
  std::vector<gpdb_pose> in(hands.size()), res(hands.size());
  for (size_t i = 0; i < hands.size(); i++) in[i] = hands[i]->raw();
  const int n = gpdb_find_clusters(ctx_, in.data(), (int)in.size(), min_inliers, res.data());
  if (n < 0) {
    printf("ERROR: %s\n", gpdb_last_error(ctx_));
    return out;
  }
  for (int i = 0; i < n; i++) out.push_back(std::make_unique<candidate::Hand>(res[i]));
  return out;
}

std::vector<double> GraspDetector::candidateSamplePositions(const util::Cloud &cloud) {
  std::vector<double> out;
  if (!ctx_ || !ensureCloud(cloud)) return out;
  std::vector<int> idx;
  if (!sample_indices_of(ctx_, cloud, idx) || idx.empty()) return out;
  gpdb_result r;
  if (gpdb_hand_search(ctx_, idx.data(), (int)idx.size(), &r) < 0) {
    printf("ERROR: %s\n", gpdb_last_error(ctx_));
    return out;
  }
  int last_slot = -1;
  for (int i = 0; i < r.n_candidates; i++) {  // candidates are in (sample slot, pose slot) order
    if (r.candidates[i].sample_slot == last_slot) continue;
    last_slot = r.candidates[i].sample_slot;
    for (int k = 0; k < 3; k++) out.push_back(r.candidates[i].sample[k]);
  }
  gpdb_free_result(&r);
  return out;
}

std::vector<std::unique_ptr<candidate::Hand>> GraspDetector::classifyAtPositions(const util::Cloud &cloud,
                                                                                const std::vector<double> &positions,
                                                                                double min_score) {
  std::vector<std::unique_ptr<candidate::Hand>> out;
  const int ns = (int)(positions.size() / 3);
  if (!ctx_ || !has_classifier_ || ns == 0 || !ensureCloud(cloud)) return out;
  const int first = gpdb_set_samples(ctx_, positions.data(), ns);
  if (first < 0) {
    printf("ERROR: %s\n", gpdb_last_error(ctx_));
    return out;
  }
  std::vector<int> idx(ns);
  for (int i = 0; i < ns; i++) idx[i] = first + i;
  gpdb_result r;
  if (gpdb_detect(ctx_, idx.data(), ns, &r) < 0) {
    printf("ERROR: %s\n", gpdb_last_error(ctx_));
    return out;
  }
  for (int i = 0; i < r.n_candidates; i++)
    if ((double)r.candidates[i].score > min_score) out.push_back(std::make_unique<candidate::Hand>(r.candidates[i]));
  gpdb_free_result(&r);
  return out;
}

std::vector<std::unique_ptr<candidate::Hand>> GraspDetector::detectGraspsMultiGpu(const util::Cloud &cloud, int num_gpus) {
  std::vector<std::unique_ptr<candidate::Hand>> hands;
  if (num_gpus <= 1) return detectGrasps(cloud);
  if (cloud.size() == 0 || !has_classifier_ || cloud.getNormals().size() != 3 * cloud.size()) {
    printf("ERROR: detectGraspsMultiGpu needs a processed cloud with normals and classifier weights\n");
    return hands;
  }
  std::vector<int> idx = cloud.getSampleIndices();
  if (idx.empty()) {
    printf("ERROR: no sample indices\n");
    return hands;
  }
  char uid[GPDB_COMM_ID_BYTES];
  if (gpdb_comm_unique_id(uid) != GPDB_OK) {
    printf("ERROR: %s\n", gpdb_last_error(nullptr));
    return hands;
  }
  std::vector<std::vector<gpdb_pose>> per_rank(num_gpus);
  std::vector<int> rc(num_gpus, 0), total(num_gpus, 0);
  // phase 1, before any collective: one context per device + the weights. A rank that failed here would leave the others
  // blocked in ncclCommInitRank, so nothing collective starts unless every context exists.
  std::vector<gpdb_ctx *> ctxs(num_gpus, nullptr);
  bool all_ok = true;
  for (int r = 0; r < num_gpus && all_ok; r++) {
    gpdb_params p = params_;
    p.device = r;
    if (gpdb_create(&p, &ctxs[r]) != GPDB_OK ||
        gpdb_load_weights_file(ctxs[r], model_file_.empty() ? nullptr : model_file_.c_str(), weights_file_.c_str()) != GPDB_OK) {
      printf("ERROR (GPU %d): %s\n", r, gpdb_last_error(ctxs[r]));
      all_ok = false;
    }
  }
  if (!all_ok) {
    for (gpdb_ctx *c : ctxs)
      if (c) gpdb_destroy(c);
    return hands;
  }
  // phase 2: one host thread per rank (the collectives block until every rank has joined)
  std::vector<std::thread> th;
  for (int r = 0; r < num_gpus; r++)
    th.emplace_back([&, r]() {
      gpdb_ctx *c = ctxs[r];
      if (gpdb_comm_init(c, uid, r, num_gpus) != GPDB_OK) {
        printf("ERROR (GPU %d): %s\n", r, gpdb_last_error(c));
        rc[r] = -1;
      }
      if (rc[r] == 0) {
        int n = r == 0 ? gpdb_set_cloud_bcast(c, 0, cloud.getPoints().data(), cloud.getNormals().data(),
                                              cloud.getCameraSource().empty() ? nullptr : cloud.getCameraSource().data(),
                                              (int)cloud.size(), cloud.getViewPoints().data(), cloud.numCameras())
                       : gpdb_set_cloud_bcast(c, 0, nullptr, nullptr, nullptr, 0, nullptr, 0);
        gpdb_result res;
        if (n < 0 || gpdb_detect_sharded(c, idx.data(), (int)idx.size(), &res) < 0) {
          printf("ERROR (GPU %d): %s\n", r, gpdb_last_error(c));
          rc[r] = -1;
        } else {
          // this rank's num_selected best (ties keep the (sample, pose) order): the global top-k is among them
          std::vector<gpdb_pose> loc(res.candidates, res.candidates + res.n_candidates);
          std::stable_sort(loc.begin(), loc.end(), [](const gpdb_pose &a, const gpdb_pose &b) { return a.score > b.score; });
          if ((int)loc.size() > num_selected_) loc.resize(num_selected_);
          per_rank[r] = std::move(loc);
          total[r] = res.n_total_candidates;
          gpdb_free_result(&res);
        }
      }
      gpdb_destroy(c);
    });
  for (auto &t : th) t.join();
  for (int r = 0; r < num_gpus; r++)
    if (rc[r] != 0) return hands;
  std::vector<gpdb_pose> all;
  for (auto &v : per_rank) all.insert(all.end(), v.begin(), v.end());  // rank order = sample order
  std::stable_sort(all.begin(), all.end(), [](const gpdb_pose &a, const gpdb_pose &b) { return a.score > b.score; });
  if ((int)all.size() > num_selected_) all.resize(num_selected_);
  printf("Number of grasp candidates within workspace and gripper width: %d (on %d GPUs)\n", total[0], num_gpus);
  for (auto &p : all) hands.push_back(std::make_unique<candidate::Hand>(p));
  return hands;
}

std::vector<std::unique_ptr<candidate::Hand>> GraspDetector::detectGrasps(const util::Cloud &cloud) {
  std::vector<std::unique_ptr<candidate::Hand>> hands_out;
  if (cloud.size() == 0) {
    printf("ERROR: Point cloud is empty!");
    return hands_out;
  }
  if (!ctx_ || !has_classifier_) {
    printf("ERROR: detector not initialised (%s)\n", ctx_ ? "no classifier weights" : gpdb_last_error(nullptr));
    return hands_out;
  }
  if (!ensureCloud(cloud)) return hands_out;
  std::vector<int> idx;
  if (!sample_indices_of(ctx_, cloud, idx)) return hands_out;
  gpdb_result r;
  // steps 1-4 + selectGrasps in one call: the num_selected best hands are picked on the device and only they are
  // copied back (grasp_detector.cpp:222-283,405-420)
  int n = gpdb_detect_select(ctx_, idx.data(), (int)idx.size(), num_selected_, &r);
  if (n < 0) {
    printf("ERROR: %s\n", gpdb_last_error(ctx_));
    return hands_out;
  }
  printf("Generated %d hand sets.\n", r.n_samples);
  printf("Number of grasp candidates within workspace and gripper width: %d\n", r.n_total_candidates);
  printf("Selecting the %d highest scoring grasps ...\n", num_selected_);
  std::vector<std::unique_ptr<candidate::Hand>> hands;
  for (int i = 0; i < n; i++) hands.push_back(std::make_unique<candidate::Hand>(r.candidates[i]));
  last_ms_candidates = r.ms_candidates;
  last_ms_images = r.ms_images;
  last_ms_classify = r.ms_classify;
  gpdb_free_result(&r);
  if (cluster_grasps_) {  // 6. Cluster the grasps (grasp_detector.cpp:283-301)
    std::vector<std::unique_ptr<candidate::Hand>> clusters = findClustersOnDevice(hands, min_inliers_);
    printf("Found %d clusters.\n", (int)clusters.size());
    if (clusters.size() <= 3) {
      printf("Not enough clusters found! Adding all grasps from previous step.");
      for (auto &h : hands) clusters.push_back(std::move(h));
    }
    hands = std::move(clusters);
  }
  std::sort(hands.begin(), hands.end(), [](const std::unique_ptr<candidate::Hand> &a, const std::unique_ptr<candidate::Hand> &b) {
    return a->getScore() > b->getScore();
  });
  printf("======== Selected grasps ========\n");
  for (size_t i = 0; i < hands.size(); i++) std::cout << "Grasp " << i << ": " << hands[i]->getScore() << "\n";
  printf("======== RUNTIMES (device) ========\n 1. Candidate generation: %3.4fs\n 2. Descriptor extraction: %3.4fs\n"
         " 3. Classification: %3.4fs\n==========\n",
         last_ms_candidates * 1e-3, last_ms_images * 1e-3, last_ms_classify * 1e-3);
  return hands;
}

// ---- SequentialImportanceSampling (sequential_importance_sampling.cpp) -------------------------------------------------
SequentialImportanceSampling::SequentialImportanceSampling(const std::string &config_filename) {
  util::ConfigFile config_file(config_filename);
  config_file.ExtractKeys();
  num_init_samples_ = config_file.getValueOfKey<int>("num_init_samples", 50);  // :19-31
  num_iterations_ = config_file.getValueOfKey<int>("num_iterations", 5);
  num_samples_ = config_file.getValueOfKey<int>("num_samples_per_iteration", 50);
  prob_rand_samples_ = config_file.getValueOfKey<double>("prob_rand_samples", 0.3);
  radius_ = config_file.getValueOfKey<double>("standard_deviation", 0.02);
  sampling_method_ = config_file.getValueOfKey<int>("sampling_method", 0);
  min_score_ = config_file.getValueOfKey<double>("min_score", 0);
  workspace_ = config_file.getValueOfKeyAsStdVectorDouble("workspace", "-1 1 -1 1 -1 1");
  if (workspace_.size() != 6) workspace_ = {-1, 1, -1, 1, -1, 1};
  grasp_detector_ = std::make_unique<GraspDetector>(config_filename);
  clustering_ = std::make_unique<Clustering>(config_file.getValueOfKey<int>("min_inliers", 1));
}

std::vector<std::unique_ptr<candidate::Hand>> SequentialImportanceSampling::detectGrasps(util::Cloud &cloud) {
  std::vector<std::unique_ptr<candidate::Hand>> none;
  evaluated_.clear();
  kept_.clear();
  if (cloud.size() == 0) {
    printf("Error: Point cloud is empty!");
    return none;
  }
  std::mt19937 gen(seed_);
  auto uniform_index = [&](size_t n) { return (size_t)(gen() % (unsigned long)n); };  // rand() % n upstream
  // 1. Find initial grasp hypotheses (:68-79)
  cloud.setSamples({});
  cloud.subsample(num_init_samples_);
  for (int i : cloud.getSampleIndices())
    for (int k = 0; k < 3; k++) evaluated_.push_back((double)cloud.getPoints()[3 * (size_t)i + k]);
  kept_ = grasp_detector_->candidateSamplePositions(cloud);
  printf("Initially detected grasp candidates: %zu\n", kept_.size() / 3);
  if (kept_.empty()) return none;
  const int num_rand_samples = (int)(prob_rand_samples_ * num_samples_);  // :100-101
  const int num_gauss_samples = num_samples_ - num_rand_samples;
  const double sigma = radius_;
  const double term = 1.0 / std::sqrt(std::pow(2.0 * M_PI, 3.0) * std::pow(sigma, 3.0));
  std::normal_distribution<double> distr{0.0, sigma};
  const std::vector<int> init_indices = cloud.getSampleIndices();
  // 2. Find grasp hypotheses using importance sampling (:109-160)
  for (int it = 0; it < num_iterations_; it++) {
    std::vector<double> samples(3 * (size_t)num_samples_, 0.0);
    const size_t m = kept_.size() / 3;
    int j = 0;
    while (j < num_gauss_samples) {  // 2.1 samples close to existing affordances (:187-236)
      const size_t idx = uniform_index(m);
      double x[3];
      for (int k = 0; k < 3; k++) x[k] = kept_[3 * idx + k] + distr(gen);
      if (sampling_method_ == 1) {  // MAX_OF_GAUSSIANS: rejection sampling (:213-234)
        auto dens = [&](size_t h) {
          double d2 = 0;
          for (int k = 0; k < 3; k++) d2 += (x[k] - kept_[3 * h + k]) * (x[k] - kept_[3 * h + k]);
          return term * std::exp((-1.0 / (2.0 * sigma)) * d2);
        };
        double maxp = 0;
        for (size_t h = 0; h < m; h++) maxp = std::max(maxp, dens(h));
        if (!(dens(idx) >= maxp)) continue;
      }
      for (int k = 0; k < 3; k++) samples[3 * (size_t)j + k] = x[k];
      j++;
    }
    int i = 0, guard = 0;
    while (i < num_rand_samples && guard++ < 1000000) {  // 2.2 uniform samples inside the workspace (:239-270)
      const int pi = init_indices.empty() ? (int)uniform_index(cloud.size()) : init_indices[uniform_index(init_indices.size())];
      const double sx = cloud.getPoints()[3 * (size_t)pi], sy = cloud.getPoints()[3 * (size_t)pi + 1], sz = cloud.getPoints()[3 * (size_t)pi + 2];
      if (sx >= workspace_[0] && sx <= workspace_[1] && sy >= workspace_[2] && sy <= workspace_[3] && sz >= workspace_[4] &&
          sz <= workspace_[5]) {
        samples[3 * (size_t)(num_gauss_samples + i)] = sx;
        samples[3 * (size_t)(num_gauss_samples + i) + 1] = sy;
        samples[3 * (size_t)(num_gauss_samples + i) + 2] = sz;
        i++;
      }
    }
    // 2.3 evaluate grasp hypotheses at <samples> (:129-144)
    cloud.setSamples(samples);
    evaluated_.insert(evaluated_.end(), samples.begin(), samples.end());
    std::vector<double> fresh = grasp_detector_->candidateSamplePositions(cloud);
    kept_.insert(kept_.end(), fresh.begin(), fresh.end());
    printf("Added %zu grasp candidates in round %d. Total: %zu.\n", fresh.size() / 3, it, kept_.size() / 3);
  }
  cloud.setSamples({});
  // 3. Classify the grasps (:168-170), 4. cluster them (:177-179)
  std::vector<std::unique_ptr<candidate::Hand>> valid = grasp_detector_->classifyAtPositions(cloud, kept_, min_score_);
  printf("Valid grasps: %zu\n", valid.size());
  if (clustering_->getMinInliers() > 0) valid = grasp_detector_->findClustersOnDevice(valid, clustering_->getMinInliers());
  printf("Final result: found %zu grasps.\n", valid.size());
  return valid;
}

}  // namespace gpd

// ------------------------------------------------------------------------------------------------
// The reference's C interface for Python callers (src/detect_grasps_python.cpp)
// ------------------------------------------------------------------------------------------------
namespace {
std::vector<Grasp *> g_grasp_arrays;  // arrays handed out, with their lengths, so that freeMemoryGrasps can free members
std::vector<int> g_grasp_counts;

gpd::util::Cloud make_cloud(float *points, float *normals, int *camera_index, float *view_points, int size, int nv) {
  std::vector<float> xyz(points, points + 3 * (size_t)size);
  std::vector<double> nrm;
  if (normals) nrm.assign(normals, normals + 3 * (size_t)size);  // viewPointsToMatrix(normals, size): 3 x N
  std::vector<int> cam(camera_index, camera_index + (size_t)nv * size);
  std::vector<double> vp(view_points, view_points + 3 * (size_t)nv);
  return gpd::util::Cloud(xyz, nrm, cam, vp);
}

// handsToGraspsStruct (detect_grasps_python.cpp:251-295); images (optional) -> Grasp.image as ints, else {-1}
int hands_to_structs(const std::vector<std::unique_ptr<gpd::candidate::Hand>> &hands, const std::vector<std::vector<uint8_t>> *images,
                     int, Grasp **grasps_out) {
  const int n = (int)hands.size();
  Grasp *g = new Grasp[n > 0 ? n : 1];
  for (int i = 0; i < n; i++) {
    const gpdb_pose &p = hands[i]->raw();
    g[i].pos = new double[3]{p.position[0], p.position[1], p.position[2]};
    g[i].orient = new double[4];
    gpdQuaternionFromMatrix(p.frame, g[i].orient);
    g[i].sample = new double[3]{p.sample[0], p.sample[1], p.sample[2]};
    g[i].score = hands[i]->getScore();
    g[i].label = hands[i]->isFullAntipodal();
    if (images && (size_t)i < images->size()) {
      const std::vector<uint8_t> &im = (*images)[i];
      g[i].image = new int[im.size() > 0 ? im.size() : 1];
      for (size_t k = 0; k < im.size(); k++) g[i].image[k] = (int)im[k];
    } else {
      g[i].image = new int[1]{-1};
    }
  }
  g_grasp_arrays.push_back(g);
  g_grasp_counts.push_back(n);
  *grasps_out = g;
  return n;
}

int detect_to_structs(char *config_filename, gpd::util::Cloud &cloud, Grasp **grasps_out) {
  if (!config_filename || !grasps_out) return -1;
  *grasps_out = nullptr;
  gpd::GraspDetector detector(config_filename);  // detect_grasps_python.cpp:298-308
  detector.preprocessPointCloud(cloud);
  std::vector<std::unique_ptr<gpd::candidate::Hand>> hands = detector.detectGrasps(cloud);
  return hands_to_structs(hands, nullptr, 0, grasps_out);
}

// initCloud (detect_grasps_python.cpp:212-237)
gpd::util::Cloud init_cloud(char *pcd_filename, char *normals_filename, float *view_points, int num_view_points) {
  std::vector<double> vp(view_points, view_points + 3 * (size_t)num_view_points);
  gpd::util::Cloud cloud(std::string(pcd_filename), vp);
  if (cloud.size() == 0) {
    printf("Error: Input point cloud is empty or does not exist!\n");
    return cloud;
  }
  if (normals_filename && std::string(normals_filename).size() > 0) {
    cloud.setNormalsFromFile(normals_filename);
    printf("Loaded surface normals from file: %s\n", normals_filename);
  }
  return cloud;
}
}  // namespace

extern "C" {

void gpdQuaternionFromMatrix(const double *m, double *q) {
  auto M = [&](int r, int c) { return m[c * 3 + r]; };
  double t = M(0, 0) + M(1, 1) + M(2, 2);
  if (t > 0.0) {
    t = std::sqrt(t + 1.0);
    q[3] = 0.5 * t;
    t = 0.5 / t;
    q[0] = (M(2, 1) - M(1, 2)) * t;
    q[1] = (M(0, 2) - M(2, 0)) * t;
    q[2] = (M(1, 0) - M(0, 1)) * t;
  } else {
    int i = 0;
    if (M(1, 1) > M(0, 0)) i = 1;
    if (M(2, 2) > M(i, i)) i = 2;
    const int j = (i + 1) % 3, k = (j + 1) % 3;
    t = std::sqrt(M(i, i) - M(j, j) - M(k, k) + 1.0);
    q[i] = 0.5 * t;
    t = 0.5 / t;
    q[3] = (M(k, j) - M(j, k)) * t;
    q[j] = (M(j, i) + M(i, j)) * t;
    q[k] = (M(k, i) + M(i, k)) * t;
  }
}

int gpdSubsample(int n_points, const int *plane_idx, int n_plane, int num_samples, int *out) {
  gpd::util::Cloud cloud(std::vector<float>(3 * (size_t)std::max(n_points, 0), 0.0f), {}, {}, {0.0, 0.0, 0.0});
  if (n_plane > 0) cloud.setPlaneIndices(std::vector<int>(plane_idx, plane_idx + n_plane));
  cloud.subsample(num_samples);
  const std::vector<int> &s = cloud.getSampleIndices();
  std::copy(s.begin(), s.end(), out);
  return (int)s.size();
}

int gpdConfigGet(const char *file, const char *key, const char *def, char *out, int out_len) {
  gpd::util::ConfigFile cfg(file);
  const bool ok = cfg.ExtractKeys();
  std::snprintf(out, (size_t)out_len, "%s", cfg.getValueOfKeyAsString(key, def).c_str());
  return ok ? 1 : 0;
}
double gpdConfigGetDouble(const char *file, const char *key, double def) {
  gpd::util::ConfigFile cfg(file);
  cfg.ExtractKeys();
  return cfg.getValueOfKey<double>(key, def);
}
int gpdConfigGetInt(const char *file, const char *key, int def) {
  gpd::util::ConfigFile cfg(file);
  cfg.ExtractKeys();
  return cfg.getValueOfKey<int>(key, def);
}
int gpdConfigGetBool(const char *file, const char *key, int def) {
  gpd::util::ConfigFile cfg(file);
  cfg.ExtractKeys();
  return cfg.getValueOfKey<bool>(key, def != 0) ? 1 : 0;
}
int gpdConfigGetDoubles(const char *file, const char *key, const char *def, double *out, int cap) {
  gpd::util::ConfigFile cfg(file);
  cfg.ExtractKeys();
  std::vector<double> v = cfg.getValueOfKeyAsStdVectorDouble(key, def);
  for (size_t i = 0; i < v.size() && (int)i < cap; i++) out[i] = v[i];
  return (int)v.size();
}

void gpdHandGeometry(const char *file, double out[5]) {
  gpd::candidate::HandGeometry g{std::string(file)};
  out[0] = g.finger_width_; out[1] = g.outer_diameter_; out[2] = g.depth_; out[3] = g.height_; out[4] = g.init_bite_;
}
void gpdImageGeometry(const char *file, double out[3], int out2[2]) {
  gpd::descriptor::ImageGeometry g{std::string(file)};
  out[0] = g.outer_diameter_; out[1] = g.depth_; out[2] = g.height_; out2[0] = g.size_; out2[1] = g.num_channels_;
}

int gpdFindClusters(const gpdb_pose *hands, int n, int min_inliers, int remove_inliers, gpdb_pose *out) {
  std::vector<std::unique_ptr<gpd::candidate::Hand>> list;
  for (int i = 0; i < n; i++) list.push_back(std::make_unique<gpd::candidate::Hand>(hands[i]));
  auto clusters = gpd::Clustering(min_inliers).findClusters(list, remove_inliers != 0);
  for (size_t i = 0; i < clusters.size(); i++) out[i] = clusters[i]->raw();
  return (int)clusters.size();
}

int detectGraspsInCloud(char *config_filename, float *points, int *camera_index, float *view_points, int size,
                        int num_view_points, struct Grasp **grasps_out) {
  if (!points || !camera_index || !view_points || size <= 0 || num_view_points <= 0) return -1;
  gpd::util::Cloud cloud = make_cloud(points, nullptr, camera_index, view_points, size, num_view_points);
  return detect_to_structs(config_filename, cloud, grasps_out);
}

int detectGraspsInCloudNormals(char *config_filename, float *points, float *normals, int *camera_index,
                               float *view_points, int size, int num_view_points, struct Grasp **grasps_out) {
  if (!points || !normals || !camera_index || !view_points || size <= 0 || num_view_points <= 0) return -1;
  gpd::util::Cloud cloud = make_cloud(points, normals, camera_index, view_points, size, num_view_points);
  return detect_to_structs(config_filename, cloud, grasps_out);
}

// detectGraspsInFile (detect_grasps_python.cpp:468-488): cloud from a .pcd / .ply file, optional normals file ("" = none)
int detectGraspsInFile(char *config_filename, char *pcd_filename, char *normals_filename, float *view_points, int num_view_points,
                       struct Grasp **grasps_out) {
  if (!config_filename || !pcd_filename || !view_points || num_view_points <= 0 || !grasps_out) return 0;
  *grasps_out = nullptr;
  gpd::util::Cloud cloud = init_cloud(pcd_filename, normals_filename, view_points, num_view_points);
  if (cloud.size() == 0) return 0;
  return detect_to_structs(config_filename, cloud, grasps_out);
}

// generateGraspCandidatesInFile (detect_grasps_python.cpp:530-549): preprocessing + hand search, no classification
int generateGraspCandidatesInFile(char *config_filename, char *pcd_filename, char *normals_filename, float *view_points,
                                  int num_view_points, struct Grasp **grasps_out) {
  if (!config_filename || !pcd_filename || !view_points || num_view_points <= 0 || !grasps_out) return 0;
  *grasps_out = nullptr;
  gpd::util::Cloud cloud = init_cloud(pcd_filename, normals_filename, view_points, num_view_points);
  if (cloud.size() == 0) return 0;
  gpd::GraspDetector detector(config_filename);
  detector.preprocessPointCloud(cloud);
  std::vector<std::unique_ptr<gpd::candidate::Hand>> hands = detector.generateGraspCandidates(cloud);
  return hands_to_structs(hands, nullptr, 0, grasps_out);
}

// detectAndEvalGrasps (detect_grasps_python.cpp:490-528): candidates + images in the camera cloud, labels against the
// ground-truth mesh cloud (points_gt / normals_gt, 3 x size_gt). Grasp.image = the hand's own image as ints (HWC); the
// reference's cvMatToArray never fills its array and passes images[0] for every hand.
int detectAndEvalGrasps(char *config_filename, float *points, int *camera_index, float *view_points, int size, int num_view_points,
                        float *points_gt, float *normals_gt, int size_gt, struct Grasp **grasps_out) {
  if (!config_filename || !points || !camera_index || !view_points || size <= 0 || num_view_points <= 0 || !points_gt ||
      !normals_gt || size_gt <= 0 || !grasps_out)
    return 0;
  *grasps_out = nullptr;
  gpd::util::Cloud cloud = make_cloud(points, nullptr, camera_index, view_points, size, num_view_points);
  std::vector<int> ones((size_t)size_gt, 1);  // createGroundTruthCloud (:178-190): one camera at the origin seeing everything
  float origin[3] = {0.f, 0.f, 0.f};
  gpd::util::Cloud mesh_cloud = make_cloud(points_gt, normals_gt, ones.data(), origin, size_gt, 1);
  gpd::GraspDetector detector(config_filename);
  detector.preprocessPointCloud(cloud);
  std::vector<std::unique_ptr<gpd::candidate::Hand>> hands;
  std::vector<std::vector<uint8_t>> images;
  if (!detector.createGraspImages(cloud, hands, images)) {
    printf("No grasps found!\n");
    return 0;
  }
  printf("Created %d grasps and %d images.\n", (int)hands.size(), (int)images.size());
  detector.evalGroundTruth(mesh_cloud, hands);
  return hands_to_structs(hands, &images, 0, grasps_out);
}

int CopyAndFree(float *in, float *out, int n) {  // detect_grasps_python.cpp:603-607
  if (!in || !out || n < 0) return -1;
  memcpy(out, in, sizeof(float) * (size_t)n);
  delete[] in;
  return 0;
}

int freeMemoryGrasps(struct Grasp *in) {
  if (!in) return 0;
  for (size_t a = 0; a < g_grasp_arrays.size(); a++)
    if (g_grasp_arrays[a] == in) {
      for (int i = 0; i < g_grasp_counts[a]; i++) {
        delete[] in[i].pos;
        delete[] in[i].orient;
        delete[] in[i].sample;
        delete[] in[i].image;
      }
      g_grasp_arrays.erase(g_grasp_arrays.begin() + a);
      g_grasp_counts.erase(g_grasp_counts.begin() + a);
      break;
    }
  delete[] in;
  return 0;
}

}  // extern "C"
