// C++ host layer over the C ABI (include/ftkb200.h): the operator surface of
//   ftk::critical_point_tracker_2d_regular   ref: include/ftk/filters/critical_point_tracker_2d_regular.hh:51-140
//   ftk::critical_point_tracker_3d_regular   ref: include/ftk/filters/critical_point_tracker_3d_regular.hh:58-90
// with the same method names, argument meaning and call order (set_domain / set_array_domain /
// set_*_field_source / initialize / push_*_snapshot / advance_timestep / update_timestep / finalize /
// get_traced_critical_points / get_critical_points), so that the reference's front ends
// (json_interface.hh:606-725, python/pyftk.cpp:93-142) compile against these classes after a
// namespace change.  Everything numerical happens behind ftkb_* in libftkb200.so on the GPU;
// this header only marshals arguments and turns the C ABI's flat results into the reference's
// result containers.  Errors of the C ABI become std::runtime_error (the reference calls exit()).
//
// Header-only, C++17, no dependency besides ftkb200.h.  Not a copy of the reference's headers:
// the containers below carry only what the tracking path produces.
#ifndef FTK_B200_CRITICAL_POINT_TRACKER_REGULAR_HH
#define FTK_B200_CRITICAL_POINT_TRACKER_REGULAR_HH

#include <algorithm>
#include <array>
#include <cstdint>
#include <cstring>
#include <fstream>
#include <iomanip>
#include <limits>
#include <map>
#include <ostream>
#include <sstream>
#include <stdexcept>
#include <string>
#include <vector>

#include "../ftkb200.h"

namespace ftk_b200 {

// field sources (ref: include/ftk/filters/critical_point_tracker.hh:21-25)
enum { SOURCE_NONE = FTKB_SOURCE_NONE, SOURCE_GIVEN = FTKB_SOURCE_GIVEN, SOURCE_DERIVED = FTKB_SOURCE_DERIVED };

// critical point types (ref: include/ftk/numeric/critical_point_type.hh:10-36)
enum : unsigned {
  CRITICAL_POINT_2D_UNKNOWN = 0, CRITICAL_POINT_2D_DEGENERATE = 1, CRITICAL_POINT_2D_MINIMUM = 2, CRITICAL_POINT_2D_REPELLING = 2,
  CRITICAL_POINT_2D_SADDLE = 4, CRITICAL_POINT_2D_MAXIMUM = 8, CRITICAL_POINT_2D_ATTRACTING = 8,
  CRITICAL_POINT_2D_ATTRACTING_FOCUS = 16, CRITICAL_POINT_2D_REPELLING_FOCUS = 32, CRITICAL_POINT_2D_CENTER = 64,
  CRITICAL_POINT_3D_UNKNOWN = 0, CRITICAL_POINT_3D_DEGENERATE = 1, CRITICAL_POINT_3D_MINIMUM = 2, CRITICAL_POINT_3D_SADDLE = 4,
  CRITICAL_POINT_3D_MAXIMUM = 8
};

// ref: critical_point_type.hh:95-118
inline std::string critical_point_type_to_string(int cpdims, unsigned type, bool scalar) {
  if (cpdims == 2 || (cpdims == 3 && scalar)) {
    switch (type) {
      case 1: return "degenerate";
      case 2: return scalar ? "min" : "repelling";
      case 4: return "saddle";
      case 8: return scalar ? "max" : "attracting";
      case 16: return (!scalar && cpdims == 2) ? "attracting_focus" : "unknown";
      case 32: return (!scalar && cpdims == 2) ? "repelling_focus" : "unknown";
      case 64: return (!scalar && cpdims == 2) ? "center" : "unknown";
      default: return "unknown";
    }
  }
  return "unknown";
}

// ftk::lattice(starts, sizes) (ref: include/ftk/mesh/lattice.hh:16-69)
class lattice {
 public:
  lattice() {}
  lattice(const std::vector<int> &starts, const std::vector<int> &sizes) : starts_(starts), sizes_(sizes) {
    if (starts.size() != sizes.size()) throw std::invalid_argument("lattice: starts and sizes differ in length");
  }
  size_t nd() const { return sizes_.size(); }
  int start(size_t i) const { return starts_[i]; }
  int size(size_t i) const { return sizes_[i]; }
  int lower_bound(size_t i) const { return starts_[i]; }
  int upper_bound(size_t i) const { return starts_[i] + sizes_[i] - 1; }
  const std::vector<int> &starts() const { return starts_; }
  const std::vector<int> &sizes() const { return sizes_; }
  size_t n() const { size_t p = 1; for (int s : sizes_) p *= (size_t)s; return p; }

 private:
  std::vector<int> starts_, sizes_;
};

// dense array, dimension 0 fastest (ref: include/ftk/ndarray.hh:129-135,724-737); only what the
// tracker's inputs need.  A view over memory the caller owns (host, or device with on_device()).
template <typename T>
class ndarray {
 public:
  ndarray() {}
  explicit ndarray(const std::vector<size_t> &shape) { reshape(shape); }
  void reshape(const std::vector<size_t> &shape) {
    dims_ = shape;
    if (!borrowed_) own_.assign(nelem(), T());
  }
  // borrow caller memory (no copy); device = the pointer is CUDA device memory: on the tracker's device for one device, on any
  // visible device for a tracker on several devices (set_device_ids), whose devices copy it from there
  static ndarray wrap(const T *p, const std::vector<size_t> &shape, bool device = false) {
    ndarray a;
    a.dims_ = shape; a.ext_ = p; a.borrowed_ = true; a.device_ = device;
    return a;
  }
  size_t nd() const { return dims_.size(); }
  size_t dim(size_t i) const { return dims_[i]; }
  const std::vector<size_t> &shape() const { return dims_; }
  size_t nelem() const { size_t p = dims_.empty() ? 0 : 1; for (size_t d : dims_) p *= d; return p; }
  bool empty() const { return nelem() == 0; }
  bool on_device() const { return device_; }
  const T *data() const { return borrowed_ ? ext_ : own_.data(); }
  T *data() { if (borrowed_) throw std::logic_error("ndarray: borrowed arrays are read-only"); return own_.data(); }
  T &operator[](size_t i) { return data()[i]; }
  const T &operator[](size_t i) const { return data()[i]; }
  T &operator()(size_t i0, size_t i1) { return data()[i0 + dims_[0] * i1]; }
  T &operator()(size_t i0, size_t i1, size_t i2) { return data()[i0 + dims_[0] * (i1 + dims_[1] * i2)]; }
  T &operator()(size_t i0, size_t i1, size_t i2, size_t i3) { return data()[i0 + dims_[0] * (i1 + dims_[1] * (i2 + dims_[2] * i3))]; }

 private:
  std::vector<size_t> dims_;
  std::vector<T> own_;
  const T *ext_ = nullptr;
  bool borrowed_ = false, device_ = false;
};

// one critical point (ref: include/ftk/features/feature_point.hh:15-120)
struct feature_point_t {
  std::array<double, 3> x{{0, 0, 0}};
  double t = 0.0;
  int timestep = 0;
  std::array<double, 3> scalar{{0, 0, 0}};
  std::array<double, 3> v{{0, 0, 0}};
  unsigned int type = 0;
  bool ordinal = false;
  unsigned long long tag = 0;   // 64-bit element id (the reference's int tag overflows on large grids, SURVEY.md A8)
  unsigned long long id = 0;    // trajectory id
  // our additions: the discrete element the point lives on
  std::array<int, 4> corner{{0, 0, 0, 0}};
  int simplex_type = 0;

  // same text as feature_point_t::print (feature_point.hh:82-100)
  std::ostream &print(std::ostream &os, const std::vector<std::string> &scalar_components) const {
    os << "x=(" << x[0] << ", " << x[1] << ", " << x[2] << "), ";
    os << "t=" << t << ", ";
    for (size_t k = 0; k < scalar_components.size(); k++) os << scalar_components[k] << "=" << scalar[k] << ", ";
    os << "v=(" << v[0] << ", " << v[1] << ", " << v[2] << "), ";
    os << "type=" << type << ", timestep=" << timestep << ", ordinal=" << ordinal << ", tag=" << tag << ", id=" << id;
    return os;
  }
};

// ---- binary archives: the byte layout of the reference's DIY serialization (little endian, no padding) ----------
// feature_point.hh:160-188: x[3] t timestep(int) scalar[FTK_CP_MAX_NUM_VARS = 3] v[3] type(unsigned) ordinal(bool) tag id = 105 bytes
namespace bin {
template <typename T> inline void put(std::ostream &os, const T &v) { os.write(reinterpret_cast<const char *>(&v), sizeof(T)); }
template <typename T> inline bool get(std::istream &is, T &v) { is.read(reinterpret_cast<char *>(&v), sizeof(T)); return (bool)is; }
inline void put_point(std::ostream &os, const feature_point_t &p) {
  for (double v : p.x) put(os, v);
  put(os, p.t); put(os, (int)p.timestep);
  for (double v : p.scalar) put(os, v);
  for (double v : p.v) put(os, v);
  put(os, (unsigned int)p.type); put(os, (unsigned char)(p.ordinal ? 1 : 0)); put(os, (unsigned long long)p.tag); put(os, (unsigned long long)p.id);
}
inline bool get_point(std::istream &is, feature_point_t &p) {
  unsigned char o = 0;
  for (double &v : p.x) get(is, v);
  get(is, p.t); get(is, p.timestep);
  for (double &v : p.scalar) get(is, v);
  for (double &v : p.v) get(is, v);
  get(is, p.type); get(is, o); get(is, p.tag);
  p.ordinal = o != 0;
  return get(is, p.id);
}
}  // namespace bin

// one trajectory (ref: include/ftk/features/feature_curve.hh:8-54,145-184)
struct feature_curve_t : public std::vector<feature_point_t> {
  int id = 0;
  bool complete = false, loop = false;
  std::array<double, 3> max{{0, 0, 0}}, min{{0, 0, 0}}, persistence{{0, 0, 0}};
  std::array<double, 3> bbmin{{0, 0, 0}}, bbmax{{0, 0, 0}};
  double tmin = 0, tmax = 0;
  unsigned int consistent_type = 0;

  void relabel(int i) { id = i; for (auto &p : *this) p.id = (unsigned long long)i; }

  void update_statistics() {
    if (empty()) return;
    const double lo = std::numeric_limits<double>::lowest(), hi = std::numeric_limits<double>::max();
    max.fill(lo); min.fill(hi); bbmax.fill(lo); bbmin.fill(hi);
    tmax = lo; tmin = hi;
    for (const auto &p : *this) {
      for (int k = 0; k < 3; k++) {
        max[k] = std::max(max[k], p.scalar[k]); min[k] = std::min(min[k], p.scalar[k]);
        bbmax[k] = std::max(bbmax[k], p.x[k]); bbmin[k] = std::min(bbmin[k], p.x[k]);
      }
      tmax = std::max(tmax, p.t); tmin = std::min(tmin, p.t);
    }
    for (int k = 0; k < 3; k++) persistence[k] = max[k] - min[k];
    consistent_type = front().type;
    for (const auto &p : *this)
      if (p.type != consistent_type) { consistent_type = 0; break; }
  }

  // ref: feature_curve.hh discard_interval_points (critical_point_tracker_2d_regular.hh:219-222)
  void discard_interval_points() {
    erase(std::remove_if(begin(), end(), [](const feature_point_t &p) { return !p.ordinal; }), end());
  }
};

// the tracker's result (ref: include/ftk/features/feature_curve_set.hh: a multimap id -> curve)
struct feature_curve_set_t : public std::multimap<int, feature_curve_t> {
  int add(const feature_curve_t &c) {
    const int id = empty() ? 0 : (rbegin()->first + 1);
    auto it = insert(std::make_pair(id, c));
    it->second.relabel(id);
    return id;
  }

  // same layout as feature_curve_set_t::write_text (feature_curve_set.hh:180-229), including its
  // "bbmin=(a, b, c, " quirk (the closing parenthesis is never written there)
  void write_text(std::ostream &os, const std::vector<std::string> &scalar_components) const {
    os << "#trajectories=" << size() << std::endl;
    for (const auto &kv : *this) {
      const auto &c = kv.second;
      os << "--trajectory " << kv.first << ", ";
      const size_t ns = scalar_components.size();
      if (ns > 0) {
        const char *names[3] = {"min=(", "max=(", "persistence=("};
        const std::array<double, 3> *vals[3] = {&c.min, &c.max, &c.persistence};
        for (int q = 0; q < 3; q++) {
          os << names[q];
          for (size_t k = 0; k < ns; k++) os << (*vals[q])[k] << (k + 1 < ns ? ", " : "), ");
        }
      }
      os << "bbmin=(";
      for (int k = 0; k < 3; k++) os << c.bbmin[k] << ", ";
      os << "bbmax=(";
      for (int k = 0; k < 3; k++) os << c.bbmax[k] << ", ";
      os << "tmin=" << c.tmin << ", tmax=" << c.tmax << ", ";
      os << "consistent_type=" << c.consistent_type << ", ";
      os << "loop=" << c.loop << std::endl;
      for (const auto &p : c) { os << "---"; p.print(os, scalar_components) << std::endl; }
    }
  }

  // the reference's binary archive: diy::save(bb, feature_curve_set_t) (feature_curve_set.hh:92-100) = count, then per curve
  // its id and diy::Serialization<feature_curve_t>::save (feature_curve.hh:472-487): complete, max, min, persistence, bbmin, bbmax,
  // tmin, tmax, consistent_type, size, points.  (The loop flag is not part of the reference's archive.)
  void write_binary(std::ostream &os) const {
    bin::put(os, (unsigned long long)size());
    for (const auto &kv : *this) {
      const auto &c = kv.second;
      bin::put(os, (int)kv.first);
      bin::put(os, (unsigned char)(c.complete ? 1 : 0));
      for (const auto *a : {&c.max, &c.min, &c.persistence, &c.bbmin, &c.bbmax})
        for (double v : *a) bin::put(os, v);
      bin::put(os, c.tmin); bin::put(os, c.tmax); bin::put(os, (unsigned int)c.consistent_type);
      bin::put(os, (unsigned long long)c.size());
      for (const auto &p : c) bin::put_point(os, p);
    }
  }
  bool read_binary(std::istream &is) {     // diy::load: every curve is relabelled with its id and inserted
    unsigned long long n = 0;
    if (!bin::get(is, n)) return false;
    for (unsigned long long i = 0; i < n; i++) {
      int id = 0;
      unsigned char complete = 0;
      feature_curve_t c;
      bin::get(is, id); bin::get(is, complete);
      c.complete = complete != 0;
      for (auto *a : {&c.max, &c.min, &c.persistence, &c.bbmin, &c.bbmax})
        for (double &v : *a) bin::get(is, v);
      bin::get(is, c.tmin); bin::get(is, c.tmax); bin::get(is, c.consistent_type);
      unsigned long long np = 0;
      if (!bin::get(is, np)) return false;
      c.resize(np);
      for (auto &p : c)
        if (!bin::get_point(is, p)) return false;
      c.relabel(id);
      insert(std::make_pair(id, c));
    }
    return true;
  }

  // keys of the reference's JSON archive (feature_curve_set.hh:79-89, feature_curve.hh:437-451, feature_point.hh:129-145)
  void write_json(std::ostream &os) const {
    os << std::setprecision(17) << "{\"trajs\":[";
    bool first = true;
    for (const auto &kv : *this) {
      const auto &c = kv.second;
      os << (first ? "" : ",") << "{\"id\":" << c.id;
      auto arr = [&](const char *k, const std::array<double, 3> &a) { os << ",\"" << k << "\":[" << num(a[0]) << "," << num(a[1]) << "," << num(a[2]) << "]"; };
      arr("max", c.max); arr("min", c.min); arr("persistence", c.persistence); arr("bbmin", c.bbmin); arr("bbmax", c.bbmax);
      os << ",\"tmin\":" << num(c.tmin) << ",\"tmax\":" << num(c.tmax) << ",\"consistent_type\":" << c.consistent_type << ",\"traj\":[";
      for (size_t i = 0; i < c.size(); i++) { os << (i ? "," : ""); point_json(os, c[i]); }
      os << "]}";
      first = false;
    }
    os << "]}" << std::endl;
  }

  static std::string num(double v) {
    if (v != v || v - v != 0.0) return "null";   // JSON has no NaN / Inf (nlohmann writes null as well)
    std::ostringstream s;
    s << std::setprecision(17) << v;
    return s.str();
  }
  static void point_json(std::ostream &os, const feature_point_t &p) {
    os << "{\"x\":[" << num(p.x[0]) << "," << num(p.x[1]) << "," << num(p.x[2]) << "],\"t\":" << num(p.t) << ",\"timestep\":" << p.timestep
       << ",\"scalar\":[" << num(p.scalar[0]) << "," << num(p.scalar[1]) << "," << num(p.scalar[2]) << "],\"v\":[" << num(p.v[0]) << "," << num(p.v[1]) << ","
       << num(p.v[2]) << "],\"type\":" << p.type << ",\"ordinal\":" << (p.ordinal ? "true" : "false") << ",\"tag\":" << p.tag << ",\"id\":" << p.id << "}";
  }
};

// ------------------------------------------------------------------------------------------------
// the tracker classes
// ------------------------------------------------------------------------------------------------
class critical_point_tracker_regular {
 public:
  explicit critical_point_tracker_regular(int nd) : nd_(nd) {}
  virtual ~critical_point_tracker_regular() { reset(); }
  critical_point_tracker_regular(const critical_point_tracker_regular &) = delete;
  critical_point_tracker_regular &operator=(const critical_point_tracker_regular &) = delete;

  // ---- configuration: regular_tracker.hh:24-27, critical_point_tracker.hh:26-52, filter.hh:25-51, tracker.hh:49-76
  void set_domain(const lattice &l) { domain_ = l; }
  void set_array_domain(const lattice &l) { array_domain_ = l; }
  void set_scalar_field_source(int s) { scalar_source_ = s; }
  void set_vector_field_source(int s) { vector_source_ = s; }
  void set_jacobian_field_source(int s) { jacobian_source_ = s; }
  void set_jacobian_symmetric(bool b) { symmetric_ = b; }
  void set_type_filter(unsigned int f) { use_type_filter_ = true; type_filter_ = f; }
  void set_enable_robust_detection(bool b) { robust_ = b; }
  void set_enable_computing_degrees(bool b) { degrees_ = b; }
  // critical_point_tracker.hh:38; trajectories then grow after every interval sweep (trace_critical_points_online, hh:522-641)
  void set_enable_streaming_trajectories(bool b) { streaming_ = b; }
  // physical coordinates: regular_tracker.hh:38-40 (applied at initialize())
  void set_coords_bounds(const std::vector<double> &bounds) { coords_mode_ = FTKB_COORDS_BOUNDS; coords_ = bounds; }
  void set_coords_rectilinear(const std::vector<ndarray<double>> &rc) {
    coords_mode_ = FTKB_COORDS_RECTILINEAR;
    coords_.clear();
    for (const auto &a : rc) coords_.insert(coords_.end(), a.data(), a.data() + a.nelem());
  }
  void set_coords_explicit(const ndarray<double> &e) { coords_mode_ = FTKB_COORDS_EXPLICIT; coords_.assign(e.data(), e.data() + e.nelem()); }
  void set_enable_discarding_interval_points(bool b) { discard_interval_ = b; }
  void set_enable_discarding_degenerate_points(bool b) { discard_degenerate_ = b; }
  void set_scalar_components(const std::vector<std::string> &c) { scalar_components_ = c; }
  const std::vector<std::string> &get_scalar_components() const { return scalar_components_; }
  void set_number_of_threads(int) {}                 // the sweep runs on the GPU
  void use_accelerator(const std::string &name) {
    if (name != "cuda" && name != "b200" && name != "ftkb200")
      throw std::runtime_error("ftk_b200 runs on CUDA sm_100a only; there is no CPU or other back end");
  }
  void use_accelerator(int) {}
  // filter.hh:47-51: one id = that device; several = the tracker is served by all of them (ftkb_group: time chunks of
  // set_time_chunk() timesteps go round the devices; results equal the one-device run)
  void set_device_ids(const std::vector<int> &ids) { device_ids_ = ids; if (!ids.empty()) device_ = ids[0]; }
  void set_time_chunk(int timesteps) { time_chunk_ = timesteps >= 0 ? timesteps : 8; }     // 0: z-slabs (3D) instead of time chunks
  void set_start_timestep(int t) { start_timestep_ = t; }
  void set_current_timestep(int t) { start_timestep_ = t; }
  // time-slab sharding: running min non-zero |v| inherited from the slabs before this one
  void set_initial_resolution(double r) { resolution_init_ = r; }

  void initialize() {
    if ((int)array_domain_.nd() != nd_) throw std::runtime_error("ftk_b200: set_array_domain() must be called with an nd-dimensional lattice before initialize()");
    if (domain_.nd() == 0) domain_ = array_domain_;
    if ((int)domain_.nd() != nd_) throw std::runtime_error("ftk_b200: domain dimensionality mismatch");
    reset();
    ftkb_config cfg;
    std::memset(&cfg, 0, sizeof(cfg));
    cfg.abi_version = FTKB_ABI_VERSION;
    cfg.nd = nd_;
    for (int i = 0; i < 3; i++) {
      const bool used = i < nd_;
      cfg.dims[i] = used ? array_domain_.size(i) : 1;
      cfg.lb[i] = used ? domain_.lower_bound(i) - array_domain_.start(i) : 0;
      cfg.ub[i] = used ? domain_.upper_bound(i) - array_domain_.start(i) : 0;
    }
    cfg.scalar_source = scalar_source_; cfg.vector_source = vector_source_; cfg.jacobian_source = jacobian_source_;
    cfg.jacobian_symmetric = symmetric_; cfg.robust_detection = robust_; cfg.compute_degrees = degrees_;
    cfg.use_type_filter = use_type_filter_; cfg.type_filter = type_filter_;
    cfg.start_timestep = start_timestep_; cfg.device = device_; cfg.resolution_init = resolution_init_;
    if (device_ids_.size() > 1) {
      std::vector<int32_t> ids(device_ids_.begin(), device_ids_.end());
      const int rcg = ftkb_group_create(&cfg, ids.data(), (int32_t)ids.size(), time_chunk_, &group_);
      if (rcg != FTKB_OK) throw std::runtime_error("ftkb_group_create failed (device ids?)");
      if (streaming_) gcheck(ftkb_group_set_streaming_trajectories(group_, 1));
      if (coords_mode_ != FTKB_COORDS_SIMPLE) gcheck(ftkb_group_set_coords(group_, coords_mode_, coords_.data(), coords_.size()));
      return;
    }
    const int rc = ftkb_create(&cfg, &ctx_);
    if (rc != FTKB_OK) throw std::runtime_error(std::string("ftkb_create: ") + ftkb_last_error(nullptr));
    if (streaming_) check(ftkb_set_streaming_trajectories(ctx_, 1));
    if (coords_mode_ != FTKB_COORDS_SIMPLE) check(ftkb_set_coords(ctx_, coords_mode_, coords_.data(), coords_.size()));
  }

  void reset() {
    if (group_) { ftkb_group_destroy(group_); group_ = nullptr; ctx_ = nullptr; }       // (the group owns its root context)
    if (ctx_) { ftkb_destroy(ctx_); ctx_ = nullptr; }
    traced_.clear();
    points_valid_ = false;
    finalized_ = false;
    sweeps_ = refreshed_sweeps_ = 0;
  }

  // ---- inputs: critical_point_tracker.hh:202-229 ------------------------------------------------
  void push_field_data_snapshot(const ndarray<double> &scalar, const ndarray<double> &vector, const ndarray<double> &jacobian) {
    need();
    size_t nvert = 1;
    for (int i = 0; i < nd_; i++) nvert *= (size_t)array_domain_.size(i);
    auto ptr = [&](const ndarray<double> &a, size_t count, const char *what) -> const double * {
      if (a.empty()) return nullptr;
      if (a.nelem() != count) throw std::runtime_error(std::string("ftk_b200: ") + what + " snapshot has the wrong number of elements");
      return a.data();
    };
    const double *s = ptr(scalar, nvert, "scalar"), *v = ptr(vector, nvert * nd_, "vector"), *j = ptr(jacobian, nvert * nd_ * nd_, "jacobian");
    const bool dev = scalar.on_device() || vector.on_device() || jacobian.on_device();
    if (group_)
      gcheck(dev ? ftkb_group_push_snapshot_device(group_, s, v, j) : ftkb_group_push_snapshot(group_, s, v, j));
    else
    check(ftkb_push_snapshot(ctx_, s, v, j, dev ? FTKB_MEM_DEVICE : FTKB_MEM_HOST));
    points_valid_ = false;
  }
  // A snapshot in pieces along the slowest axis (z in 3D, y in 2D), as a producer decomposed over several GPUs holds it: piece i
  // is a device ndarray view (ndarray::wrap(p, shape, true), on any visible device) of planes [first[i], first[i] + its last
  // dimension); an array not passed is an empty list.  Only on several devices (set_device_ids): every device copies the planes
  // it needs from the pieces that hold them (ftkb_group_push_pieces_device).  The caller synchronises its producer first.
  void push_field_data_snapshot_pieces(const std::vector<int> &first, const std::vector<ndarray<double>> &scalar,
                                       const std::vector<ndarray<double>> &vector = {}, const std::vector<ndarray<double>> &jacobian = {}) {
    need();
    if (!group_) throw std::runtime_error("ftk_b200: snapshot pieces need a tracker on several devices (set_device_ids)");
    std::vector<ftkb_piece> pieces(first.size(), ftkb_piece{});
    for (auto *a : {&scalar, &vector, &jacobian})
      if (!a->empty() && a->size() != first.size()) throw std::runtime_error("ftk_b200: pass one array per piece");
    for (size_t i = 0; i < first.size(); i++) {
      ftkb_piece &p = pieces[i];
      p.first = first[i];
      const ndarray<double> *arrays[3] = {scalar.empty() ? nullptr : &scalar[i], vector.empty() ? nullptr : &vector[i], jacobian.empty() ? nullptr : &jacobian[i]};
      const double **ptrs[3] = {&p.scalar, &p.vector, &p.jacobian};
      for (int k = 0; k < 3; k++) {
        const ndarray<double> *a = arrays[k];
        if (!a || a->empty()) continue;
        if (!a->on_device()) throw std::runtime_error("ftk_b200: snapshot pieces are device arrays");
        *ptrs[k] = a->data();
        p.count = (int32_t)a->dim(a->nd() - 1);
      }
    }
    gcheck(ftkb_group_push_pieces_device(group_, pieces.data(), (int32_t)pieces.size()));
    points_valid_ = false;
  }
  void push_scalar_field_snapshot(const ndarray<double> &scalar) { push_field_data_snapshot(scalar, ndarray<double>(), ndarray<double>()); }
  void push_vector_field_snapshot(const ndarray<double> &vector) { push_field_data_snapshot(ndarray<double>(), vector, ndarray<double>()); }
  // float32 host snapshots (raw float32 series; the reference's streams widen them on the host): they travel as float32 and are
  // widened on the device.  Several devices: widened here, then pushed like any host snapshot.
  void push_field_data_snapshot(const ndarray<float> &scalar, const ndarray<float> &vector) {
    need();
    size_t nvert = 1;
    for (int i = 0; i < nd_; i++) nvert *= (size_t)array_domain_.size(i);
    if (!scalar.empty() && scalar.nelem() != nvert) throw std::runtime_error("ftk_b200: scalar snapshot has the wrong number of elements");
    if (!vector.empty() && vector.nelem() != nvert * nd_) throw std::runtime_error("ftk_b200: vector snapshot has the wrong number of elements");
    if (scalar.on_device() || vector.on_device()) throw std::runtime_error("ftk_b200: float32 snapshots are host arrays");
    if (group_) {
      std::vector<double> s(scalar.data(), scalar.data() + scalar.nelem()), v(vector.data(), vector.data() + vector.nelem());
      gcheck(ftkb_group_push_snapshot(group_, s.empty() ? nullptr : s.data(), v.empty() ? nullptr : v.data(), nullptr));
    } else
    check(ftkb_push_snapshot_f32(ctx_, scalar.empty() ? nullptr : scalar.data(), vector.empty() ? nullptr : vector.data()));
    points_valid_ = false;
  }
  void push_scalar_field_snapshot(const ndarray<float> &scalar) { push_field_data_snapshot(scalar, ndarray<float>()); }
  void push_vector_field_snapshot(const ndarray<float> &vector) { push_field_data_snapshot(ndarray<float>(), vector); }
  // device-side generator (no host data): FTKB_SYN_* kinds of ftkb200.h
  void push_synthetic_snapshot(int kind, const std::vector<double> &params, double t) {
    need();
    if (group_) gcheck(ftkb_group_push_synthetic(group_, kind, params.data(), (int)params.size(), t));
    else
    check(ftkb_push_synthetic(ctx_, kind, params.data(), (int)params.size(), t));
    points_valid_ = false;
  }

  // ---- stepping: critical_point_tracker.hh:841-848, *_regular.hh update_timestep ------------------
  void update_timestep() { need(); if (group_) gcheck(ftkb_group_update_timestep(group_)); else check(ftkb_update_timestep(ctx_)); points_valid_ = false; sweeps_++; }
  bool advance_timestep() { need(); if (group_) gcheck(ftkb_group_advance_timestep(group_)); else check(ftkb_advance_timestep(ctx_)); points_valid_ = false; sweeps_++; return true; }
  int get_current_timestep() const { int32_t t = start_timestep_; if (ctx_) ftkb_current_timestep(ctx_, &t); return t; }

  // ---- finalize: critical_point_tracker_2d_regular.hh:143-225, critical_point_tracker.hh:668-817 --
  void finalize() {
    need();
    ensure_root();     // several devices: merged into one context on the first device, traced there
    check(ftkb_finalize(ctx_));
    finalized_ = true;
    fetch_points();
    uint64_t nt = 0;
    check(ftkb_num_trajectories(ctx_, &nt));
    std::vector<uint64_t> off(nt + 1), idx(points_.size() ? points_.size() : 1);
    std::vector<uint8_t> loop(nt ? nt : 1);
    check(ftkb_get_trajectories(ctx_, off.data(), idx.data(), loop.data()));
    std::vector<uint8_t> complete(nt ? nt : 1);
    check(ftkb_get_trajectory_complete(ctx_, complete.data()));
    traced_.clear();
    for (uint64_t i = 0; i < nt; i++) {
      feature_curve_t c;
      for (uint64_t k = off[i]; k < off[i + 1]; k++) c.push_back(points_[idx[k]]);
      c.loop = loop[i] != 0;
      c.complete = complete[i] != 0;  // only the online tracer sets it (critical_point_tracker.hh:603)
      if (discard_interval_) c.discard_interval_points();
      if (discard_degenerate_) c.erase(std::remove_if(c.begin(), c.end(), [](const feature_point_t &p) { return p.type == 1; }), c.end());
      c.update_statistics();
      traced_.add(c);
    }
  }

  // ---- trajectory post-processing: feature_curve_set_post_processor.hh:23-70 (op list), json_interface.hh:758-800
  // ("legacy[:duration_threshold[:discard_interval_points[:derive_velocities]]]").  The curve operations run in the
  // library (ftkb_curveset_*); the traced set is replaced by the processed curves, in the multimap's order.
  void post_process(const std::string &ops = "legacy") {
    need();
    ftkb_curveset *cs = nullptr;
    check(ftkb_get_curveset(ctx_, &cs));
    if (ftkb_curveset_post_process(cs, ops.c_str()) != FTKB_OK) {
      const std::string msg = ftkb_curveset_last_error(cs);
      ftkb_curveset_destroy(cs);
      throw std::runtime_error("ftk_b200: " + msg);
    }
    load_curveset(cs);
    ftkb_curveset_destroy(cs);
  }

  // ---- results: critical_point_tracker.hh:68-69,105, critical_point_tracker_regular.hh:24-38 ------
  const feature_curve_set_t &get_traced_critical_points() const { return traced_; }
  // With streaming trajectories the reference's traced set is live: trace_critical_points_online updates it after every interval
  // sweep.  So before finalize, after any sweep since the last call, this refreshes it from the trajectories grown so far (the
  // const overload returns it as last refreshed).
  feature_curve_set_t &get_traced_critical_points() {
    if (streaming_ && !finalized_ && (ctx_ || group_) && refreshed_sweeps_ != sweeps_) {
      ftkb_curveset *cs = nullptr;
      int32_t grown_through = 0;
      if (group_) gcheck(ftkb_group_get_live_curveset(group_, &grown_through, &cs));
      else check(ftkb_get_live_curveset(ctx_, &grown_through, &cs));
      load_curveset(cs);
      ftkb_curveset_destroy(cs);
      refreshed_sweeps_ = sweeps_;
    }
    return traced_;
  }
  std::vector<feature_point_t> get_critical_points() { need(); fetch_points(); return points_; }
  std::vector<feature_point_t> get_discrete_critical_points() { return get_critical_points(); }

  void write_traced_critical_points_text(std::ostream &os) const { traced_.write_text(os, scalar_components_); }
  void write_traced_critical_points_text(const std::string &f) const { std::ofstream o(f); write_traced_critical_points_text(o); }
  void write_traced_critical_points_json(const std::string &f) const { std::ofstream o(f); traced_.write_json(o); }
  // critical_point_tracker.hh:339-364: diy::serializeToFile(get_critical_points() / traced_critical_points, filename)
  void write_traced_critical_points_binary(const std::string &f) const { std::ofstream o(f, std::ios::binary); traced_.write_binary(o); }
  bool read_traced_critical_points_binary(const std::string &f) { std::ifstream i(f, std::ios::binary); traced_.clear(); return i && traced_.read_binary(i); }
  void write_critical_points_binary(const std::string &f) {
    const std::vector<feature_point_t> pts = ctx_ ? get_critical_points() : points_;
    std::ofstream o(f, std::ios::binary);
    bin::put(o, (unsigned long long)pts.size());
    for (const auto &p : pts) bin::put_point(o, p);
  }
  bool read_critical_points_binary(const std::string &f) {      // put_critical_points: the points become the tracker's discrete set
    std::ifstream i(f, std::ios::binary);
    unsigned long long n = 0;
    if (!i || !bin::get(i, n)) return false;
    points_.assign(n, feature_point_t());
    for (auto &p : points_)
      if (!bin::get_point(i, p)) return false;
    points_valid_ = true;
    return true;
  }

  // ---- sliced output: critical_point_tracker.hh:819-835 (slice_traced_critical_points), :465-474 (text) ----
  void slice_traced_critical_points() {
    sliced_.clear();
    for (const auto &kv : traced_)
      for (const auto &cp : kv.second)
        if (cp.ordinal) sliced_[cp.timestep].push_back(cp);
  }
  const std::map<int, std::vector<feature_point_t>> &get_sliced_critical_points() const { return sliced_; }
  void write_sliced_critical_points_text(int t, std::ostream &os) const {
    const auto it = sliced_.find(t);
    if (it == sliced_.end()) return;
    for (const auto &cp : it->second) cp.print(os, scalar_components_) << std::endl;
  }
  void write_sliced_critical_points_text(int t, const std::string &f) const { std::ofstream o(f); write_sliced_critical_points_text(t, o); }
  // feature_curve_set_t::intercept (feature_curve_set.hh:534-545) through the library's curve set
  void intercept_traced_critical_points(int t0, int t1) { post_process("intercept:" + std::to_string(t0) + ":" + std::to_string(t1)); }
  void write_critical_points_text(std::ostream &os) { for (const auto &p : get_critical_points()) p.print(os, scalar_components_) << std::endl; }
  void write_critical_points_text(const std::string &f) { std::ofstream o(f); write_critical_points_text(o); }
  void write_critical_points_json(const std::string &f) {
    std::ofstream o(f);
    o << "[";
    const auto pts = get_critical_points();
    for (size_t i = 0; i < pts.size(); i++) { o << (i ? "," : ""); feature_curve_set_t::point_json(o, pts[i]); }
    o << "]" << std::endl;
  }

  ftkb_stats stats() {
    need();
    ftkb_stats s;
    if (group_) { ensure_root(); gcheck(ftkb_group_get_stats(group_, &s, nullptr)); }     // sums over the chunks of all devices
    else check(ftkb_get_stats(ctx_, &s));
    return s;
  }
  ftkb_ctx *handle() { return ctx_; }

 protected:
  void need() const { if (!ctx_ && !group_) throw std::runtime_error("ftk_b200: initialize() has not been called"); }
  // several devices: every result getter works on the merged context (ftkb_group_finalize)
  void ensure_root() { if (group_ && !ctx_) gcheck(ftkb_group_finalize(group_, &ctx_)); }
  void gcheck(int rc) const { if (rc != FTKB_OK) throw std::runtime_error(std::string("ftk_b200: ") + ftkb_group_last_error(group_)); }
  void check(int rc) const { if (rc != FTKB_OK) throw std::runtime_error(std::string("ftk_b200: ") + ftkb_last_error(ctx_)); }
  // the curves of a library curve set, in its multimap order, as the traced set
  void load_curveset(const ftkb_curveset *cs) {
    uint64_t nc = 0, np = 0;
    ftkb_curveset_size(cs, &nc, &np);
    std::vector<ftkb_curve_info> infos(nc ? nc : 1);
    std::vector<ftkb_curve_point> pts(np ? np : 1);
    ftkb_curveset_get(cs, infos.data(), pts.data());
    traced_.clear();
    for (uint64_t i = 0; i < nc; i++) {
      const ftkb_curve_info &in = infos[i];
      feature_curve_t c;
      for (uint64_t k = in.first; k < in.first + in.count; k++) {
        feature_point_t p = to_feature_point(pts[k].p);
        p.v = {{pts[k].v[0], pts[k].v[1], pts[k].v[2]}};
        p.id = (unsigned long long)pts[k].id;
        c.push_back(p);
      }
      c.id = in.id; c.loop = in.loop != 0; c.complete = in.complete != 0; c.consistent_type = in.consistent_type;
      c.tmin = in.tmin; c.tmax = in.tmax;
      c.min = {{in.smin, 0, 0}}; c.max = {{in.smax, 0, 0}}; c.persistence = {{in.persistence, 0, 0}};
      c.bbmin = {{in.bbmin[0], in.bbmin[1], in.bbmin[2]}}; c.bbmax = {{in.bbmax[0], in.bbmax[1], in.bbmax[2]}};
      traced_.insert(std::make_pair(in.id, c));
    }
  }


  void fetch_points() {
    if (points_valid_) return;
    uint64_t n = 0;
    ensure_root();
    check(ftkb_num_points(ctx_, &n));
    std::vector<ftkb_point> raw(n ? n : 1);
    if (n) check(ftkb_get_points(ctx_, raw.data(), n));
    points_.assign(n, feature_point_t());
    for (uint64_t i = 0; i < n; i++) points_[i] = to_feature_point(raw[i]);
    points_valid_ = true;
  }

  feature_point_t to_feature_point(const ftkb_point &r) const {
    const unsigned long long ntypes = nd_ == 2 ? 12 : 60;
    feature_point_t p;
    {
      p.x = {{r.x[0], r.x[1], r.x[2]}};
      // the library works in array-relative vertex coordinates; the reference's grid-unit positions are absolute
      // (simplex_coordinates, REGULAR_COORDS_SIMPLE: X = vertices).  Bounds coordinates are array-relative there too.
      if (coords_mode_ == FTKB_COORDS_SIMPLE) for (int j = 0; j < nd_; j++) p.x[j] += (double)array_domain_.start(j);
      p.t = r.t;
      p.timestep = r.timestep;
      p.scalar = {{r.scalar, 0.0, 0.0}};
      p.type = r.cp_type;
      p.ordinal = r.ordinal != 0;
      p.corner = {{r.corner[0], r.corner[1], r.corner[2], r.corner[3]}};
      p.simplex_type = r.simplex_type;
      // element id in the spirit of simplicial_regular_mesh_element::to_integer (simplicial_regular_mesh.hh:495-502): corner rank
      // over domain x time, times the number of types, plus the type -- in 64 bits
      unsigned long long rank = 0, prod = 1;
      for (int j = 0; j < nd_; j++) { rank += (unsigned long long)(r.corner[j] - (domain_.lower_bound(j) - array_domain_.start(j))) * prod; prod *= (unsigned long long)domain_.size(j); }
      rank += (unsigned long long)r.corner[3] * prod;
      p.tag = rank * ntypes + (unsigned long long)r.simplex_type;
    }
    return p;
  }

  int nd_;
  ftkb_ctx *ctx_ = nullptr;
  ftkb_group *group_ = nullptr;        // several devices: ctx_ is the group's root context once finalize() has run
  std::vector<int> device_ids_;
  int time_chunk_ = 8;
  lattice domain_, array_domain_;
  int scalar_source_ = SOURCE_NONE, vector_source_ = SOURCE_NONE, jacobian_source_ = SOURCE_NONE;
  bool symmetric_ = false, robust_ = true, degrees_ = false, use_type_filter_ = false, discard_interval_ = false, discard_degenerate_ = false, streaming_ = false;
  int coords_mode_ = FTKB_COORDS_SIMPLE;
  std::vector<double> coords_;
  unsigned int type_filter_ = 0;
  int start_timestep_ = 0, device_ = 0;
  double resolution_init_ = 0.0;
  std::vector<std::string> scalar_components_{"scalar"};
  std::vector<feature_point_t> points_;
  bool points_valid_ = false;
  bool finalized_ = false;
  uint64_t sweeps_ = 0, refreshed_sweeps_ = 0;     // update / advance calls; their count at the last refresh of traced_
  feature_curve_set_t traced_;
  std::map<int, std::vector<feature_point_t>> sliced_;
};

struct critical_point_tracker_2d_regular : public critical_point_tracker_regular {
  critical_point_tracker_2d_regular() : critical_point_tracker_regular(2) {}
  template <typename Comm> explicit critical_point_tracker_2d_regular(const Comm &) : critical_point_tracker_regular(2) {}
};

struct critical_point_tracker_3d_regular : public critical_point_tracker_regular {
  critical_point_tracker_3d_regular() : critical_point_tracker_regular(3) {}
  template <typename Comm> explicit critical_point_tracker_3d_regular(const Comm &) : critical_point_tracker_regular(3) {}
};

}  // namespace ftk_b200
#endif
