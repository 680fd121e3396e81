// Host side of the engine: the stateful context behind the C ABI (include/ftkb200.h).
//
// Mirrors the control flow of ftk::critical_point_tracker_{2d,3d}_regular
//   push_*_snapshot   ref: critical_point_tracker_2d_regular.hh:238-261, _3d_regular.hh:125-148
//   update_timestep   ref: critical_point_tracker_2d_regular.hh:263-433, _3d_regular.hh:150-308
//   advance_timestep  ref: critical_point_tracker.hh:841-848
//   finalize          ref: critical_point_tracker.hh:668-817, geometry/cc2curves.hh:10-122
// but keeps every field layer resident in HBM, never materialises the Jacobian and runs all
// per-simplex work in the CUDA kernels of kernels.cu.  There is no CPU code path for the sweep.
#include <algorithm>
#include <cfloat>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <deque>
#include <mutex>
#include <set>
#include <string>
#include <thread>
#include <atomic>
#include <vector>

#include <memory>
#include "kernels.h"
#include "online.h"
#include "curves.h"

using namespace ftkb;

namespace {

thread_local std::string g_create_error;

struct Layer {
  double *S = nullptr, *V = nullptr, *J = nullptr;
  bool ownS = false, ownV = false, ownJ = false;
  int slot = 0;                  // resolution slot
  bool res_pending = false;      // min non-zero |v| not computed yet: the fused scan produces it
  uint4 *cells = nullptr;        // this layer's range cells (kernels.cu, "range cells")
  bool cells_valid = false;
  bool cells_foreign = false;    // the cells belong to a peer process (remote snapshot) or were exported: never recycled
};

// The scans a context's input can still use.  Each input has a fast scan and a slower one that takes every input; a context
// starts at the fastest its configuration and the environment switches allow and only ever moves down (fall_back).
enum class Scans : uint8_t {
  keys2d,       // 2D scalar input: high-word key build kernel
  f32_2d,       //   fp32-range build kernel: NaN / Inf / >= 2^1000 scalars, FTKB_SCAN2D=f32
  fused3d,      // 3D scalar input: gradient fused into the TMA-staged range-cell scan
  gradient3d,   //   gradient materialised: odd W, robust detection off, NaN / Inf / >= 2^1000, no TMA descriptor, FTKB_SCAN3D=plain
  vcells,       // vector input: range-cell scan, each layer streamed once
  twolayer,     //   both layers re-read every step + resolution pass: |v| >= 2^1000 / Inf, 3D odd W or robust detection off, FTKB_VSCAN=twolayer
};

}  // namespace

// host arrays that are filled completely right after they are sized (by a device-to-host copy or a loop): no value-initialisation
// pass over tens of megabytes first
template <class T>
struct NoInitAlloc : std::allocator<T> {
  template <class U> struct rebind { using other = NoInitAlloc<U>; };
  template <class U, class... A>
  void construct(U *q, A &&...a) {
    if constexpr (sizeof...(A) > 0) ::new ((void *)q) U(std::forward<A>(a)...);
  }
};
template <class T> using RawVec = std::vector<T, NoInitAlloc<T>>;

struct ftkb_ctx {
  ftkb_config cfg{};
  int n = 0;                     // spatial dims
  size_t nvert = 0;
  uint64_t ncore = 0;
  int n_ord = 0, n_int = 0;
  cudaStream_t stream = nullptr;
  cudaEvent_t ev[8] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};   // 0-2: sweep, 3: spare, 4-5: derive, 6-7: stopwatch
  bool derive_timed = false;
  std::string error;

  bool slab = false;             // the context holds a z-slab of a larger array (cfg.slab_*)
  void *d_f32 = nullptr;         // staging of float32 snapshots (ftkb_push_snapshot_f32)
  size_t f32_cap = 0;
  std::deque<Layer> layers;
  std::vector<double *> freeS, freeV, freeJ;   // buffer pools
  int current_timestep = 0;
  double resolution = DBL_MAX;
  double factor = 1.0;
  int nbits = 0;
  int next_slot = 0;
  int sm_count = 148;
  Scans scans = Scans::keys2d;
  std::vector<uint4 *> freeCells;
  std::vector<uint4 *> exportedCells;   // handed to a peer process (ftkb_export_layer_cells): freed at destroy only
  size_t ncells = 0;             // cells per layer (fixed by the dims)

  // device scalars: [0..7] per-layer resolution bits, [8] worklist count, [9] point count, [10] unique count, [11] poison,
  // [12] the second worklist counter (deferred steps alternate), [13] ticket of the test kernel's blocks, [14] second poison flag
  unsigned long long *d_scalars = nullptr;
  unsigned long long *h_scalars = nullptr;     // pinned mirror
  static constexpr int SLOT_WL = 8, SLOT_PT = 9, SLOT_UQ = 10, SLOT_POISON = 11, SLOT_WL2 = 12, SLOT_TICKET = 13, SLOT_POISON2 = 14, NSLOTS = 16;

  // ---- deferred ("sync-free") steps ------------------------------------------------------------------------------
  // ftkb_update_timestep enqueues scan + test and returns; the test kernel's last block publishes the counters into the
  // mapped ring below and re-arms the device counters.  The step is confirmed -- counters read, statistics updated --
  // AFTER the next step has been enqueued (or by any call that needs results: drain()).  A step that turns out to have
  // run with a stale quantisation factor, or whose buffers overflowed, is replayed synchronously together with
  // whatever was enqueued behind it.  Layers popped in between wait in `limbo`.
  struct Pending {
    int ring = 0, evset = 0, pops = 0, nbits = 0, wl_sel = 0, timestep = 0;
    uint64_t seq = 0, npts_before = 0, pt_cap = 0;     // pt_cap: the point buffer's capacity this step ran with
    bool has_next = false;
    int res_slots[2] = {-1, -1};     // resolution slots this step's scan fills
  };
  bool defer = true;                 // FTKB_DEFER=0: every step synchronous (the round-1 behaviour)
  std::deque<Pending> pend;
  std::deque<Layer> limbo;
  unsigned long long *h_ring = nullptr;        // pinned + mapped: RING entries of 8 u64
  static constexpr int RING = 4;
  uint64_t step_seq = 0;
  bool primed = false;               // the previous deferred step left the device counters armed for the next one
  int wl_sel = 0;                    // worklist counter of the next deferred step: 0 = SLOT_WL, 1 = SLOT_WL2
  cudaEvent_t dev[2][3] = {{nullptr, nullptr, nullptr}, {nullptr, nullptr, nullptr}};
  bool push_d2h_outstanding = false; // a push queued a resolution read-back the next sweep must wait for
  uint64_t wl_hint = 1 << 16;        // surviving cubes expected by the next test kernel (sizes its grid)
  cudaEvent_t ev_input = nullptr;    // orders device inputs after their producer stream (ftkb_set_producer_stream)
  cudaStream_t producer = nullptr;
  cudaStream_t stream2 = nullptr;    // deferred steps: the test kernels' stream
  cudaEvent_t ev_join = nullptr;
  bool debug_timing = false;         // FTKB_DEBUG_TIMING=1: report the sweep stream's idle time between scans at destroy
  double gap_ms = 0; uint64_t gap_n = 0, last_confirmed_seq = 0;
  std::vector<float> gaps, tl_scan_end, tl_test_end;
  cudaEvent_t dbg_prev = nullptr; bool dbg_prev_valid = false;
  double host_wait_us = 0, host_enq_us = 0; uint64_t host_wait_n = 0, host_enq_n = 0;
  bool last_test_overlapped = false; // where the previous deferred step's test kernel went
  bool has_producer = false;

  unsigned long long *d_wl = nullptr;          // worklist of the synchronous steps and of the even deferred ones
  unsigned long long *d_wl2 = nullptr;         // worklist of the odd deferred steps (a test kernel overlaps the next scan)
  int last_wl_sel = 0;
  uint64_t wl_cap = 0, last_wl = 0;
  ftkb_point *d_pts = nullptr;
  uint64_t pt_cap = 0, npts = 0;
  uint64_t max_step_points = 0;          // most points one confirmed step has produced (sizes the buffer ahead of deferred steps)
  std::vector<ftkb_point *> retired_pts; // point buffers replaced while steps were in flight; freed once nothing is

  // finalize scratch (sort keys / indices, cub temp storage, neighbour lists, union-find parents): kept between calls, grown on demand
  struct Scratch { void *p = nullptr; size_t cap = 0; bool in_slab = false; };
  void *fz_slab = nullptr;          // one allocation behind the slots a finalize plans together (scratch_plan)
  size_t fz_slab_cap = 0;
  Scratch fz[14];          // 10, 11: the streaming grow step's neighbour lists and counts; 12, 13: the sorted records and their keys
  void *grow_stage = nullptr;   // page-locked staging of a grow step's batch
  size_t grow_stage_cap = 0;

  // sorted / traced results (host)
  bool sorted = false, traced = false;
  RawVec<ftkb_point> pts_sorted;
  ftkb_point *d_pts_sorted = nullptr;          // device copy of the sorted unique points
  unsigned long long *d_keys_sorted = nullptr;
  uint64_t nsorted = 0;
  RawVec<uint64_t> labels;
  RawVec<int32_t> deg;
  std::vector<uint64_t> traj_off, traj_idx;
  std::vector<uint8_t> traj_loop, traj_complete;

  // physical coordinates (regular_tracker.hh:38-40)
  int coords_mode = 0, coords_ncomp = 0;
  double coords_bounds[6] = {0, 0, 0, 0, 0, 0};
  double *d_coords = nullptr;

  // streaming trajectories (critical_point_tracker.hh:38,522-641): grown on the host after every interval sweep
  bool streaming = false;
  std::unique_ptr<ftkb::OnlineTracer> online;
  uint64_t grown = 0;            // d_pts[0 .. grown) have been through a grow step
  int grown_through = 0;         // the last timestep whose grow step has run (start_timestep - 1: none)
  bool grow_failed = false;      // a grow step threw: every later call that depends on the trajectories reports it

  // d_pts[begin, end) = the points of the confirmed sweep of timestep start_timestep + k (steps[k]); a replay only redoes steps
  // that were not confirmed, from the point count they started at, so a confirmed step's points stay where they are
  struct StepRange { uint64_t begin = 0, end = 0; bool interval = false; };
  std::vector<StepRange> steps;

  ftkb_stats stats{};
};

#define CK(call)                                                                                         \
  do {                                                                                                   \
    cudaError_t e_ = (call);                                                                             \
    if (e_ != cudaSuccess) {                                                                             \
      c->error = std::string(#call) + ": " + cudaGetErrorString(e_);                                     \
      return e_ == cudaErrorMemoryAllocation ? FTKB_ERR_NOMEM : FTKB_ERR_CUDA;                           \
    }                                                                                                    \
  } while (0)

static int fail(ftkb_ctx *c, int code, const std::string &msg) {
  if (c) c->error = msg;
  else g_create_error = msg;
  return code;
}

// pooled device scratch of ensure_sorted / ftkb_finalize: slot i holds at least `bytes`
// Every cudaMalloc of a finalize showed up in its wall time (0.1 .. 30 ms each, depending on what the process freed before): the slots
// one finalize needs are planned together and carved out of ONE allocation.  bytes[i] == 0: slot i is left alone.
static int scratch_plan(ftkb_ctx *c, const size_t *bytes, int nslots) {
  bool enough = true;
  size_t total = 0;
  for (int i = 0; i < nslots; i++)
    if (bytes[i]) { enough = enough && c->fz[i].cap >= bytes[i]; total += (bytes[i] + bytes[i] / 4 + 511) / 256 * 256; }
  if (enough) return FTKB_OK;
  for (int i = 0; i < (int)(sizeof(c->fz) / sizeof(c->fz[0])); i++)
    if (c->fz[i].in_slab) c->fz[i] = ftkb_ctx::Scratch{};
  if (c->fz_slab_cap < total) {
    cudaFree(c->fz_slab);
    c->fz_slab = nullptr; c->fz_slab_cap = 0;
    if (cudaMalloc(&c->fz_slab, total) != cudaSuccess) { cudaGetLastError(); c->error = "finalize: out of device memory"; return FTKB_ERR_NOMEM; }
    c->fz_slab_cap = total;
  }
  size_t off = 0;
  for (int i = 0; i < nslots; i++) {
    if (!bytes[i]) continue;
    ftkb_ctx::Scratch &s = c->fz[i];
    if (s.p && !s.in_slab) cudaFree(s.p);
    const size_t sz = (bytes[i] + bytes[i] / 4 + 511) / 256 * 256;
    s.p = (char *)c->fz_slab + off; s.cap = sz; s.in_slab = true;
    off += sz;
  }
  return FTKB_OK;
}

static int scratch(ftkb_ctx *c, int i, size_t bytes, void **out) {
  ftkb_ctx::Scratch &s = c->fz[i];
  if (s.cap < bytes) {
    if (!s.in_slab) cudaFree(s.p);
    s.in_slab = false;
    s.p = nullptr; s.cap = 0;
    const size_t want = bytes + bytes / 4 + 256;
    if (cudaMalloc(&s.p, want) != cudaSuccess) { cudaGetLastError(); c->error = "finalize: out of device memory"; return FTKB_ERR_NOMEM; }
    s.cap = want;
  }
  *out = s.p;
  return FTKB_OK;
}

static int check_launch(ftkb_ctx *c, const char *what) {
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return fail(c, FTKB_ERR_CUDA, std::string(what) + ": " + cudaGetErrorString(e));
  return FTKB_OK;
}

// ------------------------------------------------------------------------------------------------
extern "C" int ftkb_abi_version(void) { return FTKB_ABI_VERSION; }

extern "C" int ftkb_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
  int usable = 0;
  for (int i = 0; i < n; i++) {
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, i) == cudaSuccess && prop.major == 10) usable++;
  }
  return usable;
}

extern "C" const char *ftkb_last_error(const ftkb_ctx *c) { return c ? c->error.c_str() : g_create_error.c_str(); }

static void release_layer(ftkb_ctx *c, Layer &l) {
  if (l.ownS && l.S) c->freeS.push_back(l.S);
  if (l.ownV && l.V) c->freeV.push_back(l.V);
  if (l.ownJ && l.J) c->freeJ.push_back(l.J);
  if (l.cells && !l.cells_foreign) c->freeCells.push_back(l.cells);
  l = Layer();
}

static void fill_trace_params(const ftkb_ctx *c, TraceParams &tp);
static int drain(ftkb_ctx *c);

extern "C" void ftkb_destroy(ftkb_ctx *c) {
  if (!c) return;
  if (c->debug_timing && c->gaps.size() > 8) {
    auto med = [](std::vector<float> v) { std::sort(v.begin(), v.end()); return 1e3 * v[v.size() / 2]; };
    std::fprintf(stderr, "[ftkb] deferred steps, relative to the previous scan's end (medians over %zu): scan starts +%.1f us, ends +%.1f us, test ends +%.1f us\n",
                 c->gaps.size(), med(c->gaps), med(c->tl_scan_end), med(c->tl_test_end));
    std::fprintf(stderr, "[ftkb] host: %.1f us to enqueue a step, %.1f us blocked per confirmation (avg over %llu / %llu)\n",
                 c->host_enq_us / std::max<uint64_t>(1, c->host_enq_n), c->host_wait_us / std::max<uint64_t>(1, c->host_wait_n),
                 (unsigned long long)c->host_enq_n, (unsigned long long)c->host_wait_n);
  }
  cudaSetDevice(c->cfg.device);
  if (c->stream) cudaStreamSynchronize(c->stream);
  for (auto &l : c->layers) release_layer(c, l);
  for (auto &l : c->limbo) release_layer(c, l);
  c->limbo.clear();
  for (auto *p : c->freeS) cudaFree(p);
  for (auto *p : c->freeV) cudaFree(p);
  for (auto *p : c->freeJ) cudaFree(p);
  for (auto *p : c->freeCells) cudaFree(p);
  for (auto *p : c->exportedCells) cudaFree(p);
  cudaFree(c->d_scalars);
  if (c->h_scalars) cudaFreeHost(c->h_scalars);
  if (c->grow_stage) cudaFreeHost(c->grow_stage);
  for (ftkb_point *q : c->retired_pts) cudaFree(q);
  if (c->h_ring) cudaFreeHost(c->h_ring);
  for (auto &es : c->dev) for (auto &e : es) if (e) cudaEventDestroy(e);
  if (c->ev_input) cudaEventDestroy(c->ev_input);
  if (c->dbg_prev) cudaEventDestroy(c->dbg_prev);
  cudaFree(c->d_wl);
  cudaFree(c->d_wl2);
  if (c->stream2) { cudaStreamSynchronize(c->stream2); cudaStreamDestroy(c->stream2); }
  if (c->ev_join) cudaEventDestroy(c->ev_join);
  cudaFree(c->d_pts);
  cudaFree(c->d_coords);
  cudaFree(c->d_f32);
  for (auto &s : c->fz) if (!s.in_slab) cudaFree(s.p);
  cudaFree(c->fz_slab);
  for (auto &e : c->ev) if (e) cudaEventDestroy(e);
  if (c->stream) cudaStreamDestroy(c->stream);
  delete c;
}

extern "C" int ftkb_create(const ftkb_config *cfg, ftkb_ctx **out) {
  if (!cfg || !out) return fail(nullptr, FTKB_ERR_INVALID, "ftkb_create: null argument");
  *out = nullptr;
  if (cfg->abi_version != FTKB_ABI_VERSION) return fail(nullptr, FTKB_ERR_INVALID, "ftkb_create: ABI version mismatch");
  if (cfg->nd != 2 && cfg->nd != 3) return fail(nullptr, FTKB_ERR_INVALID, "ftkb_create: nd must be 2 or 3");
  const int n = cfg->nd;
  for (int j = 0; j < n; j++) {
    if (cfg->dims[j] < 2) return fail(nullptr, FTKB_ERR_INVALID, "ftkb_create: array dims must be >= 2");
    if (cfg->lb[j] < 0 || cfg->ub[j] > cfg->dims[j] - 1 || cfg->lb[j] > cfg->ub[j])
      return fail(nullptr, FTKB_ERR_INVALID, "ftkb_create: domain must lie inside the array");
  }
  if (cfg->start_timestep < 0) return fail(nullptr, FTKB_ERR_INVALID, "ftkb_create: start_timestep must be >= 0");
  // no CPU fallback: a Blackwell device is required
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
    cudaGetLastError();
    return fail(nullptr, FTKB_ERR_NO_DEVICE, "ftkb_create: no CUDA device (this engine has no CPU fallback)");
  }
  if (cfg->device < 0 || cfg->device >= ndev) return fail(nullptr, FTKB_ERR_NO_DEVICE, "ftkb_create: device ordinal out of range");
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, cfg->device) != cudaSuccess || prop.major != 10)
    return fail(nullptr, FTKB_ERR_NO_DEVICE, "ftkb_create: device is not compute capability 10.x (kernels are built for sm_100a only)");

  if (cfg->slab_global_dim != 0) {
    if (n != 3) return fail(nullptr, FTKB_ERR_INVALID, "ftkb_create: spatial slabs are 3D (along z)");
    if (cfg->slab_offset < 0 || cfg->slab_offset + cfg->dims[2] > cfg->slab_global_dim || cfg->slab_global_lb < 0 ||
        cfg->slab_global_ub >= cfg->slab_global_dim || cfg->slab_global_lb > cfg->slab_global_ub ||
        cfg->slab_offset + cfg->lb[2] < cfg->slab_global_lb || cfg->slab_offset + cfg->ub[2] > cfg->slab_global_ub)
      return fail(nullptr, FTKB_ERR_INVALID, "ftkb_create: the slab does not lie inside the whole array / domain");
  }
  ftkb_ctx *c = new ftkb_ctx();
  c->cfg = *cfg;
  c->slab = cfg->slab_global_dim != 0;
  c->sm_count = prop.multiProcessorCount > 0 ? prop.multiProcessorCount : 148;
  {
    // the 3D range-cell scans need TMA-compatible rows (W even) and the exact early-out (robust detection on)
    auto env_is = [](const char *name, const char *value) { const char *e = std::getenv(name); return e && std::string(e) == value; };
    if (cfg->vector_source == FTKB_SOURCE_GIVEN)
      c->scans = (n == 2 || (cfg->robust_detection && cfg->dims[0] % 2 == 0)) && !env_is("FTKB_VSCAN", "twolayer") ? Scans::vcells : Scans::twolayer;
    else if (n == 3)
      c->scans = cfg->vector_source == FTKB_SOURCE_DERIVED && cfg->robust_detection && cfg->dims[0] % 2 == 0 && !env_is("FTKB_SCAN3D", "plain")
                     ? Scans::fused3d : Scans::gradient3d;
    else
      c->scans = env_is("FTKB_SCAN2D", "f32") ? Scans::f32_2d : Scans::keys2d;
  }
  c->n = n;
  c->nvert = (size_t)cfg->dims[0] * cfg->dims[1] * (n == 3 ? cfg->dims[2] : 1);
  c->ncore = 1;
  for (int j = 0; j < n; j++) c->ncore *= (uint64_t)(cfg->ub[j] - cfg->lb[j] + 1);
  // element keys pack (x, y, z, t, type) into 64 bits
  {
    const long double cap = 18446744073709551616.0L / (long double)(1ull << (KEY_TIME_BITS + KEY_TYPE_BITS));
    long double key_cells = (long double)c->ncore;
    if (c->slab) key_cells = key_cells / (long double)(cfg->ub[2] - cfg->lb[2] + 1) * (long double)(cfg->slab_global_ub - cfg->slab_global_lb + 1);
    if (key_cells >= cap) { delete c; return fail(nullptr, FTKB_ERR_OVERFLOW, "ftkb_create: domain too large for 64-bit element ids"); }
  }
  const MeshTables &mt = mesh_tables(n + 1);
  c->n_ord = (int)mt.ordinal_types[n].size();
  c->n_int = (int)mt.interval_types[n].size();
  c->current_timestep = cfg->start_timestep;
  c->grown_through = cfg->start_timestep - 1;
  c->resolution =cfg->resolution_init > 0 ? cfg->resolution_init : DBL_MAX;

  auto bail = [&](const std::string &m, int code) { g_create_error = m; ftkb_destroy(c); return code; };
  cudaError_t e;
  if ((e = cudaSetDevice(cfg->device)) != cudaSuccess) return bail(std::string("cudaSetDevice: ") + cudaGetErrorString(e), FTKB_ERR_CUDA);
  if ((e = cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking)) != cudaSuccess) return bail(std::string("cudaStreamCreate: ") + cudaGetErrorString(e), FTKB_ERR_CUDA);
  for (auto &ev : c->ev)
    if ((e = cudaEventCreate(&ev)) != cudaSuccess) return bail(std::string("cudaEventCreate: ") + cudaGetErrorString(e), FTKB_ERR_CUDA);
  if ((e = cudaMalloc(&c->d_scalars, sizeof(unsigned long long) * ftkb_ctx::NSLOTS)) != cudaSuccess) return bail("cudaMalloc(scalars) failed", FTKB_ERR_NOMEM);
  if ((e = cudaMallocHost(&c->h_scalars, sizeof(unsigned long long) * ftkb_ctx::NSLOTS)) != cudaSuccess) return bail("cudaMallocHost failed", FTKB_ERR_NOMEM);
  std::memset(c->h_scalars, 0, sizeof(unsigned long long) * ftkb_ctx::NSLOTS);
  if ((e = cudaHostAlloc(&c->h_ring, sizeof(unsigned long long) * 8 * ftkb_ctx::RING, cudaHostAllocMapped | cudaHostAllocPortable)) != cudaSuccess) return bail("cudaHostAlloc(ring) failed", FTKB_ERR_NOMEM);
  std::memset(c->h_ring, 0xff, sizeof(unsigned long long) * 8 * ftkb_ctx::RING);
  for (auto &es : c->dev)
    for (auto &ev : es)
      if ((e = cudaEventCreate(&ev)) != cudaSuccess) return bail(std::string("cudaEventCreate: ") + cudaGetErrorString(e), FTKB_ERR_CUDA);
  if ((e = cudaEventCreateWithFlags(&c->ev_input, cudaEventDisableTiming)) != cudaSuccess) return bail(std::string("cudaEventCreate: ") + cudaGetErrorString(e), FTKB_ERR_CUDA);
  if (const char *d = std::getenv("FTKB_DEFER")) c->defer = std::string(d) != "0";
  cudaMemsetAsync(c->d_scalars, 0, sizeof(unsigned long long) * ftkb_ctx::NSLOTS, c->stream);
  c->wl_cap = std::max<uint64_t>(1 << 16, c->ncore / 64);
  if (const char *w = std::getenv("FTKB_WL_CAP")) c->wl_cap = std::max<uint64_t>(1, std::strtoull(w, nullptr, 10));   // tests: force the overflow path
  if ((e = cudaMalloc(&c->d_wl, sizeof(unsigned long long) * c->wl_cap)) != cudaSuccess) return bail("cudaMalloc(worklist) failed", FTKB_ERR_NOMEM);
  if ((e = cudaMalloc(&c->d_wl2, sizeof(unsigned long long) * c->wl_cap)) != cudaSuccess) return bail("cudaMalloc(worklist) failed", FTKB_ERR_NOMEM);
  {
    // the exact tests of deferred step k run on their own (high-priority) stream next to the scan of step k+1
    int lo = 0, hi = 0;
    cudaDeviceGetStreamPriorityRange(&lo, &hi);
    if ((e = cudaStreamCreateWithPriority(&c->stream2, cudaStreamNonBlocking, hi)) != cudaSuccess) return bail(std::string("cudaStreamCreate: ") + cudaGetErrorString(e), FTKB_ERR_CUDA);
    if ((e = cudaEventCreateWithFlags(&c->ev_join, cudaEventDisableTiming)) != cudaSuccess) return bail(std::string("cudaEventCreate: ") + cudaGetErrorString(e), FTKB_ERR_CUDA);
    if (const char *o = std::getenv("FTKB_DEBUG_TIMING")) c->debug_timing = std::string(o) == "1";
    if (c->debug_timing) cudaEventCreate(&c->dbg_prev);
  }
  c->pt_cap = cfg->point_capacity ? cfg->point_capacity : (1 << 20);      // 75 MB of 180 GB: growth (a cudaMalloc in the middle of the step loop) starts late
  if ((e = cudaMalloc(&c->d_pts, sizeof(ftkb_point) * c->pt_cap)) != cudaSuccess) return bail("cudaMalloc(points) failed", FTKB_ERR_NOMEM);
  DeviceMeshTables t2, t3;
  fill_device_tables(3, &t2);
  fill_device_tables(4, &t3);
  upload_mesh_tables(t2, t3);
  init_kernel_attributes();
  if ((e = cudaStreamSynchronize(c->stream)) != cudaSuccess) return bail(std::string("init: ") + cudaGetErrorString(e), FTKB_ERR_CUDA);
  *out = c;
  return FTKB_OK;
}

static int take_buffer(ftkb_ctx *c, std::vector<double *> &pool, size_t count, double **out) {
  if (pool.empty() && !c->pend.empty() && c->layers.size() + c->limbo.size() >= 4) {
    // buffers of layers that enqueued steps still read come back once those steps are confirmed
    const int rc = drain(c);
    if (rc) return rc;
  }
  if (!pool.empty()) { *out = pool.back(); pool.pop_back(); return FTKB_OK; }
  CK(cudaMalloc(out, sizeof(double) * count));
  return FTKB_OK;
}

// resolution of the layer's vector field into its slot; the value reaches the host asynchronously
static int queue_resolution(ftkb_ctx *c, Layer &l, bool fused_in_gradient) {
  if (!fused_in_gradient) launch_resolution(l.V, (uint64_t)c->nvert * c->n, c->d_scalars + l.slot, c->stream);
  c->stats.kernel_launches += fused_in_gradient ? 0 : 1;
  CK(cudaMemcpyAsync(c->h_scalars + l.slot, c->d_scalars + l.slot, sizeof(unsigned long long), cudaMemcpyDeviceToHost, c->stream));
  c->stats.d2h_bytes += 8;
  c->push_d2h_outstanding = true;
  return check_launch(c, "resolution");
}

static bool aligned16(const void *a) { return (uintptr_t)a % 16 == 0; }

// the sweep derives the vector field from layer l0's scalars on the fly (SweepParams::fused)
static bool derives_vectors(const ftkb_ctx *c, const Layer &l0) {
  return !l0.V && l0.S && c->cfg.vector_source == FTKB_SOURCE_DERIVED && (c->n == 2 || c->scans == Scans::fused3d);
}

// the scan derives the layer's gradient on the fly, or streams its vectors into range cells, and folds the layer's min
// non-zero |v| into that pass
static bool scan_resolves(const ftkb_ctx *c, const Layer &l) {
  return l.V ? c->scans == Scans::vcells && aligned16(l.V) : derives_vectors(c, l) && (c->n == 2 || aligned16(l.S));
}

static int derive_layer(ftkb_ctx *c, Layer &l) {
  // slot <- all ones: above the bit pattern of every finite double, so the kernels' atomicMin on the
  // bit patterns of |v| works unchanged and "nothing found" reads back as DBL_MAX (slot_value).
  // Layers whose resolution the scan produces (res_pending) only mark the host mirror: the sweep's one
  // host-to-device copy of the counter block resets the device slot (no separate memset per push).
  bool fused = false;
  if (scan_resolves(c, l)) {
    // the first sweep that reads this layer computes its resolution
    l.res_pending = true;
    c->h_scalars[l.slot] = ~0ull;
    return FTKB_OK;
  }
  CK(cudaMemsetAsync(c->d_scalars + l.slot, 0xff, sizeof(unsigned long long), c->stream));
  if (!l.V && c->cfg.vector_source == FTKB_SOURCE_DERIVED && l.S) {
    int rc = take_buffer(c, c->freeV, c->nvert * c->n, &l.V);
    if (rc) return rc;
    l.ownV = true;
    CK(cudaEventRecord(c->ev[4], c->stream));
    launch_gradient(c->n, l.S, l.V, c->cfg.dims[0], c->cfg.dims[1], c->n == 3 ? c->cfg.dims[2] : 1, c->d_scalars + l.slot, c->stream);
    CK(cudaEventRecord(c->ev[5], c->stream));
    c->derive_timed = true;
    c->stats.kernel_launches++;
    fused = true;
  }
  if (l.V) {
    int rc = queue_resolution(c, l, fused);
    if (rc) return rc;
  }
  return check_launch(c, "derive");
}

static int new_layer(ftkb_ctx *c, Layer &l) {
  if (c->layers.size() >= 4) return fail(c, FTKB_ERR_INVALID, "push: more than 4 resident snapshots (call advance_timestep)");
  l.slot = c->next_slot;
  c->next_slot = (c->next_slot + 1) % 8;
  return FTKB_OK;
}

// Peer access of `device` to `peer` (device arrays of a group's push may live on any device): enabled once per (destination,
// source) pair where the hardware allows it; without it cudaMemcpyPeerAsync still copies, staged by the driver.  Leaves `device`
// current.
cudaError_t ftkb::enable_peer_access(int device, int peer) {
  static std::mutex m;
  static std::set<std::pair<int, int>> done;
  cudaError_t e = cudaSetDevice(device);
  if (e != cudaSuccess || device == peer) return e;
  std::lock_guard<std::mutex> lk(m);
  if (done.count({device, peer})) return cudaSuccess;
  int can = 0;
  if ((e = cudaDeviceCanAccessPeer(&can, device, peer)) != cudaSuccess) return e;
  if (can && (e = cudaDeviceEnablePeerAccess(peer, 0)) != cudaSuccess) {
    if (e != cudaErrorPeerAccessAlreadyEnabled) return e;
    cudaGetLastError();
  }
  done.insert({device, peer});
  return cudaSuccess;
}

// the ingest of every push: the layer is copied from `segs`, which tile the array in plane order (one segment covering it all
// for host input and for borrowed arrays); device arrays (FTKB_MEM_DEVICE) are read on each segment's device, the context's own
// or any other.  A segment's `after`, if not null, is an event its copies wait for (it replaces the context's own producer stream).
static int push_snapshot(ftkb_ctx *c, const ftkb::Segment *segs, int nsegs, int where) {
  const double *scalar = segs[0].scalar, *vector = segs[0].vector, *jacobian = segs[0].jacobian;
  if (where < FTKB_MEM_HOST || where > FTKB_MEM_DEVICE_BORROW) return fail(c, FTKB_ERR_INVALID, "push: bad memory kind");
  if (c->cfg.scalar_source == FTKB_SOURCE_GIVEN && !scalar) return fail(c, FTKB_ERR_INVALID, "push: scalar field is GIVEN but no scalar array was passed");
  if (c->cfg.vector_source == FTKB_SOURCE_GIVEN && !vector) return fail(c, FTKB_ERR_INVALID, "push: vector field is GIVEN but no vector array was passed");
  if (c->cfg.vector_source == FTKB_SOURCE_DERIVED && !vector && !scalar) return fail(c, FTKB_ERR_INVALID, "push: vector field is DERIVED but no scalar array was passed");
  if (c->cfg.jacobian_source == FTKB_SOURCE_GIVEN && !jacobian) return fail(c, FTKB_ERR_INVALID, "push: jacobian is GIVEN but no jacobian array was passed");
  CK(cudaSetDevice(c->cfg.device));
  const int extent = c->n == 3 ? c->cfg.dims[2] : c->cfg.dims[1];
  for (int i = 0, next = 0; i < nsegs; next += segs[i++].count) {
    const ftkb::Segment &s = segs[i];
    if (s.first != next || s.count < 1 || (i == nsegs - 1 && s.first + s.count != extent) || (where == FTKB_MEM_DEVICE_BORROW && nsegs != 1) ||
        !s.scalar != !scalar || !s.vector != !vector || !s.jacobian != !jacobian)
      return fail(c, FTKB_ERR_INVALID, "push: segments do not tile the array with the same arrays");
    for (const double *q : {s.scalar, s.vector, s.jacobian})
      if ((uintptr_t)q % 8 != 0) return fail(c, FTKB_ERR_INVALID, "push: arrays must be 8-byte aligned");
  }
  Layer l;
  int rc = new_layer(c, l);
  if (rc) return rc;
  bool ordered = false;
  for (int i = 0; i < nsegs; i++)
    if (segs[i].after) { CK(cudaStreamWaitEvent(c->stream, segs[i].after, 0)); ordered = true; }
  if (!ordered && where != FTKB_MEM_HOST && c->has_producer) {
    // device inputs are written by the caller's stream: everything this context enqueues from here on runs after the
    // work queued there so far (the context's own stream is non-blocking: the legacy default stream orders nothing)
    CK(cudaEventRecord(c->ev_input, c->producer));
    CK(cudaStreamWaitEvent(c->stream, c->ev_input, 0));
  }
  const size_t plane = c->nvert / (size_t)extent;
  // one copy per segment of array `a`, whose vertices hold `per` doubles each
  auto ingest = [&](const double *ftkb::Segment::*a, size_t per, std::vector<double *> &pool, double **dst, bool *own) -> int {
    if (!(segs[0].*a)) return FTKB_OK;
    if (where == FTKB_MEM_DEVICE_BORROW) { *dst = const_cast<double *>(segs[0].*a); *own = false; return FTKB_OK; }
    int r = take_buffer(c, pool, c->nvert * per, dst);
    if (r) return r;
    *own = true;
    for (int i = 0; i < nsegs; i++) {
      const ftkb::Segment &s = segs[i];
      double *to = *dst + (size_t)s.first * plane * per;
      const size_t bytes = sizeof(double) * (size_t)s.count * plane * per;
      if (where == FTKB_MEM_DEVICE && s.device != c->cfg.device)
        CK(cudaMemcpyPeerAsync(to, c->cfg.device, s.*a, s.device, bytes, c->stream));
      else
        CK(cudaMemcpyAsync(to, s.*a, bytes, where == FTKB_MEM_HOST ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToDevice, c->stream));
      if (where == FTKB_MEM_HOST) c->stats.h2d_bytes += bytes;
    }
    return FTKB_OK;
  };
  if ((rc = ingest(&ftkb::Segment::scalar, 1, c->freeS, &l.S, &l.ownS))) { release_layer(c, l); return rc; }
  if ((rc = ingest(&ftkb::Segment::vector, c->n, c->freeV, &l.V, &l.ownV))) { release_layer(c, l); return rc; }
  if ((rc = ingest(&ftkb::Segment::jacobian, c->n * c->n, c->freeJ, &l.J, &l.ownJ))) { release_layer(c, l); return rc; }
  if ((rc = derive_layer(c, l))) { release_layer(c, l); return rc; }
  // copied inputs (host or device) are borrowed only until return: the caller may free or overwrite them right away
  if (where != FTKB_MEM_DEVICE_BORROW) CK(cudaStreamSynchronize(c->stream));
  c->layers.push_back(l);
  return FTKB_OK;
}

extern "C" int ftkb_push_snapshot(ftkb_ctx *c, const double *scalar, const double *vector, const double *jacobian, int where) {
  if (!c) return FTKB_ERR_INVALID;
  ftkb::Segment s;           // the whole array as one segment
  s.count = c->n == 3 ? c->cfg.dims[2] : c->cfg.dims[1];
  s.scalar = scalar; s.vector = vector; s.jacobian = jacobian;
  s.device = c->cfg.device;
  return push_snapshot(c, &s, 1, where);
}

int ftkb::push_segments(ftkb_ctx *c, const Segment *segs, int n) {
  if (!c || !segs || n < 1) return FTKB_ERR_INVALID;
  for (int i = 0; i < n; i++) CK(ftkb::enable_peer_access(c->cfg.device, segs[i].device));
  return push_snapshot(c, segs, n, FTKB_MEM_DEVICE);
}

// A snapshot that exists as float32 (raw float32 file series: the reference widens them on the host, ndarray.hh read_binary_file):
// it travels over PCIe as float32 and is widened on the device, into the same resident fp64 layer the other pushes produce.
extern "C" int ftkb_push_snapshot_f32(ftkb_ctx *c, const float *scalar, const float *vector) {
  if (!c) return FTKB_ERR_INVALID;
  if (c->cfg.jacobian_source == FTKB_SOURCE_GIVEN) return fail(c, FTKB_ERR_INVALID, "push_snapshot_f32: a GIVEN jacobian has no float32 form");
  if (c->cfg.scalar_source == FTKB_SOURCE_GIVEN && !scalar) return fail(c, FTKB_ERR_INVALID, "push: scalar field is GIVEN but no scalar array was passed");
  if (c->cfg.vector_source == FTKB_SOURCE_GIVEN && !vector) return fail(c, FTKB_ERR_INVALID, "push: vector field is GIVEN but no vector array was passed");
  if (c->cfg.vector_source == FTKB_SOURCE_DERIVED && !vector && !scalar) return fail(c, FTKB_ERR_INVALID, "push: vector field is DERIVED but no scalar array was passed");
  if ((uintptr_t)scalar % 4 != 0 || (uintptr_t)vector % 4 != 0) return fail(c, FTKB_ERR_INVALID, "push: arrays must be 4-byte aligned");
  CK(cudaSetDevice(c->cfg.device));
  Layer l;
  int rc = new_layer(c, l);
  if (rc) return rc;
  const size_t nS = c->nvert, nV = c->nvert * c->n;
  const size_t need = 4 * std::max(scalar ? nS : 0, vector ? nV : 0) + 16;
  if (c->f32_cap < need) {
    cudaFree(c->d_f32);
    c->d_f32 = nullptr; c->f32_cap = 0;
    CK(cudaMalloc(&c->d_f32, need));
    c->f32_cap = need;
  }
  auto ingest = [&](const float *src, size_t count, std::vector<double *> &pool, double **dst, bool *own) -> int {
    if (!src) return FTKB_OK;
    const int r = take_buffer(c, pool, count, dst);
    if (r) return r;
    *own = true;
    CK(cudaMemcpyAsync(c->d_f32, src, 4 * count, cudaMemcpyHostToDevice, c->stream));
    launch_widen_f32(static_cast<const float *>(c->d_f32), *dst, count, c->stream);
    c->stats.h2d_bytes += 4 * count;
    c->stats.kernel_launches++;
    return check_launch(c, "widen");
  };
  if ((rc = ingest(scalar, nS, c->freeS, &l.S, &l.ownS))) { release_layer(c, l); return rc; }
  if ((rc = ingest(vector, nV, c->freeV, &l.V, &l.ownV))) { release_layer(c, l); return rc; }
  if ((rc = derive_layer(c, l))) { release_layer(c, l); return rc; }
  CK(cudaStreamSynchronize(c->stream));      // the host buffer is borrowed only until return
  c->layers.push_back(l);
  return FTKB_OK;
}

extern "C" int ftkb_set_producer_stream(ftkb_ctx *c, void *stream, int enable) {
  if (!c) return FTKB_ERR_INVALID;
  c->producer = reinterpret_cast<cudaStream_t>(stream);
  c->has_producer = enable != 0;
  return FTKB_OK;
}

extern "C" int ftkb_push_synthetic(ftkb_ctx *c, int kind, const double *params, int nparams, double t) {
  if (!c) return FTKB_ERR_INVALID;
  if (nparams < 0 || nparams > 8 || (nparams && !params)) return fail(c, FTKB_ERR_INVALID, "push_synthetic: bad params");
  const bool vector_kind = kind == FTKB_SYN_DOUBLE_GYRE || kind == FTKB_SYN_ABC || kind == FTKB_SYN_TORNADO;
  const bool ok2 = kind == FTKB_SYN_WOVEN || kind == FTKB_SYN_DOUBLE_GYRE || kind == FTKB_SYN_MERGER;
  if (kind < 0 || kind > FTKB_SYN_TORNADO || (ok2 && c->n != 2) || ((kind == FTKB_SYN_ABC || kind == FTKB_SYN_TORNADO) && c->n != 3))
    return fail(c, FTKB_ERR_INVALID, "push_synthetic: generator does not match the context's dimensionality");
  if (vector_kind ? c->cfg.vector_source != FTKB_SOURCE_GIVEN : c->cfg.scalar_source != FTKB_SOURCE_GIVEN)
    return fail(c, FTKB_ERR_INVALID, "push_synthetic: generator kind does not match the configured field sources");
  CK(cudaSetDevice(c->cfg.device));
  double p[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  for (int i = 0; i < nparams; i++) p[i] = params[i];
  Layer l;
  int rc = new_layer(c, l);
  if (rc) return rc;
  double **dst = vector_kind ? &l.V : &l.S;
  if ((rc = take_buffer(c, vector_kind ? c->freeV : c->freeS, vector_kind ? c->nvert * c->n : c->nvert, dst))) { release_layer(c, l); return rc; }
  (vector_kind ? l.ownV : l.ownS) = true;
  launch_synthetic(kind, c->n, c->cfg.dims[0], c->cfg.dims[1], c->n == 3 ? c->cfg.dims[2] : 1, p, t, *dst, c->stream,
                   c->slab ? c->cfg.slab_offset : 0, c->slab ? c->cfg.slab_global_dim : 0);
  c->stats.kernel_launches++;
  if ((rc = derive_layer(c, l))) { release_layer(c, l); return rc; }
  c->layers.push_back(l);
  return FTKB_OK;
}

static int resolve_pending(ftkb_ctx *c, Layer &l);

static double slot_value(const ftkb_ctx *c, int slot) {
  double v;
  std::memcpy(&v, c->h_scalars + slot, 8);
  return (c->h_scalars[slot] >> 52) >= 0x7ff ? DBL_MAX : v;    // untouched slot (all ones): no non-zero finite value
}

extern "C" int ftkb_last_layer_resolution(ftkb_ctx *c, double *res) {
  if (!c || !res) return FTKB_ERR_INVALID;
  if (c->layers.empty()) return fail(c, FTKB_ERR_INVALID, "last_layer_resolution: no resident snapshot");
  CK(cudaSetDevice(c->cfg.device));
  { const int rc = drain(c); if (rc) return rc; }
  Layer &l = c->layers.back();
  if (l.res_pending) {
    const int rc = resolve_pending(c, l);
    if (rc) return rc;
  }
  CK(cudaStreamSynchronize(c->stream));
  *res = (l.V || l.S) ? slot_value(c, l.slot) : DBL_MAX;
  return FTKB_OK;
}

extern "C" int ftkb_set_resolution(ftkb_ctx *c, double res) {
  if (!c) return FTKB_ERR_INVALID;
  if (!c->pend.empty()) {           // applies to the sweeps that follow, not to those in flight
    cudaSetDevice(c->cfg.device);
    const int rc = drain(c);
    if (rc) return rc;
  }
  if (res > 0 && res < c->resolution) c->resolution = res;
  return FTKB_OK;
}

extern "C" int ftkb_current_timestep(const ftkb_ctx *c, int32_t *t) {
  if (!c || !t) return FTKB_ERR_INVALID;
  *t = c->current_timestep;
  return FTKB_OK;
}

static int grow_points(ftkb_ctx *c, uint64_t need) {
  uint64_t cap = c->pt_cap;
  while (cap < need) cap *= 2;
  ftkb_point *np = nullptr;
  CK(cudaMalloc(&np, sizeof(ftkb_point) * cap));
  CK(cudaMemcpyAsync(np, c->d_pts, sizeof(ftkb_point) * c->npts, cudaMemcpyDeviceToDevice, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  cudaFree(c->d_pts);
  c->d_pts = np;
  c->pt_cap = cap;
  return FTKB_OK;
}

static int nbits_of(double resolution) {
  // ref: critical_point_tracker.hh:850-864
  int nbits = (int)std::ceil(std::log2(1.0 / resolution));
  const int minbits = 8, maxbits = 21;
  return std::max(minbits, std::min(nbits, maxbits));
}

// set_coords_bounds / set_coords_rectilinear / set_coords_explicit (regular_tracker.hh:38-40): the coordinates the
// per-simplex test interpolates (simplex_coordinates, critical_point_tracker_2d_regular.hh:494-526, ..._3d_regular.hh:343-379).
// A z-slab takes the whole array's coordinates (its rectilinear z array has slab_global_dim values).
extern "C" int ftkb_set_coords(ftkb_ctx *c, int mode, const double *data, uint64_t n) {
  if (!c || mode < FTKB_COORDS_SIMPLE || mode > FTKB_COORDS_EXPLICIT || (mode != FTKB_COORDS_SIMPLE && !data)) return FTKB_ERR_INVALID;
  CK(cudaSetDevice(c->cfg.device));
  const uint64_t W = c->cfg.dims[0], H = c->cfg.dims[1], D = c->n == 3 ? (c->slab ? c->cfg.slab_global_dim : c->cfg.dims[2]) : 0;
  if (mode == FTKB_COORDS_BOUNDS && n != 2u * c->n) return fail(c, FTKB_ERR_INVALID, "set_coords: bounds take 2 * nd values");
  if (mode == FTKB_COORDS_RECTILINEAR && n != W + H + D) return fail(c, FTKB_ERR_INVALID, "set_coords: rectilinear coordinates take W + H [+ D] values");
  if (mode == FTKB_COORDS_EXPLICIT && (n % (W * H) != 0 || n / (W * H) < (c->n == 3 ? 3u : 2u)))
    return fail(c, FTKB_ERR_INVALID, "set_coords: explicit coordinates are (ncomp, W, H) with ncomp >= nd");
  { const int rc = drain(c); if (rc) return rc; }
  CK(cudaStreamSynchronize(c->stream));
  cudaFree(c->d_coords);
  c->d_coords = nullptr;
  c->coords_mode = mode;
  c->coords_ncomp = mode == FTKB_COORDS_EXPLICIT ? (int)(n / (W * H)) : 0;
  if (mode == FTKB_COORDS_BOUNDS) for (uint64_t k = 0; k < n; k++) c->coords_bounds[k] = data[k];
  if (mode == FTKB_COORDS_RECTILINEAR || mode == FTKB_COORDS_EXPLICIT) {
    CK(cudaMalloc(&c->d_coords, 8 * n));
    CK(cudaMemcpy(c->d_coords, data, 8 * n, cudaMemcpyHostToDevice));
    c->stats.h2d_bytes += 8 * n;
  }
  return FTKB_OK;
}

static void fill_sweep_geometry(const ftkb_ctx *c, SweepParams &p) {
  p.coords_mode = c->coords_mode;
  p.coords_ncomp = c->coords_ncomp;
  for (int k = 0; k < 6; k++) p.coords_bounds[k] = c->coords_bounds[k];
  p.coords = c->d_coords;
  p.nd = c->n;
  p.sm_count = c->sm_count;
  p.W = c->cfg.dims[0]; p.H = c->cfg.dims[1]; p.D = c->n == 3 ? c->cfg.dims[2] : 1;
  p.coords_D = c->slab ? c->cfg.slab_global_dim : p.D;
  for (int j = 0; j < 3; j++) {
    const bool used = j < c->n;
    p.lb[j] = used ? c->cfg.lb[j] : 0;
    p.ub[j] = used ? c->cfg.ub[j] : 0;
    p.nc[j] = p.ub[j] - p.lb[j] + 1;
    p.vmax[j] = p.ub[j];   // vertices outside the domain belong to no valid simplex: keep them out of the cube ranges
    p.voff[j] = 0; p.rank_lb[j] = p.lb[j]; p.rank_nc[j] = p.nc[j];
  }
  if (c->slab) {           // a z-slab of a larger array: ranks / positions / corners in the whole lattice's frame
    p.voff[2] = c->cfg.slab_offset;
    p.rank_lb[2] = c->cfg.slab_global_lb;
    p.rank_nc[2] = c->cfg.slab_global_ub - c->cfg.slab_global_lb + 1;
  }
}

// scalar build kernels: key filter of the layer's min non-zero |v| against the running minimum known now (kernels.h);
// gradient2D scales the differences by W - 1 / H - 1 (grad.hh:24-27), gradient3D halves them (grad.hh:140-144)
static void set_key_filter(const ftkb_ctx *c, SweepParams &p) {
  for (int j = 0; j < 3; j++)
    p.res_thr[j] = res_threshold_key(c->resolution, c->n == 2 ? (double)(c->cfg.dims[j < 2 ? j : 0] - 1) : 0.5);
}

// quantisation factor 2^nbits and the fp32 thresholds of the scans' exclusion test
static void set_factor(SweepParams &p, int nbits) {
  p.nbits = nbits;
  p.factor = (double)(uint64_t)(1 << nbits);
  p.thrp_f = (float)((1.0 / p.factor) * (1.0 + 1.0 / 1048576.0));
  p.thr2_f = (float)(2.0 / p.factor);
  p.lim_f = (float)(0.999 * 4.5e18 / (p.factor * p.factor));
}

// strips x row chunks of the fused 2D scan.  aligned: 16-byte aligned rows, range-cell kernels on CTA tiles of 7 x 62 corner
// columns, 3 CTAs per SM; otherwise the register kernel on strips of 60 corner columns, 2 blocks of 8 warps per SM
static void fused2d_decomposition(const ftkb_ctx *c, SweepParams &p, bool aligned) {
  if (aligned) {
    // just under eight waves of CTAs (costs differ: border strips, cold paths; the last, partly filled wave runs at low occupancy:
    // measured on C2, rows 36 / 45 / 54 / 63 / 90 = 9.8 / 7.8 / 6.5 / 5.6 / 3.9 waves: 0.153 / 0.145 / 0.148 / 0.150 / 0.163 ms),
    // at least two cell blocks per chunk
    const int R = SCAN2D_CELL_ROWS;
    p.nsx = std::max(1, (p.W + 7 * 62 - 1) / (7 * 62));
    const int64_t want = std::max<int64_t>(1, (8 * (int64_t)c->sm_count * 3) / p.nsx);
    p.rows = std::max(2 * R, (int)((p.H + want - 1) / want));
    p.rows = (p.rows + R - 1) / R * R;      // chunks start on cell-block boundaries
    p.rows = std::min(p.rows, 64 * R);      // the key kernel keeps one fail bit per block of a chunk
  } else {    // about two equal waves of warps over the resident slots
    p.nsx = std::max(1, (p.W - 1 + 59) / 60);
    int64_t nsy = (2 * (int64_t)c->sm_count * 2 * 8) / p.nsx;
    nsy = std::max<int64_t>(1, std::min<int64_t>(nsy, (p.H + 31) / 32));
    p.rows = (int)((p.H + nsy - 1) / nsy);
  }
  p.nsy = (p.H + p.rows - 1) / p.rows;
  p.nsz = 1;
}

// tiles x z chunks of the 3D range-cell scans (scalar and vector input)
static void fused3d_decomposition(const ftkb_ctx *c, SweepParams &p) {
  p.nsx = (p.W + F3_STRIDE - 1) / F3_STRIDE;
  p.nsy = (p.H + F3_TROWS - 1) / F3_TROWS;
  const int64_t tiles = (int64_t)p.nsx * p.nsy;
  // two CTAs per SM.  CTA costs differ (edge tiles, cold paths), so aim for about six waves of CTAs and let the
  // hardware scheduler balance them, but keep at least 16 planes per CTA (3 halo planes are re-read per chunk)
  const int64_t slots = 2 * (int64_t)c->sm_count;
  const int64_t nsz = std::max<int64_t>(1, std::min<int64_t>((6 * slots + tiles - 1) / tiles, std::max(1, p.D / 16)));
  p.rows = (int)((p.D + nsz - 1) / nsz);
  p.rows = std::min(p.rows, 63);       // the build kernels keep one fail bit per corner plane of a chunk
  p.nsz = (p.D + p.rows - 1) / p.rows;
}

// vector input, range-cell scan: warps = strips of 62 corner columns x row chunks (2D), tiles x plane chunks (3D)
static void vcells_decomposition(const ftkb_ctx *c, SweepParams &p) {
  if (c->n == 3) { fused3d_decomposition(c, p); return; }
  // two CTAs of 8 warps per SM, about six waves; chunks are multiples of the cell block
  const int R = VSCAN2D_CELL_ROWS;
  p.nsx = std::max(1, (p.W + 61) / 62);
  const int64_t want = std::max<int64_t>(1, (6 * (int64_t)c->sm_count * 16) / p.nsx);
  p.rows = std::max(2 * R, (int)((p.H + want - 1) / want));
  p.rows = (p.rows + R - 1) / R * R;
  p.nsy = (p.H + p.rows - 1) / p.rows;
  p.nsz = 1;
}

static int ensure_cells(ftkb_ctx *c, Layer &l, const SweepParams &p) {
  if (l.cells) return FTKB_OK;
  if (!c->ncells) c->ncells = c->n == 3 ? scan3d_cells_per_layer(p) : (p.fused ? scan2d_cells_per_layer(p) : vscan2d_cells_per_layer(p));
  if (!c->freeCells.empty()) { l.cells = c->freeCells.back(); c->freeCells.pop_back(); return FTKB_OK; }
  CK(cudaMalloc(&l.cells, sizeof(uint4) * c->ncells));
  return FTKB_OK;
}

// a resident layer of the fused 3D path gets its gradient materialised after all (non-finite or huge scalars)
static int materialise_gradient(ftkb_ctx *c, Layer &l) {
  if (l.V || !l.S) return FTKB_OK;
  CK(cudaMemsetAsync(c->d_scalars + l.slot, 0xff, sizeof(unsigned long long), c->stream));
  int rc = take_buffer(c, c->freeV, c->nvert * c->n, &l.V);
  if (rc) return rc;
  l.ownV = true;
  l.cells_valid = false;
  launch_gradient(c->n, l.S, l.V, c->cfg.dims[0], c->cfg.dims[1], c->n == 3 ? c->cfg.dims[2] : 1, c->d_scalars + l.slot, c->stream);
  c->stats.kernel_launches++;
  l.res_pending = false;
  CK(cudaMemcpyAsync(c->h_scalars + l.slot, c->d_scalars + l.slot, sizeof(unsigned long long), cudaMemcpyDeviceToHost, c->stream));
  c->stats.d2h_bytes += 8;
  c->push_d2h_outstanding = true;
  return check_launch(c, "gradient");
}

// The context's input moves down to its slower scan for good (Scans): values the float keys cannot order (NaN, Inf,
// |v| >= 2^1000), no TMA descriptor, or 3D layers of both forms.  Every layer's range cells are dropped, those that came from a
// peer included; in 3D the resident layers get their gradient materialised instead.
static int fall_back(ftkb_ctx *c) {
  switch (c->scans) {
    case Scans::keys2d: c->scans = Scans::f32_2d; break;
    case Scans::fused3d: c->scans = Scans::gradient3d; break;
    case Scans::vcells: c->scans = Scans::twolayer; break;
    default: break;
  }
  if (c->scans != Scans::gradient3d) {
    for (Layer &l : c->layers) l.cells_valid = false;
    return FTKB_OK;
  }
  for (Layer &l : c->layers) {
    const int rc = materialise_gradient(c, l);
    if (rc) return rc;
  }
  CK(cudaStreamSynchronize(c->stream));
  return FTKB_OK;
}

static bool rows_aligned16(const ftkb_ctx *c, const double *a, const double *b) {
  return (c->cfg.dims[0] % 2 == 0) && aligned16(a) && (!b || aligned16(b));
}

// The scan of a sweep over layers l0, l1 (l1 == l0 without a next layer).  launch is the kernel family's launcher; cells: a
// range-cell scan, whose layers keep their cells from one step to the next.
struct Scan {
  void (*launch)(const SweepParams &, cudaStream_t);
  bool cells;
};

// Chooses the scan from the context's Scans and the two layers, and sets p.fused, p.keys2d, the TMA descriptors and the grid
// decomposition.  Choices that depend on the layers hold for this sweep only: misaligned 2D rows take the register kernel,
// a misaligned vector layer the two-layer scan.  launch == nullptr: the fused 3D scan has no TMA descriptor (driver entry
// point or alignment) for a layer, and the context has to fall back before it sweeps.
static Scan choose_scan(const ftkb_ctx *c, const Layer &l0, const Layer &l1, SweepParams &p) {
  p.fused = derives_vectors(c, l0);
  if (p.fused && c->n == 3) {
    if (!encode_scalar_tmap3d(l0.S, p.W, p.H, p.D, &p.tmap[0]) || !encode_scalar_tmap3d(l1.S, p.W, p.H, p.D, &p.tmap[1])) return {nullptr, false};
    fused3d_decomposition(c, p);
    return {launch_scan3d_cells, true};
  }
  if (p.fused) {
    const bool aligned = rows_aligned16(c, l0.S, l1.S);    // the range-cell kernels need 16-byte aligned rows
    fused2d_decomposition(c, p, aligned);
    p.keys2d = c->scans == Scans::keys2d;
    return {aligned ? launch_scan2d_cells : launch_scan, aligned};
  }
  if (l0.V && l1.V && scan_resolves(c, l0) && scan_resolves(c, l1)) {
    vcells_decomposition(c, p);
    return {launch_vscan_cells, true};
  }
  // two-layer scans of vector layers: strips of 31 corners x 64 rows (2D) / x 15 rows x 32 planes (3D)
  p.nsx = (p.nc[0] + 30) / 31;
  if (c->n == 2) {
    p.rows = 64;
    p.nsy = (p.nc[1] + p.rows - 1) / p.rows;
    p.nsz = 1;
  } else {
    p.rows = 32;
    p.nsy = (p.nc[1] + 14) / 15;
    p.nsz = (p.nc[2] + p.rows - 1) / p.rows;
  }
  return {launch_scan, false};
}

// what every sweep over l0, l1 shares (the quantisation factor, the key filter and the buffers aside), and its scan
static Scan sweep_setup(const ftkb_ctx *c, const Layer &l0, const Layer &l1, bool has_next, SweepParams &p) {
  fill_sweep_geometry(c, p);
  p.t = c->current_timestep;
  p.has_next = has_next;
  p.no_filter = (c->n == 3 && !c->cfg.robust_detection);
  p.scalar_source = l0.S ? c->cfg.scalar_source : FTKB_SOURCE_NONE;
  p.jacobian_source = c->cfg.jacobian_source;
  p.jacobian_symmetric = c->cfg.jacobian_symmetric;
  // 2D: jacobian2D<double,true> on the scalar path, <double,false> when the vector field was pushed
  p.derived_symmetric = c->cfg.vector_source == FTKB_SOURCE_DERIVED;
  p.robust = c->cfg.robust_detection;
  p.compute_degrees = c->cfg.compute_degrees;
  p.use_type_filter = c->cfg.use_type_filter;
  p.type_filter = c->cfg.type_filter;
  p.L[0] = {l0.S, l0.V, l0.J};
  p.L[1] = {l1.S, l1.V, l1.J};
  p.poison = c->d_scalars + ftkb_ctx::SLOT_POISON;
  p.wl_count = c->d_scalars + ftkb_ctx::SLOT_WL;
  p.pt_count = c->d_scalars + ftkb_ctx::SLOT_PT;
  p.ticket = c->d_scalars + ftkb_ctx::SLOT_TICKET;
  return choose_scan(c, l0, l1, p);
}

// min non-zero |v| of a layer that no sweep has streamed yet, outside a sweep (time-slab halos, z-slab groups, vector layers
// pushed further ahead than the sweep reads): the layer's own scan streams it once -- its range cells and min |v| -- and tests
// no cube
static int resolve_pending(ftkb_ctx *c, Layer &l) {
  const bool vector_input = l.V != nullptr;
  c->primed = false;
  CK(cudaMemsetAsync(c->d_scalars + l.slot, 0xff, sizeof(unsigned long long), c->stream));   // (a pending layer's device slot is reset lazily)
  SweepParams p{};
  const Scan s = sweep_setup(c, l, l, false, p);
  if (!s.launch) return fall_back(c);        // the materialised gradient brings the layer's min |v|
  if (vector_input && (!s.cells || l.cells_valid)) {
    l.res_pending = false;
    return queue_resolution(c, l, false);
  }
  set_key_filter(c, p);
  p.keys2d = 0;                              // 2D: the fp32-range build, which orders every value (no poison flag to read back)
  p.nbits = vector_input ? (c->nbits ? c->nbits : 8) : (c->n == 3 ? 8 : 0);
  if (!vector_input) { p.thrp_f = 1.f; p.thr2_f = 1.f; p.lim_f = 0.f; }
  p.res_slot[0] = c->d_scalars + l.slot;
  p.wl = c->d_wl; p.wl_cap = 0;
  if (s.cells) {
    // the build keeps the real domain: the cells need its masks
    const int rc = ensure_cells(c, l, p);
    if (rc) return rc;
    p.sum_mode = SUM_BUILD; p.build_layer = 0; p.sum_out = l.cells;
  } else {
    p.lb[1] = 1; p.ub[1] = 0;                // the register kernel over an empty domain: gradient and min |v| only
  }
  const bool keyed = vector_input || c->n == 3;   // the key scans raise the poison flag
  if (keyed) CK(cudaMemsetAsync(p.poison, 0, sizeof(unsigned long long), c->stream));
  s.launch(p, c->stream);
  c->stats.kernel_launches++;
  CK(cudaMemcpyAsync(c->h_scalars + l.slot, c->d_scalars + l.slot, sizeof(unsigned long long), cudaMemcpyDeviceToHost, c->stream));
  if (keyed) CK(cudaMemcpyAsync(c->h_scalars + ftkb_ctx::SLOT_POISON, p.poison, sizeof(unsigned long long), cudaMemcpyDeviceToHost, c->stream));
  c->stats.d2h_bytes += keyed ? 16 : 8;
  int rc = check_launch(c, "resolution (scan)");
  if (rc) return rc;
  if (!keyed) {
    l.cells_valid = l.cells_valid || s.cells;
    l.res_pending = false;
    c->push_d2h_outstanding = true;
    return FTKB_OK;
  }
  CK(cudaStreamSynchronize(c->stream));
  if (!c->h_scalars[ftkb_ctx::SLOT_POISON]) {
    l.cells_valid = true;
    l.res_pending = false;
    return FTKB_OK;
  }
  // values the float keys cannot order: a 3D scalar layer gets its gradient (and with it its min |v|), a vector layer the
  // plain resolution pass
  if ((rc = fall_back(c)) || !vector_input) return rc;
  CK(cudaMemsetAsync(c->d_scalars + l.slot, 0xff, sizeof(unsigned long long), c->stream));
  l.res_pending = false;
  return queue_resolution(c, l, false);
}

// ref: critical_point_tracker_{2d,3d}_regular::update_timestep (xl == NONE branch)
// grow(), critical_point_tracker_2d_regular.hh:288-329 / ..._3d_regular.hh:173-200: the punctured simplices found since
// the last grow step (the reference clears discrete_critical_points after each) go to the host-side online tracer
static int wait_grow(ftkb_ctx *c) {
  return c->grow_failed ? FTKB_ERR_NOMEM : FTKB_OK;
}

// one grow step over d_pts[grown .. end), the batch of timestep t
static int grow_trajectories(ftkb_ctx *c, uint64_t end, int t) {
  const uint64_t n = end - c->grown;
  if (n >= 0xffffffffull) return fail(c, FTKB_ERR_OVERFLOW, "more than 2^32 punctured simplices in one step");
  { const int rc = wait_grow(c); if (rc) return rc; }
  // The device prepares the batch: element keys -> radix sort -> unique -> for every element the batch indices of its punctured
  // neighbours, itself included (the same binary search as the offline trace).  The host walk then only chases index lists
  // (OnlineTracer::grow_sorted).
  // staging: {keys, nine neighbour indices, count} per element -- the records themselves stay on the device: finalize maps the
  // trajectories' keys onto the sorted points
  const size_t per = 8 + 4 * 9 + 1;
  if (n && c->grow_stage_cap < per * n) {
    if (c->grow_stage) cudaFreeHost(c->grow_stage);
    c->grow_stage = nullptr; c->grow_stage_cap = 0;
    const size_t want = per * (n + n / 2 + 1024);
    if (cudaMallocHost(&c->grow_stage, want) != cudaSuccess) { cudaGetLastError(); return fail(c, FTKB_ERR_NOMEM, "streaming grow step: out of page-locked memory"); }
    c->grow_stage_cap = want;
  }
  uint64_t *h_keys = (uint64_t *)c->grow_stage;
  uint32_t *h_nb = (uint32_t *)(h_keys + n);
  uint8_t *h_cnt = (uint8_t *)(h_nb + 9 * n);
  uint64_t nu = n;
  if (n) {
    TraceParams tp{};
    fill_trace_params(c, tp);
    unsigned long long *k0 = nullptr, *k1 = nullptr;
    uint32_t *i0 = nullptr, *i1 = nullptr, *d_nb = nullptr;
    uint8_t *d_cnt = nullptr;
    void *temp = nullptr;
    unsigned long long *d_nu = c->d_scalars + ftkb_ctx::SLOT_UQ;
    { int rs = scratch(c, 0, 8 * n, (void **)&k0); if (!rs) rs = scratch(c, 1, 8 * n, (void **)&k1); if (!rs) rs = scratch(c, 2, 4 * n, (void **)&i0);
      if (!rs) rs = scratch(c, 3, 4 * n, (void **)&i1);
      if (!rs) rs = scratch(c, 10, 4 * 9 * n, (void **)&d_nb); if (!rs) rs = scratch(c, 11, n, (void **)&d_cnt); if (rs) return rs; }
    CK(cudaEventRecord(c->ev[0], c->stream));
    launch_point_keys(c->d_pts + c->grown, n, tp, k0, i0, c->stream);
    const size_t tb = std::max(sort_pairs_u64(nullptr, 0, k0, k1, i0, i1, n, c->stream), unique_by_key_u64(nullptr, 0, k1, i1, k0, i0, d_nu, n, c->stream));
    { const int rs = scratch(c, 4, tb, &temp); if (rs) return rs; }
    sort_pairs_u64(temp, tb, k0, k1, i0, i1, n, c->stream);
    unique_by_key_u64(temp, tb, k1, i1, k0, i0, d_nu, n, c->stream);
    tp.keys = k0;
    launch_batch_neighbors(tp, d_nu, n, c->d_pts + c->grown, i0, nullptr, d_nb, d_cnt, c->stream);
    CK(cudaEventRecord(c->ev[1], c->stream));
    CK(cudaMemcpyAsync(c->h_scalars + ftkb_ctx::SLOT_UQ, d_nu, 8, cudaMemcpyDeviceToHost, c->stream));
    CK(cudaMemcpyAsync(h_keys, k0, 8 * n, cudaMemcpyDeviceToHost, c->stream));
    CK(cudaMemcpyAsync(h_nb, d_nb, 4 * 9 * n, cudaMemcpyDeviceToHost, c->stream));
    CK(cudaMemcpyAsync(h_cnt, d_cnt, n, cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    { const int rc = check_launch(c, "streaming grow step (batch preparation)"); if (rc) return rc; }
    nu = c->h_scalars[ftkb_ctx::SLOT_UQ];
    float ms = 0;
    CK(cudaEventElapsedTime(&ms, c->ev[0], c->ev[1]));
    c->stats.ms_finalize_device += ms;
    c->stats.kernel_launches += 4;
    c->stats.d2h_bytes += per * n + 8;
  }
  try {
    const auto t0 = std::chrono::steady_clock::now();
    if (n) c->online->grow_sorted(nullptr, h_keys, (uint32_t)nu, h_nb, h_cnt);
    else c->online->grow(nullptr, 0);
    c->stats.ms_finalize_host += std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
  }
  catch (const std::bad_alloc &) { c->grow_failed = true; return fail(c, FTKB_ERR_NOMEM, "streaming grow step: out of memory (trajectories are incomplete)"); }
  catch (const std::exception &e) { c->grow_failed = true; return fail(c, FTKB_ERR_INVALID, std::string("streaming grow step: ") + e.what()); }
  c->grown = end;
  c->grown_through = t;
  c->traced = false;
  return FTKB_OK;
}

// a streaming context that sweeps nothing itself (the merged context of a device group, include/ftkb200.h): one grow step over
// the imported points that follow those grown so far, the batch of timestep t
int ftkb::grow_imported(ftkb_ctx *c, int t) {
  if (!c || !c->streaming) return FTKB_ERR_INVALID;
  CK(cudaSetDevice(c->cfg.device));
  return grow_trajectories(c, c->npts, t);
}

// the sweep of timestep t has been confirmed with d_pts[begin, end) as its points (a second sweep of the same timestep appends)
static void record_step(ftkb_ctx *c, int t, uint64_t begin, uint64_t end, bool interval) {
  const size_t k = (size_t)(t - c->cfg.start_timestep);
  if (k >= c->steps.size()) {
    c->steps.resize(k + 1);
    c->steps[k].begin = begin;
  }
  c->steps[k].end = end;
  c->steps[k].interval = c->steps[k].interval || interval;
}

int ftkb::confirmed_through(const ftkb_ctx *c) { return c->cfg.start_timestep + (int)c->steps.size() - 1; }

int ftkb::import_step(ftkb_ctx *dst, ftkb_ctx *src, int t, bool *interval) {
  const size_t k = (size_t)(t - src->cfg.start_timestep);
  if (!dst->streaming || t < src->cfg.start_timestep || k >= src->steps.size())
    return fail(dst, FTKB_ERR_INVALID, "import_step: timestep " + std::to_string(t) + " has no confirmed sweep");
  ftkb_ctx *c = dst;        // (CK reports to c)
  const ftkb_ctx::StepRange r = src->steps[k];
  *interval = r.interval;
  const uint64_t n = r.end - r.begin;
  if (!n) return FTKB_OK;
  const int dd = dst->cfg.device, sd = src->cfg.device;
  if (!src->retired_pts.empty()) {
    // the source's point buffer was replaced while steps were in flight: its confirmed points reach the new buffer by a copy
    // queued on its stream
    CK(cudaSetDevice(sd));
    CK(cudaEventRecord(src->ev[3], src->stream));
    CK(cudaSetDevice(dd));
    CK(cudaStreamWaitEvent(dst->stream, src->ev[3], 0));
  }
  CK(cudaSetDevice(dd));
  if (dst->npts + n > dst->pt_cap) {
    const int rc = grow_points(dst, dst->npts + n);
    if (rc) return rc;
  }
  if (dd == sd) {
    CK(cudaMemcpyAsync(dst->d_pts + dst->npts, src->d_pts + r.begin, sizeof(ftkb_point) * n, cudaMemcpyDeviceToDevice, dst->stream));
  } else {
    CK(enable_peer_access(dd, sd));
    CK(cudaMemcpyPeerAsync(dst->d_pts + dst->npts, dd, src->d_pts + r.begin, sd, sizeof(ftkb_point) * n, dst->stream));
  }
  // complete before the source's owner may move its buffer again
  CK(cudaStreamSynchronize(dst->stream));
  dst->npts += n;
  dst->stats.points = dst->npts;
  dst->sorted = false;
  dst->traced = false;
  return FTKB_OK;
}

extern "C" int ftkb_set_streaming_trajectories(ftkb_ctx *c, int enable) {
  if (!c) return FTKB_ERR_INVALID;
  if (c->stats.scan_launches || c->npts) return fail(c, FTKB_ERR_INVALID, "set_streaming_trajectories: call it before the first update_timestep");
  if (c->slab && enable) return fail(c, FTKB_ERR_INVALID, "set_streaming_trajectories: not available on a spatial slab");
  c->streaming = enable != 0;
  c->grow_failed = false;
  c->online.reset(c->streaming ? new ftkb::OnlineTracer(c->n, c->cfg.lb, c->cfg.ub) : nullptr);
  c->grown = 0;
  c->grown_through = c->cfg.start_timestep - 1;
  return FTKB_OK;
}

// ---- deferred steps: confirmation, replay ------------------------------------------------------------------------
static int update_impl(ftkb_ctx *c, bool allow_defer);

static void absorb_resolutions(ftkb_ctx *c, const ftkb_ctx::Pending &pd) {
  const volatile unsigned long long *r = c->h_ring + 8 * pd.ring;
  if (r[5] != pd.seq) return;
  for (int k = 0; k < 2; k++)
    if (pd.res_slots[k] >= 0) {
      c->h_scalars[pd.res_slots[k]] = r[3 + k];
      c->resolution = std::min(c->resolution, slot_value(c, pd.res_slots[k]));
    }
}

// the oldest enqueued step failed (a buffer overflowed, or the scan met values its keys cannot order): everything that
// was enqueued is discarded and redone synchronously, with the popped layers put back for the duration
static int replay(ftkb_ctx *c, bool poison) {
  CK(cudaStreamSynchronize(c->stream));
  CK(cudaStreamSynchronize(c->stream2));
  for (const auto &pd : c->pend) absorb_resolutions(c, pd);      // a scan's min |v| is valid whatever happened to the counters
  std::vector<int> pops;
  for (const auto &pd : c->pend) pops.push_back(pd.pops);
  const uint64_t npts0 = c->pend.front().npts_before;
  c->pend.clear();
  c->primed = false;
  while (!c->limbo.empty()) {
    c->layers.push_front(c->limbo.back());
    c->limbo.pop_back();
    c->current_timestep--;
  }
  c->npts = npts0;
  c->stats.points = npts0;
  c->sorted = false;
  c->traced = false;
  if (poison) {
    const int rc = fall_back(c);
    if (rc) return rc;
  }
  c->stats.sweeps_repeated += pops.size();
  for (size_t i = 0; i < pops.size(); i++) {
    const int rc = update_impl(c, false);
    if (rc) return rc;
    for (int j = 0; j < pops[i] && !c->layers.empty(); j++) {
      release_layer(c, c->layers.front());
      c->layers.pop_front();
      c->current_timestep++;
    }
  }
  return FTKB_OK;
}

static int confirm_front(ftkb_ctx *c) {
  const ftkb_ctx::Pending pd = c->pend.front();
  const auto tw0 = std::chrono::steady_clock::now();
  CK(cudaEventSynchronize(c->dev[pd.evset][2]));
  if (c->debug_timing) { c->host_wait_us += std::chrono::duration<double, std::micro>(std::chrono::steady_clock::now() - tw0).count(); c->host_wait_n++; }
  const volatile unsigned long long *r = c->h_ring + 8 * pd.ring;
  if (r[5] != pd.seq) return fail(c, FTKB_ERR_CUDA, "deferred step: the test kernel did not publish its counters");
  const uint64_t nwl = r[0], npt = r[1];
  const bool poison = r[2] != 0;
  c->stats.d2h_bytes += 48;
  absorb_resolutions(c, pd);
  // the step ran with the factor known when it was enqueued; the layers it resolved may have lowered the running minimum
  // (critical_point_tracker.hh:850-864) -- then it, and whatever was enqueued behind it, is redone with the right factor
  const bool stale = nbits_of(c->resolution) != pd.nbits;
  if (poison || stale || nwl > c->wl_cap || npt > pd.pt_cap) return replay(c, poison);
  c->nbits = pd.nbits;
  c->factor = (double)(uint64_t)(1 << pd.nbits);
  float ms_scan = 0, ms_test = 0;
  CK(cudaEventElapsedTime(&ms_scan, c->dev[pd.evset][0], c->dev[pd.evset][1]));
  CK(cudaEventElapsedTime(&ms_test, c->dev[pd.evset][1], c->dev[pd.evset][2]));
  c->stats.ms_scan += ms_scan; c->stats.ms_test += ms_test; c->stats.last_ms_scan = ms_scan;
  if (c->debug_timing) {
    // timeline of the deferred steps (diagnostic, FTKB_DEBUG_TIMING=1): scan start / scan end / test end relative to the
    // previous confirmed step's scan end
    float s0 = 0, s1 = 0, s2 = 0;
    if (c->dbg_prev_valid && cudaEventElapsedTime(&s0, c->dbg_prev, c->dev[pd.evset][0]) == cudaSuccess &&
        cudaEventElapsedTime(&s1, c->dbg_prev, c->dev[pd.evset][1]) == cudaSuccess && cudaEventElapsedTime(&s2, c->dbg_prev, c->dev[pd.evset][2]) == cudaSuccess) {
      c->gaps.push_back(s0);
      c->tl_scan_end.push_back(s1);
      c->tl_test_end.push_back(s2);
    } else cudaGetLastError();
    // keep this step's scan-end time in an event of its own (the per-step events are re-recorded two steps later)
    std::swap(c->dbg_prev, c->dev[pd.evset][1]);
    c->dbg_prev_valid = true;
  }
  c->stats.scan_launches++;
  c->stats.cells_scanned += c->ncore;
  c->stats.cells_refined += nwl;
  c->last_wl = nwl;
  c->last_wl_sel = pd.wl_sel;
  c->wl_hint = nwl;
  c->stats.simplices_tested += c->ncore * (uint64_t)(c->n_ord + (pd.has_next ? c->n_int : 0));
  if (npt != c->npts) { c->sorted = false; c->traced = false; }
  if (npt > c->npts) c->max_step_points = std::max(c->max_step_points, npt - c->npts);
  record_step(c, pd.timestep, pd.npts_before, npt, pd.has_next);
  c->npts = npt;
  c->stats.points = npt;
  for (int j = 0; j < pd.pops && !c->limbo.empty(); j++) {
    release_layer(c, c->limbo.front());
    c->limbo.pop_front();
  }
  c->pend.pop_front();
  if (!c->pend.empty()) c->pend.front().npts_before = c->npts;
  return FTKB_OK;
}

// confirm every enqueued step (any call that needs results, or that touches the stream's state, starts here)
static int drain(ftkb_ctx *c) {
  while (!c->pend.empty()) {
    const int rc = confirm_front(c);
    if (rc) return rc;
  }
  if (!c->retired_pts.empty()) {
    CK(cudaStreamSynchronize(c->stream));          // the copy out of a retired buffer is stream-ordered
    for (ftkb_point *q : c->retired_pts) cudaFree(q);
    c->retired_pts.clear();
  }
  return FTKB_OK;
}

// Deferred steps: grow the point buffer BEFORE a step can overflow it -- an overflow is only noticed one step later and costs a
// drain and a replay of everything in flight.  The steps in flight keep the old buffer; the copy into the new one is ordered
// behind their test kernels, the old buffer is freed at the next drain (cudaFree would synchronise the device here).
static int grow_points_ahead(ftkb_ctx *c) {
  const uint64_t per = c->max_step_points;
  if (!per) return FTKB_OK;
  const uint64_t need = c->npts + (c->pend.size() + 2) * (per + per / 2);
  if (need <= c->pt_cap) return FTKB_OK;
  uint64_t cap = 4 * c->pt_cap;                      // in big steps: every growth costs a cudaMalloc in the middle of the step loop
  while (cap < need) cap *= 2;
  if (cap >= 0xffffffffull) return FTKB_OK;          // (the overflow path reports it)
  ftkb_point *np = nullptr;
  if (cudaMalloc(&np, sizeof(ftkb_point) * cap) != cudaSuccess) { cudaGetLastError(); return FTKB_OK; }   // the overflow path will say so if it matters
  if (!c->pend.empty()) CK(cudaStreamWaitEvent(c->stream, c->dev[c->pend.back().evset][2], 0));
  CK(cudaMemcpyAsync(np, c->d_pts, sizeof(ftkb_point) * c->pt_cap, cudaMemcpyDeviceToDevice, c->stream));
  c->retired_pts.push_back(c->d_pts);
  c->d_pts = np;
  c->pt_cap = cap;
  return FTKB_OK;
}

static int test_grid(const ftkb_ctx *c) {
  const uint64_t cpb = c->n == 2 ? 10 : 2;           // cubes per block and round of test_kernel
  const uint64_t want = (c->wl_hint * 2 + 256 + cpb - 1) / cpb;
  return (int)std::max<uint64_t>(8, std::min<uint64_t>(want, (uint64_t)c->sm_count * 8));
}

extern "C" int ftkb_update_timestep(ftkb_ctx *c) {
  if (!c) return FTKB_ERR_INVALID;
  return update_impl(c, c->defer);
}

// arm the device counters from the host mirror; the same copy resets the resolution slots whose mirror is all ones
static int arm_counters(ftkb_ctx *c) {
  for (int k : {ftkb_ctx::SLOT_WL, ftkb_ctx::SLOT_WL2, ftkb_ctx::SLOT_UQ, ftkb_ctx::SLOT_POISON, ftkb_ctx::SLOT_POISON2, ftkb_ctx::SLOT_TICKET})
    c->h_scalars[k] = 0;
  c->h_scalars[ftkb_ctx::SLOT_PT] = c->npts;
  CK(cudaMemcpyAsync(c->d_scalars, c->h_scalars, 15 * sizeof(unsigned long long), cudaMemcpyHostToDevice, c->stream));
  return FTKB_OK;
}

// One sweep: the scan between ev[0] and ev[1] on the context's stream, then the exact test up to ev[2] on stream ts, behind
// test_after as well if that is given.  A range-cell scan streams each layer once (the step that first sees it) and reads
// its cells after that; the very first step streams both layers.
static int launch_sweep(ftkb_ctx *c, const Scan &s, SweepParams &p, Layer &l0, Layer &l1, cudaEvent_t *ev, cudaStream_t ts,
                        cudaEvent_t test_after) {
  CK(cudaEventRecord(ev[0], c->stream));
  if (!s.cells) {
    s.launch(p, c->stream);
  } else if (!l0.cells_valid) {
    p.sum_in[0] = l0.cells; p.sum_in[1] = l1.cells;
    p.sum_mode = p.has_next ? SUM_BUILD : SUM_BUILD_TEST1; p.build_layer = 0; p.sum_out = l0.cells;
    s.launch(p, c->stream);
    l0.cells_valid = true;
    if (p.has_next) {
      c->stats.kernel_launches++;
      p.sum_mode = l1.cells_valid ? SUM_TEST2 : SUM_BUILD_TEST2; p.build_layer = 1; p.sum_out = l1.cells;
      s.launch(p, c->stream);
      l1.cells_valid = true;
    }
  } else {
    p.sum_in[0] = l0.cells; p.sum_in[1] = l1.cells;
    if (p.has_next && !l1.cells_valid) {
      p.sum_mode = SUM_BUILD_TEST2; p.build_layer = 1; p.sum_out = l1.cells;
      l1.cells_valid = true;
    } else {
      p.sum_mode = p.has_next ? SUM_TEST2 : SUM_TEST1;
    }
    s.launch(p, c->stream);
  }
  CK(cudaEventRecord(ev[1], c->stream));
  if (test_after) CK(cudaStreamWaitEvent(c->stream, test_after, 0));
  if (ts != c->stream) CK(cudaStreamWaitEvent(ts, ev[1], 0));
  launch_test(p, ts);
  CK(cudaEventRecord(ev[2], ts));
  c->stats.kernel_launches += 2;
  return check_launch(c, "sweep");
}

// ---- deferred step: enqueue and return; the previous one is confirmed behind it ------------------------------------
static int enqueue_step(ftkb_ctx *c, const Scan &s, SweepParams &p, Layer &l0, Layer &l1, int nbits) {
  const bool has_next = p.has_next;
  if (has_next && !l1.cells) {
    // (an empty pool means one more buffer: with a step in flight four layers hold cells -- the one in limbo, the two being
    // swept and the one being built; confirming the step in flight first would serialise the steps again)
    const int rc0 = ensure_cells(c, l1, p);
    if (rc0) return rc0;
  }
  set_factor(p, nbits);
  p.test_blocks = test_grid(c);
  const auto te0 = std::chrono::steady_clock::now();
  ftkb_ctx::Pending pd;
  pd.seq = ++c->step_seq;
  pd.ring = (int)(pd.seq % ftkb_ctx::RING);
  pd.evset = (int)(pd.seq & 1);
  pd.has_next = has_next;
  pd.nbits = nbits;
  pd.npts_before = c->npts;                 // exact for the oldest enqueued step (set again when it becomes the oldest)
  pd.timestep = c->current_timestep;
  Layer *lay[2] = {&l0, &l1};
  for (int k = 0; k < (has_next ? 2 : 1); k++)
    if (lay[k]->res_pending) {
      p.res_slot[k] = c->d_scalars + lay[k]->slot;
      pd.res_slots[k] = lay[k]->slot;
      lay[k]->res_pending = false;          // this scan produces it; the value reaches the host at confirmation
    }
  pd.wl_sel = c->wl_sel;
  p.wl = c->wl_sel ? c->d_wl2 : c->d_wl; p.wl_cap = c->wl_cap;
  { const int rcg = grow_points_ahead(c); if (rcg) return rcg; }
  p.pts = c->d_pts; p.pt_cap = c->pt_cap;
  pd.pt_cap = c->pt_cap;
  // worklist, its counter and the poison flag alternate between two sets: the test kernel of this step may still run
  // (on stream2) while the scan of the next step fills the other set; each test kernel re-arms its own set when done
  p.wl_count = c->d_scalars + (c->wl_sel ? ftkb_ctx::SLOT_WL2 : ftkb_ctx::SLOT_WL);
  p.poison = c->d_scalars + (c->wl_sel ? ftkb_ctx::SLOT_POISON2 : ftkb_ctx::SLOT_POISON);
  p.step_out = c->h_ring + 8 * pd.ring;     // pinned + mapped, unified addressing: the device writes it in place
  p.step_seq = pd.seq;
  // resolution slots are handed out in push order: the layer the scan of step k+1 / k+2 resolves sits 2 / 3 places
  // behind the current front, resident already or still to be pushed.  This step's test kernel re-arms the slot for
  // step k+2 (step k+1's scan may already be running by then; its slot was re-armed by the previous test kernel).
  auto slot_at = [&](size_t idx) { return idx < c->layers.size() ? c->layers[idx].slot : (int)((c->next_slot + (idx - c->layers.size())) % 8); };
  p.res_reset = c->d_scalars + slot_at(3);
  if (!c->primed) {
    // first deferred step after a synchronous one: arm the device counters once
    if (c->layers.size() < 3) c->h_scalars[slot_at(2)] = ~0ull;      // the layer the next step's scan resolves (not pushed yet)
    const int rc = arm_counters(c);
    if (rc) return rc;
  }
  // a test kernel with a GPU's worth of work (feature-dense fields: 1e5 .. 1e6 surviving cubes) gains nothing next to the
  // following scan -- the two take turns on the SMs, measured 0.90 .. 1.64 ms per step against 0.95 in a row -- so only
  // the small, latency-bound ones go to the second stream
  const bool overlap = c->wl_hint < 100000;
  // test kernels share one ticket counter: never two at once
  const cudaEvent_t test_after = !overlap && c->last_test_overlapped && !c->pend.empty() ? c->dev[c->pend.back().evset][2] : nullptr;
  c->last_test_overlapped = overlap;
  const int rc = launch_sweep(c, s, p, l0, l1, c->dev[pd.evset], overlap ? c->stream2 : c->stream, test_after);
  if (rc) return rc;
  c->pend.push_back(pd);
  c->primed = true;
  c->wl_sel ^= 1;
  if (c->debug_timing) { c->host_enq_us += std::chrono::duration<double, std::micro>(std::chrono::steady_clock::now() - te0).count(); c->host_enq_n++; }
  while (c->pend.size() > 1) {
    const int rc2 = confirm_front(c);
    if (rc2) return rc2;
  }
  return FTKB_OK;
}

// ---- synchronous step: confirmed before it returns; redone until the factor is right and the buffers were big enough --
static int sync_step(ftkb_ctx *c, const Scan &s, SweepParams &p, Layer &l0, Layer &l1, int nbits) {
  { const int rc = drain(c); if (rc) return rc; }
  c->primed = false;
  const bool has_next = p.has_next;
  Layer *lay[2] = {&l0, &l1};
  for (int attempt = 0; attempt < 12; attempt++) {
    set_factor(p, nbits);
    p.res_slot[0] = p.res_slot[1] = nullptr;
    bool pending = false;
    if (p.fused || s.cells)
      for (int k = 0; k < (has_next ? 2 : 1); k++)
        if (lay[k]->res_pending) { p.res_slot[k] = c->d_scalars + lay[k]->slot; pending = true; }
    p.wl = c->d_wl; p.wl_cap = c->wl_cap;
    p.pts = c->d_pts; p.pt_cap = c->pt_cap;
    p.test_blocks = test_grid(c);
    int rc = arm_counters(c);
    if (!rc && s.cells) rc = ensure_cells(c, l0, p);
    if (!rc && s.cells && has_next) rc = ensure_cells(c, l1, p);
    if (!rc) rc = launch_sweep(c, s, p, l0, l1, c->ev, c->stream, nullptr);
    if (rc) return rc;
    if (pending) {   // slots 0..7 hold the per-layer resolutions, 8..11 the counters: one copy
      CK(cudaMemcpyAsync(c->h_scalars, c->d_scalars, 12 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, c->stream));
      c->stats.d2h_bytes += 64;
    } else {
      CK(cudaMemcpyAsync(c->h_scalars + ftkb_ctx::SLOT_WL, c->d_scalars + ftkb_ctx::SLOT_WL, 32, cudaMemcpyDeviceToHost, c->stream));
    }
    CK(cudaStreamSynchronize(c->stream));
    c->stats.d2h_bytes += 32;
    if ((p.fused || s.cells) && c->h_scalars[ftkb_ctx::SLOT_POISON]) {
      // a value the scan's float keys cannot order (NaN / Inf / >= 2^1000): redo the step with the slower scan
      c->stats.sweeps_repeated++;
      const int rc2 = fall_back(c);
      return rc2 ? rc2 : update_impl(c, false);
    }
    float ms_scan = 0, ms_test = 0;
    CK(cudaEventElapsedTime(&ms_scan, c->ev[0], c->ev[1]));
    CK(cudaEventElapsedTime(&ms_test, c->ev[1], c->ev[2]));
    c->stats.ms_scan += ms_scan; c->stats.ms_test += ms_test; c->stats.last_ms_scan = ms_scan;
    c->stats.scan_launches++;
    if (pending) {
      for (int k = 0; k < (has_next ? 2 : 1); k++)
        if (lay[k]->res_pending) {
          lay[k]->res_pending = false;
          c->resolution = std::min(c->resolution, slot_value(c, lay[k]->slot));
        }
      const int nb = nbits_of(c->resolution);
      if (nb != nbits) {           // the speculated factor was stale: repeat the sweep with the right one
        nbits = nb;
        c->stats.sweeps_repeated++;
        continue;
      }
    }
    const uint64_t nwl = c->h_scalars[ftkb_ctx::SLOT_WL], npt = c->h_scalars[ftkb_ctx::SLOT_PT];
    c->wl_hint = std::min<uint64_t>(nwl, c->wl_cap);
    if (nwl > c->wl_cap) {           // worklist overflow: grow and redo the step (inputs are still resident)
      cudaFree(c->d_wl); cudaFree(c->d_wl2);
      c->d_wl = c->d_wl2 = nullptr;
      c->wl_cap = nwl + nwl / 8 + 1024;
      CK(cudaMalloc(&c->d_wl, sizeof(unsigned long long) * c->wl_cap));
      CK(cudaMalloc(&c->d_wl2, sizeof(unsigned long long) * c->wl_cap));
      c->wl_hint = nwl;
      c->stats.sweeps_repeated++;
      continue;
    }
    if (npt > c->pt_cap) {
      int rc2 = grow_points(c, npt);
      if (rc2) return rc2;
      c->stats.sweeps_repeated++;
      continue;
    }
    c->nbits = nbits;
    c->factor = p.factor;
    c->stats.cells_scanned += c->ncore;
    c->stats.cells_refined += nwl;
    c->last_wl = nwl;
    c->last_wl_sel = 0;
    c->stats.simplices_tested += c->ncore * (uint64_t)(c->n_ord + (has_next ? c->n_int : 0));
    if (npt != c->npts) { c->sorted = false; c->traced = false; }
    record_step(c, c->current_timestep, c->npts, npt, has_next);
    c->npts = npt;
    c->stats.points = npt;
    if (c->streaming && has_next) { const int rc2 = grow_trajectories(c, c->npts, c->current_timestep); if (rc2) return rc2; }
    return FTKB_OK;
  }
  return fail(c, FTKB_ERR_CUDA, "update_timestep: buffers kept overflowing");
}

static int update_impl(ftkb_ctx *c, bool allow_defer) {
  if (c->layers.empty()) return fail(c, FTKB_ERR_INVALID, "update_timestep: no snapshot has been pushed");
  CK(cudaSetDevice(c->cfg.device));
  bool may_defer = allow_defer && !c->streaming && !c->push_d2h_outstanding;
  if (!may_defer) { const int rc = drain(c); if (rc) return rc; }
  if (c->n == 3 && c->scans == Scans::fused3d && c->cfg.vector_source == FTKB_SOURCE_DERIVED) {
    // a layer whose pointer TMA cannot take was materialised at push time: the sweep cannot mix the two forms
    bool anyV = false, anyS = false;
    for (const Layer &l : c->layers) { anyV = anyV || l.V; anyS = anyS || (!l.V && l.S); }
    if (anyV && anyS) {
      int rc = drain(c);
      if (!rc) rc = fall_back(c);
      if (rc) return rc;
      may_defer = false;
    }
  }
  if (c->n == 3 && c->scans != Scans::fused3d) {
    // scalar layers that reached the context without their gradient (remote snapshots): materialise it
    bool any = false;
    for (Layer &l : c->layers)
      if (!l.V && l.S && c->cfg.vector_source == FTKB_SOURCE_DERIVED) {
        int rc = drain(c);
        if (!rc) rc = materialise_gradient(c, l);
        if (rc) return rc;
        any = true;
      }
    if (any) { CK(cudaStreamSynchronize(c->stream)); may_defer = false; }
  }
  const bool has_next = c->layers.size() >= 2;
  Layer &l0 = c->layers[0], &l1 = c->layers[has_next ? 1 : 0];
  SweepParams p{};
  const Scan s = sweep_setup(c, l0, l1, has_next, p);
  if (!s.launch) {
    int rc = drain(c);
    if (!rc) rc = fall_back(c);
    return rc ? rc : update_impl(c, allow_defer);
  }
  if (!l0.V && !p.fused) return fail(c, FTKB_ERR_INVALID, "update_timestep: the snapshot has no vector field");
  if (c->current_timestep + 1 >= (1 << KEY_TIME_BITS)) return fail(c, FTKB_ERR_OVERFLOW, "update_timestep: timestep exceeds the element id range");
  if (c->push_d2h_outstanding) {
    CK(cudaStreamSynchronize(c->stream));   // resolutions of layers derived at push time are on the host now
    c->push_d2h_outstanding = false;
  }
  // derive timing of the most recent gradient launch
  if (c->derive_timed) {
    float ms = 0;
    if (cudaEventElapsedTime(&ms, c->ev[4], c->ev[5]) == cudaSuccess) { c->stats.ms_derive += ms; c->stats.last_ms_derive = ms; }
    else cudaGetLastError();
    c->derive_timed = false;
  }
  if (has_next && !l1.V && !(p.fused && l1.S)) return fail(c, FTKB_ERR_INVALID, "update_timestep: the next snapshot has no vector field");
  {
    // vector input: the range-cell scan streams each layer once and produces its min |v|; layers it cannot take now
    // (pushed further ahead than this sweep reads) get the plain resolution pass
    bool any = false;
    for (size_t k = 0; k < c->layers.size(); k++) {
      Layer &l = c->layers[k];
      if (l.V && l.res_pending && !(s.cells && !p.fused && k < 2)) {
        int rc = drain(c);
        if (!rc) rc = resolve_pending(c, l);
        if (rc) return rc;
        any = true;
      }
    }
    if (any) { CK(cudaStreamSynchronize(c->stream)); c->push_d2h_outstanding = false; may_defer = false; }
  }
  if (has_next && p.fused && l1.V) return fail(c, FTKB_ERR_INVALID, "update_timestep: resident snapshots mix derived and given vector fields");
  // ref: critical_point_tracker.hh:850-864 (running minimum over every resident snapshot, every sweep).
  // Layers whose resolution the fused scan still has to produce are left out here: the sweep runs with
  // the factor known so far and is repeated if the completed minimum changes nbits (nbits only ever
  // grows and is clamped to [8, 21], so at most 13 sweeps of a whole run are repeated).
  for (const Layer &l : c->layers)
    if ((l.V || l.S) && !l.res_pending) c->resolution = std::min(c->resolution, slot_value(c, l.slot));
  set_key_filter(c, p);
  if (has_next && p.scalar_source != FTKB_SOURCE_NONE && !l1.S) return fail(c, FTKB_ERR_INVALID, "update_timestep: the next snapshot has no scalar field");
  const int nbits = nbits_of(c->resolution);
  if (may_defer && s.cells && l0.cells_valid && !p.no_filter) return enqueue_step(c, s, p, l0, l1, nbits);
  return sync_step(c, s, p, l0, l1, nbits);
}

extern "C" int ftkb_advance_timestep(ftkb_ctx *c) {
  if (!c) return FTKB_ERR_INVALID;
  const int rc = ftkb_update_timestep(c);
  if (rc) return rc;
  if (!c->layers.empty()) {
    if (!c->pend.empty()) {
      // an enqueued step still reads this layer: it is released when that step has been confirmed
      c->limbo.push_back(c->layers.front());
      c->pend.back().pops++;
    } else {
      release_layer(c, c->layers.front());
    }
    c->layers.pop_front();
  }
  c->current_timestep++;
  return FTKB_OK;
}

// ------------------------------------------------------------------------------------------------
// results
// ------------------------------------------------------------------------------------------------
static void fill_trace_params(const ftkb_ctx *c, TraceParams &tp) {
  tp.nd = c->n;
  for (int j = 0; j < 3; j++) {
    const bool used = j < c->n;
    tp.lb[j] = used ? c->cfg.lb[j] : 0;
    tp.ub[j] = used ? c->cfg.ub[j] : 0;
  }
  if (c->slab) { tp.lb[2] = c->cfg.slab_global_lb; tp.ub[2] = c->cfg.slab_global_ub; }    // the points carry whole-array corners
  tp.ny = tp.ub[1] - tp.lb[1] + 1;
  tp.nz = tp.ub[2] - tp.lb[2] + 1;
}

// FTKB_DEBUG_TIMING=1: wall-clock laps of the finalize phases on stderr
struct Laps {
  bool on;
  const char *what;
  std::chrono::steady_clock::time_point t;
  std::string line;
  Laps(bool enabled, const char *w) : on(enabled), what(w), t(std::chrono::steady_clock::now()) {}
  void lap(const char *name) {
    if (!on) return;
    const auto now = std::chrono::steady_clock::now();
    char buf[96];
    std::snprintf(buf, sizeof(buf), " %s=%.2f", name, std::chrono::duration<double, std::milli>(now - t).count());
    line += buf;
    t = now;
  }
  ~Laps() { if (on) std::fprintf(stderr, "[ftkb timing] %s (ms):%s\n", what, line.c_str()); }
};

// sort the punctured simplices by element order and drop duplicates (std::map semantics of the
// reference's discrete_critical_points, critical_point_tracker_regular.hh:13-38)
static int ensure_sorted(ftkb_ctx *c) {
  CK(cudaSetDevice(c->cfg.device));
  { const int rc = drain(c); if (rc) return rc; }
  if (c->sorted) return FTKB_OK;
  c->d_pts_sorted = nullptr;         // (slots 12 / 13 of the finalize scratch: nothing to free here)
  c->d_keys_sorted = nullptr;
  c->pts_sorted.clear();
  c->nsorted = 0;
  const uint64_t n = c->npts;
  if (n == 0) { c->sorted = true; return FTKB_OK; }
  if (n >= 0xffffffffull) return fail(c, FTKB_ERR_OVERFLOW, "more than 2^32 punctured simplices");
  TraceParams tp{};
  fill_trace_params(c, tp);
  const auto tw0 = std::chrono::steady_clock::now();
  Laps laps(c->debug_timing, "sort");
  unsigned long long *k0 = nullptr, *k1 = nullptr;
  uint32_t *i0 = nullptr, *i1 = nullptr;
  void *temp = nullptr;
#define CKC(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { c->error = std::string(#call) + ": " + cudaGetErrorString(e_); return FTKB_ERR_CUDA; } } while (0)
  {
    // everything this sort and the trace after it will ask for (the cub sizes are queries: nothing is launched)
    const size_t tb0 = std::max(sort_pairs_u64(nullptr, 0, nullptr, nullptr, nullptr, nullptr, n, c->stream),
                                unique_by_key_u64(nullptr, 0, nullptr, nullptr, nullptr, nullptr, c->d_scalars + ftkb_ctx::SLOT_UQ, n, c->stream));
    const size_t plan[14] = {8 * n, 8 * n, 4 * n, 4 * n, tb0, c->streaming ? 0 : 4 * 8 * n, c->streaming ? 0 : 4 * n, c->streaming ? 0 : 4 * n, c->streaming ? 0 : 4 * n,
                             0, 0, 0, sizeof(ftkb_point) * n, 8 * n};
    const int rp = scratch_plan(c, plan, 14);
    if (rp) return rp;
  }
  { int rs = scratch(c, 0, 8 * n, (void **)&k0); if (!rs) rs = scratch(c, 1, 8 * n, (void **)&k1); if (!rs) rs = scratch(c, 2, 4 * n, (void **)&i0);
    if (!rs) rs = scratch(c, 3, 4 * n, (void **)&i1); if (rs) return rs; }
  CKC(cudaEventRecord(c->ev[0], c->stream));
  launch_point_keys(c->d_pts, n, tp, k0, i0, c->stream);
  size_t tb = std::max(sort_pairs_u64(nullptr, 0, k0, k1, i0, i1, n, c->stream),
                       unique_by_key_u64(nullptr, 0, k1, i1, k0, i0, c->d_scalars + ftkb_ctx::SLOT_UQ, n, c->stream));
  { const int rs = scratch(c, 4, tb, &temp); if (rs) return rs; }
  sort_pairs_u64(temp, tb, k0, k1, i0, i1, n, c->stream);
  unique_by_key_u64(temp, tb, k1, i1, k0, i0, c->d_scalars + ftkb_ctx::SLOT_UQ, n, c->stream);
  CKC(cudaMemcpyAsync(c->h_scalars + ftkb_ctx::SLOT_UQ, c->d_scalars + ftkb_ctx::SLOT_UQ, 8, cudaMemcpyDeviceToHost, c->stream));
  CKC(cudaStreamSynchronize(c->stream));
  const uint64_t nu = c->h_scalars[ftkb_ctx::SLOT_UQ];
  laps.lap("sort+unique");
  { int rs = scratch(c, 12, sizeof(ftkb_point) * nu, (void **)&c->d_pts_sorted); if (!rs) rs = scratch(c, 13, 8 * nu, (void **)&c->d_keys_sorted); if (rs) return rs; }
  launch_gather_points(c->d_pts, i0, nu, c->d_pts_sorted, c->stream);
  CKC(cudaMemcpyAsync(c->d_keys_sorted, k0, 8 * nu, cudaMemcpyDeviceToDevice, c->stream));      // unique sorted keys
  CKC(cudaEventRecord(c->ev[1], c->stream));
  laps.lap("malloc+gather");
  // the sorted records stay on the device: ftkb_get_points copies them straight into the caller's array, and the few host-side
  // users (curve sets) fetch them on demand (host_points) -- a copy of 72 bytes per record into fresh pageable memory costs more
  // than the sort
  CKC(cudaStreamSynchronize(c->stream));
  laps.lap("sync");
  CKC(cudaGetLastError());
  float ms = 0;
  CKC(cudaEventElapsedTime(&ms, c->ev[0], c->ev[1]));
  c->stats.ms_finalize_device += ms;
  c->stats.kernel_launches += 4;
  c->nsorted = nu;
  c->stats.ms_sort_wall += std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - tw0).count();
#undef CKC
  c->sorted = true;
  return FTKB_OK;
}

// host copy of the sorted records, made when somebody on the host needs it
static int host_points(ftkb_ctx *c) {
  const int rc = ensure_sorted(c);
  if (rc) return rc;
  if (c->pts_sorted.size() == c->nsorted) return FTKB_OK;
  c->pts_sorted.resize(c->nsorted);
  if (c->nsorted) {
    CK(cudaMemcpyAsync(c->pts_sorted.data(), c->d_pts_sorted, sizeof(ftkb_point) * c->nsorted, cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    c->stats.d2h_bytes += sizeof(ftkb_point) * c->nsorted;
  }
  return FTKB_OK;
}

extern "C" int ftkb_num_points(ftkb_ctx *c, uint64_t *n) {
  if (!c || !n) return FTKB_ERR_INVALID;
  const int rc = ensure_sorted(c);
  if (rc) return rc;
  *n = c->nsorted;
  return FTKB_OK;
}

extern "C" int ftkb_get_points(ftkb_ctx *c, ftkb_point *out, uint64_t cap) {
  if (!c || (!out && cap)) return FTKB_ERR_INVALID;
  const int rc = ensure_sorted(c);
  if (rc) return rc;
  if (cap < c->nsorted) return fail(c, FTKB_ERR_INVALID, "get_points: output buffer too small");
  if (!c->nsorted) return FTKB_OK;
  if (c->pts_sorted.size() == c->nsorted) { std::memcpy(out, c->pts_sorted.data(), sizeof(ftkb_point) * c->nsorted); return FTKB_OK; }
  CK(cudaSetDevice(c->cfg.device));
  CK(cudaMemcpyAsync(out, c->d_pts_sorted, sizeof(ftkb_point) * c->nsorted, cudaMemcpyDeviceToHost, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  c->stats.d2h_bytes += sizeof(ftkb_point) * c->nsorted;
  return FTKB_OK;
}

extern "C" int ftkb_import_points(ftkb_ctx *c, const ftkb_point *pts, uint64_t n) {
  if (!c || (!pts && n)) return FTKB_ERR_INVALID;
  // a streaming context grows its trajectories from its own sweeps; one that holds no snapshot and has swept nothing takes
  // imports instead, and grows them step by step with ftkb::grow_imported
  if (c->streaming && (c->stats.scan_launches || !c->layers.empty()))
    return fail(c, FTKB_ERR_INVALID, "import_points: not available on a streaming context that sweeps");
  if (!n) return FTKB_OK;
  CK(cudaSetDevice(c->cfg.device));
  { const int rc = drain(c); if (rc) return rc; }
  c->primed = false;
  if (c->npts + n > c->pt_cap) {
    const int rc = grow_points(c, c->npts + n);
    if (rc) return rc;
  }
  CK(cudaMemcpyAsync(c->d_pts + c->npts, pts, sizeof(ftkb_point) * n, cudaMemcpyHostToDevice, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  c->stats.h2d_bytes += sizeof(ftkb_point) * n;
  c->npts += n;
  c->stats.points = c->npts;
  c->sorted = false;
  c->traced = false;
  return FTKB_OK;
}

// A streaming context's trajectories grown so far, in id order, as CSR over its sorted points (traj_*): what ftkb_finalize
// publishes, and what ftkb_get_live_curveset reads at any time.  Points that no grow step has seen yet are among the sorted
// points but on no trajectory.
static int publish_grown(ftkb_ctx *c) {
  { const int rc = wait_grow(c); if (rc) return rc; }
  { const int rc = ensure_sorted(c); if (rc) return rc; }
  const uint64_t n = c->nsorted;
  const auto t0 = std::chrono::steady_clock::now();
  c->traj_off.assign(1, 0);
  c->traj_idx.clear();
  c->traj_loop.clear();
  c->traj_complete.clear();
  std::vector<uint64_t> keys(n);
  if (n) {      // the sorted points' element keys (the device sorted by them)
    CK(cudaMemcpyAsync(keys.data(), c->d_keys_sorted, 8 * n, cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    c->stats.d2h_bytes += 8 * n;
  }
  const std::vector<uint64_t> &streamed = c->online->keys();
  for (const ftkb::OnlineCurve &cv : c->online->curves()) {
    for (const uint32_t g : cv.idx) {
      const uint64_t key = streamed[g];
      const auto it = std::lower_bound(keys.begin(), keys.end(), key);
      if (it == keys.end() || *it != key) return fail(c, FTKB_ERR_INVALID, "a streamed point is missing from the sorted points");
      c->traj_idx.push_back((uint64_t)(it - keys.begin()));
    }
    c->traj_loop.push_back(cv.loop);
    c->traj_complete.push_back(cv.complete);
    c->traj_off.push_back(c->traj_idx.size());
  }
  c->stats.ms_finalize_host += std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
  return FTKB_OK;
}

// ref: critical_point_tracker.hh:668-817 trace_critical_points_offline; cc2curves.hh:10-122
extern "C" int ftkb_finalize(ftkb_ctx *c) {
  if (!c) return FTKB_ERR_INVALID;
  int rc = drain(c);
  if (rc) return rc;
  if (c->traced) return FTKB_OK;
  rc = ensure_sorted(c);
  if (rc) return rc;
  const uint64_t n = c->nsorted;
  Laps laps(c->debug_timing, "trace");
  c->labels.clear(); c->deg.clear();
  if (c->streaming) { c->labels.assign(n, 0); c->deg.assign(n, 0); }     // (not computed: zeros)
  else { c->labels.resize(n); c->deg.resize(n); }                       // every entry is written below
  c->traj_off.assign(1, 0);
  c->traj_idx.clear();
  c->traj_loop.clear();
  c->traj_complete.clear();
  if (c->streaming) {
    // "done" (critical_point_tracker_2d_regular.hh:150-151): the grown trajectories as they stand; the component labels /
    // degrees of the offline trace are not computed
    { const int rc2 = publish_grown(c); if (rc2) return rc2; }
    c->traced = true;
    return FTKB_OK;
  }
  if (n == 0) { c->traced = true; return FTKB_OK; }

  // device: neighbour search among punctured simplices + union-find (all nodes / ordinary nodes)
  TraceParams tp{};
  fill_trace_params(c, tp);
  tp.n = n;
  tp.keys = c->d_keys_sorted;
  tp.pts = c->d_pts_sorted;
  const auto tw0 = std::chrono::steady_clock::now();
  uint32_t *d_nb = nullptr, *d_pa = nullptr, *d_po = nullptr;
  int32_t *d_deg = nullptr;
#define CKC(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { c->error = std::string(#call) + ": " + cudaGetErrorString(e_); return FTKB_ERR_CUDA; } } while (0)
  { int rs = scratch(c, 5, 4 * 8 * n, (void **)&d_nb); if (!rs) rs = scratch(c, 6, 4 * n, (void **)&d_pa); if (!rs) rs = scratch(c, 7, 4 * n, (void **)&d_po);
    if (!rs) rs = scratch(c, 8, 4 * n, (void **)&d_deg); if (rs) return rs; }
  tp.nb = d_nb; tp.deg = d_deg; tp.parent_all = d_pa; tp.parent_ord = d_po;
  laps.lap("host_assign+scratch");
  CKC(cudaEventRecord(c->ev[0], c->stream));
  launch_neighbors(tp, c->stream);
  launch_union_find(tp, c->stream);
  CKC(cudaEventRecord(c->ev[1], c->stream));
  c->stats.kernel_launches += 3;
  RawVec<uint32_t> nb(8 * n), pa(n), po(n);
  laps.lap("host_vectors");
  CKC(cudaMemcpyAsync(nb.data(), d_nb, 4 * 8 * n, cudaMemcpyDeviceToHost, c->stream));
  CKC(cudaMemcpyAsync(pa.data(), d_pa, 4 * n, cudaMemcpyDeviceToHost, c->stream));
  CKC(cudaMemcpyAsync(po.data(), d_po, 4 * n, cudaMemcpyDeviceToHost, c->stream));
  CKC(cudaMemcpyAsync(c->deg.data(), d_deg, 4 * n, cudaMemcpyDeviceToHost, c->stream));
  CKC(cudaStreamSynchronize(c->stream));
  CKC(cudaGetLastError());
  float ms = 0;
  CKC(cudaEventElapsedTime(&ms, c->ev[0], c->ev[1]));
  c->stats.ms_finalize_device += ms;
  c->stats.d2h_bytes += 4 * 11 * n;
  laps.lap("kernels+d2h");
#undef CKC

  // host: order every trajectory with the reference's deterministic walk (cc2curves.hh:46-108)
  const auto t0 = std::chrono::steady_clock::now();
  for (uint64_t i = 0; i < n; i++) c->labels[i] = pa[i];
  std::vector<uint8_t> visited(n, 0);
  auto ordinary = [&](uint32_t i) { return c->deg[i] <= 2; };
  auto next_unvisited = [&](uint32_t cur, uint32_t &out) {
    for (int q = 0; q < 8; q++) {
      const uint32_t j = nb[(size_t)cur * 8 + q];
      if (j == 0xffffffffu) break;
      if (ordinary(j) && !visited[j]) { out = j; return true; }
    }
    return false;
  };
  // The walks of different trajectories touch disjoint nodes (a trajectory is one connected component of the ordinary nodes),
  // so they run on several host threads; the trajectories are then laid out in seed order, as the serial walk would.
  std::vector<uint32_t> seeds;
  for (uint64_t seed = 0; seed < n; seed++)
    if (ordinary((uint32_t)seed) && po[seed] == seed) seeds.push_back((uint32_t)seed);   // the smallest member starts the walk
  const size_t S = seeds.size();
  laps.lap("seeds");
  struct Piece { uint32_t thread; uint64_t off, len; uint8_t loop; };
  std::vector<Piece> pieces(S);
  const unsigned hw = std::thread::hardware_concurrency();
  const size_t nthr = std::max<size_t>(1, std::min<size_t>({(size_t)16, (size_t)(hw ? hw : 1), (size_t)(n / 65536 + 1)}));
  std::vector<std::vector<uint32_t>> bufs(nthr);
  std::atomic<size_t> next{0};
  const size_t batch = std::max<size_t>(1, std::min<size_t>(64, S / (nthr * 8)));      // few long trajectories: one seed at a time
  auto work = [&](const uint32_t tid) {
    std::vector<uint32_t> &out = bufs[tid];
    std::vector<uint32_t> fwd, bwd;
    for (;;) {
      const size_t s0 = next.fetch_add(batch), s1 = std::min(S, s0 + batch);
      if (s0 >= S) break;
      for (size_t si = s0; si < s1; si++) {
        const uint32_t seed = seeds[si];
        fwd.clear(); bwd.clear();
        visited[seed] = 1;
        uint32_t sn[8]; int nsn = 0;
        for (int q = 0; q < 8; q++) {
          const uint32_t j = nb[(size_t)seed * 8 + q];
          if (j == 0xffffffffu) break;
          if (ordinary(j)) sn[nsn++] = j;
        }
        for (int dir = 0; dir < 2 && nsn > 0; dir++) {
          uint32_t cur = dir == 0 ? sn[0] : sn[nsn - 1];
          while (true) {
            if (!visited[cur]) { (dir == 0 ? fwd : bwd).push_back(cur); visited[cur] = 1; }
            uint32_t nx;
            if (!next_unvisited(cur, nx)) break;
            cur = nx;
          }
          if (nsn == 1) break;
        }
        const uint64_t start = out.size();
        for (size_t k = bwd.size(); k > 0; k--) out.push_back(bwd[k - 1]);
        out.push_back(seed);
        for (uint32_t v : fwd) out.push_back(v);
        const uint64_t len = out.size() - start;
        bool loop = false;
        if (len > 1) {   // is_loop: the back is a neighbour of the front (cc2curves.hh:113-122)
          const uint64_t front = out[start], back = out.back();
          for (int q = 0; q < 8; q++) loop = loop || nb[front * 8 + q] == back;
        }
        pieces[si] = Piece{tid, start, len, (uint8_t)loop};
      }
    }
  };
  if (nthr == 1) work(0);
  else {
    std::vector<std::thread> pool;
    for (uint32_t t = 0; t < nthr; t++) pool.emplace_back(work, t);
    for (auto &th : pool) th.join();
  }
  laps.lap("walk");
  c->traj_idx.reserve(n);
  for (size_t si = 0; si < S; si++) {
    const Piece &pc = pieces[si];
    const uint32_t *src = bufs[pc.thread].data() + pc.off;
    c->traj_idx.insert(c->traj_idx.end(), src, src + pc.len);
    c->traj_loop.push_back(pc.loop);
    c->traj_off.push_back(c->traj_idx.size());
  }
  laps.lap("layout");
  c->stats.ms_finalize_host += std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
  c->stats.ms_trace_wall += std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - tw0).count();
  c->traced = true;
  return FTKB_OK;
}

extern "C" int ftkb_num_trajectories(ftkb_ctx *c, uint64_t *n) {
  if (!c || !n) return FTKB_ERR_INVALID;
  if (!c->traced) return fail(c, FTKB_ERR_INVALID, "num_trajectories: call finalize first");
  *n = c->traj_loop.size();
  return FTKB_OK;
}

extern "C" int ftkb_get_trajectory_complete(ftkb_ctx *c, uint8_t *complete) {
  if (!c || !complete) return FTKB_ERR_INVALID;
  if (!c->traced) return fail(c, FTKB_ERR_INVALID, "get_trajectory_complete: call finalize first");
  for (size_t k = 0; k < c->traj_loop.size(); k++) complete[k] = k < c->traj_complete.size() ? c->traj_complete[k] : 0;
  return FTKB_OK;
}

extern "C" int ftkb_get_trajectories(ftkb_ctx *c, uint64_t *offsets, uint64_t *point_idx, uint8_t *loop) {
  if (!c || !offsets) return FTKB_ERR_INVALID;
  if (!c->traced) return fail(c, FTKB_ERR_INVALID, "get_trajectories: call finalize first");
  std::memcpy(offsets, c->traj_off.data(), 8 * c->traj_off.size());
  if (point_idx && !c->traj_idx.empty()) std::memcpy(point_idx, c->traj_idx.data(), 8 * c->traj_idx.size());
  if (loop && !c->traj_loop.empty()) std::memcpy(loop, c->traj_loop.data(), c->traj_loop.size());
  return FTKB_OK;
}

// ------------------------------------------------------------------------------------------------
// time-slab halo through peer memory
// ------------------------------------------------------------------------------------------------
extern "C" int ftkb_ipc_export(const void *dev_ptr, ftkb_ipc_handle *out) {
  if (!dev_ptr || !out) return FTKB_ERR_INVALID;
  typedef CUresult (*RangeFn)(CUdeviceptr *, size_t *, CUdeviceptr);
  static RangeFn range = nullptr;
  if (!range) {
    void *fp = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuMemGetAddressRange", &fp, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess) { cudaGetLastError(); return FTKB_ERR_CUDA; }
    range = reinterpret_cast<RangeFn>(fp);
  }
  CUdeviceptr base = 0;
  size_t size = 0;
  if (range(&base, &size, (CUdeviceptr)(uintptr_t)dev_ptr) != CUDA_SUCCESS) return FTKB_ERR_CUDA;
  cudaIpcMemHandle_t h;
  if (cudaIpcGetMemHandle(&h, reinterpret_cast<void *>(base)) != cudaSuccess) { cudaGetLastError(); return FTKB_ERR_CUDA; }
  static_assert(sizeof(h) == 64, "cudaIpcMemHandle_t is 64 bytes");
  std::memcpy(out->bytes, &h, 64);
  out->offset = (uint64_t)((uintptr_t)dev_ptr - (uintptr_t)base);
  return FTKB_OK;
}

extern "C" int ftkb_ipc_import(const ftkb_ipc_handle *h, int device, void **dev_ptr) {
  if (!h || !dev_ptr) return FTKB_ERR_INVALID;
  if (cudaSetDevice(device) != cudaSuccess) { cudaGetLastError(); return FTKB_ERR_NO_DEVICE; }
  cudaIpcMemHandle_t ih;
  std::memcpy(&ih, h->bytes, 64);
  void *base = nullptr;
  if (cudaIpcOpenMemHandle(&base, ih, cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) { cudaGetLastError(); return FTKB_ERR_CUDA; }
  *dev_ptr = static_cast<char *>(base) + h->offset;
  return FTKB_OK;
}

extern "C" int ftkb_ipc_close(void *dev_ptr, const ftkb_ipc_handle *h) {
  if (!dev_ptr || !h) return FTKB_ERR_INVALID;
  if (cudaIpcCloseMemHandle(static_cast<char *>(dev_ptr) - h->offset) != cudaSuccess) { cudaGetLastError(); return FTKB_ERR_CUDA; }
  return FTKB_OK;
}

extern "C" int ftkb_export_layer_cells(ftkb_ctx *c, int index, void **cells, uint64_t *bytes, double *resolution) {
  if (!c || !cells || !bytes) return FTKB_ERR_INVALID;
  if (index < 0 || (size_t)index >= c->layers.size()) return fail(c, FTKB_ERR_INVALID, "export_layer_cells: no such resident layer");
  { const int rc = drain(c); if (rc) return rc; }
  if ((size_t)index >= c->layers.size()) return fail(c, FTKB_ERR_INVALID, "export_layer_cells: no such resident layer");
  Layer &l = c->layers[index];
  if (!l.cells || !l.cells_valid) return fail(c, FTKB_ERR_INVALID, "export_layer_cells: the layer has no range cells yet (a sweep must have read it)");
  CK(cudaSetDevice(c->cfg.device));
  CK(cudaStreamSynchronize(c->stream));
  if (!l.cells_foreign) { l.cells_foreign = true; c->exportedCells.push_back(l.cells); }
  *cells = l.cells;
  *bytes = (uint64_t)c->ncells * sizeof(uint4);
  if (resolution) *resolution = l.res_pending ? DBL_MAX : slot_value(c, l.slot);
  return FTKB_OK;
}

extern "C" int ftkb_push_snapshot_remote(ftkb_ctx *c, const double *scalar, const double *vector, const void *cells, double resolution) {
  if (!c || !cells || (!scalar && !vector)) return FTKB_ERR_INVALID;
  if (c->cfg.jacobian_source == FTKB_SOURCE_GIVEN) return fail(c, FTKB_ERR_INVALID, "push_snapshot_remote: a GIVEN jacobian cannot be remote");
  if (c->cfg.vector_source == FTKB_SOURCE_GIVEN ? !vector : !scalar) return fail(c, FTKB_ERR_INVALID, "push_snapshot_remote: the field the sweep reads is missing");
  CK(cudaSetDevice(c->cfg.device));
  if ((uintptr_t)scalar % 8 != 0 || (uintptr_t)vector % 8 != 0 || (uintptr_t)cells % 16 != 0)
    return fail(c, FTKB_ERR_INVALID, "push_snapshot_remote: arrays must be 8-byte aligned, cells 16-byte aligned");
  Layer l;
  int rc = new_layer(c, l);
  if (rc) return rc;
  l.S = const_cast<double *>(scalar);
  l.V = const_cast<double *>(vector);
  l.cells = reinterpret_cast<uint4 *>(const_cast<void *>(cells));
  l.cells_valid = true;
  l.cells_foreign = true;
  l.res_pending = false;
  // the owner's min non-zero |v| of this layer, as the sweep would have produced it
  unsigned long long bits;
  const double r = resolution > 0 ? resolution : DBL_MAX;
  std::memcpy(&bits, &r, 8);
  if (!(resolution > 0) || resolution >= DBL_MAX) bits = ~0ull;
  c->h_scalars[l.slot] = bits;
  CK(cudaMemcpyAsync(c->d_scalars + l.slot, c->h_scalars + l.slot, sizeof(unsigned long long), cudaMemcpyHostToDevice, c->stream));
  c->layers.push_back(l);
  return FTKB_OK;
}

// the curve set of the trajectories in traj_* over the sorted points
static int build_curveset(ftkb_ctx *c, ftkb_curveset **out) {
  const uint64_t ntraj = c->traj_off.empty() ? 0 : c->traj_off.size() - 1;
  static const uint64_t zero = 0;
  { const int rch = host_points(c); if (rch) return rch; }
  const int rc = ftkb_curveset_create(c->pts_sorted.data(), c->pts_sorted.size(), ntraj ? c->traj_off.data() : &zero, c->traj_idx.data(),
                                      c->traj_loop.data(), ntraj, out);
  if (rc == FTKB_OK)   // streaming: feature_curve_t::complete as the grow steps left it (curves are in id order)
    for (size_t k = 0; k < c->traj_complete.size() && k < (*out)->curves.size(); k++) (*out)->curves[k].complete = c->traj_complete[k] != 0;
  return rc;
}

extern "C" int ftkb_get_curveset(ftkb_ctx *c, ftkb_curveset **out) {
  if (!c || !out) return FTKB_ERR_INVALID;
  if (!c->traced) return fail(c, FTKB_ERR_INVALID, "get_curveset: call finalize first");
  return build_curveset(c, out);
}

extern "C" int ftkb_get_live_curveset(ftkb_ctx *c, int32_t *grown_through, ftkb_curveset **out) {
  if (!c || !grown_through || !out) return fail(c, FTKB_ERR_INVALID, "get_live_curveset: null argument");
  *out = nullptr;
  if (!c->streaming) return fail(c, FTKB_ERR_INVALID, "get_live_curveset: streaming trajectories are off (ftkb_set_streaming_trajectories)");
  CK(cudaSetDevice(c->cfg.device));
  { const int rc = drain(c); if (rc) return rc; }
  // after finalize traj_* hold what it published; before, they are rebuilt from the tracer (traced stays false, so the
  // finalize-only getters still refuse, and any later sweep, grow or import makes the next query rebuild them)
  if (!c->traced) { const int rc = publish_grown(c); if (rc) return rc; }
  const int rc = build_curveset(c, out);
  if (rc == FTKB_OK) *grown_through = c->grown_through;
  return rc;
}

extern "C" int ftkb_get_component_labels(ftkb_ctx *c, uint64_t *labels) {
  if (!c || !labels) return FTKB_ERR_INVALID;
  if (!c->traced) return fail(c, FTKB_ERR_INVALID, "get_component_labels: call finalize first");
  if (!c->labels.empty()) std::memcpy(labels, c->labels.data(), 8 * c->labels.size());
  return FTKB_OK;
}

extern "C" int ftkb_get_degrees(ftkb_ctx *c, int32_t *deg) {
  if (!c || !deg) return FTKB_ERR_INVALID;
  if (!c->traced) return fail(c, FTKB_ERR_INVALID, "get_degrees: call finalize first");
  if (!c->deg.empty()) std::memcpy(deg, c->deg.data(), 4 * c->deg.size());
  return FTKB_OK;
}

extern "C" int ftkb_get_last_worklist(ftkb_ctx *c, uint64_t *out, uint64_t cap, uint64_t *n) {
  if (!c || !n || (!out && cap)) return FTKB_ERR_INVALID;
  CK(cudaSetDevice(c->cfg.device));
  { const int rc = drain(c); if (rc) return rc; }
  CK(cudaStreamSynchronize(c->stream));
  const uint64_t have = std::min<uint64_t>(c->last_wl, c->wl_cap);
  *n = have;
  const uint64_t m = std::min(have, cap);
  if (m) CK(cudaMemcpy(out, c->last_wl_sel ? c->d_wl2 : c->d_wl, sizeof(uint64_t) * m, cudaMemcpyDeviceToHost));
  return FTKB_OK;
}

extern "C" int ftkb_get_layer(ftkb_ctx *c, int index, double *scalar, double *vector) {
  if (!c || (!scalar && !vector)) return FTKB_ERR_INVALID;
  CK(cudaSetDevice(c->cfg.device));
  { const int rc = drain(c); if (rc) return rc; }
  if (index < 0 || (size_t)index >= c->layers.size()) return fail(c, FTKB_ERR_INVALID, "get_layer: no such resident snapshot");
  const Layer &l = c->layers[index];
  if ((scalar && !l.S) || (vector && !l.V)) return fail(c, FTKB_ERR_INVALID, "get_layer: the snapshot does not hold that field");
  CK(cudaStreamSynchronize(c->stream));
  if (scalar) CK(cudaMemcpy(scalar, l.S, sizeof(double) * c->nvert, cudaMemcpyDeviceToHost));
  if (vector) CK(cudaMemcpy(vector, l.V, sizeof(double) * c->nvert * c->n, cudaMemcpyDeviceToHost));
  c->stats.d2h_bytes += sizeof(double) * c->nvert * ((scalar ? 1 : 0) + (vector ? c->n : 0));
  return FTKB_OK;
}

// page-locked host memory for callers that feed snapshots from files or generators: copies from it run at full PCIe speed and
// do not go through the driver's staging buffers (the CLI's double-buffered reader, stream.hh:1607-1699 in the reference)
// CPUs on the socket the device's PCIe root hangs off (sysfs local_cpulist), restricted to what the thread may run on
static bool device_local_cpus(int device, cpu_set_t *set) {
  char bus[32] = {0};
  if (cudaDeviceGetPCIBusId(bus, sizeof(bus) - 1, device) != cudaSuccess) { cudaGetLastError(); return false; }
  for (char *q = bus; *q; q++) *q = (char)std::tolower((unsigned char)*q);
  FILE *f = std::fopen((std::string("/sys/bus/pci/devices/") + bus + "/local_cpulist").c_str(), "r");
  if (!f) return false;
  char line[4096];
  const bool got = std::fgets(line, sizeof(line), f) != nullptr;
  std::fclose(f);
  cpu_set_t allowed;
  if (!got || sched_getaffinity(0, sizeof(allowed), &allowed) != 0) return false;
  CPU_ZERO(set);
  int n = 0;
  for (const char *q = line; *q && *q != '\n';) {          // "0-31,64-95"
    char *e = nullptr;
    long a = std::strtol(q, &e, 10), b = a;
    if (e == q) break;
    if (*e == '-') { q = e + 1; b = std::strtol(q, &e, 10); }
    for (long i = a; i <= b && i < CPU_SETSIZE; i++)
      if (CPU_ISSET(i, &allowed)) { CPU_SET(i, set); n++; }
    if (*e != ',') break;
    q = e + 1;
  }
  return n > 0;
}

// The calling thread (and the threads it creates afterwards) run on the CPUs next to `device` from here on: page-locked
// buffers it allocates and the driver's staging copies then live in that socket's memory, so host<->device copies of several
// devices do not all cross the inter-socket link or drain one socket's DRAM (e2e at 4 and 8 ranks).
extern "C" int ftkb_bind_thread_to_device(int device) {
  cpu_set_t set;
  if (!device_local_cpus(device, &set)) return 0;
  if (sched_setaffinity(0, sizeof(set), &set) != 0) return 0;
  return CPU_COUNT(&set);
}

extern "C" int ftkb_host_alloc(uint64_t bytes, void **out) {
  if (!out || !bytes) return FTKB_ERR_INVALID;
  *out = nullptr;
  // pages are placed where the allocating thread runs: next to the current device for the duration of the call
  cpu_set_t before, local;
  int device = 0;
  bool moved = false;
  if (cudaGetDevice(&device) == cudaSuccess && sched_getaffinity(0, sizeof(before), &before) == 0 && device_local_cpus(device, &local))
    moved = sched_setaffinity(0, sizeof(local), &local) == 0;
  const cudaError_t e = cudaHostAlloc(out, bytes, cudaHostAllocPortable);
  if (moved) sched_setaffinity(0, sizeof(before), &before);
  if (e != cudaSuccess) { cudaGetLastError(); return FTKB_ERR_NOMEM; }
  return FTKB_OK;
}

extern "C" void ftkb_host_free(void *p) {
  if (p && cudaFreeHost(p) != cudaSuccess) cudaGetLastError();
}

extern "C" int ftkb_get_stats(ftkb_ctx *c, ftkb_stats *out) {
  if (!c || !out) return FTKB_ERR_INVALID;
  if (!c->pend.empty()) {
    cudaSetDevice(c->cfg.device);
    const int rc = drain(c);
    if (rc) return rc;
  }
  { const int rc = wait_grow(c); if (rc) return rc; }
  c->stats.scaling_factor = c->factor;
  c->stats.resolution = c->resolution;
  *out = c->stats;
  return FTKB_OK;
}

extern "C" int ftkb_reset_stats(ftkb_ctx *c) {
  if (!c) return FTKB_ERR_INVALID;
  if (!c->pend.empty()) {
    cudaSetDevice(c->cfg.device);
    const int rc = drain(c);
    if (rc) return rc;
  }
  { const int rc = wait_grow(c); if (rc) return rc; }
  const uint64_t pts = c->stats.points;
  c->stats = ftkb_stats{};
  c->stats.points = pts;
  return FTKB_OK;
}

extern "C" int ftkb_synchronize(ftkb_ctx *c) {
  if (!c) return FTKB_ERR_INVALID;
  CK(cudaSetDevice(c->cfg.device));
  { const int rc = drain(c); if (rc) return rc; }
  CK(cudaStreamSynchronize(c->stream));
  CK(cudaStreamSynchronize(c->stream2));
  return wait_grow(c);
}

extern "C" int ftkb_timer_start(ftkb_ctx *c) {
  if (!c) return FTKB_ERR_INVALID;
  CK(cudaSetDevice(c->cfg.device));
  CK(cudaEventRecord(c->ev[6], c->stream));
  return FTKB_OK;
}

extern "C" int ftkb_timer_stop(ftkb_ctx *c, double *ms) {
  if (!c || !ms) return FTKB_ERR_INVALID;
  CK(cudaSetDevice(c->cfg.device));
  CK(cudaEventRecord(c->ev_join, c->stream2));      // the last test kernel belongs to the timed work
  CK(cudaStreamWaitEvent(c->stream, c->ev_join, 0));
  CK(cudaEventRecord(c->ev[7], c->stream));
  CK(cudaEventSynchronize(c->ev[7]));
  float f = 0;
  CK(cudaEventElapsedTime(&f, c->ev[6], c->ev[7]));
  *ms = f;
  return FTKB_OK;
}

// ------------------------------------------------------------------------------------------------
// mesh tables (host only)
// ------------------------------------------------------------------------------------------------
extern "C" int ftkb_mesh_ntypes(int nd_mesh, int k, int scope) {
  if ((nd_mesh != 3 && nd_mesh != 4) || k < 0 || k > nd_mesh) return -1;
  const MeshTables &m = mesh_tables(nd_mesh);
  return scope == 0 ? m.ntypes(k) : scope == 1 ? (int)m.ordinal_types[k].size() : (int)m.interval_types[k].size();
}

extern "C" int ftkb_mesh_unit_simplex(int nd_mesh, int k, int type, int32_t *out) {
  if ((nd_mesh != 3 && nd_mesh != 4) || k < 0 || k > nd_mesh || !out) return -1;
  const MeshTables &m = mesh_tables(nd_mesh);
  if (type < 0 || type >= m.ntypes(k)) return -1;
  for (int i = 0; i <= k; i++)
    for (int j = 0; j < nd_mesh; j++) out[i * nd_mesh + j] = (m.unit[k][type][i] >> j) & 1;
  return 0;
}

extern "C" int ftkb_mesh_scope_type(int nd_mesh, int k, int scope, int itype) {
  if ((nd_mesh != 3 && nd_mesh != 4) || k < 0 || k > nd_mesh) return -1;
  const MeshTables &m = mesh_tables(nd_mesh);
  const std::vector<int> *v = scope == 1 ? &m.ordinal_types[k] : scope == 2 ? &m.interval_types[k] : nullptr;
  if (!v) return itype;
  return itype >= 0 && itype < (int)v->size() ? (*v)[itype] : -1;
}

static int copy_offsets(const std::vector<TypeOffset> &v, int nd, int32_t *out) {
  for (size_t i = 0; i < v.size(); i++) {
    out[i * (nd + 1)] = v[i].type;
    for (int j = 0; j < nd; j++) out[i * (nd + 1) + 1 + j] = v[i].off[j];
  }
  return (int)v.size();
}

extern "C" int ftkb_mesh_sides(int nd_mesh, int k, int type, int32_t *out) {
  if ((nd_mesh != 3 && nd_mesh != 4) || k < 0 || k > nd_mesh || !out) return -1;
  const MeshTables &m = mesh_tables(nd_mesh);
  if (type < 0 || type >= m.ntypes(k)) return -1;
  return copy_offsets(m.sides[k][type], nd_mesh, out);
}

extern "C" int ftkb_mesh_side_of(int nd_mesh, int k, int type, int32_t *out) {
  if ((nd_mesh != 3 && nd_mesh != 4) || k < 0 || k > nd_mesh || !out) return -1;
  const MeshTables &m = mesh_tables(nd_mesh);
  if (type < 0 || type >= m.ntypes(k)) return -1;
  return copy_offsets(m.side_of[k][type], nd_mesh, out);
}
