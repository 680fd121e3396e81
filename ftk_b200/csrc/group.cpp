// Several GPUs behind one tracker: ftkb_group (include/ftkb200.h).
//
// The reference plumbs a device list into every filter (filter.hh:47-51 set_device_ids) and decomposes the work
// with DIY/MPI (regular_tracker.hh:120-151).  Here ONE process drives N devices through N ordinary contexts:
//
//   time chunks   timesteps are cut into chunks of `chunk_timesteps`; chunk c = steps [cB, (c+1)B) is swept by its own
//                 context on device c mod N and owns every simplex whose corner time lies in the chunk (the face-ownership
//                 rule of SURVEY.md 8e).  It needs layers cB .. (c+1)B: the first layer of chunk c+1 is pushed to both
//                 contexts (halo = one layer).
//   workers       one host thread per device executes that device's commands (push / advance / update) in order, so the
//                 caller's thread only hands snapshots over; devices sweep their chunks concurrently.  Host snapshots are
//                 borrowed until the push returns, exactly as with a single context.
//   factor        the quantisation factor is a running quantity (critical_point_tracker.hh:850-864).  A chunk inherits the
//                 running minimum of min non-zero |v| from its predecessor.  It may start before the predecessor has finished
//                 as soon as the minimum known so far already saturates the factor (2^21: nothing later can change it);
//                 until then chunks run one after another.  Results therefore equal the one-device run bit for bit.
//   merge         ftkb_group_finalize collects the (sparse) punctured simplices of every chunk into one context on the first
//                 device and runs the union-find + ordering there: components that cross chunk boundaries are united by
//                 the same neighbour search that unites them inside a chunk.
//   streaming     the merged context exists from the first push and grows during the run.  Chunks and slabs keep sweeping
//                 deferred; once the sweep of timestep t is confirmed (by every slab, or by the chunk that owns t) and t-1 has
//                 been grown, the points of that sweep are copied to the merged context's device (peer copies, no host) and the
//                 reference's grow step runs over them -- the batch a single streaming context grows at t (ordinal sweep at t +
//                 interval sweep [t, t+1]).  Slabs are grown by the caller's thread after every sweep, chunks by a thread of the
//                 merged context's own.  The last ordinal sweep's points join no trajectory, as on one device.
//                 Locks: a chunk's `m` (its context) may be taken before the group's `m`, never after; `root_m` (the merged
//                 context) before a chunk's `m`.
//   coordinates   physical coordinates (ftkb_group_set_coords) are kept here and handed to every chunk context as it is
//                 created and to every slab context at once; a slab looks them up in the whole array's frame.
#include <algorithm>
#include <atomic>
#include <cfloat>
#include <climits>
#include <cmath>
#include <condition_variable>
#include <cstring>
#include <deque>
#include <functional>
#include <memory>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include <cuda_runtime.h>

#include "../../include/ftkb200.h"
#include "online.h"

namespace {

struct Worker {
  std::thread th;
  std::mutex m;
  std::condition_variable cv, cv_space;
  std::deque<std::function<void()>> q;
  bool stop = false;
  void start(int device) {
    th = std::thread([this, device] {
      ftkb_bind_thread_to_device(device);      // host-side staging of this device's snapshots stays in the socket next to it
      for (;;) {
        std::function<void()> f;
        {
          std::unique_lock<std::mutex> lk(m);
          cv.wait(lk, [this] { return stop || !q.empty(); });
          if (q.empty()) return;
          f = std::move(q.front());
          q.pop_front();
        }
        cv_space.notify_one();
        f();
      }
    });
  }
  void post(std::function<void()> f) {
    {
      std::unique_lock<std::mutex> lk(m);
      cv_space.wait(lk, [this] { return q.size() < 256; });      // the caller never runs unboundedly ahead of a device
      q.push_back(std::move(f));
    }
    cv.notify_one();
  }
  void join() {
    { std::lock_guard<std::mutex> lk(m); stop = true; }
    cv.notify_one();
    if (th.joinable()) th.join();
  }
};

// completion flag a caller can wait on
struct Done {
  std::mutex m;
  std::condition_variable cv;
  bool done = false;
  int rc = FTKB_OK;
  void set(int r) { { std::lock_guard<std::mutex> lk(m); rc = r; done = true; } cv.notify_all(); }
  int wait() { std::unique_lock<std::mutex> lk(m); cv.wait(lk, [this] { return done; }); return rc; }
};

struct Chunk {
  int index = 0, device = 0;
  std::mutex m;                          // ctx: held by the worker around every call into it, and by the grower while it copies
  ftkb_ctx *ctx = nullptr;               // created by the device's worker when the chunk may start
  int confirmed = INT_MIN;               // streaming: the last timestep whose sweep ctx has confirmed (under the group's m)
  bool finished = false;                 // every sweep of the chunk has been confirmed
  double resolution_out = DBL_MAX;       // running minimum after the chunk (valid once finished)
  std::vector<ftkb_point> points;
  ftkb_stats stats{};
};

int nbits_of(double res) {
  if (!(res > 0) || res >= DBL_MAX) return 8;
  const int nb = (int)std::ceil(std::log2(1.0 / res));
  return nb < 8 ? 8 : (nb > 21 ? 21 : nb);
}

}  // namespace

// spatial mode (chunk_timesteps == 0, 3D): device s holds planes [a0, a1] of every snapshot -- its corner planes plus the ghost
// planes its stencils reach (the reference's spatial decomposition, regular_tracker.hh:126-149)
struct Slab {
  int device = 0, c0 = 0, c1 = 0, a0 = 0, a1 = 0;
  ftkb_ctx *ctx = nullptr;
  std::vector<ftkb_point> points;
  ftkb_stats stats{};
};

// an event a device push records on a producer's stream, kept by the group for the next push
struct ProducerEvent {
  cudaEvent_t ev = nullptr;
  int device = -1;
  cudaError_t record(cudaStream_t stream, int dev);
  void destroy();
};

struct ftkb_group {
  ftkb_config cfg{};
  std::vector<int> devices;
  int B = 8;
  bool spatial = false;
  std::vector<Slab> slabs;
  double running = DBL_MAX;                        // spatial mode: running minimum of min non-zero |v| over the whole array
  std::vector<std::unique_ptr<Worker>> workers;
  std::deque<std::unique_ptr<Chunk>> chunks;       // by index
  mutable std::mutex m;                            // protects chunk state shared between workers
  std::condition_variable cv;
  double saturating = 0.0;                         // a running minimum known to saturate the factor (0: not known yet)
  int npushed = 0, nadvanced = 0;
  int nintervals = 0;                              // intervals [t, t+1] swept so far, from start_timestep on
  bool streaming = false;                          // grow trajectories on the merged context (ftkb_group_set_streaming_trajectories)
  int coords_mode = FTKB_COORDS_SIMPLE;            // ftkb_group_set_coords, handed to every chunk context
  std::vector<double> coords;
  cudaStream_t producer = nullptr;                 // ftkb_group_set_producer_stream: device pushes wait for the work queued there
  bool has_producer = false;
  ProducerEvent ev_producer;                       // recorded on `producer` by every device push
  std::vector<ProducerEvent> ev_pieces;            // piece pushes: one per producer stream the pieces name
  std::atomic<int> failed{FTKB_OK};
  mutable std::string error;                       // (set by refusals of const queries too)
  ftkb_ctx *root = nullptr;
  // streaming: the merged context grows during the run
  std::mutex root_m;                               // root, while the grower may use it
  int imported = 0;                                // sweeps of timesteps start .. start + imported - 1 are in root (grown if intervals)
  std::thread grower;                              // time chunks: imports and grows in time order (grow_in_time_order)
  bool grower_stop = false;                        // (under m) finalize: every chunk has been imported

  Chunk *chunk(int c) {
    std::lock_guard<std::mutex> lk(m);
    while ((int)chunks.size() <= c) {
      std::unique_ptr<Chunk> ch(new Chunk());
      ch->index = (int)chunks.size();
      ch->device = devices[ch->index % devices.size()];
      chunks.push_back(std::move(ch));
    }
    return chunks[c].get();
  }
  void fail(int rc, const std::string &msg) {
    std::lock_guard<std::mutex> lk(m);
    if (failed.load() == FTKB_OK) { failed.store(rc); error = msg; }
    cv.notify_all();
  }
  // runs on the chunk's worker: wait until the chunk may start, then create its context
  int ensure_ctx(Chunk *ch) {
    if (ch->ctx) return FTKB_OK;
    double res_init = cfg.resolution_init;
    if (ch->index > 0) {
      std::unique_lock<std::mutex> lk(m);
      Chunk *prev = chunks[ch->index - 1].get();
      cv.wait(lk, [&] { return failed.load() != FTKB_OK || prev->finished || saturating > 0.0; });
      if (failed.load() != FTKB_OK) return failed.load();
      res_init = prev->finished ? prev->resolution_out : saturating;
      if (res_init >= DBL_MAX) res_init = 0.0;
    }
    ftkb_config c = cfg;
    c.device = ch->device;
    c.start_timestep = cfg.start_timestep + ch->index * B;
    c.resolution_init = res_init;
    ftkb_ctx *ctx = nullptr;
    int rc = ftkb_create(&c, &ctx);
    if (rc) { fail(rc, std::string("chunk context: ") + ftkb_last_error(nullptr)); return rc; }
    if (coords_mode != FTKB_COORDS_SIMPLE && (rc = ftkb_set_coords(ctx, coords_mode, coords.data(), coords.size())))
      fail(rc, std::string("chunk context: ") + ftkb_last_error(ctx));
    std::lock_guard<std::mutex> lk(ch->m);
    ch->ctx = ctx;
    return rc;
  }
  // streaming: tell the grower how far the chunk's context has confirmed its sweeps (ct from ftkb::confirmed_through)
  void note_confirmed(Chunk *ch, int ct) {
    { std::lock_guard<std::mutex> lk(m); ch->confirmed = ct; }
    cv.notify_all();
  }
  // after a sweep of a chunk: publish a saturating minimum as soon as one is known (lets the next chunk start early)
  void publish_resolution(Chunk *ch) {
    { std::lock_guard<std::mutex> lk(m); if (saturating > 0.0) return; }
    ftkb_stats st;
    if (ftkb_get_stats(ch->ctx, &st) != FTKB_OK) return;          // (confirms the chunk's sweeps: only until saturation is known)
    if (nbits_of(st.resolution) == 21) {
      { std::lock_guard<std::mutex> lk(m); saturating = st.resolution; }
      cv.notify_all();
    }
  }
  void finish_chunk(Chunk *ch) {
    ftkb_stats st{};
    int rc, last = INT_MIN;
    {
      std::lock_guard<std::mutex> lk(ch->m);
      rc = ftkb_get_stats(ch->ctx, &st);              // (confirms every sweep)
      last = ftkb::confirmed_through(ch->ctx);
      uint64_t n = 0;
      if (!rc && !streaming) rc = ftkb_num_points(ch->ctx, &n);
      if (!rc && !streaming) { ch->points.resize(n); rc = ftkb_get_points(ch->ctx, ch->points.data(), n); }
      if (rc) fail(rc, std::string("chunk ") + std::to_string(ch->index) + ": " + ftkb_last_error(ch->ctx));
    }
    if (streaming && !rc) {
      // the grower copies the points of every sweep from the chunk's device: the context stays until it has
      note_confirmed(ch, last);
      std::unique_lock<std::mutex> lk(m);
      cv.wait(lk, [&] { return failed.load() != FTKB_OK || cfg.start_timestep + imported > last; });
    }
    ch->stats = st;
    {
      std::lock_guard<std::mutex> lk(ch->m);
      ftkb_destroy(ch->ctx);            // its layers and buffers go back to the device; the points stay on the host (or in root)
      ch->ctx = nullptr;
    }
    { std::lock_guard<std::mutex> lk(m); ch->resolution_out = st.resolution; ch->finished = true; }
    cv.notify_all();
  }
};

extern "C" const char *ftkb_group_last_error(const ftkb_group *g) { return g ? g->error.c_str() : "null group"; }

extern "C" int ftkb_group_create(const ftkb_config *cfg, const int32_t *device_ids, int32_t n_devices, int32_t chunk_timesteps, ftkb_group **out) {
  if (!cfg || !out || !device_ids || n_devices < 1 || n_devices > 64 || chunk_timesteps < 0) return FTKB_ERR_INVALID;
  *out = nullptr;
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) { cudaGetLastError(); return FTKB_ERR_NO_DEVICE; }
  for (int i = 0; i < n_devices; i++)
    if (device_ids[i] < 0 || device_ids[i] >= ndev) return FTKB_ERR_NO_DEVICE;
  ftkb_group *g = new ftkb_group();
  g->cfg = *cfg;
  g->devices.assign(device_ids, device_ids + n_devices);
  g->B = chunk_timesteps;
  g->spatial = chunk_timesteps == 0;
  if (g->spatial) {
    // z-slabs: the domain's corner planes are split evenly; slab s also sweeps the corner plane above its last one (the flat
    // simplices of that plane are found twice and merged as one), and its array reaches two planes past every vertex it uses
    // (gradient of the Jacobian's neighbours); the first / last slab hold the array's end planes so that min non-zero |v|
    // still covers the whole array
    const int D = cfg->dims[2], glb = cfg->lb[2], gub = cfg->ub[2], nplanes = gub - glb + 1;
    if (cfg->nd != 3 || nplanes < 2 * n_devices) { delete g; return FTKB_ERR_INVALID; }
    g->running = cfg->resolution_init > 0 ? cfg->resolution_init : DBL_MAX;
    for (int s = 0; s < n_devices; s++) {
      Slab sl;
      sl.device = device_ids[s];
      const int c0 = glb + (int)((long long)nplanes * s / n_devices), c1 = glb + (int)((long long)nplanes * (s + 1) / n_devices) - 1;
      const int vtop = std::min(c1 + 1, gub);
      sl.c0 = c0;
      sl.c1 = c1;
      sl.a0 = s == 0 ? 0 : std::max(0, c0 - 2);
      sl.a1 = s == n_devices - 1 ? D - 1 : std::min(D - 1, vtop + 2);
      ftkb_config c = *cfg;
      c.device = sl.device;
      c.dims[2] = sl.a1 - sl.a0 + 1;
      c.lb[2] = c0 - sl.a0;
      c.ub[2] = vtop - sl.a0;
      c.slab_offset = sl.a0;
      c.slab_global_dim = D;
      c.slab_global_lb = glb;
      c.slab_global_ub = gub;
      const int rc = ftkb_create(&c, &sl.ctx);
      if (rc) {
        for (auto &x : g->slabs) ftkb_destroy(x.ctx);
        delete g;
        return rc;
      }
      g->slabs.push_back(sl);
    }
  }
  for (int i = 0; i < n_devices; i++) {
    g->workers.emplace_back(new Worker());
    g->workers.back()->start(device_ids[i]);
  }
  *out = g;
  return FTKB_OK;
}

extern "C" void ftkb_group_destroy(ftkb_group *g) {
  if (!g) return;
  g->fail(FTKB_ERR_INVALID, "group destroyed");            // releases workers that wait for a predecessor
  for (auto &w : g->workers) w->join();
  if (g->grower.joinable()) g->grower.join();
  for (auto &ch : g->chunks) if (ch->ctx) ftkb_destroy(ch->ctx);
  for (auto &sl : g->slabs) if (sl.ctx) ftkb_destroy(sl.ctx);
  if (g->root) ftkb_destroy(g->root);
  g->ev_producer.destroy();
  for (auto &e : g->ev_pieces) e.destroy();
  delete g;
}

// ---- streaming: the merged context grows during the run ---------------------------------------------------------------------
// one timestep into the merged context: the points of its sweep from every context that swept it, then the grow step if that sweep
// covered an interval (the last ordinal sweep's points are imported and never grown)
static int import_and_grow(ftkb_group *g, const std::vector<ftkb_ctx *> &from, int t) {
  bool interval = false;
  for (ftkb_ctx *c : from) {
    bool iv = false;
    const int rc = ftkb::import_step(g->root, c, t, &iv);
    if (rc) return rc;
    interval = interval || iv;
  }
  return interval ? ftkb::grow_imported(g->root, t) : FTKB_OK;
}

// time chunks: the grower thread.  Timestep t is imported and grown once the chunk that owns it has confirmed its sweep and t-1
// is done; it stops when finalize says every chunk has been imported, or at the first failure.
static void grow_in_time_order(ftkb_group *g) {
  for (;;) {
    const int t = g->cfg.start_timestep + g->imported;
    const size_t c = (size_t)(g->imported / g->B);
    Chunk *ch = nullptr;
    {
      std::unique_lock<std::mutex> lk(g->m);
      auto ready = [&] { return c < g->chunks.size() && g->chunks[c]->confirmed >= t; };
      g->cv.wait(lk, [&] { return g->failed.load() != FTKB_OK || g->grower_stop || ready(); });
      if (g->failed.load() != FTKB_OK || !ready()) return;
      ch = g->chunks[c].get();
    }
    int rc;
    std::string msg;
    {
      std::lock_guard<std::mutex> rl(g->root_m);
      std::lock_guard<std::mutex> cl(ch->m);
      // (no context: a failure elsewhere let its chunk finish without waiting)
      rc = ch->ctx ? import_and_grow(g, {ch->ctx}, t) : FTKB_ERR_INVALID;
      if (rc) msg = ch->ctx ? ftkb_last_error(g->root) : "the chunk's context is gone";
    }
    if (rc) { g->fail(rc, "streaming grow of timestep " + std::to_string(t) + ": " + msg); return; }
    { std::lock_guard<std::mutex> lk(g->m); g->imported++; }
    g->cv.notify_all();
  }
}

// the merged context of a streaming group, from its first push on (and, for time chunks, its grower)
static int ensure_root(ftkb_group *g) {
  if (!g->streaming || g->root) return FTKB_OK;
  ftkb_config c = g->cfg;
  c.device = g->devices[0];
  int rc = ftkb_create(&c, &g->root);
  if (rc) { g->error = std::string("merged context: ") + ftkb_last_error(nullptr); return rc; }
  if ((rc = ftkb_set_streaming_trajectories(g->root, 1))) { g->error = std::string("merged context: ") + ftkb_last_error(g->root); return rc; }
  if (!g->spatial) g->grower = std::thread(grow_in_time_order, g);
  return FTKB_OK;
}

// z-slabs, on the caller's thread while the workers are idle: every timestep that all slabs have confirmed since the last call,
// in time order, the slabs' points in slab order (the flat simplices of a cut plane come twice: the grow step's sort drops one)
static int slabs_grow(ftkb_group *g) {
  if (!g->streaming) return FTKB_OK;
  std::vector<ftkb_ctx *> from;
  for (Slab &sl : g->slabs) from.push_back(sl.ctx);
  for (;;) {
    const int t = g->cfg.start_timestep + g->imported;
    for (ftkb_ctx *c : from) if (ftkb::confirmed_through(c) < t) return FTKB_OK;
    const int rc = import_and_grow(g, from, t);
    if (rc) { g->error = "streaming grow of timestep " + std::to_string(t) + ": " + ftkb_last_error(g->root); return rc; }
    g->imported++;
  }
}

// ---- spatial mode: every device works on every step ------------------------------------------------------------------------
// run f(slab) on every device's worker and wait for all
static int on_all_slabs(ftkb_group *g, std::function<int(Slab &)> f, const char *what) {
  std::vector<std::shared_ptr<Done>> waits;
  for (size_t s = 0; s < g->slabs.size(); s++) {
    std::shared_ptr<Done> d(new Done());
    waits.push_back(d);
    Slab *sl = &g->slabs[s];
    g->workers[s]->post([g, sl, f, d, what] {
      int rc = g->failed.load();
      if (!rc) {
        rc = f(*sl);
        if (rc) g->fail(rc, std::string(what) + ": " + ftkb_last_error(sl->ctx));
      }
      d->set(rc);
    });
  }
  int rc = FTKB_OK;
  for (auto &d : waits) { const int r = d->wait(); if (r && !rc) rc = r; }
  return rc;
}

// The quantisation factor must be the undivided run's on every slab: until the running minimum saturates it, the slabs
// resolve the new layer first (a cells-only build for scalar input, a reduction for vector input), the minima are combined
// and handed back before anyone sweeps.  Once saturated (nbits = 21) nothing can change the factor and the step is skipped.
static int spatial_sync_resolution(ftkb_group *g) {
  if (nbits_of(g->running) == 21) return FTKB_OK;
  std::vector<double> res(g->slabs.size(), DBL_MAX);
  int rc = on_all_slabs(g, [&](Slab &sl) { return ftkb_last_layer_resolution(sl.ctx, &res[&sl - g->slabs.data()]); }, "resolution");
  if (rc) return rc;
  for (double r : res) if (r > 0 && r < g->running) g->running = r;
  if (g->running < DBL_MAX) {
    const double run = g->running;
    rc = on_all_slabs(g, [run](Slab &sl) { return ftkb_set_resolution(sl.ctx, run); }, "set_resolution");
  }
  return rc;
}

static int spatial_push(ftkb_group *g, std::function<int(Slab &)> push) {
  int rc = on_all_slabs(g, push, "push");
  if (!rc) rc = spatial_sync_resolution(g);
  g->npushed++;
  return rc;
}

// ---- options: set before the first push ---------------------------------------------------------------------------------------
extern "C" int ftkb_group_set_coords(ftkb_group *g, int mode, const double *data, uint64_t n) {
  if (!g) return FTKB_ERR_INVALID;
  if (g->npushed) { g->error = "set_coords: call it before the first push"; return FTKB_ERR_INVALID; }
  // the sizes of ftkb_set_coords, in the whole array's frame (a chunk context checks them again when it is created)
  const uint64_t W = g->cfg.dims[0], H = g->cfg.dims[1], D = g->cfg.nd == 3 ? g->cfg.dims[2] : 0, nd = g->cfg.nd;
  const bool ok = mode == FTKB_COORDS_SIMPLE ||
                  (data && ((mode == FTKB_COORDS_BOUNDS && n == 2 * nd) || (mode == FTKB_COORDS_RECTILINEAR && n == W + H + D) ||
                            (mode == FTKB_COORDS_EXPLICIT && n % (W * H) == 0 && n / (W * H) >= nd)));
  if (!ok) { g->error = "set_coords: unknown mode, or a size that does not fit the array"; return FTKB_ERR_INVALID; }
  g->coords_mode = mode;
  g->coords.assign(data, data + (mode == FTKB_COORDS_SIMPLE ? 0 : n));
  if (!g->spatial) return FTKB_OK;
  return on_all_slabs(g, [g](Slab &sl) { return ftkb_set_coords(sl.ctx, g->coords_mode, g->coords.data(), g->coords.size()); }, "set_coords");
}

extern "C" int ftkb_group_set_streaming_trajectories(ftkb_group *g, int enable) {
  if (!g) return FTKB_ERR_INVALID;
  if (g->npushed) { g->error = "set_streaming_trajectories: call it before the first push"; return FTKB_ERR_INVALID; }
  g->streaming = enable != 0;
  return FTKB_OK;
}

// hand one snapshot to chunk c's context (runs on that device's worker)
static void post_push(ftkb_group *g, int c, std::function<int(ftkb_ctx *)> push, std::shared_ptr<Done> done) {
  Chunk *ch = g->chunk(c);
  Worker *w = g->workers[ch->index % g->workers.size()].get();
  w->post([g, ch, push, done] {
    int rc = g->failed.load();
    if (!rc) rc = g->ensure_ctx(ch);
    if (!rc) {
      std::lock_guard<std::mutex> lk(ch->m);
      rc = push(ch->ctx);
      if (rc) g->fail(rc, std::string("push: ") + ftkb_last_error(ch->ctx));
    }
    if (done) done->set(rc);
  });
}

static int push_layer(ftkb_group *g, std::function<int(ftkb_ctx *)> push, bool wait) {
  if (g->failed.load()) return g->failed.load();
  const int k = g->npushed++;
  const int c = k / g->B;
  std::vector<std::shared_ptr<Done>> waits;
  auto mk = [&]() -> std::shared_ptr<Done> { if (!wait) return nullptr; waits.emplace_back(new Done()); return waits.back(); };
  // the first layer of a chunk is also the last layer (halo) of the chunk before it
  if (k % g->B == 0 && k > 0) post_push(g, c - 1, push, mk());
  post_push(g, c, push, mk());
  int rc = FTKB_OK;
  for (auto &d : waits) { const int r = d->wait(); if (r && !rc) rc = r; }
  return rc;
}

// Where a snapshot's arrays come from: pieces that tile the whole array in plane order along its slowest axis (z in 3D, y in 2D),
// in the whole array's frame.  Host memory comes as one piece; CUDA device memory as one piece or several, each on any device
// (in the group or not), every copy from a piece ordered after its `after` when that is set.  Either way the arrays are borrowed
// only until the push returns.
struct Source {
  bool on_device = false;
  std::vector<ftkb::Segment> pieces;
  size_t plane = 0, n = 0;                     // doubles per plane of a scalar array; components per vertex of a vector
  Source(const ftkb_config &cfg, bool device) : on_device(device), n((size_t)cfg.nd) {
    plane = (size_t)cfg.dims[0] * (cfg.nd == 3 ? (size_t)cfg.dims[1] : 1);
  }
  int extent() const { return pieces.back().first + pieces.back().count; }
  // the plan for a destination that holds planes [a0, a1]: one segment per intersecting piece, in the destination's frame
  std::vector<ftkb::Segment> cut(int a0, int a1) const {
    std::vector<ftkb::Segment> out;
    for (const ftkb::Segment &p : pieces) {
      const int lo = std::max(a0, p.first), hi = std::min(a1 + 1, p.first + p.count);
      if (lo >= hi) continue;
      const size_t o = plane * (size_t)(lo - p.first);
      ftkb::Segment s = p;
      s.first = lo - a0;
      s.count = hi - lo;
      s.scalar = p.scalar ? p.scalar + o : nullptr;
      s.vector = p.vector ? p.vector + n * o : nullptr;
      s.jacobian = p.jacobian ? p.jacobian + n * n * o : nullptr;
      out.push_back(s);
    }
    return out;
  }
  int push(ftkb_ctx *c, int a0, int a1) const {
    const std::vector<ftkb::Segment> segs = cut(a0, a1);
    if (!on_device) return ftkb_push_snapshot(c, segs[0].scalar, segs[0].vector, segs[0].jacobian, FTKB_MEM_HOST);
    return ftkb::push_segments(c, segs.data(), (int)segs.size());
  }
};

// The first layer of chunk c > 0 arrives while chunk c-1 may still have to finish before chunk c's context can exist (it
// inherits the running minimum), and chunk c-1 finishes with an advance the caller only issues after this push has returned.
// So that layer is copied to the new chunk's device right away, into buffers of the group, and handed to the context later.
struct Staged { double *S = nullptr, *V = nullptr, *J = nullptr; };

static int push_snapshot(ftkb_group *g, const Source src) {
  { const int rc = ensure_root(g); if (rc) return rc; }
  const int last = src.extent() - 1;
  if (g->spatial)
    // every device copies its planes (ghost planes included) over its own link, concurrently
    return spatial_push(g, [=](Slab &sl) { return src.push(sl.ctx, sl.a0, sl.a1); });
  const int k = g->npushed;
  if (k % g->B != 0 || k == 0)
    // borrowed until return: wait for the copy
    return push_layer(g, [=](ftkb_ctx *c) { return src.push(c, 0, last); }, true);
  g->npushed++;
  const int c = k / g->B;
  std::shared_ptr<Done> d_halo(new Done()), d_stage(new Done());
  post_push(g, c - 1, [=](ftkb_ctx *x) { return src.push(x, 0, last); }, d_halo);   // halo of the chunk before
  Chunk *ch = g->chunk(c);
  Worker *w = g->workers[ch->index % g->workers.size()].get();
  std::shared_ptr<Staged> st(new Staged());
  w->post([=] {
    int rc = g->failed.load();
    cudaStream_t s = nullptr;      // device source: the copies run here, after the producers
    auto ck = [&](cudaError_t e) {
      if (e == cudaSuccess || rc) return;
      cudaGetLastError();
      rc = e == cudaErrorMemoryAllocation ? FTKB_ERR_NOMEM : FTKB_ERR_CUDA;
      g->fail(rc, std::string("group: staging the first layer of a chunk failed: ") + cudaGetErrorString(e));
    };
    auto up = [&](const double *ftkb::Segment::*a, size_t per, double **dst) {
      if (!(src.pieces[0].*a) || rc) return;
      ck(cudaMalloc(dst, src.plane * per * (last + 1) * sizeof(double)));
      for (const ftkb::Segment &p : src.pieces) {
        if (rc) return;
        double *to = *dst + src.plane * per * (size_t)p.first;
        const size_t bytes = src.plane * per * (size_t)p.count * sizeof(double);
        if (!src.on_device) ck(cudaMemcpy(to, p.*a, bytes, cudaMemcpyHostToDevice));
        else if (p.device == ch->device) ck(cudaMemcpyAsync(to, p.*a, bytes, cudaMemcpyDeviceToDevice, s));
        else ck(cudaMemcpyPeerAsync(to, ch->device, p.*a, p.device, bytes, s));
      }
    };
    if (!rc) ck(cudaSetDevice(ch->device));
    if (src.on_device) {
      for (const ftkb::Segment &p : src.pieces) ck(ftkb::enable_peer_access(ch->device, p.device));
      ck(cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking));
      for (const ftkb::Segment &p : src.pieces)
        if (p.after) ck(cudaStreamWaitEvent(s, p.after, 0));
    }
    up(&ftkb::Segment::scalar, 1, &st->S); up(&ftkb::Segment::vector, src.n, &st->V); up(&ftkb::Segment::jacobian, src.n * src.n, &st->J);
    if (s) { ck(cudaStreamSynchronize(s)); cudaStreamDestroy(s); }
    d_stage->set(rc);
  });
  w->post([=] {
    int rc = g->failed.load();
    if (!rc) rc = g->ensure_ctx(ch);
    if (!rc) {
      std::lock_guard<std::mutex> lk(ch->m);
      rc = ftkb_push_snapshot(ch->ctx, st->S, st->V, st->J, FTKB_MEM_DEVICE);      // copied (and synchronised) before it returns
      if (rc) g->fail(rc, std::string("push: ") + ftkb_last_error(ch->ctx));
    }
    cudaSetDevice(ch->device);
    cudaFree(st->S); cudaFree(st->V); cudaFree(st->J);
  });
  const int r1 = d_halo->wait(), r2 = d_stage->wait();
  return r1 ? r1 : r2;
}

// the whole array as one piece
static Source whole(const ftkb_group *g, const double *scalar, const double *vector, const double *jacobian, bool on_device, int device,
                    cudaEvent_t after) {
  Source src(g->cfg, on_device);
  ftkb::Segment p;
  p.count = g->cfg.dims[g->cfg.nd - 1];
  p.scalar = scalar; p.vector = vector; p.jacobian = jacobian;
  p.device = device;
  p.after = after;
  src.pieces.push_back(p);
  return src;
}

extern "C" int ftkb_group_push_snapshot(ftkb_group *g, const double *scalar, const double *vector, const double *jacobian) {
  if (!g) return FTKB_ERR_INVALID;
  if (g->failed.load()) return g->failed.load();
  return push_snapshot(g, whole(g, scalar, vector, jacobian, false, -1, nullptr));
}

extern "C" int ftkb_group_set_producer_stream(ftkb_group *g, void *stream, int enable) {
  if (!g) return FTKB_ERR_INVALID;
  g->producer = reinterpret_cast<cudaStream_t>(stream);
  g->has_producer = enable != 0;
  return FTKB_OK;
}

// The checks a device push makes of its arrays (the whole snapshot, or one piece of it): every non-null array is CUDA device
// memory, 8-byte aligned, and on the same device as the others, which goes to *device.  Returns what is wrong, or "".
static std::string device_of(const double *const arrays[3], int *device) {
  static const char *const names[3] = {"scalar", "vector", "jacobian"};
  *device = -1;
  for (int i = 0; i < 3; i++) {
    if (!arrays[i]) continue;
    cudaPointerAttributes a{};
    if (cudaPointerGetAttributes(&a, arrays[i]) != cudaSuccess) { cudaGetLastError(); a.type = cudaMemoryTypeUnregistered; }
    if (a.type != cudaMemoryTypeDevice) return std::string("the ") + names[i] + " array is not CUDA device memory (host, unregistered and managed memory are refused)";
    if ((uintptr_t)arrays[i] % 8 != 0) return std::string("the ") + names[i] + " array is not 8-byte aligned";
    if (*device >= 0 && a.device != *device) return std::string("the ") + names[i] + " array is on another device than the arrays before it";
    *device = a.device;
  }
  return *device < 0 ? "no array was passed" : "";
}

// Records `ev` on `stream`, which lives on `dev` (NULL: the legacy default stream of `dev`), creating it there, or again when
// the event it kept from an earlier push is on another device.
cudaError_t ProducerEvent::record(cudaStream_t stream, int dev) {
  int cur = 0;
  cudaError_t e = cudaGetDevice(&cur);
  if (!e) e = cudaSetDevice(dev);
  if (!e && ev && device != dev) { e = cudaEventDestroy(ev); ev = nullptr; }
  if (!e && !ev && !(e = cudaEventCreateWithFlags(&ev, cudaEventDisableTiming))) device = dev;
  if (!e) e = cudaEventRecord(ev, stream);
  cudaSetDevice(cur);
  if (e) cudaGetLastError();
  return e;
}

void ProducerEvent::destroy() {
  if (!ev) return;
  int cur = 0;
  cudaGetDevice(&cur);
  cudaSetDevice(device);
  cudaEventDestroy(ev);
  cudaSetDevice(cur);
  ev = nullptr;
}

extern "C" int ftkb_group_push_snapshot_device(ftkb_group *g, const double *scalar, const double *vector, const double *jacobian) {
  if (!g) return FTKB_ERR_INVALID;
  if (g->failed.load()) return g->failed.load();
  // a rejected push leaves the group as it was: the caller may push a valid snapshot next
  auto reject = [g](const std::string &msg) { std::lock_guard<std::mutex> lk(g->m); g->error = "push_snapshot_device: " + msg; return FTKB_ERR_INVALID; };
  const double *arrays[3] = {scalar, vector, jacobian};
  int device = -1;
  const std::string why = device_of(arrays, &device);
  if (!why.empty()) return reject(why);
  cudaEvent_t after = nullptr;
  if (g->has_producer) {
    // one event is enough: this push returns only after every copy that waits for it has completed.  The stream may live on
    // another device than the arrays: `device` stays the arrays' own, the source of every copy.
    int stream_device = device;
    if (g->producer && cudaStreamGetDevice(g->producer, &stream_device) != cudaSuccess) { cudaGetLastError(); return reject("the producer stream is not a valid CUDA stream"); }
    const cudaError_t e = g->ev_producer.record(g->producer, stream_device);
    if (e) { std::lock_guard<std::mutex> lk(g->m); g->error = std::string("push_snapshot_device: producer event: ") + cudaGetErrorString(e); return FTKB_ERR_CUDA; }
    after = g->ev_producer.ev;
  }
  return push_snapshot(g, whole(g, scalar, vector, jacobian, true, device, after));
}

extern "C" int ftkb_group_push_pieces_device(ftkb_group *g, const ftkb_piece *pieces, int32_t n) {
  if (!g) return FTKB_ERR_INVALID;
  if (g->failed.load()) return g->failed.load();
  // everything is checked before anything is enqueued: a rejected push leaves the group as it was
  auto reject = [g](const std::string &msg) { std::lock_guard<std::mutex> lk(g->m); g->error = "push_pieces_device: " + msg; return FTKB_ERR_INVALID; };
  if (!pieces || n < 1) return reject("no pieces were passed (n = " + std::to_string(n) + ")");
  const ftkb_config &cfg = g->cfg;
  const long long extent = cfg.dims[cfg.nd - 1];
  const char *axis = cfg.nd == 3 ? "z plane" : "y row";
  Source src(cfg, true);
  std::vector<int> stream_devices;         // the device of every piece's stream (NULL: the legacy stream of the piece's device)
  long long next = 0;
  for (int i = 0; i < n; i++) {
    const ftkb_piece &p = pieces[i];
    const std::string who = "piece " + std::to_string(i) + ": ";
    if (p.count < 1) return reject(who + "count is " + std::to_string(p.count) + " (a piece holds at least one " + axis + ")");
    if (p.first != next)
      return reject(who + "starts at " + axis + " " + std::to_string(p.first) + " where " + std::to_string(next) + " was expected (" +
                    (p.first > next ? "a gap" : "an overlap, or pieces out of order") + "; pieces tile the array in order)");
    if (next + p.count > extent)
      return reject(who + "ends at " + axis + " " + std::to_string(next + p.count) + ", past the array's " + std::to_string(extent));
    next += p.count;
    const double *arrays[3] = {p.scalar, p.vector, p.jacobian}, *first[3] = {pieces[0].scalar, pieces[0].vector, pieces[0].jacobian};
    static const char *const names[3] = {"scalar", "vector", "jacobian"};
    for (int a = 0; a < 3; a++)
      if (!arrays[a] != !first[a])
        return reject(who + (arrays[a] ? "passes a " : "lacks the ") + names[a] + " array" + (arrays[a] ? " that piece 0 lacks" : " that piece 0 passes") +
                      " (every piece passes the same arrays)");
    int device = -1;
    const std::string why = device_of(arrays, &device);
    if (!why.empty()) return reject(who + why);
    int stream_device = device;
    if (p.has_stream && p.stream && cudaStreamGetDevice(reinterpret_cast<cudaStream_t>(p.stream), &stream_device) != cudaSuccess) {
      cudaGetLastError();
      return reject(who + "its stream is not a valid CUDA stream");
    }
    ftkb::Segment s;
    s.first = p.first; s.count = p.count;
    s.scalar = p.scalar; s.vector = p.vector; s.jacobian = p.jacobian;
    s.device = device;
    src.pieces.push_back(s);
    stream_devices.push_back(stream_device);
  }
  if (next != extent)
    return reject("piece " + std::to_string(n - 1) + ": the pieces end at " + axis + " " + std::to_string(next) + ", the array has " + std::to_string(extent));
  const ftkb_piece &p0 = pieces[0];
  if ((cfg.scalar_source == FTKB_SOURCE_GIVEN && !p0.scalar) || (cfg.vector_source == FTKB_SOURCE_DERIVED && !p0.vector && !p0.scalar))
    return reject("piece 0: lacks the scalar array, which the configuration's sources need");
  if (cfg.vector_source == FTKB_SOURCE_GIVEN && !p0.vector) return reject("piece 0: lacks the vector array, which the configuration's sources need");
  if (cfg.jacobian_source == FTKB_SOURCE_GIVEN && !p0.jacobian) return reject("piece 0: lacks the jacobian array, which the configuration's sources need");
  // one event per producer stream named by the pieces (pieces written by the same stream share it), kept for the next push:
  // enough for the same reason as ftkb_group_set_producer_stream's single event
  std::vector<std::pair<cudaStream_t, int>> streams;
  for (int i = 0; i < n; i++) {
    if (!pieces[i].has_stream) continue;
    const std::pair<cudaStream_t, int> key(reinterpret_cast<cudaStream_t>(pieces[i].stream), stream_devices[i]);
    size_t e = std::find(streams.begin(), streams.end(), key) - streams.begin();
    if (e == streams.size()) {
      streams.push_back(key);
      if (g->ev_pieces.size() < streams.size()) g->ev_pieces.emplace_back();
      const cudaError_t r = g->ev_pieces[e].record(key.first, key.second);
      if (r) { std::lock_guard<std::mutex> lk(g->m); g->error = "push_pieces_device: piece " + std::to_string(i) + ": producer event: " + cudaGetErrorString(r); return FTKB_ERR_CUDA; }
    }
    src.pieces[i].after = g->ev_pieces[e].ev;
  }
  return push_snapshot(g, src);
}

extern "C" int ftkb_group_get_slab(const ftkb_group *g, int32_t s, int32_t planes[4]) {
  if (!g || !planes) return FTKB_ERR_INVALID;
  if (!g->spatial || s < 0 || s >= (int32_t)g->slabs.size()) {
    std::lock_guard<std::mutex> lk(g->m);
    g->error = !g->spatial ? "get_slab: the group runs time chunks, not z-slabs"
                           : "get_slab: slab " + std::to_string(s) + " does not exist (the group has " + std::to_string(g->slabs.size()) + ")";
    return FTKB_ERR_INVALID;
  }
  const Slab &sl = g->slabs[s];
  planes[0] = sl.c0; planes[1] = sl.c1; planes[2] = sl.a0; planes[3] = sl.a1;
  return FTKB_OK;
}

extern "C" int ftkb_group_push_synthetic(ftkb_group *g, int kind, const double *params, int nparams, double t) {
  if (!g || nparams < 0 || nparams > 8 || (nparams && !params)) return FTKB_ERR_INVALID;
  std::vector<double> p(params, params + nparams);
  { const int rc = ensure_root(g); if (rc) return rc; }
  if (g->spatial) return spatial_push(g, [=](Slab &sl) { return ftkb_push_synthetic(sl.ctx, kind, p.data(), (int)p.size(), t); });
  return push_layer(g, [=](ftkb_ctx *c) { return ftkb_push_synthetic(c, kind, p.data(), (int)p.size(), t); }, false);
}

static int post_sweep(ftkb_group *g, int step, bool advance) {
  if (g->failed.load()) return g->failed.load();
  const int c = step / g->B;
  Chunk *ch = g->chunk(c);
  Worker *w = g->workers[ch->index % g->workers.size()].get();
  const bool last_of_chunk = advance && (step + 1) % g->B == 0;
  w->post([g, ch, advance, last_of_chunk] {
    int rc = g->failed.load();
    if (!rc) rc = g->ensure_ctx(ch);
    if (rc) return;
    int ct = INT_MIN;
    {
      std::lock_guard<std::mutex> lk(ch->m);
      rc = advance ? ftkb_advance_timestep(ch->ctx) : ftkb_update_timestep(ch->ctx);
      if (rc) { g->fail(rc, std::string("sweep: ") + ftkb_last_error(ch->ctx)); return; }
      g->publish_resolution(ch);
      ct = ftkb::confirmed_through(ch->ctx);
    }
    if (g->streaming) g->note_confirmed(ch, ct);
    if (last_of_chunk || !advance) g->finish_chunk(ch);
  });
  return FTKB_OK;
}

extern "C" int ftkb_group_advance_timestep(ftkb_group *g) {
  if (!g) return FTKB_ERR_INVALID;
  if (g->npushed < g->nadvanced + 2) { g->error = "advance_timestep: two snapshots are needed"; return FTKB_ERR_INVALID; }
  g->nintervals = std::max(g->nintervals, g->nadvanced + 1);
  if (g->spatial) {
    g->nadvanced++;
    const int rc = on_all_slabs(g, [](Slab &sl) { return ftkb_advance_timestep(sl.ctx); }, "sweep");
    return rc ? rc : slabs_grow(g);
  }
  return post_sweep(g, g->nadvanced++, true);
}

extern "C" int ftkb_group_update_timestep(ftkb_group *g) {
  if (!g) return FTKB_ERR_INVALID;
  if (g->npushed < g->nadvanced + 1) { g->error = "update_timestep: no snapshot has been pushed"; return FTKB_ERR_INVALID; }
  if (g->npushed >= g->nadvanced + 2) g->nintervals = std::max(g->nintervals, g->nadvanced + 1);     // the next snapshot is there
  if (g->spatial) {
    const int rc = on_all_slabs(g, [](Slab &sl) { return ftkb_update_timestep(sl.ctx); }, "sweep");
    return rc ? rc : slabs_grow(g);
  }
  return post_sweep(g, g->nadvanced, false);
}

// The merged context on the first device: the punctured simplices of every chunk or slab, sorted and deduplicated there, then
// traced offline -- or, with streaming trajectories, the context that has grown them during the run: it publishes what it grew.
static int build_root(ftkb_group *g, const std::vector<const std::vector<ftkb_point> *> &parts) {
  int rc = FTKB_OK;
  if (g->streaming) {
    if ((rc = ensure_root(g))) return rc;
  } else {
    if (g->root) { ftkb_destroy(g->root); g->root = nullptr; }
    ftkb_config c = g->cfg;
    c.device = g->devices[0];
    rc = ftkb_create(&c, &g->root);
    if (rc) { g->error = ftkb_last_error(nullptr); return rc; }
    // (the flat simplices of a cut plane were found by both neighbouring slabs: the root's sort drops the duplicates)
    for (auto *p : parts)
      if (!rc && !p->empty()) rc = ftkb_import_points(g->root, p->data(), p->size());
  }
  if (!rc) rc = ftkb_finalize(g->root);
  if (rc) g->error = ftkb_last_error(g->root);
  return rc;
}

extern "C" int ftkb_group_finalize(ftkb_group *g, ftkb_ctx **root) {
  if (!g || !root) return FTKB_ERR_INVALID;
  *root = nullptr;
  if (g->spatial) {
    const bool streaming = g->streaming;
    int rc = on_all_slabs(g, [streaming](Slab &sl) {
      uint64_t n = 0;
      int r = ftkb_get_stats(sl.ctx, &sl.stats);
      if (!r && !streaming) r = ftkb_num_points(sl.ctx, &n);
      if (!r && !streaming) { sl.points.resize(n); r = ftkb_get_points(sl.ctx, sl.points.data(), n); }
      return r;
    }, "collect");
    if (!rc) rc = slabs_grow(g);     // streaming: what the last sweeps confirmed, the last ordinal sweep included
    if (rc) return rc;
    std::vector<const std::vector<ftkb_point> *> parts;
    for (auto &sl : g->slabs) parts.push_back(&sl.points);
    if ((rc = build_root(g, parts))) return rc;
    *root = g->root;
    return FTKB_OK;
  }
  // wait for every device's queue to drain
  std::vector<std::shared_ptr<Done>> waits;
  for (auto &w : g->workers) {
    std::shared_ptr<Done> d(new Done());
    waits.push_back(d);
    w->post([d] { d->set(FTKB_OK); });
  }
  for (auto &d : waits) d->wait();
  if (g->failed.load()) return g->failed.load();
  // chunks that never reached their last sweep (the series ended inside them, without a final update): collect them as they are
  for (auto &ch : g->chunks)
    if (ch->ctx && !ch->finished) g->finish_chunk(ch.get());
  if (g->grower.joinable()) {
    // every chunk has finished, so every sweep has been imported: the grower has nothing left to wait for
    { std::lock_guard<std::mutex> lk(g->m); g->grower_stop = true; }
    g->cv.notify_all();
    g->grower.join();
  }
  if (g->failed.load()) return g->failed.load();
  std::vector<const std::vector<ftkb_point> *> parts;
  for (auto &ch : g->chunks) parts.push_back(&ch->points);
  const int rc = build_root(g, parts);
  if (rc) return rc;
  *root = g->root;
  return FTKB_OK;
}

extern "C" int ftkb_group_get_live_curveset(ftkb_group *g, int32_t *grown_through, ftkb_curveset **out) {
  if (!g) return FTKB_ERR_INVALID;
  auto refuse = [g](const std::string &msg) { std::lock_guard<std::mutex> lk(g->m); g->error = "get_live_curveset: " + msg; return FTKB_ERR_INVALID; };
  if (!grown_through || !out) return refuse("null argument");
  *out = nullptr;
  if (!g->streaming) return refuse("streaming trajectories are off (ftkb_group_set_streaming_trajectories)");
  if (g->failed.load()) return g->failed.load();
  int rc = ensure_root(g);
  if (rc) return rc;
  if (g->spatial) {
    // confirm the slabs' deferred sweeps, then import and grow them
    rc = on_all_slabs(g, [](Slab &sl) { ftkb_stats st; return ftkb_get_stats(sl.ctx, &st); }, "confirm");
    if (!rc) rc = slabs_grow(g);
    if (rc) return rc;
  } else if (g->nintervals > 0) {
    // the chunk that swept the last interval confirms it (its worker runs this behind that sweep), then the grower catches up
    Chunk *ch = g->chunk((g->nintervals - 1) / g->B);
    g->workers[ch->index % g->workers.size()]->post([g, ch] {
      int ct = INT_MIN;
      {
        std::lock_guard<std::mutex> lk(ch->m);
        if (!ch->ctx) return;
        ftkb_stats st;
        const int r = ftkb_get_stats(ch->ctx, &st);
        if (r) { g->fail(r, std::string("confirm: ") + ftkb_last_error(ch->ctx)); return; }
        ct = ftkb::confirmed_through(ch->ctx);
      }
      g->note_confirmed(ch, ct);
    });
    std::unique_lock<std::mutex> lk(g->m);
    g->cv.wait(lk, [g] { return g->failed.load() != FTKB_OK || g->imported >= g->nintervals; });
    if (g->failed.load()) return g->failed.load();
  }
  std::lock_guard<std::mutex> rl(g->root_m);
  rc = ftkb_get_live_curveset(g->root, grown_through, out);
  if (rc) { std::lock_guard<std::mutex> lk(g->m); g->error = std::string("get_live_curveset: ") + ftkb_last_error(g->root); }
  return rc;
}

extern "C" int ftkb_group_get_stats(ftkb_group *g, ftkb_stats *sum, int32_t *chunks_done) {
  if (!g || !sum) return FTKB_ERR_INVALID;
  std::lock_guard<std::mutex> lk(g->m);
  ftkb_stats s{};
  int done = 0;
  for (auto &sl : g->slabs) {          // spatial mode: as collected by ftkb_group_finalize
    const ftkb_stats &t = sl.stats;
    s.simplices_tested += t.simplices_tested; s.cells_scanned += t.cells_scanned; s.cells_refined += t.cells_refined;
    s.points += t.points; s.kernel_launches += t.kernel_launches; s.h2d_bytes += t.h2d_bytes; s.d2h_bytes += t.d2h_bytes;
    s.ms_derive += t.ms_derive; s.ms_scan += t.ms_scan; s.ms_test += t.ms_test;
    s.scan_launches += t.scan_launches; s.sweeps_repeated += t.sweeps_repeated;
    s.scaling_factor = t.scaling_factor; s.resolution = t.resolution;
    done++;
  }
  for (auto &ch : g->chunks) {
    if (!ch->finished) continue;
    done++;
    const ftkb_stats &t = ch->stats;
    s.simplices_tested += t.simplices_tested; s.cells_scanned += t.cells_scanned; s.cells_refined += t.cells_refined;
    s.points += t.points; s.kernel_launches += t.kernel_launches; s.h2d_bytes += t.h2d_bytes; s.d2h_bytes += t.d2h_bytes;
    s.ms_derive += t.ms_derive; s.ms_scan += t.ms_scan; s.ms_test += t.ms_test;
    s.scan_launches += t.scan_launches; s.sweeps_repeated += t.sweeps_repeated;
    s.scaling_factor = t.scaling_factor; s.resolution = t.resolution;
  }
  *sum = s;
  if (chunks_done) *chunks_done = done;
  return FTKB_OK;
}
