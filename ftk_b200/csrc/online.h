// Streaming trajectories: the reference's trace_critical_points_online (critical_point_tracker.hh:522-641),
// the grow step run after every interval sweep when set_enable_streaming_trajectories(true).
#pragma once
#include <cstdint>
#include <deque>
#include <vector>

#include <cuda_runtime.h>

#include "../../include/ftkb200.h"
#include "mesh_tables.h"

namespace ftkb {

// a trajectory = indices into OnlineTracer::keys() / point() (every punctured simplex is stored once, in the order it arrived)
struct OnlineCurve {
  std::deque<uint32_t> idx;
  bool loop = false, complete = false;
  OnlineCurve() = default;
  OnlineCurve(const OnlineCurve &) = default;
  OnlineCurve &operator=(const OnlineCurve &) = default;
  // noexcept so that a growing std::vector<OnlineCurve> moves its curves instead of copying them
  OnlineCurve(OnlineCurve &&o) noexcept : idx(std::move(o.idx)), loop(o.loop), complete(o.complete) {}
  OnlineCurve &operator=(OnlineCurve &&o) noexcept { idx = std::move(o.idx); loop = o.loop; complete = o.complete; return *this; }
};

class OnlineTracer {
 public:
  OnlineTracer(int nd, const int32_t lb[3], const int32_t ub[3]);
  // one grow() = one call of trace_critical_points_online on the punctured simplices found since the last one
  // (host only: the batch comes in any order, duplicates allowed; neighbours are found through a hash of the batch)
  void grow(const ftkb_point *pts, uint64_t n);
  // the same step on a batch the device prepared: elements in ascending element order, unique, `keys` their element keys,
  // nb[9 * i ..] the batch indices of the punctured neighbours of element i (ascending, itself included), cnt[i] how many.
  // pts == nullptr: only the keys are kept (a caller that holds the records itself and maps keys back to them)
  void grow_sorted(const ftkb_point *pts, const uint64_t *keys, uint32_t n, const uint32_t *nb, const uint8_t *cnt);
  const std::vector<OnlineCurve> &curves() const { return curves_; }
  const std::vector<uint64_t> &keys() const { return keys_; }      // element key of stored element g
  bool has_points() const { return have_points_; }
  const ftkb_point &point(uint32_t g) const;                       // record of stored element g (has_points())
  uint64_t npoints() const;      // points on trajectories
  // element key of a point (the reference's element order packed into 64 bits; same packing as the device sort)
  bool key_of(const ftkb_point &p, uint64_t &key) const { return key_at(p.corner[0], p.corner[1], p.corner[2], p.corner[3], p.simplex_type, key); }
  int neighbor_keys(uint64_t key, uint64_t out[9]) const;   // of the element with this key: ascending, the element itself included

 private:
  bool key_at(int x, int y, int z, int t, int type, uint64_t &key) const;
  void store_batch(const uint64_t *keys, uint32_t n, std::vector<ftkb_point> &&pts);

  // the walk itself; `src` answers neighbour queries on the batch (find(key), list(i), first_alive(i)); `sorted`: batch index
  // order is element order
  template <class Source>
  void walk(uint32_t n, const uint64_t *keys, bool sorted, Source src);

  int nd_;
  int32_t lb_[3], ub_[3];
  int64_t ny_, nz_;
  // neighbour candidates of every simplex type (the element itself included) in ascending element order: the order
  // of (corner + offset, type) does not depend on the corner
  struct Candidate { int8_t off[4]; int8_t type; int64_t cell_delta; int64_t key_delta; };
  Candidate cand_[60][9];
  int ncand_[60] = {};
  int ntypes_ = 0;             // 12 (2D+t) or 60 (3D+t); points with another simplex type are ignored
  std::vector<OnlineCurve> curves_;
  std::vector<uint64_t> keys_;                      // every element handed to a grow step (deduplicated per step), batch after batch
  std::vector<std::vector<ftkb_point>> batches_;    // their records, one array per batch
  std::vector<uint32_t> batch_base_;                // index of a batch's first element
  bool have_points_ = true;
};

// (context.cpp) one grow step of a streaming context over the points imported since its last one, as the batch of timestep t:
// how a device group's merged context grows the trajectories of the chunks or slabs that sweep for it (group.cpp)
int grow_imported(ftkb_ctx *c, int t);

// One source of a layer's planes [first, first + count) along the slowest axis (z in 3D, y in 2D) of the context's array: the
// arrays start at plane `first` and live on `device`; every copy from them waits for `after` unless it is null.
struct Segment {
  int first = 0, count = 0;
  const double *scalar = nullptr, *vector = nullptr, *jacobian = nullptr;
  int device = 0;
  cudaEvent_t after = nullptr;
};
// (context.cpp) ftkb_push_snapshot(c, .., FTKB_MEM_DEVICE) for a layer assembled from device segments on any devices, which tile
// the context's array in plane order and all pass the same arrays: one copy per (segment, array), a peer copy when the segment
// is on another device than the context's.  How a device group feeds its contexts from a device snapshot (one segment) or from
// snapshot pieces (group.cpp); ftkb_push_snapshot is the one-segment case for its own memory kinds.
int push_segments(ftkb_ctx *c, const Segment *segs, int n);
// (context.cpp) the last timestep whose sweep `c` has confirmed (start_timestep - 1: none yet); waits for nothing
int confirmed_through(const ftkb_ctx *c);
// (context.cpp) appends the points `src` found in its confirmed sweep of timestep t to the imported points of the streaming
// context `dst`, device to device: a peer copy when the two live on different devices, never through the host.  *interval: that
// sweep covered the interval [t, t+1] (an advance), so the points make up a grow step.  The copy is complete on return; neither
// context may be used by another thread meanwhile.
int import_step(ftkb_ctx *dst, ftkb_ctx *src, int t, bool *interval);
// (context.cpp) lets `device` read `peer`'s memory where the hardware allows it, once per pair; makes `device` current
cudaError_t enable_peer_access(int device, int peer);

}  // namespace ftkb
