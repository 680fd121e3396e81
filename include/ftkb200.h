/* ftkb200.h -- C ABI of the B200-native critical-point extraction/tracking engine.
 *
 * This is the drop-in boundary for ONE path of hguo/ftk: critical-point tracking on regular grids.
 * It replaces the reference's accelerator entry points, which are C++ free functions with C++
 * types and per-call cudaMalloc/H2D/launch/D2H/cudaFree:
 *
 *   extract_cp2dt_cuda(scope, t, domain, core, ext, Vc, Vn, Jc, Jn, Sc, Sn, use_explicit_coords, coords)
 *       ref: include/ftk/filters/critical_point_tracker_2d_regular.hh:33-47,
 *            src/filters/critical_point_tracer_2d_regular.cu:274-310
 *   extract_cp3dt_cuda(scope, t, domain4, core4, ext3, Vc, Vl, Jc, Jl, Sc, Sl)
 *       ref: include/ftk/filters/critical_point_tracker_3d_regular.hh:42-56,
 *            src/filters/critical_point_tracer_3d_regular.cu:252-276
 *
 * and, one level up, carries the whole operator surface of
 * ftk::critical_point_tracker_{2d,3d}_regular (set_domain / push_field_data_snapshot /
 * advance_timestep / update_timestep / finalize / get_traced_critical_points), so that the C++
 * shim classes (include/ftk_b200/critical_point_tracker_regular.hh), the Python module
 * (ftk_b200/) and the CLI call ONLY this ABI.  Unlike the reference entry points it is stateful:
 * field layers stay resident in HBM between calls and results are produced to match the
 * reference's CPU tracker (not its fixed-precision CUDA kernel).
 *
 * Conventions: extern "C", plain pointers and sizes.  Every function returns an int status
 * (0 = FTKB_OK) and never calls exit(); ftkb_last_error() returns a message for the last failure
 * on that context.  The caller owns every output buffer; the library owns all device memory.
 * One context is driven from one host thread at a time (internally: one device, one stream).
 * There is NO CPU fallback: ftkb_create() fails with FTKB_ERR_NO_DEVICE without a usable
 * sm_100 device.
 */
#ifndef FTKB200_H
#define FTKB200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FTKB_ABI_VERSION 2

enum {
  FTKB_OK = 0,
  FTKB_ERR_INVALID = 1,      /* bad argument / bad call order */
  FTKB_ERR_NO_DEVICE = 2,    /* no CUDA device of compute capability 10.x */
  FTKB_ERR_CUDA = 3,         /* a CUDA runtime call or kernel failed (message has the detail) */
  FTKB_ERR_NOMEM = 4,
  FTKB_ERR_OVERFLOW = 5      /* an index range does not fit the 64-bit element id */
};

/* field sources, same values as ftk::SOURCE_* (ref: include/ftk/filters/critical_point_tracker.hh:21-25) */
enum { FTKB_SOURCE_NONE = 0, FTKB_SOURCE_GIVEN = 1, FTKB_SOURCE_DERIVED = 2 };

/* where the pointers handed to ftkb_push_snapshot live */
enum {
  FTKB_MEM_HOST = 0,          /* host memory; copied to the device before the call returns */
  FTKB_MEM_DEVICE = 1,        /* device memory on the context's device; copied (D2D) before the call returns */
  FTKB_MEM_DEVICE_BORROW = 2  /* device memory used in place: must stay valid and unchanged until the sweeps that
                                 read the layer have been confirmed -- three ftkb_advance_timestep calls after the
                                 push, or the next ftkb_synchronize / ftkb_get_stats / result getter (steps are
                                 enqueued without a host round trip, see ftkb_update_timestep) */
};
/* Device inputs and streams.  The context runs on its own non-blocking stream.  A device array handed to
 * ftkb_push_snapshot must be complete when the context reads it: either the caller synchronises the stream that wrote
 * it before the push, or it names that stream once with ftkb_set_producer_stream(ctx, stream, 1) -- every device push
 * then records an event there and makes the context's stream wait for it (stream = NULL with enable = 1 is the legacy
 * default stream).  enable = 0 turns the ordering off again.  Arrays must be 8-byte aligned. */

/* synthetic generators of ftkb_push_synthetic (ref: include/ftk/ndarray/synthetic.hh) */
enum {
  FTKB_SYN_MOVING_EXTREMUM = 0, /* scalar; params: x0[nd], dir[nd]        synthetic.hh:332-354 */
  FTKB_SYN_WOVEN = 1,           /* 2D scalar; params: (none); t = time     synthetic.hh:32-48  */
  FTKB_SYN_DOUBLE_GYRE = 2,     /* 2D vector; params: A, omega, eps        synthetic.hh:130-217 */
  FTKB_SYN_ABC = 3,             /* 3D vector; params: A, B, C              synthetic.hh:239-260 */
  FTKB_SYN_MERGER = 4,          /* 2D scalar; params: (none)               synthetic.hh:262-297 */
  FTKB_SYN_TORNADO = 5          /* 3D vector; params: (none); t = integer time step   synthetic.hh:441-494 */
};

typedef struct ftkb_config {
  int32_t abi_version;        /* FTKB_ABI_VERSION */
  int32_t nd;                 /* spatial dimensionality: 2 or 3 */
  int32_t dims[3];            /* array dims W, H, D (dim 0 fastest); set_array_domain, regular_tracker.hh:27 */
  int32_t lb[3], ub[3];       /* tracker domain, inclusive; set_domain, regular_tracker.hh:24 */
  int32_t scalar_source, vector_source, jacobian_source;   /* FTKB_SOURCE_* */
  int32_t jacobian_symmetric; /* set_jacobian_symmetric */
  int32_t robust_detection;   /* 3D only; critical_point_tracker_3d_regular.hh:442 */
  int32_t compute_degrees;    /* 2D only; critical_point_tracker_2d_regular.hh:653-662 */
  int32_t use_type_filter;    /* 2D only; critical_point_tracker.hh:190-200 */
  uint32_t type_filter;
  int32_t start_timestep;     /* initial current_timestep (tracker.hh:76); a time slab starts here */
  int32_t device;             /* CUDA device ordinal */
  double  resolution_init;    /* running min non-zero |v| inherited from earlier time slabs; <= 0: DBL_MAX
                                 (critical_point_tracker.hh:850-864 keeps a running minimum over all sweeps) */
  uint64_t point_capacity;    /* initial capacity of the punctured-simplex buffer; 0: default (grows on demand) */
  /* ABI 2 -- spatial slab of a larger array (3D: slabs along z, the reference's spatial decomposition with ghost layers,
   * regular_tracker.hh:126-149).  The context holds planes [slab_offset, slab_offset + dims[2]) of an array of slab_global_dim
   * planes; lb / ub stay relative to the slab.  Everything that depends on a vertex's position in the WHOLE lattice uses the
   * global frame: the SoS vertex rank (regular_tracker.hh:188-194), the interpolated position, the reported corner, the element
   * key, the device generators.  slab_global_dim = 0: not a slab (the defaults below are then ignored). */
  int32_t slab_offset;
  int32_t slab_global_dim;
  int32_t slab_global_lb, slab_global_ub;   /* bounds of the whole tracker domain along z, in the whole array's indices */
} ftkb_config;

/* one punctured simplex; same 72-byte layout the parity oracle uses */
typedef struct ftkb_point {
  int32_t corner[4];          /* x, y, z, t of the simplex's corner (z = 0 in 2D) */
  int32_t simplex_type;       /* index among all n-simplex types of the (n+1)-D mesh */
  int32_t ordinal;            /* 1: all vertices in one time layer */
  int32_t timestep;
  uint32_t cp_type;           /* ftk critical point type bits, critical_point_type.hh:10-36 */
  double x[3], t, scalar;
} ftkb_point;

typedef struct ftkb_stats {
  uint64_t simplices_tested;  /* enumerated work items, valid or not (SURVEY.md 8d) */
  uint64_t cells_scanned;     /* space-time cubes visited by the scan kernel */
  uint64_t cells_refined;     /* cubes that survived the exact sign early-out */
  uint64_t points;            /* punctured simplices found so far */
  uint64_t kernel_launches;   /* launches of this library's own kernels */
  uint64_t h2d_bytes, d2h_bytes;
  double ms_derive;           /* device time (CUDA events on the context's stream), accumulated */
  double ms_scan;
  double ms_test;
  double ms_finalize_device;
  double ms_finalize_host;
  double last_ms_scan;        /* most recent scan launch */
  double last_ms_derive;
  double scaling_factor;      /* current quantisation factor (1 << nbits) */
  double resolution;          /* running min non-zero |v| */
  uint64_t scan_launches;     /* scan kernel launches (one per sweep, repeated sweeps included) */
  uint64_t sweeps_repeated;   /* sweeps run again: stale quantisation factor or output buffers grown */
  double ms_sort_wall;        /* host wall clock of sort + dedup + copy of the punctured simplices (ensure_sorted), accumulated */
  double ms_trace_wall;       /* host wall clock of ftkb_finalize after the sort: neighbour search, union-find, copies, ordering walk */
} ftkb_stats;

typedef struct ftkb_ctx ftkb_ctx;

int ftkb_abi_version(void);
/* number of usable devices (compute capability 10.x); 0 if none */
int ftkb_device_count(void);

int ftkb_create(const ftkb_config *cfg, ftkb_ctx **out);
void ftkb_destroy(ftkb_ctx *);
const char *ftkb_last_error(const ftkb_ctx *);   /* ctx may be NULL: last create() failure */

/* push_field_data_snapshot(scalar, vector, jacobian): critical_point_tracker.hh:202-213.
 * Arrays are dim-0-fastest: scalar (W,H[,D]); vector (n,W,H[,D]); jacobian (n,n,W,H[,D]).
 * A pointer may be NULL when its source is NONE or DERIVED. */
int ftkb_push_snapshot(ftkb_ctx *, const double *scalar, const double *vector, const double *jacobian, int where);
int ftkb_set_producer_stream(ftkb_ctx *, void *cuda_stream, int enable);
/* host snapshot that exists as float32 (raw float32 file series): travels as float32, widened to the resident fp64 layer on the
 * device -- bit-identical to widening on the host first (ndarray.hh read_binary_file + push), half the PCIe bytes */
int ftkb_push_snapshot_f32(ftkb_ctx *, const float *scalar, const float *vector);
/* device-side generator for snapshot time `t` (benchmarks; no host data involved) */
int ftkb_push_synthetic(ftkb_ctx *, int kind, const double *params, int nparams, double t);

/* physical coordinates of the grid vertices, interpolated into ftkb_point.x by the per-simplex test
 * (simplex_coordinates, critical_point_tracker_2d_regular.hh:494-526, ..._3d_regular.hh:343-379).  One entry point for the
 * reference's three setters (regular_tracker.hh:38-40):
 *   FTKB_COORDS_SIMPLE       grid units (default); data ignored
 *   FTKB_COORDS_BOUNDS       set_coords_bounds: n = 2*nd values {x0, x1, y0, y1[, z0, z1]}
 *   FTKB_COORDS_RECTILINEAR  set_coords_rectilinear: n = W + H [+ D] values, x[W] then y[H] [then z[D]]
 *   FTKB_COORDS_EXPLICIT     set_coords_explicit: (ncomp, W, H) dim-0-fastest, ncomp = n / (W*H) >= nd.  As in the reference,
 *                            3D trackers look the coordinates up by (x, y) only and report z in ftkb_point.t.
 * data is host memory, copied before the call returns; applies to the sweeps that follow. */
enum { FTKB_COORDS_SIMPLE = 0, FTKB_COORDS_BOUNDS = 1, FTKB_COORDS_RECTILINEAR = 2, FTKB_COORDS_EXPLICIT = 3 };
int ftkb_set_coords(ftkb_ctx *, int mode, const double *data, uint64_t n);

/* Sync-free steps: ftkb_update_timestep only ENQUEUES the sweep and returns; its counters are published by the device
 * into mapped host memory and read when the NEXT step has been enqueued, or by any call that needs results
 * (ftkb_get_stats, ftkb_synchronize, ftkb_finalize, the getters).  A step that ran with a stale quantisation factor
 * (the layer it resolved lowered the running minimum, critical_point_tracker.hh:850-864) or whose buffers overflowed
 * is replayed synchronously, so results never depend on the mode.  Streaming trajectories, non-robust 3D detection and
 * the two-layer scans run every step synchronously; FTKB_DEFER=0 in the environment does so for all. */
int ftkb_update_timestep(ftkb_ctx *);    /* critical_point_tracker_{2d,3d}_regular::update_timestep */
int ftkb_advance_timestep(ftkb_ctx *);   /* critical_point_tracker.hh:841-848 */
int ftkb_finalize(ftkb_ctx *);           /* trace_critical_points_offline, critical_point_tracker.hh:668-817 */
int ftkb_current_timestep(const ftkb_ctx *, int32_t *t);

/* resolution (min non-zero |v|) of the most recently pushed layer; lets time slabs exchange the
 * running minimum (SURVEY.md 8e) */
int ftkb_last_layer_resolution(ftkb_ctx *, double *res);
int ftkb_set_resolution(ftkb_ctx *, double res);   /* lower the running minimum (never raises it) */

/* punctured simplices, sorted by the reference's element order (corner x first, then type;
 * simplicial_regular_mesh.hh:327-337), duplicates removed */
int ftkb_num_points(ftkb_ctx *, uint64_t *n);
int ftkb_get_points(ftkb_ctx *, ftkb_point *out, uint64_t cap);
/* add punctured simplices found elsewhere (another time slab) before ftkb_finalize.  A streaming context (ftkb_set_streaming_trajectories)
 * takes imports only while it holds no snapshot and has swept nothing (the merged context of a group) */
int ftkb_import_points(ftkb_ctx *, const ftkb_point *pts, uint64_t n);

/* ---- time-slab halo through NVLink peer memory (SURVEY.md 8e) -------------------------------------------------
 * The slab below needs the first layer of the slab above only for its last sweep, and of that layer only (a) the
 * 16-byte range cells (DESIGN.md 4.2) and (b) the vertices around the handful of surviving cubes.  Instead of copying
 * the layer (ncclSend/Recv of 25.8 GB on the 1024^3 vector field), the owner exports IPC handles of the layer and of
 * its cells; the neighbour process maps them and pushes the layer as a REMOTE snapshot: its last sweep reads the cells
 * and the sparse vertices straight from the peer's HBM over NVLink / NVSwitch.  Replaces the MPI ghost exchange of
 * regular_tracker.hh:120-151 for the time-slab decomposition.
 *
 * ftkb_ipc_export: handle of the allocation that holds dev_ptr (cudaIpcGetMemHandle) + the pointer's offset in it.
 * ftkb_ipc_import: map it in another process of the same node (peer access enabled lazily); ftkb_ipc_close unmaps.
 * ftkb_export_layer_cells: device pointer / size of the range cells of resident layer `index` (0 = current); the
 *   buffer is pinned to the context (not recycled) until ftkb_destroy.  The cells exist once a sweep has read the layer.
 * ftkb_push_snapshot_remote: like ftkb_push_snapshot(.., FTKB_MEM_DEVICE_BORROW) for a layer whose cells and min non-zero
 *   |v| (`resolution`, from the owner's ftkb_last_layer_resolution) come with it; nothing is copied or streamed. */
typedef struct ftkb_ipc_handle { uint8_t bytes[64]; uint64_t offset; } ftkb_ipc_handle;
int ftkb_ipc_export(const void *dev_ptr, ftkb_ipc_handle *out);
int ftkb_ipc_import(const ftkb_ipc_handle *h, int device, void **dev_ptr);
int ftkb_ipc_close(void *dev_ptr, const ftkb_ipc_handle *h);
int ftkb_export_layer_cells(ftkb_ctx *, int index, void **cells, uint64_t *bytes, double *resolution /* the layer's min non-zero |v| */);
int ftkb_push_snapshot_remote(ftkb_ctx *, const double *scalar, const double *vector, const void *cells, double resolution);

/* ---- several GPUs behind one tracker (SURVEY.md 8e; the reference's filter::set_device_ids, filter.hh:47-51) ---------------
 * One process, one caller thread, N devices.  Timesteps are cut into chunks of `chunk_timesteps`; chunk c is swept by a context
 * of its own on device_ids[c mod n_devices] (a simplex belongs to the chunk that owns its corner time; the first layer of the
 * next chunk is pushed to both: a one-layer halo), one host thread per device executes that device's pushes and sweeps in
 * order, so the devices work on their chunks concurrently while the caller hands snapshots over in time order.  A chunk
 * inherits the running minimum of min non-zero |v| (the quantisation factor is a running quantity) from its predecessor; it
 * starts early once the minimum known so far saturates the factor, otherwise when the predecessor has finished -- results equal
 * the one-device run bit for bit.  ftkb_group_finalize merges the punctured simplices of all chunks into one context on
 * device_ids[0] and traces there; *root stays owned by the group and serves every getter (ftkb_get_points, ftkb_get_trajectories,
 * ftkb_get_trajectory_complete, ftkb_get_curveset ...).  cfg->device is ignored.
 * ftkb_group_push_snapshot takes HOST memory (borrowed until return); ftkb_group_push_synthetic generates on the devices.
 * ftkb_group_push_snapshot_device takes CUDA DEVICE memory on any visible device, one of the group's or not (a producer on
 * GPU 0 feeding a group of eight): every context that needs the snapshot -- a chunk's own and, for the first layer of a chunk,
 * the one-layer halo of the chunk before; or every z-slab, for its planes -- copies it from the source device on its own
 * stream, all at once: a device-to-device copy on the same device, cudaMemcpyPeerAsync (NVLink copy engines, no kernel)
 * otherwise.  Peer access is enabled once per (destination, source) pair where the hardware allows it.  Host and device pushes
 * may alternate in one series.
 * ftkb_group_set_producer_stream names the stream (on its own device; NULL: the legacy default stream of the source device)
 * that writes those arrays: every later device push records an event there and every copy waits for it.  Without it the caller
 * synchronises the producer before pushing.
 * ftkb_group_push_pieces_device takes a snapshot that lives in PIECES, the way a simulation decomposed over several GPUs holds
 * it: each piece is a contiguous range of planes along the slowest axis (z planes in 3D, y rows in 2D) in CUDA device memory
 * on any visible device.  Every context assembles its layer from the pieces that intersect the planes it needs -- a z-slab its
 * planes [a0, a1], ghost planes included; a chunk's context, the halo of the chunk before and the staged first layer of a new
 * chunk the whole array -- with one copy per (context, intersecting piece, array), on the context's stream.  A producer that
 * cuts its pieces at the slabs' array planes (ftkb_group_get_slab) sends only ghost planes from one device to another.
 *
 * Options, valid only before the first push (afterwards FTKB_ERR_INVALID):
 *   ftkb_group_set_coords                   ftkb_set_coords for the whole array: same modes and sizes, host data copied before
 *                                           the call returns; every chunk / slab context sweeps with it.
 *   ftkb_group_set_streaming_trajectories   the merged context on device_ids[0] exists from the first push and grows during the
 *                                           run: once the sweep of interval t is confirmed (by every z-slab, or by the chunk that
 *                                           owns t) and t-1 has been grown, its points are copied there device to device and the
 *                                           grow step of ftkb_set_streaming_trajectories runs over them -- the batch a single
 *                                           streaming context grows at t.  Grows run in time order, may lag the sweeps by a step
 *                                           or two (time chunks grow on a thread of their own), and ftkb_group_get_live_curveset
 *                                           reads them at any time.  ftkb_group_finalize waits for the last grow, imports the
 *                                           last ordinal sweep's points (they join no trajectory) and publishes trajectories,
 *                                           loop and complete flags as a streaming context's ftkb_finalize does.
 *
 * chunk_timesteps = 0 selects the SPATIAL decomposition instead (3D only; the reference's own, regular_tracker.hh:126-149):
 * device s holds a z-slab of every snapshot -- its share of the domain's corner planes, the corner plane above (whose flat
 * simplices both neighbours find; the merge drops the duplicates) and two ghost planes beyond every vertex it uses -- and every
 * device sweeps every step, so a host snapshot travels in N pieces over N PCIe links at once.  SoS vertex ranks, interpolated
 * positions, physical coordinates, reported corners and the device generators use the whole array's frame (ftkb_config.slab_*;
 * ftkb_set_coords on a slab context takes the whole array's coordinates); until the running
 * minimum of min non-zero |v| saturates the quantisation factor, the slabs' minima are combined before every sweep, so every
 * slab quantises exactly as the undivided run does. */
typedef struct ftkb_group ftkb_group;
int ftkb_group_create(const ftkb_config *cfg, const int32_t *device_ids, int32_t n_devices, int32_t chunk_timesteps, ftkb_group **out);
void ftkb_group_destroy(ftkb_group *);
const char *ftkb_group_last_error(const ftkb_group *);
int ftkb_group_set_coords(ftkb_group *, int mode, const double *data, uint64_t n);
int ftkb_group_set_streaming_trajectories(ftkb_group *, int enable);
int ftkb_group_push_snapshot(ftkb_group *, const double *scalar, const double *vector, const double *jacobian);
/* a snapshot in CUDA device memory on any visible device (not necessarily one of the group's): same arrays, sizes and NULL
 * rules as ftkb_group_push_snapshot; all non-NULL pointers on the same device, 8-byte aligned.  Copied: the call returns when
 * every device of the group holds its copy, so the caller may overwrite the arrays right away.  Host, unregistered and managed
 * memory, arrays on two devices and misaligned arrays are refused with FTKB_ERR_INVALID and leave the group as it was. */
int ftkb_group_push_snapshot_device(ftkb_group *, const double *scalar, const double *vector, const double *jacobian);
/* the group's counterpart of ftkb_set_producer_stream: every copy of a later device push waits for the work queued on
 * `stream` (on its own device) when the push is called; enable = 0 turns it off */
int ftkb_group_set_producer_stream(ftkb_group *, void *cuda_stream, int enable);
/* one piece of a snapshot: planes [first, first + count) of the slowest axis (z in 3D, y in 2D), each array holding exactly
 * those planes (count * H * W scalars in 3D, count * W in 2D; times n or n*n for the vector and Jacobian arrays) */
typedef struct ftkb_piece {
  const double *scalar, *vector, *jacobian; /* device memory, all on one device; NULL rules as ftkb_group_push_snapshot */
  int32_t first, count;                     /* planes [first, first + count) of the slowest axis (z in 3D, y in 2D) */
  void *stream;                             /* stream on the piece's device that writes it (NULL: that device's legacy stream) */
  int32_t has_stream;                       /* 1: every copy from this piece waits for the work queued on `stream` at the push */
  int32_t reserved;
} ftkb_piece;
/* a snapshot as n >= 1 pieces that tile the array in order: piece 0 starts at plane 0, each piece starts where the one before
 * ends, every count >= 1, and the counts add up to the extent (D in 3D, H in 2D).  Every piece passes the same arrays, which
 * meet the configuration's sources; every array is CUDA device memory, 8-byte aligned, and one piece's arrays are on one device
 * (several pieces may share a device).  Otherwise FTKB_ERR_INVALID, with a message that names the piece and the array, before
 * anything is enqueued: the group stays as it was.  Ordering is per piece: the push records one event of the group's on every
 * stream the pieces name (has_stream = 1) and every copy from those pieces waits for it; ftkb_group_set_producer_stream does
 * not apply to piece pushes.  Copied: the call returns when every device holds its copy, so the caller may overwrite or free
 * the pieces right away.  Piece, whole-device and host pushes may alternate in one series. */
int ftkb_group_push_pieces_device(ftkb_group *, const ftkb_piece *pieces, int32_t n);
/* z-slab mode: corner planes [c0, c1] slab s owns and array planes [a0, a1] it holds, so that a producer can cut its pieces
 * where only ghost planes cross devices; FTKB_ERR_INVALID in time-chunk mode */
int ftkb_group_get_slab(const ftkb_group *, int32_t s, int32_t planes[4]);
int ftkb_group_push_synthetic(ftkb_group *, int kind, const double *params, int nparams, double t);
int ftkb_group_advance_timestep(ftkb_group *);
int ftkb_group_update_timestep(ftkb_group *);
int ftkb_group_finalize(ftkb_group *, ftkb_ctx **root);
/* sums over the chunks that have finished so far (scaling_factor / resolution: the latest finished chunk's) */
int ftkb_group_get_stats(ftkb_group *, ftkb_stats *sum, int32_t *chunks_done);

/* after ftkb_finalize: trajectories as CSR over the sorted point array */
int ftkb_num_trajectories(ftkb_ctx *, uint64_t *n);
int ftkb_get_trajectories(ftkb_ctx *, uint64_t *offsets /* n+1 */, uint64_t *point_idx, uint8_t *loop /* n */);
/* label of the connected component (special nodes included) of each sorted point = index of its
 * smallest member; and the number of punctured neighbours of each sorted point */
int ftkb_get_component_labels(ftkb_ctx *, uint64_t *labels);
int ftkb_get_degrees(ftkb_ctx *, int32_t *deg);

/* ---- streaming trajectories (SURVEY.md 8f4) --------------------------------------------------------------------
 * set_enable_streaming_trajectories (critical_point_tracker.hh:38): with streaming on, every ftkb_update_timestep that
 * sweeps an interval (two resident snapshots) ends with the reference's grow step, trace_critical_points_online
 * (critical_point_tracker.hh:522-641): the punctured simplices found since the last grow step are copied to the host,
 * existing trajectories claim their neighbours greedily, and what is left starts new trajectories.  ftkb_finalize then
 * only publishes them ("done", critical_point_tracker_2d_regular.hh:150-151): the CSR of ftkb_get_trajectories is in
 * trajectory-id order, and -- as in the reference -- the punctured simplices of the last ordinal sweep belong to no
 * trajectory.  Must be called before the first ftkb_update_timestep.  ftkb_get_trajectory_complete: 1 for a trajectory
 * that a grow step found nothing to add to (feature_curve_t::complete); all 0 without streaming. */
int ftkb_set_streaming_trajectories(ftkb_ctx *, int enable);
int ftkb_get_trajectory_complete(ftkb_ctx *, uint8_t *complete /* n */);
/* the grow step by itself (host code, no device): feed it the punctured simplices of one step at a time */
typedef struct ftkb_online ftkb_online;
int ftkb_online_create(int nd, const int32_t *lb /* nd */, const int32_t *ub /* nd, inclusive */, ftkb_online **out);
void ftkb_online_destroy(ftkb_online *);
int ftkb_online_grow(ftkb_online *, const ftkb_point *pts, uint64_t n);
/* the same step over sorted neighbour lists -- the form the tracker's device-side preparation hands to the walk -- built here on
 * the host; results are identical to ftkb_online_grow */
int ftkb_online_grow_prepared(ftkb_online *, const ftkb_point *pts, uint64_t n);
int ftkb_online_size(const ftkb_online *, uint64_t *ntraj, uint64_t *npoints);
int ftkb_online_get(const ftkb_online *, uint64_t *offsets /* ntraj+1 */, ftkb_point *pts /* npoints */, uint8_t *loop, uint8_t *complete);

/* ---- trajectory post-processing (host code; SURVEY.md 8f3) ----------------------------------------------------
 * A curve set holds the traced trajectories as mutable curves -- the reference's feature_curve_set_t, a multimap
 * keyed by curve id (include/ftk/features/feature_curve_set.hh:21-70, :447-532) -- and applies the reference's
 * per-curve operations (include/ftk/features/feature_curve.hh:113-417).  ops is a comma-separated list as
 * feature_curve_set_post_processor_t takes it (include/ftk/filters/feature_curve_set_post_processor.hh:23-70):
 *   smooth_types, rotate, split, discard_interval_points, reorder, adjust_time, derive_velocity,
 *   duration_pruning:THRESHOLD, plus discard_degenerate_points, update_statistics, and
 *   legacy[:duration_threshold[:discard_interval_points[:derive_velocities]]] = json_interface::post_process()
 *   (include/ftk/filters/json_interface.hh:758-800), and intercept:T0:T1 = feature_curve_set_t::intercept
 *   (feature_curve_set.hh:534-545; the "intercepted" output type).
 * An unknown op returns FTKB_ERR_INVALID (the reference calls fatal()). */
typedef struct ftkb_curve_point {
  ftkb_point p;               /* cp_type and t are what post-processing may change */
  double v[3];                /* derive_velocity; zero before */
  int32_t id;                 /* id of the curve the point was traced into (feature_point_t::id) */
  int32_t reserved;
} ftkb_curve_point;

typedef struct ftkb_curve_info {
  int32_t id, loop, complete;
  uint32_t consistent_type;   /* 0 if the curve's points disagree, or before any update_statistics */
  uint64_t first, count;      /* the curve's points in the array ftkb_curveset_get fills */
  double tmin, tmax, bbmin[3], bbmax[3];
  double smin, smax, persistence, vmmin, vmmax;   /* statistics of scalar[0] and of |v| (feature_curve.hh:145-186) */
} ftkb_curve_info;

typedef struct ftkb_curveset ftkb_curveset;
/* trajectories as CSR over a point array (what ftkb_get_trajectories returns); curves get ids 0 .. ntraj-1 */
int ftkb_curveset_create(const ftkb_point *pts, uint64_t npts, const uint64_t *offsets, const uint64_t *point_idx,
                         const uint8_t *loop, uint64_t ntraj, ftkb_curveset **out);
/* get_traced_critical_points() of a finalized context (mid-run, of a streaming one: ftkb_get_live_curveset); the caller
 * destroys the set */
int ftkb_get_curveset(ftkb_ctx *, ftkb_curveset **out);
/* the trajectories a streaming context has grown so far, at any time during the run (the reference's traced_critical_points,
 * which trace_critical_points_online keeps current): the curve set ftkb_get_curveset builds after ftkb_finalize -- curves in id
 * order, points in trace order, loop and complete flags, statistics -- and, after ftkb_finalize, equal to it.  *grown_through
 * receives the last timestep whose grow step has run (start_timestep - 1 before the first).  The query changes no later
 * result.  A context without streaming trajectories, or a NULL argument, gets FTKB_ERR_INVALID.  The caller destroys the set. */
int ftkb_get_live_curveset(ftkb_ctx *, int32_t *grown_through, ftkb_curveset **out);
/* the same for a group with ftkb_group_set_streaming_trajectories: first waits for the grow steps of every interval the caller
 * has swept (advanced over), so that the answer equals, call for call, that of one context fed the same series */
int ftkb_group_get_live_curveset(ftkb_group *, int32_t *grown_through, ftkb_curveset **out);
void ftkb_curveset_destroy(ftkb_curveset *);
int ftkb_curveset_post_process(ftkb_curveset *, const char *ops);
int ftkb_curveset_size(const ftkb_curveset *, uint64_t *ncurves, uint64_t *npoints);
int ftkb_curveset_get(const ftkb_curveset *, ftkb_curve_info *infos /* ncurves */, ftkb_curve_point *pts /* npoints */);
/* the "sliced" output type: ordinal points of one timestep (critical_point_tracker.hh:819-835); *n receives the count,
 * at most cap points are copied */
int ftkb_curveset_slice(const ftkb_curveset *, int32_t timestep, ftkb_curve_point *out, uint64_t cap, uint64_t *n);
const char *ftkb_curveset_last_error(const ftkb_curveset *);

/* diagnostic: the cubes (linear corner index over the domain, x fastest) that the most recent sweep's
 * scan kernel left for the exact test; *n receives the count, at most cap entries are copied */
int ftkb_get_last_worklist(ftkb_ctx *, uint64_t *out, uint64_t cap, uint64_t *n);

/* diagnostic: copy resident snapshot `index` (0 = current) to host memory -- what a device-side generator
 * (ftkb_push_synthetic) produced; either pointer may be NULL */
int ftkb_get_layer(ftkb_ctx *, int index, double *scalar, double *vector);

/* page-locked (pinned, portable) host memory for snapshot buffers: ftkb_push_snapshot(FTKB_MEM_HOST) then copies at full
 * PCIe speed.  The CLI reads file series through two such buffers (one being read while the other is pushed and swept). */
int ftkb_host_alloc(uint64_t bytes, void **out);   /* placed in the memory of the socket next to the current device */
/* run the calling thread (and threads it creates later) on the CPUs next to `device` (sysfs local_cpulist): host buffers it
 * allocates afterwards are local to that device's PCIe root.  Returns the number of CPUs bound to, 0 if nothing was changed. */
int ftkb_bind_thread_to_device(int device);
void ftkb_host_free(void *p);

int ftkb_get_stats(ftkb_ctx *, ftkb_stats *out);
int ftkb_reset_stats(ftkb_ctx *);
/* block until all work queued on the context's stream is complete */
int ftkb_synchronize(ftkb_ctx *);
/* device-side stopwatch: CUDA events recorded on the context's stream (the stream every kernel of
 * this library is launched on); stop synchronises and returns the elapsed milliseconds */
int ftkb_timer_start(ftkb_ctx *);
int ftkb_timer_stop(ftkb_ctx *, double *ms);

/* implicit simplicial mesh tables (simplicial_regular_mesh.hh:620-831); no device needed.
 * nd_mesh = 3 (2D+t) or 4 (3D+t); scope: 0 all, 1 ordinal, 2 interval */
int ftkb_mesh_ntypes(int nd_mesh, int k, int scope);
int ftkb_mesh_unit_simplex(int nd_mesh, int k, int type, int32_t *out /* (k+1)*nd_mesh */);
int ftkb_mesh_scope_type(int nd_mesh, int k, int scope, int itype);
/* out[] = entries of (type, off[nd_mesh]); returns the number of entries */
int ftkb_mesh_sides(int nd_mesh, int k, int type, int32_t *out);
int ftkb_mesh_side_of(int nd_mesh, int k, int type, int32_t *out);

#ifdef __cplusplus
}
#endif
#endif
