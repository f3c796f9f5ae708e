/*
 * pyratslam_b200.h -- C ABI of the B200-native pose-cell / view-template hot path.
 *
 * This is the drop-in boundary.  The reference (bjkomer/pyratslam) has no FFI of
 * its own: its operator layer is the Python class `Convolution`
 * (ratslam/convolution.py:10-697, OpenCL via pyopencl), driven by
 * `PoseCellNetwork` (ratslam/posecell_network.py:22-353), and the numpy loop in
 * `ViewTemplates.match` (ratslam/view_templates.py:63-75).  Each entry point below
 * names the reference code it replaces.  Plain pointers and sizes only; `stream`
 * is a `cudaStream_t` passed as `void*` (NULL = legacy default stream).
 *
 * Every function returns 0 on success or a negative PRS_E_* code;
 * `prs_last_error()` gives the message of the last failure on the calling thread.
 * There is no CPU fallback: without a CUDA device every compute entry fails.
 *
 * Pose-cell state layout in HBM ("theta-major"):  state[b][th][x][y], y fastest,
 * element type float (dtype 0) or double (dtype 1).  The reference's numpy layout
 * is [x][y][th]; `prs_pc_import_xyt` / `prs_pc_export_xyt` convert.
 */
#ifndef PYRATSLAM_B200_H
#define PYRATSLAM_B200_H

#include <stddef.h>
#include <stdint.h>

#if defined(__GNUC__)
#define PRS_API __attribute__((visibility("default")))
#else
#define PRS_API
#endif

#ifdef __cplusplus
extern "C" {
#endif

#define PRS_OK 0
#define PRS_E_INVALID (-1) /* bad argument (shape, dtype, null pointer) */
#define PRS_E_CUDA (-2)    /* CUDA runtime error, see prs_last_error() */
#define PRS_E_NODEVICE (-3)
#define PRS_E_LUT_KEY (-4) /* prs_pc_update_host: the reference raises KeyError for this odometry */
#define PRS_E_RADIUS (-5)  /* prs_pc_update_host: the translation does not fit the grid */

#define PRS_F32 0
#define PRS_F64 1
#define PRS_U8 2 /* view-template libraries only */

/* per-network error bits written by the step kernels into `err[b]` */
#define PRS_ERR_LUT_KEY 1 /* fractional x offset exactly +0.5: the reference raises KeyError
                             (posecell_network.py:249) */
#define PRS_ERR_RADIUS 2  /* 3+ceil|vtrans/0.2| > min(X,Y): the reference convolves unwritten
                             memory (convolution.py:661-675) */
#define PRS_ERR_THETA 4   /* |floor(vrot/(2pi/Th)+.5)| beyond the filter table */

#define PRS_OG_RANGE 8    /* theta-origin filters are tabulated for og in [-8, 8] */

#define PRS_VT_MODE_REF 0      /* 15 windowed row offsets, view_templates.py:16-28 */
#define PRS_VT_MODE_CIRCULAR 1 /* all 32 cyclic row shifts (extension; BASELINE config 5) */

PRS_API const char* prs_last_error(void);
PRS_API int prs_version(void);
/* number of CUDA devices visible, or a negative error code */
PRS_API int prs_device_count(void);

/* ------------------------------------------------------------------ pose cells */

/* Host-side tables, all float64, computed by the caller exactly as the reference
 * computes them (numpy/scipy on the host) so that no device libm result can change
 * a filter.  Copied to the device by prs_pc_create. */
typedef struct prs_pc_config {
  int X, Y, Th;          /* PoseCellNetwork(shape), posecell_network.py:24-26 */
  int B;                 /* number of independent networks (1 for the drop-in class) */
  int dtype;             /* PRS_F32 or PRS_F64 */
  double vtrans_scale;   /* pc_vtrans_scale = 0.2, posecell_network.py:35 */
  double vrot_scale;     /* pc_vrot_scale = 2*pi/Th, posecell_network.py:36 */
  const double* ge;      /* [7]  exp(-d^2/(2 sigma_e^2)) : kernel_3d == aE ge(x)ge(x)ge - aI gi(x)gi(x)gi */
  const double* gi;      /* [7]  exp(-d^2/(2 sigma_i^2))   (posecell_network.py:97-113) */
  double aE, aI;         /* amplitudes including the 1/|sum| normalisation */
  const double* f2d;     /* [2][7][7] LUT filters F0 (origin 0,0) and F-1 (origin -1,-1),
                            posecell_network.py:50-59,210-222 */
  const double* f1d;     /* [2*PRS_OG_RANGE+1][7] theta filters for og=-8..8, posecell_network.py:224-235 */
  const double* cos_th;  /* [Th] cos((k-mid)*vrot_scale), posecell_network.py:260-261 */
  const double* sin_th;  /* [Th] sin((k-mid)*vrot_scale) */
} prs_pc_config;

typedef struct prs_pc_plan* prs_pc_handle;

/* replaces Convolution.__init__/set_params/set_text/build_program (convolution.py:11-35,37-91,94-398) */
PRS_API int prs_pc_create(const prs_pc_config* cfg, prs_pc_handle* out);
PRS_API int prs_pc_destroy(prs_pc_handle h);
/* bytes of one full state tensor [B][Th][X][Y] */
PRS_API size_t prs_pc_state_bytes(prs_pc_handle h);
/* which kernel family a step uses: 0 = generic multi-kernel path, 1 = fused SMEM-resident kernel (one CTA per
 * network), 2 = tiled large-grid kernels, 3 = one network per thread-block cluster */
#define PRS_PATH_AUTO (-1)
#define PRS_PATH_GENERIC 0
#define PRS_PATH_RESIDENT 1
#define PRS_PATH_TILED 2
#define PRS_PATH_CLUSTER 3
#define PRS_PATH_PAIR 4 /* fused SMEM-resident kernel, one network per 2-CTA cluster (float32 and float64) */
PRS_API int prs_pc_path(prs_pc_handle h);
/* choose the kernel family explicitly (PRS_PATH_*, PRS_PATH_AUTO = the plan's own choice); PRS_E_INVALID if the
 * plan's shape / dtype is not supported by that family; for tests and profiling */
PRS_API int prs_pc_set_path(prs_pc_handle h, int path);
/* Per-plan options.  PRS_OPT_ACTIVE_SET: sparsity-aware update (csrc/posecell_active.cu).  The attractor dynamics of
 * posecell_network.py:326-353 keep the activity in a compact packet (tens of non-zero cells out of thousands); with this
 * option an update does the reference's arithmetic only where the result can be non-zero and writes the state in place,
 * instead of the dense kernels whose cost does not depend on the state.  Exact for any state: a network whose non-zero
 * cells do not fit the kernel's lists / shared memory, or whose global inhibition is negative, is updated by the dense
 * kernels in the same call.  0 = off (default), 1 = the state is scanned for its non-zero cells every update,
 * 2 = the list of non-zero cells an update leaves behind is the next update's input (no pass over the state at all);
 * every library call that writes the state invalidates the lists, a caller that writes the state by other means must
 * call prs_pc_invalidate_active.  Dimensions up to 256 per axis. */
#define PRS_OPT_ACTIVE_SET 2
PRS_API int prs_pc_set_option(prs_pc_handle h, int option, int value);
/* the state was written by something other than this library's calls: forget the active lists (PRS_OPT_ACTIVE_SET = 2) */
PRS_API int prs_pc_invalidate_active(prs_pc_handle h, void* stream);

/* One PoseCellNetwork.update() for all B networks (posecell_network.py:326-353):
 *   state  : device, [B][Th][X][Y] of the plan's dtype, updated in place
 *   odom   : device, double [B][2] = (vtrans, vrot) as passed to update()
 *   gi     : device, [B] of the plan's dtype, global inhibition (posecell_network.py:34)
 *   argmax : device, int64 [B]  flat index x*Y*Th + y*Th + th of the first maximum
 *            (numpy.argmax order, posecell_network.py:317-319)
 *   total  : device, [B] of the plan's dtype, the sum before normalisation (posecell_network.py:343)
 *   err    : device, int32 [B], PRS_ERR_* bits (0 = fine)
 * Calls on one plan must be ordered by the stream(s) they are enqueued on (as for any in-place update of `state`).  On the
 * fused one-CTA-per-network path consecutive calls on a stream overlap on the device -- update n+1 of a network starts as
 * soon as its update n is complete, not when the whole launch n is (per-network sequence numbers, posecell_resident.cu);
 * a launch that was NOT ordered behind its predecessor would wait for it in vain and traps after two seconds.
 */
PRS_API int prs_pc_step(prs_pc_handle h, void* state, const double* odom, const void* gi, long long* argmax,
                void* total, int* err, void* stream);
/* T consecutive updates with odometry odom[T][B][2]; argmax[T][B], total[T][B]; err[B] is OR-ed */
PRS_API int prs_pc_run(prs_pc_handle h, void* state, const double* odom, int T, const void* gi,
               long long* argmax, void* total, int* err, void* stream);
/* Same as prs_pc_step with HOST odometry/results: H2D copy, step, D2H copy, stream sync.
 * odom_host/argmax_host/err_host should be pinned for the copies to be asynchronous. */
PRS_API int prs_pc_step_host(prs_pc_handle h, void* state, const double* odom_host, const void* gi,
                     long long* argmax_host, int* err_host, void* stream);

/* As prs_pc_step_host, but the result comes back as ONE array int32 result_host[B][4] = (x, y, th, err):
 * the arg-max already unravelled the way get_pc_max does (posecell_network.py:318) plus the PRS_ERR_* bits. */
PRS_API int prs_pc_step_host_xyz(prs_pc_handle h, void* state, const double* odom_host, const void* gi, int* result_host,
                         void* stream);
/* The same step WITHOUT the host waiting for it.  The plan keeps two slots of device staging and two copy streams:
 * the odometry of this step is copied in (from pinned odom_host) on a copy stream, the update runs on `stream`, the
 * packed result is copied out (to pinned result_host) on another copy stream.  With one step kept in flight -- two
 * (odom_host, result_host) pairs used alternately -- every step still moves its inputs in and its result out, but
 * those copies and the launch overhead overlap the neighbouring steps' kernels.  *slot_out (0 or 1) names the step for
 * prs_pc_host_result_wait, which blocks until result_host of that step is complete.  At most two steps in flight. */
PRS_API int prs_pc_step_host_xyz_async(prs_pc_handle h, void* state, const double* odom_host, const void* gi,
                               int* result_host, void* stream, int* slot_out);
PRS_API int prs_pc_host_result_wait(prs_pc_handle h, int slot);
/* PoseCellNetwork.update((vtrans, vrot)) of a single-network plan (B == 1) in one call (posecell_network.py:326-353).
 * The odometry is first checked on the host, in numpy's float64 arithmetic, for the cases the reference cannot
 * handle -- PRS_E_LUT_KEY: a fractional x offset of exactly +0.5 (KeyError, posecell_network.py:249); PRS_E_RADIUS:
 * 3 + ceil|vtrans/0.2| > min(X, Y) (convolution.py:661-675 reads unwritten memory) -- and such an update leaves the
 * state untouched.  Otherwise as prs_pc_step_host_xyz with odom_pinned[0..1] = (vtrans, vrot); both buffers pinned. */
PRS_API int prs_pc_update_host(prs_pc_handle h, void* state, double vtrans, double vrot, const void* gi,
                       double* odom_pinned, int* result_pinned, void* stream);

/* PoseCellNetwork.path_integration() alone (posecell_network.py:252-314): per-plane shifted 7x7
 * correlate + clamp, theta correlate + clamp; no attractor dynamics, no normalisation. */
PRS_API int prs_pc_path_integration(prs_pc_handle h, void* state, const double* odom, int* err, void* stream);

/* posecells[loc] += energy for network b, or for every network when b < 0 (posecell_network.py:322-324) */
PRS_API int prs_pc_inject(prs_pc_handle h, void* state, int b, int x, int y, int th, double energy, void* stream);
/* arg-max without an update (get_pc_max, posecell_network.py:317-319) */
PRS_API int prs_pc_argmax(prs_pc_handle h, const void* state, long long* argmax, void* stream);
/* Sparse read-back: the cells of network b with activity > threshold, in the reference's C order -- what the
 * viewers draw (`nonzero(pc > .002)`, simulate.py:61; ratslam_viewer.py:137) -- instead of copying the whole grid.
 *   idx_out : device int32 [max_out] flat indices x*Y*Th + y*Th + th (ascending)
 *   val_out : device [max_out] of the plan's dtype
 *   count_out : device int32, the number of cells above the threshold (may exceed max_out; the rest is dropped)
 *   work : device scratch of prs_pc_active_work_bytes(h) */
PRS_API size_t prs_pc_active_work_bytes(prs_pc_handle h);
PRS_API int prs_pc_active_cells(prs_pc_handle h, const void* state, int b, double threshold, int max_out, int* idx_out,
                        void* val_out, int* count_out, void* work, void* stream);
/* layout conversion between the reference's [B][x][y][th] and theta-major [B][th][x][y] (device to device) */
PRS_API int prs_pc_import_xyt(prs_pc_handle h, void* state, const void* xyt, void* stream);
PRS_API int prs_pc_export_xyt(prs_pc_handle h, const void* state, void* xyt, void* stream);

/* --------------------------------------------------------------- view templates */

/* Sub-sample a camera frame into a template: rows/cols strictly inside (lo, hi) with
 * (idx-lo) % step != 0 -- the boolean mask of view_templates.py:48-57 applied as in :64.
 * frame: device uint8 [im_rows][im_cols]; out: device uint8 [n_rows][n_cols]. */
PRS_API int prs_vt_extract_u8(const uint8_t* frame, int im_rows, int im_cols, int row_lo, int row_hi, int row_step,
                      int col_lo, int col_hi, int col_step, uint8_t* out, int n_rows, int n_cols, void* stream);

/* Sweep a library of n 32x32 templates against one query (ViewTemplates.match line 65 and
 * ViewTemplate.match, view_templates.py:16-28,65):
 *   key_out : device uint64, receives (min_score << 32) | (base_index + argmin), ties -> lowest
 *             index (numpy.argmin, view_templates.py:73).  n == 0 leaves key_out = UINT64_MAX.
 *   scores  : optional device uint32 [n] (u8) / float [n] (f32): per-template min score, or NULL.
 * u8: score = sum((a - b) mod 256) exactly as numpy uint8 arithmetic gives it.
 * f32: score = sum |a - b| in float32; the key holds the IEEE bits of the score. */
PRS_API int prs_vt_sweep_u8(const uint8_t* lib, long long n, const uint8_t* query, int mode, long long base_index,
                    unsigned long long* key_out, uint32_t* scores, void* stream);
PRS_API int prs_vt_sweep_f32(const float* lib, long long n, const float* query, int mode, long long base_index,
                     unsigned long long* key_out, float* scores, void* stream);
/* Bit-sliced ("packed") uint8 library: the layout the fast sweep streams.  1088 bytes per template, stored
 * in groups of 32 (see csrc/view_templates.cu).  Same scores, keys and tie-breaks as prs_vt_sweep_u8.
 *   prs_vt_packed_bytes(n)  : bytes of a packed library with room for n templates (whole groups)
 *   prs_vt_pack_u8          : convert n row-major templates src[n][32][32] into slots first..first+n-1
 *                             (the packed buffer must have been zero-filled once; ViewTemplates' append, :68-71)
 *   prs_vt_unpack_u8        : one template back to row-major (the ViewTemplate.template attribute)
 *   prs_vt_sweep_packed_u8  : query is a row-major device uint8[32][32]; scratch is a device buffer of
 *                             >= 2 KiB, private to the caller.  The query planes go through one constant-memory
 *                             buffer per device: sweeps issued on different streams (or host threads) of a device
 *                             are correct but run one after the other on the device (event-ordered, the host
 *                             does not block). */
PRS_API size_t prs_vt_packed_bytes(long long n);
PRS_API int prs_vt_pack_u8(const uint8_t* src, long long n, void* packed, long long first, void* stream);
PRS_API int prs_vt_unpack_u8(const void* packed, long long index, uint8_t* dst, void* stream);
PRS_API int prs_vt_sweep_packed_u8(const void* packed, long long n, const uint8_t* query, int mode, long long base_index,
                           unsigned long long* key_out, uint32_t* scores, void* scratch, void* stream);
/* Any template shape rows x cols (row-major library) and any max_offset (view_templates.py:14): the
 * reference's windowed match for configurations other than its 32x32 default.  Correctness path. */
PRS_API int prs_vt_sweep_any_u8(const uint8_t* lib, long long n, const uint8_t* query, int rows, int cols, int max_offset,
                        long long base_index, unsigned long long* key_out, uint32_t* scores, void* stream);
PRS_API int prs_vt_sweep_any_f32(const float* lib, long long n, const float* query, int rows, int cols, int max_offset,
                         long long base_index, unsigned long long* key_out, float* scores, void* stream);
/* HOST query in, HOST key out: H2D copy of the 1 KiB query, sweep, D2H of the 8-byte key, sync.
 * lib stays resident on the device; scratch is a device buffer of >= 1024+8 bytes. */
PRS_API int prs_vt_match_host_u8(const uint8_t* lib, long long n, const uint8_t* query_host, int mode,
                         long long base_index, unsigned long long* key_host, void* scratch, void* stream);

/* ------------------------------------------- sharded library: the MIN over ranks, on the device */

/* A very large library is split by contiguous template ranges over the ranks of a job, one process per GPU
 * (BASELINE config 5).  The reference has no counterpart (it is single-process); the semantics to keep are those of
 * `vals.index(min(vals))` / numpy.argmin over the whole list (ratslam/view_templates.py:65-73): minimum score, lowest
 * global index among equals -- i.e. the MIN of the ranks' packed keys -- followed by the strict '>' threshold test.
 *
 * prs_xchg is a small exchange buffer in device memory that the peers map through CUDA IPC (NVLink peer access):
 *   prs_xchg_create   allocate this rank's buffer (world <= 16)
 *   prs_xchg_export   64-byte cudaIpcMemHandle_t of the buffer, to be all-gathered by the host (any transport)
 *   prs_xchg_connect  open the peers' handles, handles = [world][64] in rank order (the own entry is ignored);
 *                     a world of 1 needs neither export nor connect
 *   prs_xchg_set_timeout  bound of the device-side wait for the peers (default 10 s; then status = 1)
 * One kernel per query publishes the rank's key(s) into every peer's buffer with system-scope stores, waits for the
 * peers' keys of the same query, and reduces them; every rank must issue the same sequence of exchange calls. */
typedef struct prs_xchg prs_xchg;
#define PRS_XCHG_HANDLE_BYTES 64
typedef struct prs_shard_result {
  unsigned long long key;   /* MIN over the ranks of (score << 32 | global index); UINT64_MAX: nothing compared */
  int created;              /* 1: the query became template `template_index` (appended on the owning rank) */
  int template_index;       /* what ViewTemplates.match(...).get_index() returns; -1 from prs_vt_shard_exchange */
  int n_total;              /* library size over all ranks after this query */
  int status;               /* 0 = fine, 1 = a peer did not publish within the timeout */
  unsigned long long seq;   /* sequence number of the exchange (1, 2, ...) */
} prs_shard_result;
PRS_API int prs_xchg_create(int world, int rank, prs_xchg** out);
PRS_API int prs_xchg_export(prs_xchg* x, void* handle64);
PRS_API int prs_xchg_connect(prs_xchg* x, const void* handles);
PRS_API int prs_xchg_set_timeout(prs_xchg* x, double seconds);
PRS_API int prs_xchg_destroy(prs_xchg* x);
/* MIN over the ranks of n_keys (<= 64) packed keys: keys_local is this rank's (device), keys_out receives the global
 * minima (device memory or pinned host memory; optional when result is given: result->key is the first key's minimum),
 * result (optional, device or pinned host) the status record. */
PRS_API int prs_vt_shard_exchange(prs_xchg* x, const unsigned long long* keys_local, int n_keys,
                          unsigned long long* keys_out, prs_shard_result* result, void* stream);
/* ViewTemplates.match's decision for a sharded library (view_templates.py:67-73), taken on the device by every rank
 * from the MIN of the ranks' keys: create when the library is empty or score > threshold (strict; the score is the
 * integer sum for PRS_U8, the float32 sum for PRS_F32, compared in double), else match the key's index.  On the
 * owning rank (owner != 0) a created template -- tpl, the query as a row-major 32x32 template on the device -- is
 * stored in slot n_local of lib (bit-sliced for PRS_U8, row-major for PRS_F32; the buffer must have room).
 * result: device or pinned host memory, valid once `stream` has completed. */
PRS_API int prs_vt_shard_decide(prs_xchg* x, const unsigned long long* key_local, double threshold, int dtype,
                        const void* tpl, void* lib, long long n_local, long long n_total, int owner,
                        prs_shard_result* result, void* stream);
/* Host side of a polled exchange: with `result` in pinned host memory, spin until the LAST exchange issued on x has
 * written its record (its sequence number goes out last) -- about 1 us after the kernel, where a stream
 * synchronisation costs a thread wake-up.  PRS_E_CUDA after timeout_s seconds. */
PRS_API int prs_xchg_wait(prs_xchg* x, const prs_shard_result* result_host, double timeout_s);
/* One query of a sharded library in one call: local sweep (PRS_U8: bit-sliced library + scratch >= 2 KiB as for
 * prs_vt_sweep_packed_u8; PRS_F32: row-major library), exchange (decide == 0: result->key is the MIN over the ranks;
 * decide != 0: the create-or-match decision of prs_vt_shard_decide as well), wait for the pinned record.
 * key_dev: device uint64 scratch for the local key. */
PRS_API int prs_vt_shard_query(prs_xchg* x, int dtype, void* lib, long long n_local, const void* query_dev, int mode,
                       long long base_index, unsigned long long* key_dev, void* scratch, int decide, double threshold,
                       long long n_total, int owner, prs_shard_result* result_pinned, void* stream);

/* ------------------------------------------------------------------- one frame */

/* Result of prs_frame_host (32 bytes, written to pinned host memory). */
typedef struct prs_frame_result {
  long long argmax;          /* arg-max pose cell after the update (flat index), or the previous one */
  unsigned long long key;    /* (best score << 32) | best index, UINT64_MAX if the library was empty */
  int created;               /* 1: the frame became template `template_index` */
  int template_index;        /* what ViewTemplates.match(...).get_index() returns */
  int n_templates;           /* library size after this frame */
  int pc_err;                /* PRS_ERR_* bits of the pose-cell update */
} prs_frame_result;

PRS_API size_t prs_frame_scratch_bytes(void);
/* One iteration of the ROS loop (ratslam/ros_simulate.py:98-105,134-137) with a single host sync:
 * [odom_host != NULL: pose-cell update with (vtrans, vrot)] -> frame H2D -> sub-sample -> sweep of the packed
 * uint8 library -> create-or-match on the device (a created template is packed into slot n_templates, so
 * the library must have room for n_templates + 1) -> result D2H.
 *   pc_work : device, 24 bytes (arg-max, total, err of the single network); persists between frames
 *   scratch : device, prs_frame_scratch_bytes()
 *   frame_host / odom_host / result_host : host (pinned for asynchronous copies) */
PRS_API int prs_frame_host(prs_pc_handle pc, void* pc_state, const void* gi, void* pc_work, const double* odom_host,
                   void* vt_packed, int n_templates, double threshold, int mode, const uint8_t* frame_host,
                   int im_rows, int im_cols, int row_lo, int row_hi, int row_step, int col_lo, int col_hi,
                   int col_step, void* scratch, prs_frame_result* result_host, void* stream);

/* The same frame as a replayed CUDA graph: all pointers (pinned host buffers included) are fixed at creation and
 * the library size lives in device memory, so one frame = one graph launch + one synchronisation.
 * The library must keep a free slot: recreate the plan when ViewTemplates grows its buffer.
 * prs_frame_run(plan, moved, stream): moved != 0 -> odom_host holds (vtrans, vrot) and the pose cells update first;
 * `stream` must be a non-default stream for the graph to be captured (otherwise every frame is enqueued eagerly). */
typedef struct prs_frame_plan prs_frame_plan;
PRS_API int prs_frame_create(prs_pc_handle pc, void* pc_state, const void* gi, void* pc_work, void* vt_packed,
                     int n_templates, int capacity, double threshold, int mode, int im_rows, int im_cols,
                     int row_lo, int row_hi, int row_step, int col_lo, int col_hi, int col_step, void* scratch,
                     double* odom_host, uint8_t* frame_host, prs_frame_result* result_host, prs_frame_plan** out);
PRS_API int prs_frame_destroy(prs_frame_plan* plan);
/* Put the library size back into the plan's device-side counter after templates were appended outside the plan
 * (ViewTemplates.match / create between fused frames); synchronises `stream`. */
PRS_API int prs_frame_set_count(prs_frame_plan* plan, int n_templates, void* stream);
PRS_API int prs_frame_run(prs_frame_plan* plan, int moved, void* stream);
/* prs_frame_run without the final synchronisation: the caller waits on `stream` (or an event recorded on it) before
 * reading result_host.  Two plans that share pc / pc_work / scratch / vt_packed (hence the device-side template
 * count) but have their own pinned host buffers can be launched alternately on ONE stream: the device runs the
 * frames back to back while the host prepares the next frame and digests the previous result. */
PRS_API int prs_frame_launch(prs_frame_plan* plan, int moved, void* stream);

/* View-template -> pose-cell injection inside the frame (ros_simulate.py:106-108, left commented out in the reference):
 * after the create-or-match decision and the pose-cell update, one more node adds `energy` to the cell stored with the
 * frame's template, posecells[loc_dev[template]] += energy, and keeps the plan's cached arg-max current (the injected
 * cell becomes the arg-max if it now exceeds the old one, or equals it at a lower flat index: numpy.argmax's first
 * maximum, exact for energy >= 0).  A created template's row is written on the device with the arg-max its match was
 * made with; rows of templates appended outside the plans are the caller's to fill in.  A frame whose template has the
 * row -1 leaves the state as it is and sets PRS_ERR_INJECT_LOC in its record's pc_err.  The record's arg-max stays the
 * one the match was made with; the next frame sees the injected state.  With PRS_OPT_ACTIVE_SET the carried lists are
 * invalidated, as prs_pc_inject does.
 * loc_dev: device int64 [capacity], C-order flat cell of every template, -1 = invalid; NULL turns injection off.
 *          Plans built on one library share it.
 * energy: finite and >= 0 (PRS_E_INVALID otherwise).  Changing the setting drops the plan's captured graphs. */
PRS_API int prs_frame_set_inject(prs_frame_plan* plan, double energy, long long* loc_dev);
#define PRS_ERR_INJECT_LOC 8 /* prs_frame_result.pc_err: the matched template has no valid pose cell */

/* The whole loop of ros_simulate.py:152-166 over recorded arrays in one call: frame t is staged into the pinned
 * buffers of plans[t % n_plans] and launched while earlier frames are still running; a plan is reused once its frame
 * has finished and its result has been copied to results[].  The plans must share pc / pc_state / pc_work / vt_packed /
 * scratch and differ only in their pinned host buffers; the library needs room for T more templates.
 *   frames : host uint8 [T][im_rows][im_cols]     odom : host double [T][2] = (vtrans, vrot) as given to update()
 *   moved  : host uint8 [T], 0 = the twist was below the 0.001 gate (ros_simulate.py:128): no pose-cell update
 *   results: host prs_frame_result [T]            stream: a non-default stream */
PRS_API int prs_replay_run(prs_frame_plan* const* plans, int n_plans, const uint8_t* frames, const double* odom,
                   const uint8_t* moved, int T, prs_frame_result* results, void* stream);

/* ------------------------------------------------------------ ensemble replay */

/* B independent agents in one pass (a parameter sweep of the ROS loop, ros_simulate.py:98-166): agent b is network b
 * of the pose-cell plan `pc` (B = its network count, global inhibition gi[b]) with its own packed uint8 library, match
 * threshold and injection energy, and it replays recording rec_of_dev[b] of R.  A recording is a stream of ticks, each
 * an optional gated twist and an optional image; a frame replay is the stream in which every tick has an image.  A
 * tick is ONE graph for the whole ensemble: the pose-cell update of all B networks on a side branch, one query per
 * recording, one sweep in which agent b compares against its recording's query, then per agent the create-or-match
 * decision (a created template goes into slot n_dev[b] of its library, its location row loc_dev[b][n] receives the
 * agent's arg-max) and the injection of prs_frame_set_inject.  Agent b's records equal a single-agent frame plan's on
 * its recording with threshold_dev[b], gi[b] and energy_dev[b].  Reference mode (PRS_VT_MODE_REF) only; PRS_E_INVALID
 * otherwise.
 *   pc_work       : device, B * 24 bytes: int64 arg-max [B], total [B] (8-byte slots), int32 err [B]; the arg-max must
 *                   hold each network's current arg-max (prs_pc_argmax) before the first tick
 *   libs          : device, B libraries of prs_vt_packed_bytes(capacity) bytes each, zero-filled once
 *   capacity      : templates per library, at most 65536
 *   n_dev         : device int32 [B], templates in each library; updated by every tick with an image
 *   threshold_dev : device double [B], the match thresholds as the caller gives them (create when score > threshold,
 *                   so a negative threshold creates on every frame)
 *   energy_dev    : device double [B], energy injected at the frame template's cell; a value that is not >= 0 (e.g. -1)
 *                   means no injection for that agent; NULL: no injection node at all
 *   loc_dev       : device int64 [B][capacity], C-order flat cell of every template, -1 = invalid
 *   rec_of_dev    : device int32 [B] in [0, R); the agents of one recording are best given contiguous indices (a sweep
 *                   block reloads its query when the recording changes)
 *   scratch       : device, prs_ens_scratch_bytes(pc, R, im_rows, im_cols); private to the plan.  It holds a chunk of
 *                   images of every recording ([R][chunk][im_rows][im_cols], chunk = 256 MiB / (R * frame bytes),
 *                   clamped to [1, 256]), the per-recording queries and, for R > 1, one snapshot of a network's state
 *                   per agent
 * The plan keeps pointers to all of these; they must outlive it. */
typedef struct prs_ens_plan prs_ens_plan;
PRS_API size_t prs_ens_scratch_bytes(prs_pc_handle pc, int R, int im_rows, int im_cols);
PRS_API int prs_ens_create(prs_pc_handle pc, void* pc_state, const void* gi, void* pc_work, void* libs, int capacity,
                   int* n_dev, const double* threshold_dev, const double* energy_dev, long long* loc_dev, int R,
                   const int* rec_of_dev, int mode, int im_rows, int im_cols, int row_lo, int row_hi, int row_step,
                   int col_lo, int col_hi, int col_step, void* scratch, prs_ens_plan** out);
PRS_API int prs_ens_destroy(prs_ens_plan* plan);
/* The room that prs_ens_run checks is counted in ticks with an image (one template per agent and image at most) and
 * decremented by every run.  prs_ens_refresh_room recounts it from n_dev as the libraries are now, so a plan fed in
 * pieces whose agents match more than they create keeps going without a new plan.  Synchronises `stream`. */
PRS_API int prs_ens_refresh_room(prs_ens_plan* plan, void* stream);
/* T ticks of every recording.  The caller compacts a message stream into ticks, odometry before image: an odometry
 * message directly followed by an image shares its tick, gated-out odometry makes no tick, an image with no twist
 * before it is an image-only tick, other odometry an odometry-only tick.  The pose-cell update of all B networks runs
 * when any recording moved at the tick; a network whose recording did not move, or has ended, gets the twist (0, 0),
 * and on such a "mixed" tick its state slice and its pc_work slots are saved before the update and restored after it
 * (the active-set lists are invalidated), so it ends the tick exactly as a skipped update leaves it.  An agent whose
 * recording has no image at the tick (an odometry-only tick, or past the recording's end) appends and injects nothing
 * and gets the "no frame" record: template_index -1, created 0, key ~0, n_templates unchanged, and the arg-max and
 * pc_err its update left.  A tick at which no recording has an image runs only the update (no query, sweep, decision
 * or injection).  Six graphs per plan: {no recording moved, every recording moved, mixed} x {image, none}.
 *   frames  : host, R pointers; frames[r] is uint8 [n_images[r]][im_rows][im_cols], recording r's images only, in
 *             order (may be NULL when n_images[r] = 0)
 *   odom    : host double [T][R][2] = (vtrans, vrot) of recording r's twist at tick t as given to update()
 *   gate    : host uint8 [T][R]: bit 0 = recording r has an image at tick t, bit 1 = it moved (the 0.001 twist gate,
 *             ros_simulate.py:128); 0 past the end of recording r's ticks
 *   n_images: host int32 [R], must equal the number of bit-0 ticks of each recording
 *   results : host prs_frame_result [T][B], one record per tick and agent; pc_err holds the err bits of the last
 *             update (valid where the agent's recording moved) and PRS_ERR_INJECT_LOC
 * Images, odometry and gates go to the device and the records come back one chunk of ticks at a time, one image copy
 * per recording; nothing per agent crosses the bus per tick.  Returns after one final synchronisation of `stream` (a
 * non-default stream).  PRS_E_INVALID when the libraries have no room for the ticks with an image. */
PRS_API int prs_ens_run(prs_ens_plan* plan, const uint8_t* const* frames, const double* odom, const uint8_t* gate,
                const int* n_images, int T, prs_frame_result* results, void* stream);
/* Ticks of one device chunk (the image slots of the scratch; at most 256). */
PRS_API int prs_ens_chunk(prs_ens_plan* plan);
/* Pose-cell activity capture: at every tick, each agent whose recording has an image gets an entry computed from the
 * state its match is made with -- after the tick's update (and a mixed tick's restore), before its injection: the
 * count of cells with (double)value > threshold and the first max_cells of them in C order [x][y][th], each an int32
 * flat index x*Y*Th + y*Th + th and its value in the state's dtype.  Agents without an image at the tick get count -1.
 * The capture is one node of the image ticks' graphs (on the update's branch, or before the decision on a tick without
 * update); a plan without it has no such node.  Setting it drops the captured graphs, as prs_frame_set_inject does.
 *   threshold : finite; max_cells in [0, X*Y*Th] (0: counts only)
 *   buffer    : device, prs_ens_activity_bytes(plan, max_cells) bytes, owned by the caller; NULL turns the capture off
 * With the capture on a run takes at most prs_ens_chunk(plan) ticks.  After a run, prs_ens_activity_pack packs the
 * kept cells of its ticks into one device prefix ([tick][agent] row-major, min(count, max_cells) cells per entry),
 * copies the counts to counts (host int32 [T][B]) and the number of packed cells to *total, and synchronises
 * `stream`; prs_ens_activity_copy then copies the first n packed cells to idx (host int32 [n]) and val (host, n values
 * of the state's dtype) and synchronises.  Host memory and bus traffic scale with the cells kept, not with max_cells.
 * prs_ens_activity_bytes returns 0 for a max_cells outside the range. */
PRS_API size_t prs_ens_activity_bytes(prs_ens_plan* plan, int max_cells);
PRS_API int prs_ens_set_activity(prs_ens_plan* plan, double threshold, int max_cells, void* buffer);
PRS_API int prs_ens_activity_pack(prs_ens_plan* plan, int* counts, long long* total, void* stream);
PRS_API int prs_ens_activity_copy(prs_ens_plan* plan, long long n, int* idx, void* val, void* stream);
/* Agent copies between a plan's rows (an ensemble session's reassignment of agents): move m makes row dst[m] an exact
 * copy of row src[m] as it was before the call -- the state slice, the pc_work slots, n_dev, the library groups of its
 * n_dev templates and the first n_dev entries of its location row.  Slots past n_dev are never read and an append
 * writes its slot whole, so nothing past the copied templates is cleared.  A source that is itself a destination (a
 * swap, a cycle) is gathered into the stage before any row is written; the others are read in place.  Work follows
 * the live bytes: the kernels copy the source's live groups, not the capacity.  The thresholds, inhibitions and
 * energies the plan reads are the caller's to rewrite.
 *   dst, src     : host int32 [n_moves], rows in [0, B); the dst distinct, no src equal to its dst
 *   n_templates  : host int32 [B], every row's template count as n_dev holds it (sizes the stage)
 *   stage        : device, prs_ens_copy_stage_bytes(...) bytes for these moves (a pair table and the gathered rows)
 * Asynchronous on `stream`, which also receives prs_pc_invalidate_active's reset; the next prs_ens_run on any stream
 * must be ordered after it.  prs_ens_copy_stage_bytes returns 0 for invalid moves. */
PRS_API size_t prs_ens_copy_stage_bytes(prs_ens_plan* plan, int n_moves, const int* dst, const int* src,
                                const int* n_templates);
PRS_API int prs_ens_copy_agents(prs_ens_plan* plan, int n_moves, const int* dst, const int* src, const int* n_templates,
                        void* stage, size_t stage_bytes, void* stream);
/* The same rows carried between two plans, which may live on different devices (a session's agents reassigned across
 * devices).  prs_ens_export_agents gathers rows[k] into stage row k (a row may be listed more than once); the stage then
 * depends on no plan: a header records K = n, the largest live template count, the network bytes, the dtype and the
 * pose-cell shape.  Copy it whole to the importing plan's device (prs_stage_copy), then prs_ens_import_agents writes
 * stage row k into row rows[k] (distinct) of its plan -- exactly what prs_ens_copy_agents writes -- and resets the
 * active-set lists as prs_ens_copy_agents does.  Import reads the header (it synchronises `stream` once) and refuses,
 * with PRS_E_INVALID, a stage of another row count, pose-cell shape or dtype, or with more live templates than its
 * capacity.  Import writes its pair table into the stage, so a stage is imported once.
 *   rows        : host int32 [n], rows in [0, B)
 *   n_templates : host int32 [B], every row's template count as n_dev holds it (sizes the stage)
 *   stage       : device, prs_ens_export_stage_bytes(...) bytes (0 for invalid rows or n = 0)
 * Asynchronous on `stream`; the next prs_ens_run on any stream must be ordered after the import. */
PRS_API size_t prs_ens_export_stage_bytes(prs_ens_plan* plan, int n, const int* rows, const int* n_templates);
PRS_API int prs_ens_export_agents(prs_ens_plan* plan, int n, const int* rows, const int* n_templates, void* stage,
                          size_t stage_bytes, void* stream);
PRS_API int prs_ens_import_agents(prs_ens_plan* plan, int n, const int* rows, const void* stage, size_t stage_bytes,
                          void* stream);
/* bytes from src on device src_device to dst on device dst_device, asynchronous on `stream`: cudaMemcpyPeerAsync between
 * two devices (peer access need not be enabled), cudaMemcpyAsync on one.  The stages of prs_ens_export_agents and
 * prs_em_session_export_agents cross devices this way. */
PRS_API int prs_stage_copy(void* dst, int dst_device, const void* src, int src_device, size_t bytes, void* stream);

/* ------------------------------------------------------- ensemble experience maps */

/* Every agent's linked experience map built from an ensemble's records (csrc/experience_map.cu): the per-frame update
 * of ExperienceMap(linked=True) (pyratslam_b200/experience_map.py: update, _find, _add_link, _create_linked,
 * _set_current) for B agents over T frames, one thread per agent.  Graph relaxation (ExperienceMap.iterate) stays on
 * the host.  Creation, loop-closure and link decisions, experience cells, tags and headings `th` are bit-identical to
 * the host class; positions, link lengths and link headings may differ by the ulps of the device's cos, sin, atan2 and
 * hypot.  Inputs, all device memory:
 *   argmax : int64 [T][B], the C-order flat arg-max cell of agent b at frame t
 *   tag    : int32 [T][B], the view template the experience is tagged with (the template of frame t-1, -1 at t = 0);
 *            a tag outside [0, n_templates) means no view template (the host's vt=None: no loop-closure search)
 *   tw     : double [T][2], the shared (vtrans, vrot) given to update()   moved : uint8 [T], 0 = no update this frame
 *   X, Y, Th : the pose-cell grid; delta_pc : the loop-closure radius in cells (sqrt(d2) <= delta_pc)
 * Per-frame outputs, device memory: n_exp int32 [T][B] (experiences so far), exp_id int32 [T][B] (the current
 * experience, -1 = none), em_xy double [T][B][2] (its position, 0 while there is none).
 * work: device, prs_em_work_bytes(B, T, n_templates) bytes, no initialisation needed; the map is left there.  It holds
 * these arrays, element [i][b] at index i*B + b, each starting at a multiple of 256 bytes, in this order:
 *   double exp_x[T][B], exp_y[T][B], exp_th[T][B]             experiences: position and heading
 *   double link_d[T][B], link_heading[T][B], link_facing[T][B] links, in creation order
 *   double rel[3][B]                                           rel_x, rel_y, rel_th after the last frame
 *   int64  exp_cell[T][B]                                      the experience's C-order flat cell
 *   int32  exp_tag[T][B]                                       its view template, -1 = none
 *   int32  exp_next[T][B], out_head[T][B]                      candidate lists (next experience with the same tag) and
 *                                                              out-link lists (first link starting there), -1 = end
 *   int32  link_from[T][B], link_to[T][B], link_next[T][B]     link ends; next link with the same start
 *   int32  vt_head[n_templates][B]                             first experience of each template's candidate list
 *   int32  counts[4][B]                                        experiences, links, current experience (-1 = none),
 *                                                              loop closures
 * Experience i and link l of agent b exist for i < counts[0][b] and l < counts[1][b].  Asynchronous on `stream`. */
PRS_API size_t prs_em_work_bytes(int B, int T, int n_templates);
PRS_API int prs_em_linked_run(int B, int T, int n_templates, const long long* argmax, const int* tag, const double* tw,
                      const uint8_t* moved, int X, int Y, int Th, double delta_pc, void* work, int* n_exp, int* exp_id,
                      double* em_xy, void* stream);
/* The same for agents that replayed different recordings: agent b follows recording rec_of[b] (device int32 [B], in
 * [0, R)) of tw: device double [T][R][2] and moved: device uint8 [T][R] (frames past a recording's end: moved 0). */
PRS_API int prs_em_linked_multi_run(int B, int T, int n_templates, const long long* argmax, const int* tag, int R,
                            const double* tw, const uint8_t* moved, const int* rec_of, int X, int Y, int Th,
                            double delta_pc, void* work, int* n_exp, int* exp_id, double* em_xy, void* stream);

/* Maps that continue across calls (an ensemble session fed in pieces).  The session workspace is the layout above with
 * the rows keyed by capacities instead of T -- E rows for each experience and link array, N rows of vt_head -- followed
 * by one int32 error word at byte offset prs_em_work_bytes(B, E, N).  Each moved frame adds at most one experience and
 * one link, so the caller keeps E >= max(experiences, links) so far + the frames of the next call, and N above every tag.
 *   prs_em_session_bytes(B, E, N): device bytes of such a workspace.
 *   prs_em_session_init: an empty map for every agent (vt_head -1, counts (0, 0, -1, 0), rel 0, error word 0).
 *   prs_em_session_grow: copies the maps of `src` (layout B, E0, N0) into `dst` (B, E1, N1; E1 >= E0, N1 >= N0, not
 *            overlapping src) and fills the new vt_head rows with -1; asynchronous on `stream`.
 *   prs_em_linked_resume_run: prs_em_linked_multi_run continued over T more frames: the counts, rel and the current
 *            experience's pose come from the workspace and go back to it, vt_head is not reset.  rec_of may be NULL for
 *            R = 1.  A moved frame of an agent that has no room for one more experience and link, or whose tag is >= N,
 *            sets the error word to 1 and stops that agent: nothing is written past E or N, and the caller reads the
 *            word after the call. */
PRS_API size_t prs_em_session_bytes(int B, int E, int N);
PRS_API int prs_em_session_init(int B, int E, int N, void* work, void* stream);
PRS_API int prs_em_session_grow(int B, int E0, int N0, int E1, int N1, const void* src, void* dst, void* stream);
PRS_API int prs_em_linked_resume_run(int B, int T, int E, int N, const long long* argmax, const int* tag, int R,
                             const double* tw, const uint8_t* moved, const int* rec_of, int X, int Y, int Th,
                             double delta_pc, void* work, int* n_exp, int* exp_id, double* em_xy, void* stream);
/* The same agent copies for a session workspace (B, E, N): column dst[m] receives column src[m]'s experiences and links
 * below its counts, all N rows of vt_head, rel and the counts (loop closures included).  Rows at or past the counts are
 * never read, so the destination's are not cleared.  Overwritten sources are staged as in prs_ens_copy_agents.
 *   n_rows : host int32 [B], max(experiences, links) of every column, at most E (sizes the stage)
 *   stage  : device, prs_em_session_copy_stage_bytes(...) bytes for these moves
 * Asynchronous on `stream`.  prs_em_session_copy_stage_bytes returns 0 for invalid moves. */
PRS_API size_t prs_em_session_copy_stage_bytes(int B, int E, int N, int n_moves, const int* dst, const int* src,
                                       const int* n_rows);
PRS_API int prs_em_session_copy_agents(int B, int E, int N, void* work, int n_moves, const int* dst, const int* src,
                               const int* n_rows, void* stage, size_t stage_bytes, void* stream);
/* The same columns carried between two workspaces, as prs_ens_export_agents carries plan rows: export gathers columns
 * cols[k] (repeats allowed) of a (B, E, N) workspace into a stage whose header records K = n, `rows` (the largest
 * max(experiences, links) among them) and the workspace's N; import writes stage column k into column cols[k]
 * (distinct) of a (B', E', N') workspace -- the experiences and links below the counts, the stage's N vt_head rows, rel
 * and the counts -- and sets vt_head rows [N, N') of those columns to -1, since the column's own are stale.  Import
 * synchronises `stream` once to read the header and refuses, with PRS_E_INVALID, another column count, rows > E' or
 * N > N'.  A stage is imported once.
 *   n_rows : host int32 [B], max(experiences, links) of every column, at most E (sizes the stage)
 *   stage  : device, prs_em_session_export_stage_bytes(...) bytes (0 for invalid columns or n = 0)
 * Asynchronous on `stream`. */
PRS_API size_t prs_em_session_export_stage_bytes(int B, int E, int N, int n, const int* cols, const int* n_rows);
PRS_API int prs_em_session_export_agents(int B, int E, int N, const void* work, int n, const int* cols, const int* n_rows,
                                 void* stage, size_t stage_bytes, void* stream);
PRS_API int prs_em_session_import_agents(int B, int E, int N, void* work, int n, const int* cols, const void* stage,
                                 size_t stage_bytes, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* PYRATSLAM_B200_H */
