// Shared declarations for the pyratslam_b200 CUDA library (sm_100a).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/pyratslam_b200.h"

void prs_set_error(const char* fmt, ...);

#define PRS_CUDA(call)                                                                         \
  do {                                                                                         \
    cudaError_t e_ = (call);                                                                   \
    if (e_ != cudaSuccess) {                                                                   \
      prs_set_error("%s:%d %s: %s", __FILE__, __LINE__, #call, cudaGetErrorString(e_));        \
      return PRS_E_CUDA;                                                                       \
    }                                                                                          \
  } while (0)

#define PRS_REQUIRE(cond, ...)      \
  do {                              \
    if (!(cond)) {                  \
      prs_set_error(__VA_ARGS__);   \
      return PRS_E_INVALID;         \
    }                               \
  } while (0)

#define PRS_NOG (2 * PRS_OG_RANGE + 1)

// Filter tables in the arithmetic type of the plan.  Passed to kernels by value
// (kernel parameter space = constant bank, 1960 bytes for double).
template <typename T>
struct PcTables {
  T ge[7], gi[7];    // theta and y passes of the separable E / I Gaussians
  T gex[7], gix[7];  // x pass with the amplitudes aE, aI folded in
  T f2d[2][49];      // F0 and F-1 of the path-integration LUT, [a*7+b]
  T f1d[PRS_NOG][7]; // theta filters for og = -PRS_OG_RANGE..PRS_OG_RANGE
};

// Coefficient PAIRS of the tiled float32 kernels, passed by value (constant bank): a packed FFMA2 can take such a
// pair straight from two adjacent uniform registers (one LDCU.64), which keeps them out of the register file
// and off the shared-memory pipe.
struct TlPairs {
  float2 ty[7];         // (ge[t], gi[t])      theta / y passes on (E, I)
  float2 tx[7];         // (aE*ge[t], aI*gi[t])  x pass
  float2 f2p[4][7][8];  // [(fsel_plane0 * 2 + fsel_plane1)][tap row][tap column (7 used)]: (F_p0, F_p1) of a plane pair
};

struct prs_pc_plan {
  int X, Y, Th, B, dtype;
  int device;   // the CUDA device the plan's buffers live on; every entry point checks it is current
  long long N;  // cells per network
  double vtrans_scale, vrot_scale;
  PcTables<float> tf;
  PcTables<double> td;
  TlPairs tl;
  double* cos_th;  // device [Th]
  double* sin_th;
  double* h_cos;   // host copy of cos_th (prs_pc_update_host checks the LUT key before touching the state)
  // scratch: two allocations of 2*B*N elements; s1|s2 are the halves of the first, s3|s4 of the second
  void *s1, *s2, *s3, *s4;
  int* shift;           // [B][Th][2] integer origins (ox, oy)
  unsigned char* fsel;  // [B][Th] 0 = F0, 1 = F-1
  int* ogi;             // [B] index into f1d
  int nblk_plane;       // blocks per theta plane in the generic kernels
  int np_max;           // partial-result slots per network (covers the generic and the tiled kernels)
  int tiled_ok;         // the tiled large-grid kernels support this shape/dtype
  void* part_val;       // [B][Th*nblk_plane] partial sums, later partial maxima
  long long* part_idx;  // [B][Th*nblk_plane]
  void* inv_total;      // [B]
  unsigned* done_ctr;   // [B] last-block-done counters of k_tl_theta_fin (atomicInc wraps them back to 0)
  // staging for the *_host entry points
  double* d_odom;
  long long* d_argmax;
  int* d_err;
  void* d_total;
  int* d_xyze;          // [B][4] int32 (x, y, th, err) for prs_pc_step_host_xyz
  // prs_pc_step_host_xyz replays its copy -> step -> unravel -> copy sequence as a CUDA graph on a private stream
  cudaStream_t hs;
  cudaEvent_t hev;
  cudaGraphExec_t hgraph;
  const void* hkey[4];  // (state, odom_host, gi, result_host) the graph was captured with
  int hwarm;
  // prs_pc_step on the multi-kernel paths (tiled, generic) is replayed as a graph too: eight dependent launches
  // are CPU-enqueue bound otherwise
  cudaStream_t ss;
  cudaEvent_t sev_in, sev_out;
  cudaGraphExec_t sgraph;
  const void* skey[6];  // (state, odom, gi, argmax, total, err)
  int swarm;
  // prs_pc_step_host_xyz_async: two slots of device staging, copies on their own streams so that the odometry of
  // step t+1 goes in and the result of step t-1 comes out while the kernel of step t runs
  cudaStream_t cs_in, cs_out;
  cudaEvent_t ev_h2d[2], ev_k[2], ev_done[2], ev_d2h[2];
  double* d_odom2[2];
  int* d_xyze2[2];
  int pipe_slot, pipe_used[2];
  int forced_path;      // -1 = automatic choice, else one of the PRS_PATH_* codes (prs_pc_set_path)
  int cluster_C;        // CTAs per network of the thread-block-cluster kernel, 0 if it does not apply to this plan
  int cluster_ok;       // = cluster_C >= 2
  int cluster_pref;     // ... and the network count is small enough for it to be the automatic choice
  int resident_ok;      // the fused SMEM-resident kernel supports this shape/dtype
  int pair_ok;          // ... and so does the one-network-per-2-CTA-cluster kernel (posecell_pair.cu)
  void* tab_dev;        // device copy of PcTables<float> for the resident kernel
  unsigned* net_seq;    // [B] per-network sequence numbers of the resident kernel's overlappable launches
  unsigned res_seq;     // launches of that chain so far
  int* res_xyze;        // set around a launch by the host API: the kernel also writes (x, y, th, err) per network there
  // zero-copy host stepping (prs_pc_step_host_xyz_async with mapped pinned buffers on the fused path): no copies, no
  // events; the launch's last CTA stores the launch number into a pinned word that prs_pc_host_result_wait polls
  unsigned* res_done_ctr;   // set around a launch: device counter of finished CTAs
  unsigned* res_done_host;  // ... device alias of the pinned completion word
  unsigned res_done_val;
  unsigned* zc_ctr;         // [3] device counters, one per slot (2: the blocking call)
  unsigned* zc_done;        // [3] pinned completion words
  unsigned zc_seq[3], zc_launch;
  // active-set path (posecell_active.cu), prs_pc_set_option(PRS_OPT_ACTIVE_SET)
  int opt_active;       // 0 = off, 1 = scan the state for its non-zero cells every update, 2 = keep the list across updates
  int* al_cnt;          // [B] entries in a network's active list (may exceed al_cap: overflow)
  int* al_idx;          // [B][al_cap] flat state indices of the non-zero cells
  int* al_valid;        // [B] the list describes the state as it is (mode 2)
  int al_cap;
  int* dense_flag;      // [B] 1 = the active-set kernel left this network to the dense kernels
  int* dense_list;      // [B] the flagged networks, dense_cnt of them
  int* dense_cnt;
  const void* act_state;        // the state tensor the carried lists describe
  unsigned long long act_cond;  // conditional-graph handle the active-set kernel raises when it flags a network (0: none)
  cudaStream_t ss2;     // the stream the conditional node's body is captured on
  int* big_list;        // [B] networks whose compressed grids need the second tier's arena, dense_cnt[1] of them
  int act_threads, act_arena, act_arena1;  // arena bytes of the (second) tier; first tier's, 0 = one tier only
  // non-null while a dense launcher runs as the active-set fallback: the kernels process network b only if only_flag[b]
  // (generic kernels), the resident kernel walks only_list[0 .. *only_cnt)
  const int* only_flag;
  const int* only_list;
  const int* only_cnt;
};

int prs_pc_check_device(const prs_pc_plan* p, const char* who);

// launchers implemented per translation unit
int prs_pc_generic_step(prs_pc_plan* p, void* state, const double* odom, const void* gi, long long* argmax,
                        void* total, int* err, cudaStream_t st);
int prs_pc_generic_path_integration(prs_pc_plan* p, void* state, const double* odom, int* err, cudaStream_t st);
int prs_pc_generic_argmax(prs_pc_plan* p, const void* state, long long* argmax, cudaStream_t st);
int prs_pc_tiled_supported(const prs_pc_plan* p);
int prs_pc_tiled_step(prs_pc_plan* p, float* state, const double* odom, const float* gi, long long* argmax, float* total,
                      int* err, cudaStream_t st);
// small shared kernels (implemented in posecell_generic.cu)
int prs_pc_launch_unravel_pack(prs_pc_plan* p, const long long* argmax, const int* err, int* out, cudaStream_t st);
int prs_pc_launch_plan(prs_pc_plan* p, const double* odom, int* err, cudaStream_t st);
int prs_pc_launch_sum_final_f32(prs_pc_plan* p, int np, float* total, cudaStream_t st);
int prs_pc_launch_argmax_final_f32(prs_pc_plan* p, int np, long long* argmax, cudaStream_t st);
int prs_pc_cluster_choose(const prs_pc_plan* p, int* one_wave);
// err_store != 0: err[b] is overwritten with the update's bits (needs no zeroed buffer); 0: OR-ed into it
// argmax2 / err2: optional second destination of network b's arg-max and error bits (both or neither)
int prs_pc_cluster_step(prs_pc_plan* p, float* state, const double* odom, const float* gi, long long* argmax,
                        float* total, int* err, int err_store, cudaStream_t st, long long* argmax2 = nullptr,
                        int* err2 = nullptr);
// prs_pc_step that, where the plan's kernel can do it (the cluster path), ALSO writes the arg-max and error bits of
// every network to argmax2 / err2 (*mirrored = 1); otherwise a plain prs_pc_step (*mirrored = 0)
int prs_pc_step_mirror(prs_pc_plan* h, void* state, const double* odom, const void* gi, long long* argmax, void* total,
                       int* err, long long* argmax2, int* err2, int* mirrored, cudaStream_t st);
int prs_pc_resident_supported(const prs_pc_plan* p);
int prs_pc_pair_supported(const prs_pc_plan* p);
int prs_pc_pair_step(prs_pc_plan* p, void* state, const double* odom, int T, const void* gi, long long* argmax,
                     void* total, int* err, cudaStream_t st);
int prs_pc_resident_step(prs_pc_plan* p, void* state, const double* odom, int T, const void* gi, long long* argmax,
                         void* total, int* err, cudaStream_t st);
int prs_pc_active_supported(const prs_pc_plan* p);
int prs_pc_active_prepare(prs_pc_plan* p);
// scan + active-set update of every network (one update); networks it could not handle are flagged in p->dense_flag /
// p->dense_list for the caller's dense kernels
// part 0: the scan and the (first-tier) active-set kernel over all networks; part 1: the second tier over the networks
// the first one could not hold (a no-op for one-tier plans)
int prs_pc_active_step(prs_pc_plan* p, void* state, const double* odom, const void* gi, long long* argmax, void* total,
                       int* err, int part, cudaStream_t st);
// the active lists no longer describe the state (something else wrote it)
int prs_pc_active_invalidate(prs_pc_plan* p, cudaStream_t st);

// ordering of the packed sweeps through their per-device constant buffer (view_templates.cu, VtqScope): a caller that
// launches a GRAPH containing such a sweep brackets the launch with these (begin locks a host mutex, end releases it)
int prs_vt_pack_query_launch(const uint8_t* query, void* scratch, unsigned long long* key, cudaStream_t st);
int prs_vt_sweep_packed_planes(const void* packed, long long n, const void* planes, int mode, long long base_index,
                               unsigned long long* key_out, cudaStream_t st);
int prs_vtq_begin(cudaStream_t st);
int prs_vtq_end(cudaStream_t st);

// ---- small device helpers -------------------------------------------------
#ifdef __CUDACC__
__device__ __forceinline__ int prs_modp_dev(int v, int n) {
  int r = v % n;
  return r < 0 ? r + n : r;
}
// Global inhibition (posecell_network.py:339-340) is two masked writes, `pc[pc < gi] = 0` then `pc[pc >= gi] -= gi`.
// A cell below gi is zeroed by the first and, when 0 >= gi, lowered by gi again by the second: it ends at max(-gi, 0),
// not at 0.  Every other cell ends at a - gi.  For gi >= 0 this is max(a - gi, 0); for gi < 0 it is not.  The floor is
// +0 for gi = -0 and gi = +0 alike, as numpy's 0.0 - (-0.0).
template <typename T>
__device__ __forceinline__ T inhib_floor(T gi) {
  return gi < T(0) ? -gi : T(0);
}
// Decisions of one path-integration step for (network b, plane k): bit-for-bit the float64 arithmetic numpy
// does on the host (posecell_network.py:252-267,249,304); explicit _rn intrinsics keep the compiler from
// contracting mul+sub into an FMA.
__device__ __forceinline__ void prs_plan_cell(int b, int k, int Th, int minXY, const double* __restrict__ odom,
                                              const double* __restrict__ cos_th, const double* __restrict__ sin_th,
                                              double vtrans_scale, double vrot_scale, int* __restrict__ shift,
                                              unsigned char* __restrict__ fsel, int* __restrict__ ogi,
                                              int* __restrict__ err) {
  const int i = b * Th + k;
  const double vt = __ddiv_rn(odom[2 * b], vtrans_scale);
  const double ex = __dmul_rn(vt, cos_th[k]);
  const double ey = __dmul_rn(vt, sin_th[k]);
  const double oxd = rint(ex), oyd = rint(ey);  // numpy.around: half to even
  const double dx = __dsub_rn(ex, oxd);
  const int key = (int)__dmul_rn(dx, 10.0);  // int(): truncation toward zero
  shift[2 * i] = (int)oxd;
  shift[2 * i + 1] = (int)oyd;
  fsel[i] = key < 0 ? 1 : 0;
  int e = 0;
  if (key >= 5) e |= PRS_ERR_LUT_KEY;
  if (k == 0) {
    const double radius = ceil(fabs(vt));
    if (!(3.0 + radius <= (double)minXY)) e |= PRS_ERR_RADIUS;
    const double vr = __ddiv_rn(odom[2 * b + 1], vrot_scale);
    const double og = floor(__dadd_rn(vr, 0.5));
    if (!(fabs(og) <= 64.0)) e |= PRS_ERR_THETA;
    const int ogc = og < -(double)PRS_OG_RANGE ? -PRS_OG_RANGE : (og > (double)PRS_OG_RANGE ? PRS_OG_RANGE : (int)og);
    ogi[b] = ogc + PRS_OG_RANGE;
  }
  if (e) atomicOr(&err[b], e);  // err[] is zeroed by the caller (prs_pc_step) and OR-ed across steps (prs_pc_run)
}
#endif

__device__ __forceinline__ int wrap1(int v, int n) {  // valid for -n <= v < 2n
  v = v < 0 ? v + n : v;
  return v >= n ? v - n : v;
}
__device__ __forceinline__ int modp(int v, int n) {  // any v
  int r = v % n;
  return r < 0 ? r + n : r;
}
