// C ABI glue: error reporting, plan life-cycle and the dispatch between the generic
// multi-kernel path and the fused SMEM-resident kernel.  See include/pyratslam_b200.h.
#include <stdarg.h>
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <new>

#include "common.cuh"

static thread_local char g_err[512] = "";

void prs_set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

extern "C" const char* prs_last_error(void) { return g_err; }
extern "C" int prs_version(void) { return 100; }

extern "C" int prs_device_count(void) {
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess) {
    prs_set_error("cudaGetDeviceCount: %s", cudaGetErrorString(e));
    (void)cudaGetLastError();
    return PRS_E_NODEVICE;
  }
  return n;
}

template <typename T>
static void fill_tables(PcTables<T>& t, const prs_pc_config* c) {
  for (int i = 0; i < 7; ++i) {
    t.ge[i] = (T)c->ge[i];
    t.gi[i] = (T)c->gi[i];
    t.gex[i] = (T)(c->aE * c->ge[i]);
    t.gix[i] = (T)(c->aI * c->gi[i]);
  }
  for (int f = 0; f < 2; ++f)
    for (int i = 0; i < 49; ++i) t.f2d[f][i] = (T)c->f2d[f * 49 + i];
  for (int o = 0; o < PRS_NOG; ++o)
    for (int i = 0; i < 7; ++i) t.f1d[o][i] = (T)c->f1d[o * 7 + i];
}

static void free_plan(prs_pc_plan* p) {
  void* ptrs[] = {p->cos_th, p->sin_th, p->s1,       nullptr,      p->s3,     nullptr,     p->shift, p->fsel,
                  p->ogi,    p->part_val, p->part_idx, p->inv_total, p->d_odom, p->d_argmax, p->d_err, p->d_total,
                  p->tab_dev, p->d_xyze, p->done_ctr};
  for (void* q : ptrs)
    if (q) cudaFree(q);
  if (p->sgraph) cudaGraphExecDestroy(p->sgraph);
  if (p->sev_in) cudaEventDestroy(p->sev_in);
  if (p->sev_out) cudaEventDestroy(p->sev_out);
  if (p->ss) cudaStreamDestroy(p->ss);
  if (p->hgraph) cudaGraphExecDestroy(p->hgraph);
  if (p->hev) cudaEventDestroy(p->hev);
  if (p->hs) cudaStreamDestroy(p->hs);
  for (int i = 0; i < 2; ++i) {
    cudaEvent_t evs[4] = {p->ev_h2d[i], p->ev_k[i], p->ev_done[i], p->ev_d2h[i]};
    for (cudaEvent_t e : evs)
      if (e) cudaEventDestroy(e);
    if (p->d_odom2[i]) cudaFree(p->d_odom2[i]);
    if (p->d_xyze2[i]) cudaFree(p->d_xyze2[i]);
  }
  if (p->ss2) cudaStreamDestroy(p->ss2);
  if (p->zc_ctr) cudaFree(p->zc_ctr);
  if (p->zc_done) cudaFreeHost(p->zc_done);
  if (p->cs_in) cudaStreamDestroy(p->cs_in);
  if (p->cs_out) cudaStreamDestroy(p->cs_out);
  if (p->net_seq) cudaFree(p->net_seq);
  void* act[7] = {p->al_cnt, p->al_idx, p->al_valid, p->dense_flag, p->dense_list, p->dense_cnt, p->big_list};
  for (void* q : act)
    if (q) cudaFree(q);
  free(p->h_cos);
  delete p;
}

extern "C" int prs_pc_create(const prs_pc_config* cfg, prs_pc_handle* out) {
  PRS_REQUIRE(cfg && out, "prs_pc_create: null argument");
  PRS_REQUIRE(cfg->X >= 3 && cfg->Y >= 3 && cfg->Th >= 3,
              "prs_pc_create: every grid dimension must be >= 3 (7-tap periodic filters), got %dx%dx%d", cfg->X,
              cfg->Y, cfg->Th);
  PRS_REQUIRE(cfg->B >= 1 && cfg->B <= 65535, "prs_pc_create: B must be in [1, 65535], got %d", cfg->B);
  PRS_REQUIRE(cfg->Th <= 65535, "prs_pc_create: Th must be <= 65535");
  PRS_REQUIRE((long long)cfg->X * cfg->Y * cfg->Th < (1LL << 31), "prs_pc_create: grid too large");
  PRS_REQUIRE(cfg->dtype == PRS_F32 || cfg->dtype == PRS_F64, "prs_pc_create: dtype must be PRS_F32 or PRS_F64");
  PRS_REQUIRE(cfg->ge && cfg->gi && cfg->f2d && cfg->f1d && cfg->cos_th && cfg->sin_th, "prs_pc_create: null table");
  PRS_REQUIRE(cfg->vtrans_scale > 0 && cfg->vrot_scale > 0, "prs_pc_create: scales must be positive");
  int ndev = prs_device_count();
  if (ndev <= 0) {
    prs_set_error("prs_pc_create: no CUDA device (this library has no CPU path)");
    return PRS_E_NODEVICE;
  }
  prs_pc_plan* p = new (std::nothrow) prs_pc_plan();
  PRS_REQUIRE(p, "prs_pc_create: out of host memory");
  memset(p, 0, sizeof(*p));
  if (cudaGetDevice(&p->device) != cudaSuccess) {
    prs_set_error("prs_pc_create: cudaGetDevice failed");
    delete p;
    return PRS_E_CUDA;
  }
  p->X = cfg->X;
  p->Y = cfg->Y;
  p->Th = cfg->Th;
  p->B = cfg->B;
  p->dtype = cfg->dtype;
  p->N = (long long)cfg->X * cfg->Y * cfg->Th;
  p->vtrans_scale = cfg->vtrans_scale;
  p->vrot_scale = cfg->vrot_scale;
  p->h_cos = (double*)malloc(p->Th * sizeof(double));
  if (!p->h_cos) {
    prs_set_error("prs_pc_create: out of host memory");
    delete p;
    return PRS_E_INVALID;
  }
  memcpy(p->h_cos, cfg->cos_th, p->Th * sizeof(double));
  fill_tables(p->tf, cfg);
  fill_tables(p->td, cfg);
  for (int t = 0; t < 7; ++t) {
    p->tl.ty[t] = make_float2(p->tf.ge[t], p->tf.gi[t]);
    p->tl.tx[t] = make_float2(p->tf.gex[t], p->tf.gix[t]);
  }
  for (int c = 0; c < 4; ++c)
    for (int a = 0; a < 7; ++a)
      for (int q = 0; q < 8; ++q)
        p->tl.f2p[c][a][q] = q < 7 ? make_float2(p->tf.f2d[c >> 1][a * 7 + q], p->tf.f2d[c & 1][a * 7 + q])
                                   : make_float2(0.f, 0.f);
  const size_t es = cfg->dtype == PRS_F32 ? 4 : 8;
  const size_t sbytes = (size_t)p->B * p->N * es;
  p->nblk_plane = (p->X * p->Y + 255) / 256;
  const int tiles = ((p->X + 31) / 32) * ((p->Y + 31) / 32);  // an upper bound of the tiled path's tile count
  p->np_max = p->Th * (p->nblk_plane > tiles ? p->nblk_plane : tiles);  // >= nblk_plane * ceil(Th/8) as well
  const size_t np = (size_t)p->B * p->np_max;
#define ALLOC(ptr, bytes)                                                        \
  do {                                                                           \
    cudaError_t e_ = cudaMalloc((void**)&(ptr), (bytes));                        \
    if (e_ != cudaSuccess) {                                                     \
      prs_set_error("prs_pc_create: cudaMalloc(%zu): %s", (size_t)(bytes), cudaGetErrorString(e_)); \
      free_plan(p);                                                              \
      return PRS_E_CUDA;                                                         \
    }                                                                            \
  } while (0)
  ALLOC(p->cos_th, p->Th * sizeof(double));
  ALLOC(p->sin_th, p->Th * sizeof(double));
  ALLOC(p->shift, (size_t)p->B * p->Th * 2 * sizeof(int));
  ALLOC(p->fsel, (size_t)p->B * p->Th);
  ALLOC(p->ogi, (size_t)p->B * sizeof(int));
  ALLOC(p->part_val, np * es);
  ALLOC(p->part_idx, np * sizeof(long long));
  ALLOC(p->inv_total, (size_t)p->B * es);
  ALLOC(p->d_odom, (size_t)p->B * 2 * sizeof(double));
  ALLOC(p->d_argmax, (size_t)p->B * sizeof(long long));
  ALLOC(p->d_err, (size_t)p->B * sizeof(int));
  ALLOC(p->d_total, (size_t)p->B * es);
  ALLOC(p->d_xyze, (size_t)p->B * 4 * sizeof(int));
  ALLOC(p->done_ctr, (size_t)p->B * sizeof(unsigned));
  cudaMemset(p->done_ctr, 0, (size_t)p->B * sizeof(unsigned));
  ALLOC(p->tab_dev, sizeof(PcTables<float>));
  ALLOC(p->net_seq, (size_t)p->B * sizeof(unsigned));
  cudaMemset(p->net_seq, 0, (size_t)p->B * sizeof(unsigned));
  p->forced_path = PRS_PATH_AUTO;
  p->resident_ok = prs_pc_resident_supported(p);
  p->pair_ok = prs_pc_pair_supported(p);
  p->tiled_ok = prs_pc_tiled_supported(p);
  int one_wave = 0;
  p->cluster_C = prs_pc_cluster_choose(p, &one_wave);
  p->cluster_ok = p->cluster_C >= 2;
  // One network per cluster pays when every cluster runs at once: a single 21x21x36 network takes 10 us against
  // 16.4 us (pair kernel) / 18.5 us (one CTA per network), a 50x50x10 one 12.6 us against 19 us (tiled).
  p->cluster_pref = p->cluster_ok && one_wave;
  // The multi-kernel paths need scratch of four state tensors; it is only allocated when such a path
  // can be taken for this plan (prs_pc_set_path / path_integration allocate it lazily otherwise).
  if (!p->resident_ok && !p->pair_ok) {
    ALLOC(p->s1, 2 * sbytes);
    ALLOC(p->s3, 2 * sbytes);
    p->s2 = (char*)p->s1 + sbytes;
    p->s4 = (char*)p->s3 + sbytes;
  }
#undef ALLOC
  cudaError_t e = cudaMemcpy(p->cos_th, cfg->cos_th, p->Th * sizeof(double), cudaMemcpyHostToDevice);
  if (e == cudaSuccess) e = cudaMemcpy(p->sin_th, cfg->sin_th, p->Th * sizeof(double), cudaMemcpyHostToDevice);
  if (e == cudaSuccess) e = cudaMemcpy(p->tab_dev, &p->tf, sizeof(PcTables<float>), cudaMemcpyHostToDevice);
  if (e != cudaSuccess) {
    prs_set_error("prs_pc_create: table upload: %s", cudaGetErrorString(e));
    free_plan(p);
    return PRS_E_CUDA;
  }
  *out = p;
  return PRS_OK;
}

int prs_pc_check_device(const prs_pc_plan* p, const char* who) {
  int dev = -1;
  PRS_CUDA(cudaGetDevice(&dev));
  PRS_REQUIRE(dev == p->device, "%s: the plan was created on device %d but device %d is current", who, p->device, dev);
  return PRS_OK;
}

extern "C" int prs_pc_destroy(prs_pc_handle h) {
  if (h) free_plan(h);
  return PRS_OK;
}

extern "C" size_t prs_pc_state_bytes(prs_pc_handle h) {
  return h ? (size_t)h->B * h->N * (h->dtype == PRS_F32 ? 4 : 8) : 0;
}

static int ensure_scratch(prs_pc_handle h) {
  if (!h->s1) {
    const size_t sbytes = prs_pc_state_bytes(h);
    PRS_CUDA(cudaMalloc(&h->s1, 2 * sbytes));
    PRS_CUDA(cudaMalloc(&h->s3, 2 * sbytes));
    h->s2 = (char*)h->s1 + sbytes;
    h->s4 = (char*)h->s3 + sbytes;
  }
  return PRS_OK;
}

extern "C" int prs_pc_path(prs_pc_handle h) {
  if (!h) return PRS_PATH_GENERIC;
  if (h->forced_path >= 0) return h->forced_path;
  if (h->cluster_pref) return PRS_PATH_CLUSTER;
  // Fused kernels.  float64: the pair kernel is the only fused one.  float32: two CTAs per network finish a wave in
  // 16.4 us against 18.5 us while every CTA has an SM of its own (B <= #SM / 2); beyond that the one-CTA kernel
  // wins (0.344 ms against 0.463 ms for 4096 networks, profiles/r2_path_compare.txt).
  if (h->pair_ok && (!h->resident_ok || h->B <= 74)) return PRS_PATH_PAIR;
  return h->resident_ok ? PRS_PATH_RESIDENT : (h->tiled_ok ? PRS_PATH_TILED : PRS_PATH_GENERIC);
}

static void drop_graphs(prs_pc_handle h);

extern "C" int prs_pc_set_path(prs_pc_handle h, int path) {
  PRS_REQUIRE(h, "prs_pc_set_path: null handle");
  const bool ok = path == PRS_PATH_AUTO || path == PRS_PATH_GENERIC || (path == PRS_PATH_RESIDENT && h->resident_ok) ||
                  (path == PRS_PATH_TILED && h->tiled_ok) || (path == PRS_PATH_CLUSTER && h->cluster_ok) ||
                  (path == PRS_PATH_PAIR && h->pair_ok);
  PRS_REQUIRE(ok, "prs_pc_set_path: path %d is not available for a %dx%dx%d %s plan", path, h->X, h->Y, h->Th,
              h->dtype == PRS_F32 ? "float32" : "float64");
  if (path == PRS_PATH_GENERIC || path == PRS_PATH_TILED) {
    int rc = ensure_scratch(h);
    if (rc != PRS_OK) return rc;
  }
  h->forced_path = path;
  drop_graphs(h);
  return PRS_OK;
}

extern "C" int prs_pc_set_option(prs_pc_handle h, int option, int value) {
  PRS_REQUIRE(h, "prs_pc_set_option: null handle");
  PRS_REQUIRE(option == PRS_OPT_ACTIVE_SET, "prs_pc_set_option: unknown option %d", option);
  PRS_REQUIRE(value >= 0 && value <= 2, "prs_pc_set_option: PRS_OPT_ACTIVE_SET takes 0, 1 or 2, got %d", value);
  if (value) {
    if (int rc_ = prs_pc_check_device(h, "prs_pc_set_option")) return rc_;
    int rc = prs_pc_active_prepare(h);
    if (rc == PRS_OK && !h->resident_ok) rc = ensure_scratch(h);  // the dense fallback is then the generic path
    if (rc != PRS_OK) return rc;
    rc = prs_pc_active_invalidate(h, nullptr);
    if (rc != PRS_OK) return rc;
    PRS_CUDA(cudaStreamSynchronize(nullptr));
  }
  h->opt_active = value;
  drop_graphs(h);
  return PRS_OK;
}

extern "C" int prs_pc_invalidate_active(prs_pc_handle h, void* stream) {
  PRS_REQUIRE(h, "prs_pc_invalidate_active: null handle");
  return prs_pc_active_invalidate(h, (cudaStream_t)stream);
}

static void drop_graphs(prs_pc_handle h) {
  if (h->hgraph) {  // a captured host-step graph holds the other path's kernels
    cudaGraphExecDestroy(h->hgraph);
    h->hgraph = nullptr;
  }
  if (h->sgraph) {
    cudaGraphExecDestroy(h->sgraph);
    h->sgraph = nullptr;
  }
}

// The carried lists (PRS_OPT_ACTIVE_SET = 2) describe the state tensor of the previous call: another tensor starts afresh.
static int active_same_state(prs_pc_handle h, const void* state, cudaStream_t st) {
  if (h->act_state != state) {
    h->act_state = state;
    return prs_pc_active_invalidate(h, st);
  }
  return PRS_OK;
}

// what follows the first active-set launch: its second tier, then the dense kernels for the flagged networks
static int active_fallback(prs_pc_handle h, void* state, const double* od, const void* gi, long long* am, void* tt, int* err,
                           cudaStream_t st) {
  int rc = prs_pc_active_step(h, state, od, gi, am, tt, err, 1, st);  // second tier, if the plan has one
  if (rc != PRS_OK) return rc;
  h->only_flag = h->dense_flag, h->only_list = h->dense_list, h->only_cnt = h->dense_cnt;
  if (h->resident_ok)
    rc = prs_pc_resident_step(h, state, od, 1, gi, am, tt, err, st);
  else
    rc = prs_pc_generic_step(h, state, od, gi, am, tt, err, st);
  h->only_flag = h->only_list = h->only_cnt = nullptr;
  return rc;
}

// One update of the active-set path as a graph whose dense fall-back sits behind a CONDITIONAL node: the active-set kernel
// raises the condition (cudaGraphSetConditional) when it flags a network, otherwise the fall-back's launches -- eight of
// them for plans without the fused kernel, each a grid of early exits -- do not exist on the device's timeline at all.
// Any failure (an older driver) returns PRS_E_CUDA with *out = nullptr and the caller captures the plain sequence.
static int capture_active_graph(prs_pc_handle h, void* state, const void* gi, long long* argmax, void* total, int* err,
                                cudaGraph_t* out) {
  *out = nullptr;
  cudaStream_t ss = h->ss;
  if (!h->ss2 && cudaStreamCreateWithFlags(&h->ss2, cudaStreamNonBlocking) != cudaSuccess) return PRS_E_CUDA;
  if (cudaStreamBeginCapture(ss, cudaStreamCaptureModeThreadLocal) != cudaSuccess) return PRS_E_CUDA;
  cudaGraph_t g = nullptr, body = nullptr, done = nullptr;
  cudaStreamCaptureStatus cs;
  cudaGraphConditionalHandle hd = 0;
  const cudaGraphNode_t* deps = nullptr;
  size_t nd = 0;
  cudaGraphNode_t cn;
  cudaGraphNodeParams cp = {};
  bool ok = cudaStreamGetCaptureInfo_v2(ss, &cs, nullptr, &g, nullptr, nullptr) == cudaSuccess && g != nullptr &&
            cudaGraphConditionalHandleCreate(&hd, g, 0, cudaGraphCondAssignDefault) == cudaSuccess;
  if (ok) {
    h->act_cond = (unsigned long long)hd;
    ok = cudaMemsetAsync(err, 0, (size_t)h->B * sizeof(int), ss) == cudaSuccess &&
         prs_pc_active_step(h, state, h->d_odom, gi, argmax, total, err, 0, ss) == PRS_OK;
    h->act_cond = 0;
  }
  ok = ok && cudaStreamGetCaptureInfo_v2(ss, &cs, nullptr, &g, &deps, &nd) == cudaSuccess;
  if (ok) {
    cp.type = cudaGraphNodeTypeConditional;
    cp.conditional.handle = hd;
    cp.conditional.type = cudaGraphCondTypeIf;
    cp.conditional.size = 1;
    ok = cudaGraphAddNode(&cn, g, deps, nd, &cp) == cudaSuccess && cp.conditional.phGraph_out != nullptr;
  }
  if (ok) {
    body = cp.conditional.phGraph_out[0];
    ok = cudaStreamUpdateCaptureDependencies(ss, &cn, 1, cudaStreamSetCaptureDependencies) == cudaSuccess;
  }
  const cudaError_t e_end = cudaStreamEndCapture(ss, &done);
  ok = ok && e_end == cudaSuccess && done != nullptr;
  if (ok) {  // the body: the dense kernels for the flagged networks
    ok = cudaStreamBeginCaptureToGraph(h->ss2, body, nullptr, nullptr, 0, cudaStreamCaptureModeThreadLocal) == cudaSuccess;
    if (ok) {
      const int rc = active_fallback(h, state, h->d_odom, gi, argmax, total, err, h->ss2);
      cudaGraph_t b2 = nullptr;
      const cudaError_t e2 = cudaStreamEndCapture(h->ss2, &b2);
      ok = rc == PRS_OK && e2 == cudaSuccess;
    }
  }
  if (!ok) {
    (void)cudaGetLastError();
    if (done) cudaGraphDestroy(done);
    return PRS_E_CUDA;
  }
  *out = done;
  return PRS_OK;
}

static int step_dispatch(prs_pc_handle h, void* state, const double* odom, int T, const void* gi, long long* argmax,
                         void* total, int* err, cudaStream_t st, int err_store = 0) {
  const size_t es = h->dtype == PRS_F32 ? 4 : 8;
  if (h->opt_active) {
    // Active-set update (posecell_active.cu): scan + one CTA per network; the networks it flags (dense state, negative
    // inhibition, ...) are then updated by a dense family that processes the flagged networks only: the fused
    // one-CTA-per-network kernel where the plan has it, else the generic kernels.
    if (int rc_ = active_same_state(h, state, st)) return rc_;
    for (int t = 0; t < T; ++t) {
      const double* od = odom + (size_t)t * h->B * 2;
      long long* am = argmax + (size_t)t * h->B;
      void* tt = (char*)total + (size_t)t * h->B * es;
      int rc = prs_pc_active_step(h, state, od, gi, am, tt, err, 0, st);
      if (rc == PRS_OK) rc = active_fallback(h, state, od, gi, am, tt, err, st);
      if (rc != PRS_OK) return rc;
    }
    return PRS_OK;
  }
  const int path = prs_pc_path(h);
  if (path == PRS_PATH_RESIDENT) return prs_pc_resident_step(h, state, odom, T, gi, argmax, total, err, st);
  if (path == PRS_PATH_PAIR) return prs_pc_pair_step(h, state, odom, T, gi, argmax, total, err, st);
  for (int t = 0; t < T; ++t) {
    int rc;
    if (path == PRS_PATH_CLUSTER)
      rc = prs_pc_cluster_step(h, (float*)state, odom + (size_t)t * h->B * 2, (const float*)gi,
                               argmax + (size_t)t * h->B, (float*)total + (size_t)t * h->B, err, err_store && T == 1, st);
    else if (path == PRS_PATH_TILED)
      rc = prs_pc_tiled_step(h, (float*)state, odom + (size_t)t * h->B * 2, (const float*)gi, argmax + (size_t)t * h->B,
                             (float*)total + (size_t)t * h->B, err, st);
    else
      rc = prs_pc_generic_step(h, state, odom + (size_t)t * h->B * 2, gi, argmax + (size_t)t * h->B,
                               (char*)total + (size_t)t * h->B * es, err, st);
    if (rc != PRS_OK) return rc;
  }
  return PRS_OK;
}

static int step_enqueue(prs_pc_handle h, void* state, const double* odom, const void* gi, long long* argmax, void* total,
                        int* err, cudaStream_t st) {
  // the cluster kernel gathers its error bits and stores them: one node less on a 12 us update
  if (prs_pc_path(h) == PRS_PATH_CLUSTER && !h->opt_active) return step_dispatch(h, state, odom, 1, gi, argmax, total, err, st, 1);
  // the fused one-CTA kernel zeroes err[b] itself: a memset between two of its launches would keep the second from
  // starting while the first one's last wave runs (posecell_resident.cu, programmatic dependent launch)
  if (!(prs_pc_path(h) == PRS_PATH_RESIDENT && !h->opt_active))
    PRS_CUDA(cudaMemsetAsync(err, 0, (size_t)h->B * sizeof(int), st));
  return step_dispatch(h, state, odom, 1, gi, argmax, total, err, st);
}

extern "C" int prs_pc_step(prs_pc_handle h, void* state, const double* odom, const void* gi, long long* argmax,
                           void* total, int* err, void* stream) {
  PRS_REQUIRE(h && state && odom && gi && argmax && total && err, "prs_pc_step: null argument");
  if (int rc_ = prs_pc_check_device(h, "prs_pc_step")) return rc_;
  cudaStream_t st = (cudaStream_t)stream;
  cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
  if (st != nullptr) PRS_CUDA(cudaStreamIsCapturing(st, &cap));
  // The fused kernels are one launch; a caller that is capturing its own graph gets plain launches as well.
  const int path_now = prs_pc_path(h);
  if (((path_now == PRS_PATH_RESIDENT || path_now == PRS_PATH_PAIR || path_now == PRS_PATH_CLUSTER) && !h->opt_active) ||
      cap != cudaStreamCaptureStatusNone)
    return step_enqueue(h, state, odom, gi, argmax, total, err, st);
  // Multi-kernel paths: replay the launch sequence as a graph on a private stream, ordered after the caller's
  // stream on entry and before it on exit (no host synchronisation).
  if (!h->ss) {
    PRS_CUDA(cudaStreamCreateWithFlags(&h->ss, cudaStreamNonBlocking));
    PRS_CUDA(cudaEventCreateWithFlags(&h->sev_in, cudaEventDisableTiming));
    PRS_CUDA(cudaEventCreateWithFlags(&h->sev_out, cudaEventDisableTiming));
  }
  // the odometry pointer usually changes from call to call: it is staged into the plan's own buffer outside the
  // graph, so that the captured launches only see fixed addresses
  const void* key[6] = {state, h->d_odom, gi, argmax, total, err};
  bool same = h->sgraph != nullptr;
  for (int i = 0; i < 6 && same; ++i) same = key[i] == h->skey[i];
  if (!same && h->swarm < 2) {  // first calls: eager on the caller's stream (lazy attributes, and short-lived users)
    ++h->swarm;
    return step_enqueue(h, state, odom, gi, argmax, total, err, st);
  }
  PRS_CUDA(cudaEventRecord(h->sev_in, st));
  PRS_CUDA(cudaStreamWaitEvent(h->ss, h->sev_in, 0));
  if (odom != h->d_odom)
    PRS_CUDA(cudaMemcpyAsync(h->d_odom, odom, (size_t)h->B * 2 * sizeof(double), cudaMemcpyDefault, h->ss));
  if (h->opt_active)  // outside the graph: a capture must not record the invalidation of another tensor's lists
    if (int rc_ = active_same_state(h, state, h->ss)) return rc_;
  if (!same) {
    if (h->sgraph) {
      cudaGraphExecDestroy(h->sgraph);
      h->sgraph = nullptr;
    }
    cudaGraph_t g = nullptr;
    if (h->opt_active) {
      if (capture_active_graph(h, state, gi, argmax, total, err, &g) == PRS_OK &&
          cudaGraphInstantiate(&h->sgraph, g, 0) != cudaSuccess) {
        (void)cudaGetLastError();
        h->sgraph = nullptr;
      }
      if (g) cudaGraphDestroy(g);
      g = nullptr;
    }
    if (!h->sgraph) {
      PRS_CUDA(cudaStreamBeginCapture(h->ss, cudaStreamCaptureModeThreadLocal));
      int rc = step_enqueue(h, state, h->d_odom, gi, argmax, total, err, h->ss);
      cudaError_t e = cudaStreamEndCapture(h->ss, &g);
      if (rc != PRS_OK || e != cudaSuccess) {
        if (g) cudaGraphDestroy(g);
        if (rc == PRS_OK) prs_set_error("prs_pc_step: graph capture failed: %s", cudaGetErrorString(e));
        return rc != PRS_OK ? rc : PRS_E_CUDA;
      }
      PRS_CUDA(cudaGraphInstantiate(&h->sgraph, g, 0));
      cudaGraphDestroy(g);
    }
    for (int i = 0; i < 6; ++i) h->skey[i] = key[i];
  }
  PRS_CUDA(cudaGraphLaunch(h->sgraph, h->ss));
  PRS_CUDA(cudaEventRecord(h->sev_out, h->ss));
  PRS_CUDA(cudaStreamWaitEvent(st, h->sev_out, 0));
  return PRS_OK;
}

int prs_pc_step_mirror(prs_pc_plan* h, void* state, const double* odom, const void* gi, long long* argmax, void* total,
                       int* err, long long* argmax2, int* err2, int* mirrored, cudaStream_t st) {
  *mirrored = 0;
  if (h && argmax2 && err2 && prs_pc_path(h) == PRS_PATH_CLUSTER && !h->opt_active) {
    PRS_REQUIRE(state && odom && gi && argmax && total && err, "prs_pc_step: null argument");
    if (int rc_ = prs_pc_check_device(h, "prs_pc_step")) return rc_;
    *mirrored = 1;
    return prs_pc_cluster_step(h, (float*)state, odom, (const float*)gi, argmax, (float*)total, err, 1, st, argmax2, err2);
  }
  return prs_pc_step(h, state, odom, gi, argmax, total, err, st);
}

extern "C" int prs_pc_path_integration(prs_pc_handle h, void* state, const double* odom, int* err, void* stream) {
  PRS_REQUIRE(h && state && odom && err, "prs_pc_path_integration: null argument");
  if (int rc_ = prs_pc_check_device(h, "prs_pc_path_integration")) return rc_;
  cudaStream_t st = (cudaStream_t)stream;
  int rc = ensure_scratch(h);
  if (rc != PRS_OK) return rc;
  PRS_CUDA(cudaMemsetAsync(err, 0, (size_t)h->B * sizeof(int), st));
  if (int rc_ = prs_pc_active_invalidate(h, st)) return rc_;
  return prs_pc_generic_path_integration(h, state, odom, err, st);
}

extern "C" int prs_pc_run(prs_pc_handle h, void* state, const double* odom, int T, const void* gi, long long* argmax,
                          void* total, int* err, void* stream) {
  PRS_REQUIRE(h && state && odom && gi && argmax && total && err, "prs_pc_run: null argument");
  if (int rc_ = prs_pc_check_device(h, "prs_pc_run")) return rc_;
  PRS_REQUIRE(T >= 0, "prs_pc_run: negative step count");
  cudaStream_t st = (cudaStream_t)stream;
  if (T == 0 || !(prs_pc_path(h) == PRS_PATH_RESIDENT && !h->opt_active))
    PRS_CUDA(cudaMemsetAsync(err, 0, (size_t)h->B * sizeof(int), st));
  if (T == 0) return PRS_OK;
  return step_dispatch(h, state, odom, T, gi, argmax, total, err, st);
}

extern "C" int prs_pc_step_host(prs_pc_handle h, void* state, const double* odom_host, const void* gi,
                                long long* argmax_host, int* err_host, void* stream) {
  PRS_REQUIRE(h && state && odom_host && gi && argmax_host && err_host, "prs_pc_step_host: null argument");
  if (int rc_ = prs_pc_check_device(h, "prs_pc_step_host")) return rc_;
  cudaStream_t st = (cudaStream_t)stream;
  PRS_CUDA(cudaMemcpyAsync(h->d_odom, odom_host, (size_t)h->B * 2 * sizeof(double), cudaMemcpyHostToDevice, st));
  int rc = prs_pc_step(h, state, h->d_odom, gi, h->d_argmax, h->d_total, h->d_err, st);
  if (rc != PRS_OK) return rc;
  PRS_CUDA(cudaMemcpyAsync(argmax_host, h->d_argmax, (size_t)h->B * sizeof(long long), cudaMemcpyDeviceToHost, st));
  PRS_CUDA(cudaMemcpyAsync(err_host, h->d_err, (size_t)h->B * sizeof(int), cudaMemcpyDeviceToHost, st));
  PRS_CUDA(cudaStreamSynchronize(st));
  return PRS_OK;
}

// device-side alias of a pinned (hence mapped) host buffer, or null
static void* mapped_alias(const void* p) {
  cudaPointerAttributes a;
  if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
    cudaGetLastError();
    return nullptr;
  }
  return a.type == cudaMemoryTypeHost ? a.devicePointer : nullptr;
}

// prs_pc_step followed by the (x, y, th, err) packing of its result into `xyze` (device or mapped host memory): the fused
// one-CTA kernel writes the packed record itself (one kernel less between two updates -- which is also what lets two
// updates of the overlapped host API overlap), every other path launches the small packing kernel.
static int step_and_pack(prs_pc_handle h, void* state, const double* odom, const void* gi, int* xyze, cudaStream_t st) {
  const bool fused = prs_pc_path(h) == PRS_PATH_RESIDENT && !h->opt_active;
  h->res_xyze = fused ? xyze : nullptr;
  int rc = prs_pc_step(h, state, odom, gi, h->d_argmax, h->d_total, h->d_err, st);
  h->res_xyze = nullptr;
  if (rc != PRS_OK || fused) return rc;
  return prs_pc_launch_unravel_pack(h, h->d_argmax, h->d_err, xyze, st);
}

static int step_host_xyz_enqueue(prs_pc_handle h, void* state, const double* odom_host, const void* gi, int* result_host,
                                 cudaStream_t st) {
  // A handful of networks: with pinned host buffers the kernels read the odometry and write the packed result in
  // place (zero-copy), which takes the two copy nodes -- most of a 12 us update's overhead -- out of the chain.
  if (h->B <= 64) {
    const double* od = (const double*)mapped_alias(odom_host);
    int* res = (int*)mapped_alias(result_host);
    if (od && res) return step_and_pack(h, state, od, gi, res, st);
  }
  PRS_CUDA(cudaMemcpyAsync(h->d_odom, odom_host, (size_t)h->B * 2 * sizeof(double), cudaMemcpyHostToDevice, st));
  int rc = step_and_pack(h, state, h->d_odom, gi, h->d_xyze, st);
  if (rc != PRS_OK) return rc;
  PRS_CUDA(cudaMemcpyAsync(result_host, h->d_xyze, (size_t)h->B * 4 * sizeof(int), cudaMemcpyDeviceToHost, st));
  return PRS_OK;
}

// Fused path with mapped pinned buffers: the kernel reads the odometry from host memory (two doubles per network, read a
// whole stage ahead of their use), writes the packed records into host memory and signals completion through a pinned
// word (slot 0 / 1: the overlapped API's two steps in flight; slot 2: the blocking call).  The stream then carries nothing
// but the update kernels, and consecutive updates overlap (posecell_resident.cu).  *launched = 0: not applicable.
static int zero_copy_submit(prs_pc_handle h, void* state, const double* odom_host, const void* gi, int* result_host,
                            cudaStream_t st, int s, int* launched) {
  *launched = 0;
  static const bool zc_on = [] {
    const char* e = getenv("PRS_HOST_ZERO_COPY");
    return !(e && atoi(e) == 0);
  }();
  if (!zc_on || prs_pc_path(h) != PRS_PATH_RESIDENT || h->opt_active) return PRS_OK;
  cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
  if (st != nullptr) PRS_CUDA(cudaStreamIsCapturing(st, &cap));
  if (cap != cudaStreamCaptureStatusNone) return PRS_OK;
  const double* od = (const double*)mapped_alias(odom_host);
  int* res = (int*)mapped_alias(result_host);
  if (!od || !res) return PRS_OK;
  if (!h->zc_ctr) {
    PRS_CUDA(cudaMalloc((void**)&h->zc_ctr, 3 * sizeof(unsigned)));
    PRS_CUDA(cudaMemset(h->zc_ctr, 0, 3 * sizeof(unsigned)));
    PRS_CUDA(cudaHostAlloc((void**)&h->zc_done, 3 * sizeof(unsigned), cudaHostAllocMapped));
    h->zc_done[0] = h->zc_done[1] = h->zc_done[2] = 0;
  }
  unsigned* done_dev = nullptr;
  PRS_CUDA(cudaHostGetDevicePointer((void**)&done_dev, h->zc_done + s, 0));
  h->zc_seq[s] = ++h->zc_launch;
  h->res_xyze = res, h->res_done_ctr = h->zc_ctr + s, h->res_done_host = done_dev, h->res_done_val = h->zc_seq[s];
  int rc = prs_pc_step(h, state, od, gi, h->d_argmax, h->d_total, h->d_err, st);
  h->res_xyze = nullptr, h->res_done_ctr = nullptr, h->res_done_host = nullptr;
  if (rc == PRS_OK) *launched = 1;
  return rc;
}

static int zero_copy_wait(prs_pc_handle h, int slot) {
  const volatile unsigned* w = h->zc_done + slot;
  const unsigned want = h->zc_seq[slot];
  struct timespec t0;
  clock_gettime(CLOCK_MONOTONIC, &t0);
  unsigned long long spins = 0;
  while ((int)(*w - want) < 0) {
#if defined(__x86_64__)
    __builtin_ia32_pause();
#endif
    if ((++spins & 0xfffff) == 0) {
      struct timespec t1;
      clock_gettime(CLOCK_MONOTONIC, &t1);
      if ((double)(t1.tv_sec - t0.tv_sec) > 30.0) {
        cudaError_t e = cudaGetLastError();
        prs_set_error("zero-copy update %u did not complete within 30 s (%s)", want, cudaGetErrorString(e));
        return PRS_E_CUDA;
      }
    }
  }
  __atomic_thread_fence(__ATOMIC_ACQUIRE);
  return PRS_OK;
}

extern "C" int prs_pc_step_host_xyz_async(prs_pc_handle h, void* state, const double* odom_host, const void* gi,
                                          int* result_host, void* stream, int* slot_out) {
  PRS_REQUIRE(h && state && odom_host && gi && result_host && slot_out, "prs_pc_step_host_xyz_async: null argument");
  if (int rc_ = prs_pc_check_device(h, "prs_pc_step_host_xyz_async")) return rc_;
  cudaStream_t st = (cudaStream_t)stream;
  {
    int launched = 0;
    const int s = h->pipe_slot;
    if (int rc = zero_copy_submit(h, state, odom_host, gi, result_host, st, s, &launched)) return rc;
    if (launched) {
      h->pipe_slot ^= 1;
      h->pipe_used[s] = 2;
      *slot_out = s;
      return PRS_OK;
    }
  }
  if (!h->cs_in) {
    PRS_CUDA(cudaStreamCreateWithFlags(&h->cs_in, cudaStreamNonBlocking));
    PRS_CUDA(cudaStreamCreateWithFlags(&h->cs_out, cudaStreamNonBlocking));
    for (int i = 0; i < 2; ++i) {
      PRS_CUDA(cudaEventCreateWithFlags(&h->ev_h2d[i], cudaEventDisableTiming));
      PRS_CUDA(cudaEventCreateWithFlags(&h->ev_k[i], cudaEventDisableTiming));
      PRS_CUDA(cudaEventCreateWithFlags(&h->ev_done[i], cudaEventDisableTiming));
      PRS_CUDA(cudaEventCreateWithFlags(&h->ev_d2h[i], cudaEventDisableTiming));
      PRS_CUDA(cudaMalloc((void**)&h->d_odom2[i], (size_t)h->B * 2 * sizeof(double)));
      PRS_CUDA(cudaMalloc((void**)&h->d_xyze2[i], (size_t)h->B * 4 * sizeof(int)));
    }
  }
  const int s = h->pipe_slot;
  h->pipe_slot ^= 1;
  // odometry in, on the copy-in stream, once the kernel that last read this slot's buffer is done
  if (h->pipe_used[s]) PRS_CUDA(cudaStreamWaitEvent(h->cs_in, h->ev_k[s], 0));
  PRS_CUDA(cudaMemcpyAsync(h->d_odom2[s], odom_host, (size_t)h->B * 2 * sizeof(double), cudaMemcpyHostToDevice, h->cs_in));
  PRS_CUDA(cudaEventRecord(h->ev_h2d[s], h->cs_in));
  PRS_CUDA(cudaStreamWaitEvent(st, h->ev_h2d[s], 0));
  if (h->pipe_used[s]) PRS_CUDA(cudaStreamWaitEvent(st, h->ev_d2h[s], 0));  // this slot's result buffer is free again
  int rc = step_and_pack(h, state, h->d_odom2[s], gi, h->d_xyze2[s], st);
  if (rc != PRS_OK) return rc;
  PRS_CUDA(cudaEventRecord(h->ev_k[s], st));
  PRS_CUDA(cudaEventRecord(h->ev_done[s], st));
  // result out, on the copy-out stream
  PRS_CUDA(cudaStreamWaitEvent(h->cs_out, h->ev_done[s], 0));
  PRS_CUDA(cudaMemcpyAsync(result_host, h->d_xyze2[s], (size_t)h->B * 4 * sizeof(int), cudaMemcpyDeviceToHost, h->cs_out));
  PRS_CUDA(cudaEventRecord(h->ev_d2h[s], h->cs_out));
  h->pipe_used[s] = 1;
  *slot_out = s;
  return PRS_OK;
}

extern "C" int prs_pc_host_result_wait(prs_pc_handle h, int slot) {
  PRS_REQUIRE(h && (slot == 0 || slot == 1) && h->pipe_used[slot], "prs_pc_host_result_wait: no step was submitted in slot %d", slot);
  if (h->pipe_used[slot] == 2) return zero_copy_wait(h, slot);  // the kernel's last CTA stores the launch number
  PRS_CUDA(cudaEventSynchronize(h->ev_d2h[slot]));
  return PRS_OK;
}

extern "C" int prs_pc_step_host_xyz(prs_pc_handle h, void* state, const double* odom_host, const void* gi,
                                    int* result_host, void* stream) {
  PRS_REQUIRE(h && state && odom_host && gi && result_host, "prs_pc_step_host_xyz: null argument");
  if (int rc_ = prs_pc_check_device(h, "prs_pc_step_host_xyz")) return rc_;
  cudaStream_t caller = (cudaStream_t)stream;
  if (h->B > 64) {  // (a handful of networks keep their graph: zero-copy there already, one launch either way)
    int launched = 0;
    if (int rc = zero_copy_submit(h, state, odom_host, gi, result_host, caller, 2, &launched)) return rc;
    if (launched) return zero_copy_wait(h, 2);
  }
  if (!h->hs) {
    PRS_CUDA(cudaStreamCreateWithFlags(&h->hs, cudaStreamNonBlocking));
    PRS_CUDA(cudaEventCreateWithFlags(&h->hev, cudaEventDisableTiming));
  }
  // whatever the caller enqueued before (inject, a posecells assignment) happens first
  PRS_CUDA(cudaEventRecord(h->hev, caller));
  PRS_CUDA(cudaStreamWaitEvent(h->hs, h->hev, 0));
  const void* key[4] = {state, odom_host, gi, result_host};
  const bool same = h->hgraph && key[0] == h->hkey[0] && key[1] == h->hkey[1] && key[2] == h->hkey[2] && key[3] == h->hkey[3];
  int rc = PRS_OK;
  if (same) {
    PRS_CUDA(cudaGraphLaunch(h->hgraph, h->hs));
  } else if (h->hwarm < 2) {  // the first calls run eagerly (lazy kernel attributes, scratch allocation)
    ++h->hwarm;
    rc = step_host_xyz_enqueue(h, state, odom_host, gi, result_host, h->hs);
    if (rc != PRS_OK) return rc;
  } else {
    if (h->hgraph) {
      cudaGraphExecDestroy(h->hgraph);
      h->hgraph = nullptr;
    }
    cudaGraph_t g = nullptr;
    PRS_CUDA(cudaStreamBeginCapture(h->hs, cudaStreamCaptureModeThreadLocal));
    rc = step_host_xyz_enqueue(h, state, odom_host, gi, result_host, h->hs);
    cudaError_t e = cudaStreamEndCapture(h->hs, &g);
    if (rc != PRS_OK || e != cudaSuccess) {
      if (g) cudaGraphDestroy(g);
      if (rc == PRS_OK) prs_set_error("prs_pc_step_host_xyz: graph capture failed: %s", cudaGetErrorString(e));
      return rc != PRS_OK ? rc : PRS_E_CUDA;
    }
    PRS_CUDA(cudaGraphInstantiate(&h->hgraph, g, 0));
    cudaGraphDestroy(g);
    for (int i = 0; i < 4; ++i) h->hkey[i] = key[i];
    PRS_CUDA(cudaGraphLaunch(h->hgraph, h->hs));
  }
  PRS_CUDA(cudaStreamSynchronize(h->hs));
  return PRS_OK;
}

// PoseCellNetwork.update((vtrans, vrot)) of a single-network plan in ONE call (posecell_network.py:326-353): the
// conditions under which the reference raises or reads unwritten memory are checked on the host first, in the same
// float64 arithmetic numpy uses (posecell_network.py:249,252-267; convolution.py:661-675), so that a rejected update
// leaves the state untouched; then the odometry goes into the caller's pinned buffer and the step runs as
// prs_pc_step_host_xyz does.  Returns PRS_OK, PRS_E_LUT_KEY (the reference's KeyError), PRS_E_RADIUS, or an error.
extern "C" int prs_pc_update_host(prs_pc_handle h, void* state, double vtrans, double vrot, const void* gi,
                                  double* odom_pinned, int* result_pinned, void* stream) {
  PRS_REQUIRE(h && state && gi && odom_pinned && result_pinned, "prs_pc_update_host: null argument");
  PRS_REQUIRE(h->B == 1, "prs_pc_update_host: the plan holds %d networks, not one", h->B);
  const volatile double vt = vtrans / h->vtrans_scale;  // volatile: every product below is rounded to double on its own
  for (int k = 0; k < h->Th; ++k) {
    const volatile double ex = vt * h->h_cos[k];
    const volatile double d = ex - rint(ex);             // numpy.around: half to even
    const volatile double d10 = d * 10.0;
    if ((long long)d10 >= 5) {
      prs_set_error("prs_pc_update_host: fractional x offset +0.5 on plane %d (the reference raises KeyError)", k);
      return PRS_E_LUT_KEY;
    }
  }
  if (3.0 + ceil(fabs(vt)) > (double)(h->X < h->Y ? h->X : h->Y)) {
    prs_set_error("prs_pc_update_host: translation of %.3g cells does not fit a %dx%d grid", (double)vt, h->X, h->Y);
    return PRS_E_RADIUS;
  }
  odom_pinned[0] = vtrans;
  odom_pinned[1] = vrot;
  return prs_pc_step_host_xyz(h, state, odom_pinned, gi, result_pinned, stream);
}
