// Sharded view-template library: the one exchange step of a query, done on the device over NVLink.
//
// The library is split by contiguous template ranges over the ranks of a job (one process per GPU).  Every rank
// sweeps its shard and holds one packed key (min score << 32 | lowest global index); the global answer is the MIN
// of those keys -- numpy.argmin over the concatenated library (ratslam/view_templates.py:65-73).  Instead of an
// NCCL all-reduce (a collective launch, three eager elementwise kernels around it and a blocking read-back: about
// 80 us per query in round 1) each rank owns a small exchange buffer that its peers map with CUDA IPC, and ONE
// small kernel per query
//   1. stores the rank's key(s) into its slot of EVERY peer's buffer (st.relaxed.sys over NVLink), then publishes
//      them with a release store of the query's sequence number,
//   2. spins (ld.acquire.sys) until the W slots of its own buffer carry that sequence number,
//   3. takes the minimum, applies the reference's create-or-match rule (strict '>', view_templates.py:67) --
//      identically on every rank -- appends the query to the owning rank's shard when a template is created, and
//   4. writes the 32-byte result straight into pinned host memory.
// Slots are double buffered by the parity of the sequence number: a rank can only publish query s+1 after it has
// seen every peer's query s, i.e. after every peer has finished reading query s-1, so two parities are enough.
// A bounded spin (default 10 s of %globaltimer) turns a missing peer into an error instead of a hung GPU.
#include <new>
#include <string.h>
#include <time.h>

#include "common.cuh"
#include "vt_pack.cuh"

namespace {

constexpr int kMaxWorld = 16;
constexpr int kMaxKeys = 64;
constexpr int kXchgThreads = 256;

struct XchgBuf {  // lives in device memory of every rank; peers write into it
  unsigned long long flag[2][kMaxWorld];           // flag[parity][p]: sequence number of rank p's last publish
  unsigned long long keys[2][kMaxWorld][kMaxKeys];  // keys[parity][p][q]
};

struct ShardDecide {
  int enabled;
  int dtype;            // PRS_F32: float32 row-major library, else bit-sliced uint8
  int owner;            // this rank appends created templates
  double threshold;
  const void* tpl;      // the query as a row-major 32x32 template (device)
  void* lib;
  long long n_local, n_total;
};

__device__ __forceinline__ void st_relaxed_sys(unsigned long long* p, unsigned long long v) {
  asm volatile("st.relaxed.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ void st_release_sys(unsigned long long* p, unsigned long long v) {
  asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ unsigned long long ld_acquire_sys(const unsigned long long* p) {
  unsigned long long v;
  asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ unsigned long long ld_relaxed_sys(const unsigned long long* p) {
  unsigned long long v;
  asm volatile("ld.relaxed.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ unsigned long long global_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}

__global__ void __launch_bounds__(kXchgThreads)
    k_vt_xchg_min(XchgBuf* const* __restrict__ peers, int W, int rank, unsigned long long* __restrict__ seq_dev,
                  const unsigned long long* __restrict__ keys_local, int Q, unsigned long long* __restrict__ keys_out,
                  prs_shard_result* __restrict__ result, unsigned long long timeout_ns, ShardDecide d) {
  __shared__ int s_timeout;
  __shared__ unsigned long long s_key0;
  const int tid = threadIdx.x;
  const unsigned long long seq = *seq_dev + 1;  // thread 0 stores it back after the last barrier
  const int par = (int)(seq & 1);
  if (tid == 0) s_timeout = 0;
  // 1. publish: my keys into my slot of every rank's buffer (mine included), then the sequence number.  Thread p does
  //    both for peer p: its release store orders its own key stores before the flag, so no block-wide system fence
  //    (MEMBAR.SC.SYS, microseconds when writes to peers are in flight) is needed in front of it.
  if (tid < W) {
    XchgBuf* pb = peers[tid];
    for (int q = 0; q < Q; ++q) st_relaxed_sys(&pb->keys[par][rank][q], keys_local[q]);
    st_release_sys(&pb->flag[par][rank], seq);
  }
  __syncthreads();  // s_timeout is initialised for the waiters below
  // 2. wait for the W publishes of this query in my own buffer
  XchgBuf* mine = peers[rank];
  if (tid < W) {
    const unsigned long long t0 = global_ns();
    while (ld_acquire_sys(&mine->flag[par][tid]) != seq) {
      if (global_ns() - t0 > timeout_ns) {
        atomicOr(&s_timeout, 1);
        break;
      }
    }
  }
  __syncthreads();
  const int timed_out = s_timeout;
  // 3. minimum over the ranks: min score, then lowest global index (numpy.argmin, view_templates.py:73)
  if (tid < Q) {
    unsigned long long m = ~0ull;
    for (int p = 0; p < W; ++p) {
      const unsigned long long k = ld_relaxed_sys(&mine->keys[par][p][tid]);
      m = k < m ? k : m;
    }
    if (timed_out) m = ~0ull;
    if (keys_out != nullptr) keys_out[tid] = m;
    if (tid == 0) s_key0 = m;
  }
  __syncthreads();
  // 4. create-or-match (view_templates.py:67-73), the same decision on every rank
  if (d.enabled) {
    const unsigned long long k = s_key0;
    const unsigned hi = (unsigned)(k >> 32);
    const double score = d.dtype == PRS_F32 ? (double)__uint_as_float(hi) : (double)hi;
    const bool create = !timed_out && (d.n_total == 0 || k == ~0ull || score > d.threshold);
    if (create && d.owner) {
      if (d.dtype == PRS_F32) {
        float* dst = (float*)d.lib + (size_t)d.n_local * 1024;
        for (int i = tid; i < 1024; i += kXchgThreads) dst[i] = ((const float*)d.tpl)[i];
      } else if (tid < 32) {
        vt_pack_row((const uint8_t*)d.tpl, (uint4*)d.lib, d.n_local, tid);
      }
    }
    if (tid == 0 && result != nullptr) {
      result->key = k;
      result->created = create ? 1 : 0;
      result->template_index = create ? (int)d.n_total : (int)(k & 0xffffffffu);
      result->n_total = (int)d.n_total + (create ? 1 : 0);
      result->status = timed_out ? 1 : 0;
    }
  } else if (tid == 0 && result != nullptr) {
    result->key = s_key0;
    result->created = 0;
    result->template_index = -1;
    result->n_total = (int)d.n_total;
    result->status = timed_out ? 1 : 0;
  }
  if (tid == 0) {
    *seq_dev = seq;
    // the sequence number is what a host that polls the (pinned) record waits for: it goes out last, as a system-scope
    // release, so that the fields above and keys_out (written before the last barrier) are visible first
    if (result != nullptr) st_release_sys(&result->seq, seq);  // a release at system scope: cumulative over the barrier above
  }
}

// device-side alias of a pinned (mapped) host pointer; device pointers pass through
void* dev_alias(void* p) {
  if (p == nullptr) return nullptr;
  cudaPointerAttributes a;
  if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
    cudaGetLastError();
    return p;
  }
  if (a.type == cudaMemoryTypeHost) return a.devicePointer;
  return p;
}

}  // namespace

struct prs_xchg {
  int world, rank, device;
  XchgBuf* local;
  XchgBuf* peers[kMaxWorld];
  bool opened[kMaxWorld];
  XchgBuf** d_peers;
  unsigned long long* d_seq;
  unsigned long long timeout_ns;
  bool connected;
  unsigned long long host_seq;  // exchanges issued so far (= the device-side sequence number once they have run)
  // prs_vt_shard_query replays a repeated query chain (pack query, sweep, exchange) as ONE graph launch on a private stream
  cudaStream_t gs;
  cudaEvent_t gev;
  void* q_stage;  // 4 KiB: the recorded chain reads the query from here (the caller's query buffer may change per call)
  cudaGraphExec_t gexec;
  unsigned long long gkey[14], glast[14];
  int gsame;
  bool capturing;  // the exchange being enqueued is recorded into a graph: its launches are counted when replayed
};

extern "C" int prs_xchg_create(int world, int rank, prs_xchg** out) {
  PRS_REQUIRE(out, "prs_xchg_create: null argument");
  PRS_REQUIRE(world >= 1 && world <= kMaxWorld && rank >= 0 && rank < world,
              "prs_xchg_create: world must be in [1, %d] and rank in [0, world), got world=%d rank=%d", kMaxWorld, world, rank);
  prs_xchg* x = new (std::nothrow) prs_xchg();
  PRS_REQUIRE(x, "prs_xchg_create: out of host memory");
  memset(x, 0, sizeof(*x));
  x->world = world;
  x->rank = rank;
  x->timeout_ns = 10ull * 1000 * 1000 * 1000;
  cudaError_t e = cudaGetDevice(&x->device);
  if (e == cudaSuccess) e = cudaMalloc((void**)&x->local, sizeof(XchgBuf));
  if (e == cudaSuccess) e = cudaMemset(x->local, 0, sizeof(XchgBuf));
  if (e == cudaSuccess) e = cudaMalloc((void**)&x->d_peers, kMaxWorld * sizeof(XchgBuf*));
  if (e == cudaSuccess) e = cudaMalloc((void**)&x->d_seq, sizeof(unsigned long long));
  if (e == cudaSuccess) e = cudaMemset(x->d_seq, 0, sizeof(unsigned long long));
  if (e == cudaSuccess) e = cudaDeviceSynchronize();
  if (e != cudaSuccess) {
    prs_set_error("prs_xchg_create: %s", cudaGetErrorString(e));
    if (x->local) cudaFree(x->local);
    if (x->d_peers) cudaFree(x->d_peers);
    if (x->d_seq) cudaFree(x->d_seq);
    delete x;
    return PRS_E_CUDA;
  }
  x->peers[rank] = x->local;
  if (world == 1) {
    e = cudaMemcpy(x->d_peers, x->peers, sizeof(x->peers), cudaMemcpyHostToDevice);
    if (e != cudaSuccess) {
      prs_set_error("prs_xchg_create: %s", cudaGetErrorString(e));
      return PRS_E_CUDA;
    }
    x->connected = true;
  }
  *out = x;
  return PRS_OK;
}

extern "C" int prs_xchg_export(prs_xchg* x, void* handle64) {
  PRS_REQUIRE(x && handle64, "prs_xchg_export: null argument");
  static_assert(sizeof(cudaIpcMemHandle_t) == PRS_XCHG_HANDLE_BYTES, "IPC handle size");
  cudaIpcMemHandle_t h;
  PRS_CUDA(cudaIpcGetMemHandle(&h, x->local));
  memcpy(handle64, &h, sizeof(h));
  return PRS_OK;
}

extern "C" int prs_xchg_connect(prs_xchg* x, const void* handles) {
  PRS_REQUIRE(x && handles, "prs_xchg_connect: null argument");
  PRS_REQUIRE(!x->connected, "prs_xchg_connect: already connected");
  for (int p = 0; p < x->world; ++p) {
    if (p == x->rank) continue;
    cudaIpcMemHandle_t h;
    memcpy(&h, (const char*)handles + (size_t)p * PRS_XCHG_HANDLE_BYTES, sizeof(h));
    void* ptr = nullptr;
    cudaError_t e = cudaIpcOpenMemHandle(&ptr, h, cudaIpcMemLazyEnablePeerAccess);
    if (e != cudaSuccess) {
      prs_set_error("prs_xchg_connect: cudaIpcOpenMemHandle(rank %d): %s", p, cudaGetErrorString(e));
      (void)cudaGetLastError();
      return PRS_E_CUDA;
    }
    x->peers[p] = (XchgBuf*)ptr;
    x->opened[p] = true;
  }
  PRS_CUDA(cudaMemcpy(x->d_peers, x->peers, sizeof(x->peers), cudaMemcpyHostToDevice));
  x->connected = true;
  return PRS_OK;
}

extern "C" int prs_xchg_set_timeout(prs_xchg* x, double seconds) {
  PRS_REQUIRE(x && seconds > 0, "prs_xchg_set_timeout: bad argument");
  x->timeout_ns = (unsigned long long)(seconds * 1e9);
  return PRS_OK;
}

extern "C" int prs_xchg_destroy(prs_xchg* x) {
  if (x) {
    cudaDeviceSynchronize();
    for (int p = 0; p < x->world; ++p)
      if (x->opened[p]) cudaIpcCloseMemHandle(x->peers[p]);
    if (x->local) cudaFree(x->local);
    if (x->d_peers) cudaFree(x->d_peers);
    if (x->d_seq) cudaFree(x->d_seq);
    if (x->gexec) cudaGraphExecDestroy(x->gexec);
    if (x->q_stage) cudaFree(x->q_stage);
    if (x->gev) cudaEventDestroy(x->gev);
    if (x->gs) cudaStreamDestroy(x->gs);
    delete x;
  }
  return PRS_OK;
}

static int xchg_launch(prs_xchg* x, const unsigned long long* keys_local, int n_keys, unsigned long long* keys_out,
                       prs_shard_result* result, const ShardDecide& d, cudaStream_t st, const char* who) {
  PRS_REQUIRE(x->connected, "%s: the exchange is not connected (prs_xchg_connect)", who);
  int dev = -1;
  PRS_CUDA(cudaGetDevice(&dev));
  PRS_REQUIRE(dev == x->device, "%s: the exchange was created on device %d but device %d is current", who, x->device, dev);
  if (!x->capturing) ++x->host_seq;
  k_vt_xchg_min<<<1, kXchgThreads, 0, st>>>(x->d_peers, x->world, x->rank, x->d_seq, keys_local, n_keys,
                                            (unsigned long long*)dev_alias(keys_out),
                                            (prs_shard_result*)dev_alias(result), x->timeout_ns, d);
  PRS_CUDA(cudaGetLastError());
  return PRS_OK;
}

extern "C" int prs_vt_shard_exchange(prs_xchg* x, const unsigned long long* keys_local, int n_keys,
                                     unsigned long long* keys_out, prs_shard_result* result, void* stream) {
  PRS_REQUIRE(x && keys_local && (keys_out || result), "prs_vt_shard_exchange: null argument");
  PRS_REQUIRE(n_keys >= 1 && n_keys <= kMaxKeys, "prs_vt_shard_exchange: n_keys must be in [1, %d], got %d", kMaxKeys, n_keys);
  ShardDecide d;
  memset(&d, 0, sizeof(d));
  return xchg_launch(x, keys_local, n_keys, keys_out, result, d, (cudaStream_t)stream, "prs_vt_shard_exchange");
}

extern "C" int prs_vt_shard_decide(prs_xchg* x, const unsigned long long* key_local, double threshold, int dtype,
                                   const void* tpl, void* lib, long long n_local, long long n_total, int owner,
                                   prs_shard_result* result, void* stream) {
  PRS_REQUIRE(x && key_local && tpl && result, "prs_vt_shard_decide: null argument");
  PRS_REQUIRE(!owner || lib, "prs_vt_shard_decide: the owning rank needs its library buffer");
  PRS_REQUIRE(dtype == PRS_F32 || dtype == PRS_U8, "prs_vt_shard_decide: dtype must be PRS_F32 or PRS_U8");
  PRS_REQUIRE(n_local >= 0 && n_total >= 0 && n_total < 0x7fffffffLL, "prs_vt_shard_decide: bad template counts");
  ShardDecide d;
  d.enabled = 1;
  d.dtype = dtype;
  d.owner = owner ? 1 : 0;
  d.threshold = threshold;
  d.tpl = tpl;
  d.lib = lib;
  d.n_local = n_local;
  d.n_total = n_total;
  return xchg_launch(x, key_local, 1, nullptr, result, d, (cudaStream_t)stream, "prs_vt_shard_decide");
}

// Host side of a polled exchange: spin on the pinned record until the kernel of the LAST issued exchange has written
// its sequence number (a stream synchronisation costs a wake-up of 5-10 us; the record arrives ~1 us after the kernel).
extern "C" int prs_xchg_wait(prs_xchg* x, const prs_shard_result* result_host, double timeout_s) {
  PRS_REQUIRE(x && result_host, "prs_xchg_wait: null argument");
  const volatile unsigned long long* seq = &result_host->seq;
  const unsigned long long want = x->host_seq;
  unsigned long long spins = 0;
  struct timespec t0;
  clock_gettime(CLOCK_MONOTONIC, &t0);
  while (*seq < want) {
#if defined(__x86_64__)
    __builtin_ia32_pause();
#endif
    if ((++spins & 0xffff) == 0) {
      struct timespec t1;
      clock_gettime(CLOCK_MONOTONIC, &t1);
      if ((double)(t1.tv_sec - t0.tv_sec) + 1e-9 * (double)(t1.tv_nsec - t0.tv_nsec) > timeout_s) {
        cudaError_t e = cudaGetLastError();
        prs_set_error("prs_xchg_wait: exchange %llu did not complete within %.1f s (%s)", want, timeout_s,
                      cudaGetErrorString(e));
        return PRS_E_CUDA;
      }
    }
  }
  __atomic_thread_fence(__ATOMIC_ACQUIRE);
  return PRS_OK;
}

// One query of a sharded library in ONE call: the local sweep (bit-sliced uint8 or float32), the exchange kernel
// (MIN over the ranks, optionally the create-or-match decision and the append) and the wait for the pinned record.
// A query chain whose arguments repeat (the steady state of matching: same library size, same buffers) is captured
// once and replayed as a single graph launch on a private stream -- five dependent launches otherwise, whose gaps are
// most of what a query costs beyond its sweep.
static int shard_query_enqueue(prs_xchg* x, int dtype, void* lib, long long n_local, const void* query_dev, int mode,
                               long long base_index, unsigned long long* key_dev, void* scratch, int decide,
                               double threshold, long long n_total, int owner, prs_shard_result* result_pinned,
                               cudaStream_t st, bool planes_ready = false) {
  int rc;
  if (dtype == PRS_U8 && planes_ready)  // the query's bit planes are in `scratch` and the key is reset already
    rc = prs_vt_sweep_packed_planes(n_local ? lib : nullptr, n_local, scratch, mode, base_index, key_dev, st);
  else if (dtype == PRS_U8)
    rc = prs_vt_sweep_packed_u8(n_local ? lib : nullptr, n_local, (const uint8_t*)query_dev, mode, base_index, key_dev,
                                nullptr, scratch, st);
  else
    rc = prs_vt_sweep_f32(n_local ? (const float*)lib : nullptr, n_local, (const float*)query_dev, mode, base_index,
                          key_dev, nullptr, st);
  if (rc != PRS_OK) return rc;
  if (decide)
    return prs_vt_shard_decide(x, key_dev, threshold, dtype, query_dev, lib, n_local, n_total, owner, result_pinned, st);
  return prs_vt_shard_exchange(x, key_dev, 1, nullptr, result_pinned, st);
}

extern "C" int prs_vt_shard_query(prs_xchg* x, int dtype, void* lib, long long n_local, const void* query_dev, int mode,
                                  long long base_index, unsigned long long* key_dev, void* scratch, int decide,
                                  double threshold, long long n_total, int owner, prs_shard_result* result_pinned,
                                  void* stream) {
  PRS_REQUIRE(x && query_dev && key_dev && result_pinned, "prs_vt_shard_query: null argument");
  PRS_REQUIRE(dtype == PRS_U8 || dtype == PRS_F32, "prs_vt_shard_query: dtype must be PRS_U8 or PRS_F32");
  cudaStream_t st = (cudaStream_t)stream;
  unsigned long long thr_bits;
  memcpy(&thr_bits, &threshold, 8);
  const unsigned long long key[14] = {(unsigned long long)dtype, (unsigned long long)(uintptr_t)lib, (unsigned long long)n_local,
                                      0ull /* the query is staged */, (unsigned long long)mode,
                                      (unsigned long long)base_index, (unsigned long long)(uintptr_t)key_dev,
                                      (unsigned long long)(uintptr_t)scratch, (unsigned long long)decide, thr_bits,
                                      (unsigned long long)n_total, (unsigned long long)owner,
                                      (unsigned long long)(uintptr_t)result_pinned, (unsigned long long)x->device};
  const bool same_as_graph = x->gexec != nullptr && memcmp(key, x->gkey, sizeof(key)) == 0;
  // a decision that may APPEND changes n_local / n_total for the next call: such chains never repeat, stay eager
  const bool repeatable = !(decide && owner);
  if (!same_as_graph) {
    if (repeatable && memcmp(key, x->glast, sizeof(key)) == 0)
      ++x->gsame;
    else
      x->gsame = 0;
    memcpy(x->glast, key, sizeof(key));
    if (!repeatable || x->gsame < 2) {  // eager on the caller's stream
      int rc = shard_query_enqueue(x, dtype, lib, n_local, query_dev, mode, base_index, key_dev, scratch, decide, threshold,
                                   n_total, owner, result_pinned, st);
      if (rc != PRS_OK) return rc;
      return prs_xchg_wait(x, result_pinned, 30.0);
    }
    // third identical call: record the chain
    if (!x->gs) {
      PRS_CUDA(cudaStreamCreateWithFlags(&x->gs, cudaStreamNonBlocking));
      PRS_CUDA(cudaEventCreateWithFlags(&x->gev, cudaEventDisableTiming));
      PRS_CUDA(cudaMalloc(&x->q_stage, 4096));
    }
    if (x->gexec) {
      cudaGraphExecDestroy(x->gexec);
      x->gexec = nullptr;
    }
    cudaGraph_t g = nullptr;
    PRS_CUDA(cudaStreamBeginCapture(x->gs, cudaStreamCaptureModeThreadLocal));
    x->capturing = true;
    int rc = shard_query_enqueue(x, dtype, lib, n_local, x->q_stage, mode, base_index, key_dev, scratch, decide, threshold,
                                 n_total, owner, result_pinned, x->gs, true);
    x->capturing = false;
    cudaError_t e = cudaStreamEndCapture(x->gs, &g);
    if (rc != PRS_OK || e != cudaSuccess) {
      if (g) cudaGraphDestroy(g);
      if (rc == PRS_OK) prs_set_error("prs_vt_shard_query: graph capture failed: %s", cudaGetErrorString(e));
      return rc != PRS_OK ? rc : PRS_E_CUDA;
    }
    PRS_CUDA(cudaGraphInstantiate(&x->gexec, g, 0));
    cudaGraphDestroy(g);
    memcpy(x->gkey, key, sizeof(key));
  }
  // replay: the query goes into the staging buffer on the caller's stream (behind whatever produced it), the graph
  // runs behind that copy and behind sweeps of other streams
  // uint8: the query's bit planes go into `scratch` and the key is reset by one small kernel on the caller's stream (the
  // chain is then constant upload, sweep, exchange); the decision kernel still reads the raw query from the staging buffer
  // when it may append, and such chains are never replayed.  float32: the raw query is staged.
  if (dtype == PRS_U8 && n_local > 0) {
    if (int rc = prs_vt_pack_query_launch((const uint8_t*)query_dev, scratch, key_dev, st)) return rc;
    if (decide) PRS_CUDA(cudaMemcpyAsync(x->q_stage, query_dev, 1024, cudaMemcpyDeviceToDevice, st));
  } else {
    if (dtype == PRS_U8) PRS_CUDA(cudaMemsetAsync(key_dev, 0xff, sizeof(unsigned long long), st));
    PRS_CUDA(cudaMemcpyAsync(x->q_stage, query_dev, dtype == PRS_U8 ? 1024 : 4096, cudaMemcpyDeviceToDevice, st));
  }
  // the recorded chain runs on the caller's own stream, right behind the staging (the private stream is only what the
  // chain was captured on): no event, no cross-stream dependency on the way to a 25 us answer
  if (int rc = prs_vtq_begin(st)) return rc;
  cudaError_t le = cudaGraphLaunch(x->gexec, st);
  ++x->host_seq;
  int rc2 = prs_vtq_end(st);
  PRS_CUDA(le);
  if (rc2 != PRS_OK) return rc2;
  return prs_xchg_wait(x, result_pinned, 30.0);
}
