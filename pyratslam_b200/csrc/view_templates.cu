// View-template library sweep (ratslam/view_templates.py:16-28,63-75) for sm_100a.
//
// One launch scores every stored 32x32 template against one query and leaves
// (min score << 32 | lowest index) in a single uint64 -- the value and the
// numpy.argmin tie-break the reference obtains with a Python list comprehension.
//
// uint8 (the ROS path, ros_simulate.py:100-101): the reference's ``abs(T - q)`` on
// uint8 arrays wraps modulo 256, so the score is  sum((T - q) mod 256).  Each lane
// owns one 4-byte column word of a template; the 16 (ref mode) or 32 (circular
// mode) query rows of that column word stay in registers for the whole sweep.
// A template row is loaded once (one 32-byte DRAM sector per 8 lanes) and used
// against every query row it is paired with; each pairing costs three integer ops
// per 4 bytes:   r = (a|H) - (q&~H)        (byte-wise subtract, no cross-byte borrow)
//                z = r ^ (~a&H) ^ (q&H)    (repair bit 7 of every byte)
//                acc = dp4a(z, 0x01010101, acc)
// The per-offset sums are reduced over the 8 lanes of a template with a halving
// butterfly, the minimum over offsets is taken, and the packed key is min-reduced
// warp -> block -> one atomicMin.
//
// float32 ("profiles", BASELINE config 5): one template per warp, lane == column,
// score = sum |T - q| accumulated in float32.
//
// Those two are the row-major kernels.  What the product runs on big libraries (further down in this file):
//   k_vt_sweep_packed_ref_ring   bit-sliced uint8 library, reference mode: 8 LOP3 + 1 POPC per 32 byte-compares,
//                                warp-private rings of TMA bulk copies, the warps of a CTA in lock step
//   k_vt_sweep_packed_circ       the same library, all 32 cyclic shifts (counters rotated in registers)
//   k_vt_sweep_f32_pair          float32 library: two columns per lane (add.f32x2), two templates per warp, rings
//   k_vt_sweep_packed_ref_small  small libraries inside replayed frames: one block per group of 32 templates
// and the frame entry points (prs_frame_*, prs_replay_run) that chain them with the pose-cell update.
#include <new>
#include <string.h>

#include <algorithm>
#include <cmath>
#include <mutex>
#include <vector>

#include "common.cuh"
#include "vt_pack.cuh"
#include "agent_moves.cuh"

namespace {

constexpr int kVtThreads = 256;
constexpr unsigned kH = 0x80808080u;

template <int MODE>
struct VtShape;
template <>
struct VtShape<PRS_VT_MODE_REF> {  // stored rows 1..30 against query rows 8..23, o = t - s in [-7, 7]
  static constexpr int T0 = 1, T1 = 31, S0 = 8, NS = 16, NOFF = 15, NACC = 16;
  __host__ __device__ static constexpr int off(int t, int s) { return t - s + 7; }
  __host__ __device__ static constexpr bool valid(int t, int s) { return t - s >= -7 && t - s <= 7; }
};
template <>
struct VtShape<PRS_VT_MODE_CIRCULAR> {  // every stored row against every query row, o = (t - s) mod 32
  static constexpr int T0 = 0, T1 = 32, S0 = 0, NS = 32, NOFF = 32, NACC = 32;
  __host__ __device__ static constexpr int off(int t, int s) { return (t - s) & 31; }
  __host__ __device__ static constexpr bool valid(int, int) { return true; }
};

__device__ __forceinline__ unsigned ld_stream_u32(const unsigned* p) {
  unsigned v;
  asm volatile("ld.global.nc.L1::no_allocate.u32 %0, [%1];" : "=r"(v) : "l"(p));
  return v;
}
__device__ __forceinline__ float ld_stream_f32(const float* p) {
  float v;
  asm volatile("ld.global.nc.L1::no_allocate.f32 %0, [%1];" : "=f"(v) : "l"(p));
  return v;
}

// Sum the per-offset accumulators over a group of LANES lanes (LANES a power of two, groups aligned),
// halving the number of live accumulators per lane at each step.  On return lane holds N_FINAL fully
// reduced accumulators acc[0..N_FINAL) whose offset indices are base + j.
template <int N, int M, typename V>
struct Butterfly {
  __device__ __forceinline__ static void run(V* acc, int lane, int& base) {
    if constexpr (M >= 1) {
      if constexpr (N > 1) {
        constexpr int h = N / 2;
        const bool up = (lane & M) != 0;
#pragma unroll
        for (int i = 0; i < h; ++i) {
          V send = up ? acc[i] : acc[i + h];
          V keep = up ? acc[i + h] : acc[i];
          acc[i] = keep + __shfl_xor_sync(0xffffffffu, send, M);
        }
        base += up ? h : 0;
        Butterfly<h, M / 2, V>::run(acc, lane, base);
      } else {
        acc[0] += __shfl_xor_sync(0xffffffffu, acc[0], M);
        Butterfly<1, M / 2, V>::run(acc, lane, base);
      }
    }
  }
};
template <int N, typename V>
struct Butterfly<N, 0, V> {
  __device__ __forceinline__ static void run(V*, int, int&) {}
};

constexpr int final_count(int n, int lanes) {
  while (lanes > 1 && n > 1) {
    n /= 2;
    lanes /= 2;
  }
  return n;
}

__device__ __forceinline__ unsigned long long warp_min_u64(unsigned long long k) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    unsigned long long k2 = __shfl_xor_sync(0xffffffffu, k, o);
    k = k2 < k ? k2 : k;
  }
  return k;
}

__device__ __forceinline__ void block_min_to_global(unsigned long long key, unsigned long long* out) {
  __shared__ unsigned long long sm[kVtThreads / 32];
  key = warp_min_u64(key);
  int w = threadIdx.x >> 5, l = threadIdx.x & 31;
  if (l == 0) sm[w] = key;
  __syncthreads();
  if (w == 0) {
    key = l < kVtThreads / 32 ? sm[l] : ~0ull;
    key = warp_min_u64(key);
    if (l == 0 && key != ~0ull) atomicMin(out, key);
  }
}

// --------------------------------------------------------------------------- uint8
template <int MODE>
__global__ void __launch_bounds__(kVtThreads)
    k_vt_sweep_u8(const uint8_t* __restrict__ lib, long long n, const uint8_t* __restrict__ query, long long base_index,
                  unsigned long long* __restrict__ key_out, uint32_t* __restrict__ scores) {
  using S = VtShape<MODE>;
  const int lane = threadIdx.x & 31;
  const int w = lane & 7;   // column word of the 32-byte row
  const int tj = lane >> 3; // template within the group of four
  // query rows of this column word, pre-split for the byte-wise subtract
  unsigned qlo[S::NS], qhi[S::NS];
#pragma unroll
  for (int s = 0; s < S::NS; ++s) {
    unsigned q = reinterpret_cast<const unsigned*>(query)[(S::S0 + s) * 8 + w];
    qlo[s] = q & ~kH;
    qhi[s] = q & kH;
  }
  const long long n_groups = (n + 3) >> 2;
  const long long warp0 = ((long long)blockIdx.x * kVtThreads + threadIdx.x) >> 5;
  const long long n_warps = ((long long)gridDim.x * kVtThreads) >> 5;
  unsigned long long best = ~0ull;
  for (long long g = warp0; g < n_groups; g += n_warps) {
    const long long ti = g * 4 + tj;
    const bool live = ti < n;
    const unsigned* tp = reinterpret_cast<const unsigned*>(lib) + (live ? ti : 0) * 256 + w;
    unsigned a[S::T1 - S::T0];
#pragma unroll
    for (int t = S::T0; t < S::T1; ++t) a[t - S::T0] = ld_stream_u32(tp + t * 8);
    unsigned acc[S::NACC];
#pragma unroll
    for (int i = 0; i < S::NACC; ++i) acc[i] = 0;
#pragma unroll
    for (int t = S::T0; t < S::T1; ++t) {
      const unsigned av = a[t - S::T0];
      const unsigned ahi = av | kH;
      const unsigned afix = ~av & kH;
#pragma unroll
      for (int s = 0; s < S::NS; ++s) {
        if (S::valid(t, S::S0 + s)) {
          unsigned z = (ahi - qlo[s]) ^ afix ^ qhi[s];
          acc[S::off(t, S::S0 + s)] = __dp4a(z, 0x01010101u, acc[S::off(t, S::S0 + s)]);
        }
      }
    }
    int obase = 0;
    Butterfly<S::NACC, 4, unsigned>::run(acc, lane, obase);
    constexpr int NF = final_count(S::NACC, 8);
    unsigned m = 0xffffffffu;
#pragma unroll
    for (int j = 0; j < NF; ++j)
      if (obase + j < S::NOFF) m = min(m, acc[j]);
    m = min(m, __shfl_xor_sync(0xffffffffu, m, 4));
    m = min(m, __shfl_xor_sync(0xffffffffu, m, 2));
    m = min(m, __shfl_xor_sync(0xffffffffu, m, 1));
    if (live) {
      unsigned long long key = ((unsigned long long)m << 32) | (unsigned long long)(base_index + ti);
      best = key < best ? key : best;
      if (scores != nullptr && w == 0) scores[ti] = m;
    }
  }
  block_min_to_global(best, key_out);
}

// --------------------------------------------------------------------------- float32
template <int MODE>
__global__ void __launch_bounds__(kVtThreads)
    k_vt_sweep_f32(const float* __restrict__ lib, long long n, const float* __restrict__ query, long long base_index,
                   unsigned long long* __restrict__ key_out, float* __restrict__ scores) {
  using S = VtShape<MODE>;
  const int lane = threadIdx.x & 31;  // column
  float q[S::NS];
#pragma unroll
  for (int s = 0; s < S::NS; ++s) q[s] = query[(S::S0 + s) * 32 + lane];
  const long long warp0 = ((long long)blockIdx.x * kVtThreads + threadIdx.x) >> 5;
  const long long n_warps = ((long long)gridDim.x * kVtThreads) >> 5;
  unsigned long long best = ~0ull;
  for (long long ti = warp0; ti < n; ti += n_warps) {
    const float* tp = lib + ti * 1024 + lane;
    float a[S::T1 - S::T0];
#pragma unroll
    for (int t = S::T0; t < S::T1; ++t) a[t - S::T0] = ld_stream_f32(tp + t * 32);
    float acc[S::NACC];
#pragma unroll
    for (int i = 0; i < S::NACC; ++i) acc[i] = 0.f;
#pragma unroll
    for (int t = S::T0; t < S::T1; ++t) {
#pragma unroll
      for (int s = 0; s < S::NS; ++s) {
        if (S::valid(t, S::S0 + s)) acc[S::off(t, S::S0 + s)] += fabsf(a[t - S::T0] - q[s]);
      }
    }
    int obase = 0;
    Butterfly<S::NACC, 16, float>::run(acc, lane, obase);
    float m = (obase < S::NOFF) ? acc[0] : INFINITY;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = fminf(m, __shfl_xor_sync(0xffffffffu, m, o));
    unsigned long long key = ((unsigned long long)__float_as_uint(m) << 32) | (unsigned long long)(base_index + ti);
    best = key < best ? key : best;
    if (scores != nullptr && lane == 0) scores[ti] = m;
  }
  block_min_to_global(best, key_out);
}

// --------------------------------------------------------------------------- sub-sampling mask
__global__ void k_vt_extract_u8(const uint8_t* __restrict__ frame, int im_cols, int row_lo, int row_step, int col_lo,
                                int col_step, uint8_t* __restrict__ out, int n_rows, int n_cols) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_rows * n_cols) return;
  int r = i / n_cols, c = i - r * n_cols;
  // n-th index strictly above lo with (idx - lo) % step != 0
  int rr = row_lo + (r / (row_step - 1)) * row_step + (r % (row_step - 1)) + 1;
  int cc = col_lo + (c / (col_step - 1)) * col_step + (c % (col_step - 1)) + 1;
  out[i] = frame[(size_t)rr * im_cols + cc];
}

int sweep_grid(long long units_per_warp_total) {
  // persistent-style grid: enough CTAs to fill 148 SMs a few times over, never more than the work
  long long warps = units_per_warp_total;
  long long blocks = (warps + (kVtThreads / 32) - 1) / (kVtThreads / 32);
  long long cap = 148LL * 8;
  if (blocks > cap) blocks = cap;
  if (blocks < 1) blocks = 1;
  return (int)blocks;
}

}  // namespace

// the boolean mask of view_templates.py:48-57 must select exactly n_rows x n_cols pixels inside the frame
static int check_mask(int im_rows, int im_cols, int row_lo, int row_hi, int row_step, int col_lo, int col_hi, int col_step,
                      int n_rows, int n_cols) {
  PRS_REQUIRE(row_step >= 2 && col_step >= 2, "prs_vt_extract_u8: step must be >= 2 (step 1 selects nothing)");
  auto count = [](int lo, int hi, int step) { return (hi - lo - 1) - (hi - lo - 1) / step; };
  PRS_REQUIRE(row_lo >= 0 && col_lo >= 0 && row_hi <= im_rows && col_hi <= im_cols && row_hi > row_lo && col_hi > col_lo,
              "prs_vt_extract_u8: ranges outside the %dx%d frame", im_rows, im_cols);
  PRS_REQUIRE(count(row_lo, row_hi, row_step) == n_rows && count(col_lo, col_hi, col_step) == n_cols,
              "prs_vt_extract_u8: mask selects %dx%d pixels, not %dx%d", count(row_lo, row_hi, row_step),
              count(col_lo, col_hi, col_step), n_rows, n_cols);
  return PRS_OK;
}

extern "C" int prs_vt_extract_u8(const uint8_t* frame, int im_rows, int im_cols, int row_lo, int row_hi, int row_step,
                                 int col_lo, int col_hi, int col_step, uint8_t* out, int n_rows, int n_cols,
                                 void* stream) {
  PRS_REQUIRE(frame && out, "prs_vt_extract_u8: null argument");
  if (int rc = check_mask(im_rows, im_cols, row_lo, row_hi, row_step, col_lo, col_hi, col_step, n_rows, n_cols)) return rc;
  int total = n_rows * n_cols;
  k_vt_extract_u8<<<(total + 255) / 256, 256, 0, (cudaStream_t)stream>>>(frame, im_cols, row_lo, row_step, col_lo,
                                                                         col_step, out, n_rows, n_cols);
  PRS_CUDA(cudaGetLastError());
  return PRS_OK;
}

extern "C" int prs_vt_sweep_u8(const uint8_t* lib, long long n, const uint8_t* query, int mode, long long base_index,
                               unsigned long long* key_out, uint32_t* scores, void* stream) {
  PRS_REQUIRE(query && key_out && n >= 0 && (lib || n == 0), "prs_vt_sweep_u8: bad argument");
  PRS_REQUIRE(mode == PRS_VT_MODE_REF || mode == PRS_VT_MODE_CIRCULAR, "prs_vt_sweep_u8: unknown mode %d", mode);
  PRS_REQUIRE(base_index >= 0 && base_index + n <= 0xffffffffLL, "prs_vt_sweep_u8: template index does not fit 32 bits");
  cudaStream_t st = (cudaStream_t)stream;
  PRS_CUDA(cudaMemsetAsync(key_out, 0xff, sizeof(unsigned long long), st));
  if (n == 0) return PRS_OK;
  int grid = sweep_grid((n + 3) / 4);
  if (mode == PRS_VT_MODE_REF)
    k_vt_sweep_u8<PRS_VT_MODE_REF><<<grid, kVtThreads, 0, st>>>(lib, n, query, base_index, key_out, scores);
  else
    k_vt_sweep_u8<PRS_VT_MODE_CIRCULAR><<<grid, kVtThreads, 0, st>>>(lib, n, query, base_index, key_out, scores);
  PRS_CUDA(cudaGetLastError());
  return PRS_OK;
}

extern "C" int prs_vt_match_host_u8(const uint8_t* lib, long long n, const uint8_t* query_host, int mode,
                                    long long base_index, unsigned long long* key_host, void* scratch, void* stream) {
  PRS_REQUIRE(query_host && key_host && scratch, "prs_vt_match_host_u8: null argument");
  cudaStream_t st = (cudaStream_t)stream;
  uint8_t* dq = (uint8_t*)scratch;
  unsigned long long* dk = (unsigned long long*)(dq + 1024);
  PRS_CUDA(cudaMemcpyAsync(dq, query_host, 1024, cudaMemcpyHostToDevice, st));
  int rc = prs_vt_sweep_u8(lib, n, dq, mode, base_index, dk, nullptr, st);
  if (rc != PRS_OK) return rc;
  PRS_CUDA(cudaMemcpyAsync(key_host, dk, sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
  PRS_CUDA(cudaStreamSynchronize(st));
  return PRS_OK;
}

// =============================================================================================
// Bit-sliced ("packed") uint8 library.
//
// The byte-wise SWAR sweep above is bound by the integer pipes (64 lanes/clk/SM on B200, measured):
// 3 instructions per 4 byte-compares = 0.50 of the HBM roof at best.  The reference score only needs
//     sum((a - b) mod 256) = sum(a) - sum(b) + 256 * #{a < b}            (checked in the CPU tests)
// so the library is stored as bit planes: for every template row, 8 words, word k holding bit k of the
// row's 32 pixels.  #{a < b} over a row pair is then 8 LOP3 (one per plane, LSB to MSB:
// lt = (~a & b) | (~(a ^ b) & lt)) and one POPC for 32 pixels -- 10 instructions per 32 compares instead
// of 24.  One lane owns one template, 32 templates are interleaved so that a warp's 128-bit loads are
// contiguous 512-byte runs, and the query planes are __constant__ operands of the LOP3s (no registers,
// no loads).  Row sums (uint16 x 32) ride along: 1088 bytes per template.
//
// Layout of one group of 32 templates (8704 uint32):
//   planes : uint4 [32 rows][2 halves][32 lanes]   .x..w = planes 4h..4h+3 of that row of template `lane`
//   rowsum : uint4 [4][32 lanes]                   16 words per lane, word w = R[2w] | R[2w+1] << 16
constexpr int kGroupU4 = kVtGroupU4;  // 2176 uint4 = 34816 bytes per 32 templates (vt_pack.cuh)

__constant__ uint32_t c_vtq[32 * 8 + 8];  // query planes [row][k], then sum(rows 8..23), sum(all rows)

// c_vtq is ONE buffer per device, and the sweeps need the planes as constant-bank operands of their LOP3s (read from
// anywhere else they cost registers the kernels do not have).  Sweeps issued on different streams -- or from different
// host threads -- of a device are therefore ordered through it: a sweep records an event behind its kernel, and the
// next writer of the buffer on another stream waits for that event on the device (no host blocking).  The host mutex
// is held from the wait to the record, so two threads cannot interleave their (write planes, sweep) pairs either.
struct VtqGuard {
  std::mutex mu;
  cudaEvent_t ev[64] = {};
  cudaStream_t last[64] = {};
  bool pending[64] = {};
};
VtqGuard g_vtq;

struct VtqScope {
  cudaStream_t st = nullptr;
  int dev = -1;
  bool locked = false;
  // `st` must not be capturing (a graph that contains a sweep is bracketed by its launcher, prs_frame_launch)
  int begin(cudaStream_t s) {
    st = s;
    PRS_CUDA(cudaGetDevice(&dev));
    PRS_REQUIRE(dev >= 0 && dev < 64, "view-template sweep: device index %d out of range", dev);
    g_vtq.mu.lock();
    locked = true;
    if (!g_vtq.ev[dev]) PRS_CUDA(cudaEventCreateWithFlags(&g_vtq.ev[dev], cudaEventDisableTiming));
    if (g_vtq.pending[dev] && g_vtq.last[dev] != st) PRS_CUDA(cudaStreamWaitEvent(st, g_vtq.ev[dev], 0));
    return PRS_OK;
  }
  int end() {
    if (!locked) return PRS_OK;
    cudaError_t e = cudaEventRecord(g_vtq.ev[dev], st);
    if (e == cudaSuccess) {
      g_vtq.pending[dev] = true;
      g_vtq.last[dev] = st;
    }
    locked = false;
    g_vtq.mu.unlock();
    PRS_CUDA(e);
    return PRS_OK;
  }
  ~VtqScope() {
    if (locked) g_vtq.mu.unlock();
  }
};

__global__ void k_vt_pack_u8(const uint8_t* __restrict__ src, long long n, uint4* __restrict__ packed,
                             long long first) {
  // one thread per (template, row)
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n * 32) return;
  const long long tl = i >> 5;
  const int t = (int)(i & 31);
  vt_pack_row(src + tl * 1024, packed, first + tl, t);
}

__global__ void k_vt_unpack_u8(const uint4* __restrict__ packed, long long ti, uint8_t* __restrict__ dst) {
  // 1024 threads: one per pixel of template ti
  const int t = threadIdx.x >> 5, c = threadIdx.x & 31;
  const uint4* grp = packed + (ti >> 5) * kGroupU4;
  const int lane = (int)(ti & 31);
  const uint4 lo = grp[(t * 2 + 0) * 32 + lane], hi = grp[(t * 2 + 1) * 32 + lane];
  const uint32_t pl[8] = {lo.x, lo.y, lo.z, lo.w, hi.x, hi.y, hi.z, hi.w};
  uint32_t px = 0;
#pragma unroll
  for (int k = 0; k < 8; ++k) px |= ((pl[k] >> c) & 1u) << k;
  dst[t * 32 + c] = (uint8_t)px;
}

__global__ void k_vt_pack_query(const uint8_t* __restrict__ q, uint32_t* __restrict__ out,
                                unsigned long long* __restrict__ key_init = nullptr) {
  // 32 threads: thread t packs row t; then the two sums.  key_init: the sweep's packed key starts at "nothing found"
  // (one graph node less than a memset of its own on the sharded query chain)
  const int t = threadIdx.x;
  if (t == 0 && key_init != nullptr) *key_init = ~0ull;
  uint32_t pl[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  uint32_t sum = 0;
  for (int c = 0; c < 32; ++c) {
    const uint32_t px = q[t * 32 + c];
    sum += px;
#pragma unroll
    for (int k = 0; k < 8; ++k) pl[k] |= ((px >> k) & 1u) << c;
  }
#pragma unroll
  for (int k = 0; k < 8; ++k) out[t * 8 + k] = pl[k];
  uint32_t mid = (t >= 8 && t < 24) ? sum : 0;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    sum += __shfl_xor_sync(0xffffffffu, sum, o);
    mid += __shfl_xor_sync(0xffffffffu, mid, o);
  }
  if (t == 0) {
    out[256] = mid;
    out[257] = sum;
  }
}

__device__ __forceinline__ uint4 ld_stream_u4(const uint4* p) {
  uint4 v;
  asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0, %1, %2, %3}, [%4];"
               : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w)
               : "l"(p));
  return v;
}

// #{pixels of the stored row that are smaller than the query row's}: bit planes (lo, hi) of the stored
// row against query row s, whose planes are constant-bank operands.  LSB to MSB; the last differing bit wins.
// One borrow step of a < q on bit plane k, (~a & q) | (~(a ^ q) & lt), is ONE three-input LOP3 (truth table 0x8e for
// inputs a, q, lt).  Written as inline PTX: left to itself the compiler re-associates the first two steps of 90 of the
// 240 chains into three LOP3s (2 182 LOP3 per 32 templates instead of 1 942).
__device__ __forceinline__ uint32_t lt_step(uint32_t a, uint32_t q, uint32_t lt) {
  uint32_t r;
  asm("lop3.b32 %0, %1, %2, %3, 0x8e;" : "=r"(r) : "r"(a), "r"(q), "r"(lt));
  return r;
}
__device__ __forceinline__ uint32_t lt_row(const uint4& lo, const uint4& hi, int s) {
  const uint32_t* q = c_vtq + s * 8;
  uint32_t lt = lt_step(lo.x, q[0], 0u);
  lt = lt_step(lo.y, q[1], lt);
  lt = lt_step(lo.z, q[2], lt);
  lt = lt_step(lo.w, q[3], lt);
  lt = lt_step(hi.x, q[4], lt);
  lt = lt_step(hi.y, q[5], lt);
  lt = lt_step(hi.z, q[6], lt);
  lt = lt_step(hi.w, q[7], lt);
  return (uint32_t)__popc(lt);
}

// one stored row T against every query row it is paired with in reference mode (o = T - s in [-7, 7], s in [8, 23])
template <int T>
__device__ __forceinline__ void ref_row(const uint4& lo, const uint4& hi, uint32_t (&cnt)[15]) {
  constexpr int s_lo = (T - 7 > 8) ? T - 7 : 8;
  constexpr int s_hi = (T + 7 < 23) ? T + 7 : 23;
#pragma unroll
  for (int s = s_lo; s <= s_hi; ++s) cnt[T - s + 7] += lt_row(lo, hi, s);
}

constexpr int kPkThreads = 128;

// ---- reference mode (15 windowed row offsets, view_templates.py:16-28), fed by warp-private rings of TMA bulk copies
// A warp that prefetches one row in registers keeps 1 KB in flight: 20 warps x 1 KB x 148 SMs = 3 MB, less than half
// of what Little's law asks for at 6.5 TB/s x ~1 us.  Here every warp owns a ring of kRingSlots slots of 2 KB (two
// stored rows of its 32 templates) with one mbarrier each; one elected lane refills a slot with one cp.async.bulk as
// soon as the warp has consumed it, so 2 kRingSlots KB per warp are always in flight and the loads cost no registers
// and no LSU issue slots beyond two LDS.128 per row.  A group is 16 ring items: rows 1..30 in pairs (rows 0 and 31
// are never read in reference mode) and the row-sum block; 16 / kRingSlots fills per slot and group is even, so the
// mbarrier parity of an item is a compile-time constant.  Four slots and five CTAs per SM are the fastest of the
// depths and grid sizes measured (profiles/r1_vt_ring_tuning.txt).
constexpr int kRingSlots = 4;
constexpr int kRingCtasPerSm = 5;
__device__ __forceinline__ uint32_t vt_smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void vt_mbar_init(uint32_t bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void vt_mbar_wait(uint32_t bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "WAIT_%=:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@!p bra WAIT_%=;\n"
      "}\n" ::"r"(bar),
      "r"(parity)
      : "memory");
}
// one ring fill: expect BYTES, then the bulk copy global -> shared that completes them on the barrier.  The
// offset is an immediate of the instruction: handed over as a pointer, every item's address becomes its own
// loop-carried 64-bit induction variable (measured: 168 registers instead of 96).
template <int OFF, int BYTES>
__device__ __forceinline__ void vt_ring_fill(uint32_t dst, const void* base, uint32_t bar) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "n"(BYTES) : "memory");
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1+%2], %3, [%4];" ::"r"(dst),
               "l"(base), "n"(OFF), "n"(BYTES), "r"(bar)
               : "memory");
}
// one elected lane of a converged warp (the form ptxas keeps on the uniform datapath)
__device__ __forceinline__ bool vt_elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n"
      ".reg .pred P;\n"
      "elect.sync _|P, 0xffffffff;\n"
      "selp.u32 %0, 1, 0, P;\n"
      "}\n"
      : "=r"(pred));
  return pred != 0;
}
__device__ __forceinline__ uint4 lds_u4(uint32_t addr) {
  uint4 v;
  asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr));
  return v;
}

// A ring item is TWO stored rows (2 KB): rows 2j+1 and 2j+2 for j < 15, then the row-sum block (j = 15).
constexpr int kItemBytes = 2048;
constexpr int kItemsPerGroup = 16;
__host__ __device__ constexpr int pk_item_off(int j) { return (j < 15 ? 2 * j + 1 : 32) * 1024; }

template <int S>
struct RingPrologue {
  __device__ __forceinline__ static void run(uint32_t ring, uint32_t bars, const char* gb) {
    if constexpr (S < kRingSlots) {
      vt_ring_fill<pk_item_off(S), kItemBytes>(ring + S * kItemBytes, gb, bars + S * 8);
      RingPrologue<S + 1>::run(ring, bars, gb);
    }
  }
};

template <int J>
struct RingItems {
  // ring / bars: shared addresses of this warp's slots and barriers; gb / nb: this group and the warp's next one.
  // The warps of the CTA meet at a barrier after every item, so that all of them execute the same stretch of the
  // (48 KB, straight-line) code at the same time; `active` is false for a warp that has run out of groups.
  __device__ __forceinline__ static void run(uint32_t ring, uint32_t bars, const char* gb, const char* nb, int lane,
                                             bool active, uint32_t (&cnt)[15], uint4 (&rs)[4]) {
    if constexpr (J < kItemsPerGroup) {
      constexpr int slot = J % kRingSlots;
      if (active) {
        const uint32_t sl = ring + slot * kItemBytes + lane * 16;
        vt_mbar_wait(bars + slot * 8, (J / kRingSlots) & 1);
        const uint4 lo0 = lds_u4(sl), hi0 = lds_u4(sl + 512), lo1 = lds_u4(sl + 1024), hi1 = lds_u4(sl + 1536);
        if constexpr (J < 15) {
          ref_row<2 * J + 1>(lo0, hi0, cnt);
          ref_row<2 * J + 2>(lo1, hi1, cnt);
        } else {
          rs[0] = lo0, rs[1] = hi0, rs[2] = lo1, rs[3] = hi1;
        }
        // the slot's contents are in registers (the compares above consumed them): refill it with item J + kRingSlots
        __syncwarp();
        if (vt_elect_one()) {
          if constexpr (J + kRingSlots < kItemsPerGroup)
            vt_ring_fill<pk_item_off(J + kRingSlots), kItemBytes>(ring + slot * kItemBytes, gb, bars + slot * 8);
          else if (nb != nullptr)
            vt_ring_fill<pk_item_off((J + kRingSlots) % kItemsPerGroup), kItemBytes>(ring + slot * kItemBytes, nb,
                                                                                    bars + slot * 8);
        }
      }
      __syncthreads();
      RingItems<J + 1>::run(ring, bars, gb, nb, lane, active, cnt, rs);
    }
  }
};

__global__ void __launch_bounds__(kPkThreads, kRingCtasPerSm)  // 96 registers: the query planes stay constant-bank operands
    k_vt_sweep_packed_ref_ring(const uint4* __restrict__ packed, long long n, long long base_index,
                               unsigned long long* __restrict__ key_out, uint32_t* __restrict__ scores,
                               const int* __restrict__ n_dev) {
  static_assert(kItemsPerGroup % kRingSlots == 0 && (kItemsPerGroup / kRingSlots) % 2 == 0,
                "the parity of an item must not depend on the group");
  extern __shared__ __align__(128) unsigned char vt_ring_smem[];
  if (n_dev != nullptr) n = *n_dev;
  const int lane = threadIdx.x & 31;
  const int wid = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0);  // warp-uniform, and known to be
  const long long n_groups = (n + 31) >> 5;
  const long long warp0 = (long long)blockIdx.x * (kPkThreads / 32) + wid;
  const long long n_warps = (long long)gridDim.x * (kPkThreads / 32);
  const uint32_t ring = vt_smem_u32(vt_ring_smem) + wid * kRingSlots * kItemBytes;
  const uint32_t bars = vt_smem_u32(vt_ring_smem) + (kPkThreads / 32) * kRingSlots * kItemBytes + wid * kRingSlots * 8;
  constexpr long long kGroupBytes = (long long)kGroupU4 * 16;
  if (vt_elect_one()) {
#pragma unroll
    for (int s = 0; s < kRingSlots; ++s) vt_mbar_init(bars + s * 8, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    if (warp0 < n_groups) {
      const char* gb = reinterpret_cast<const char*>(packed) + warp0 * kGroupBytes;
      RingPrologue<0>::run(ring, bars, gb);
    }
  }
  __syncwarp();
  unsigned long long best = ~0ull;
  // every warp of the CTA makes as many rounds as its first warp (the one with the lowest group index)
  for (long long g = warp0; g - wid < n_groups; g += n_warps) {
    const bool active = g < n_groups;
    const char* gb = reinterpret_cast<const char*>(packed) + g * kGroupBytes;
    const char* nb = (g + n_warps < n_groups) ? gb + n_warps * kGroupBytes : nullptr;
    uint32_t cnt[15];
#pragma unroll
    for (int i = 0; i < 15; ++i) cnt[i] = 0;
    uint4 rs[4] = {};
    RingItems<0>::run(ring, bars, gb, nb, lane, active, cnt, rs);
    uint32_t R[32];
#pragma unroll
    for (int w4 = 0; w4 < 4; ++w4) {
      const uint32_t ww[4] = {rs[w4].x, rs[w4].y, rs[w4].z, rs[w4].w};
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        R[(w4 * 4 + j) * 2] = ww[j] & 0xffffu;
        R[(w4 * 4 + j) * 2 + 1] = ww[j] >> 16;
      }
    }
    uint32_t A = 0;
#pragma unroll
    for (int r = 1; r <= 16; ++r) A += R[r];
    const uint32_t bq = c_vtq[256];
    uint32_t m = 0xffffffffu;
#pragma unroll
    for (int o = -7; o <= 7; ++o) {
      const uint32_t sc = A + 256u * cnt[o + 7] - bq;
      m = min(m, sc);
      if (o < 7) A = A - R[8 + o] + R[24 + o];
    }
    const long long ti = g * 32 + lane;
    if (active && ti < n) {
      const unsigned long long key = ((unsigned long long)m << 32) | (unsigned long long)(base_index + ti);
      best = key < best ? key : best;
      if (scores != nullptr) scores[ti] = m;
    }
  }
  __shared__ unsigned long long sm[kPkThreads / 32];
  best = warp_min_u64(best);
  if (lane == 0) sm[wid] = best;
  __syncthreads();
  if (threadIdx.x == 0) {
    unsigned long long k = sm[0];
#pragma unroll
    for (int i = 1; i < kPkThreads / 32; ++i) k = sm[i] < k ? sm[i] : k;
    if (k != ~0ull) atomicMin(key_out, k);
  }
}

// ---- float32 library, reference mode: two columns per lane, fed by warp-private rings ------------------------
// One template per warp with lane == column (k_vt_sweep_f32) is bound by instruction issue: two instructions per
// element-difference.  Here a lane owns two adjacent columns, so that the subtraction is one packed add.f32x2 for
// two differences (3 instructions per two) and a template needs only half a warp: a warp works on templates
// 2i and 2i+1 at once.  Every warp owns a ring of kF32PairSlots slots, a slot holds both templates' rows 1..30 (two
// bulk copies on one barrier) and is refilled after it has been compared, while the other slots are in flight.
// Three slots and two CTAs per SM are the fastest of the depths and grid sizes measured
// (profiles/r1_vt_ring_tuning.txt).  The sums are formed in another order than in k_vt_sweep_f32: scores agree to
// rounding (exactly, for integer-valued profiles), not bit for bit.
constexpr int kF32ItemBytes = 30 * 32 * 4;  // rows 1..30 of one template
constexpr int kF32RingThreads = 128;
constexpr int kF32PairSlots = 3;
constexpr int kF32PairCtasPerSm = 2;
__global__ void __launch_bounds__(kF32RingThreads)
    k_vt_sweep_f32_pair(const float* __restrict__ lib, long long n, const float* __restrict__ query, long long base_index,
                        unsigned long long* __restrict__ key_out, float* __restrict__ scores) {
  using S = VtShape<PRS_VT_MODE_REF>;
  extern __shared__ __align__(128) unsigned char vt_ring_smem[];
  const int lane = threadIdx.x & 31, half = lane >> 4, l16 = lane & 15;
  const int wid = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0);
  const long long n_pairs = (n + 1) >> 1;
  const long long warp0 = (long long)blockIdx.x * (kF32RingThreads / 32) + wid;
  const long long n_warps = (long long)gridDim.x * (kF32RingThreads / 32);
  constexpr int kSlot = 2 * kF32ItemBytes;
  const uint32_t ring = vt_smem_u32(vt_ring_smem) + wid * kF32PairSlots * kSlot;
  const uint32_t bars =
      vt_smem_u32(vt_ring_smem) + (kF32RingThreads / 32) * kF32PairSlots * kSlot + wid * kF32PairSlots * 8;
  const char* base = reinterpret_cast<const char*>(lib) + 128;  // row 1 of template 0
  auto fill = [&](uint32_t slot_addr, long long pi, uint32_t bar) {  // one elected lane
    const char* src = base + pi * 8192;
    if (2 * pi + 1 < n) {
      asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "n"(kSlot) : "memory");
      asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                       slot_addr),
                   "l"(src), "n"(kF32ItemBytes), "r"(bar)
                   : "memory");
      asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1+4096], %2, [%3];" ::"r"(
                       slot_addr + kF32ItemBytes),
                   "l"(src), "n"(kF32ItemBytes), "r"(bar)
                   : "memory");
    } else {  // odd library size: the last pair has one template
      vt_ring_fill<0, kF32ItemBytes>(slot_addr, src, bar);
    }
  };
  if (vt_elect_one()) {
#pragma unroll
    for (int s = 0; s < kF32PairSlots; ++s) vt_mbar_init(bars + s * 8, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
#pragma unroll
    for (int s = 0; s < kF32PairSlots; ++s)
      if (warp0 + s * n_warps < n_pairs) fill(ring + s * kSlot, warp0 + s * n_warps, bars + s * 8);
  }
  __syncwarp();
  float2 nq[S::NS];  // minus the query's two columns of this lane
#pragma unroll
  for (int s = 0; s < S::NS; ++s) {
    const float2 v = *reinterpret_cast<const float2*>(query + (S::S0 + s) * 32 + 2 * l16);
    nq[s] = make_float2(-v.x, -v.y);
  }
  unsigned long long best = ~0ull;
  int slot = 0;
  uint32_t parity = 0;
  for (long long pi = warp0; pi < n_pairs; pi += n_warps) {
    const uint32_t sl = ring + slot * kSlot;
    vt_mbar_wait(bars + slot * 8, parity);
    const uint32_t mine = sl + half * kF32ItemBytes + l16 * 8;
    float acc[S::NACC];
#pragma unroll
    for (int i = 0; i < S::NACC; ++i) acc[i] = 0.f;
#pragma unroll
    for (int t = S::T0; t < S::T1; ++t) {
      float2 a;
      asm volatile("ld.shared.v2.f32 {%0, %1}, [%2];" : "=f"(a.x), "=f"(a.y) : "r"(mine + (t - S::T0) * 128));
#pragma unroll
      for (int s = 0; s < S::NS; ++s) {
        if (S::valid(t, S::S0 + s)) {
          const float2 d = __fadd2_rn(a, nq[s]);
          acc[S::off(t, S::S0 + s)] = (acc[S::off(t, S::S0 + s)] + fabsf(d.x)) + fabsf(d.y);
        }
      }
    }
    // every lane's loads have been consumed by the sums above: refill the slot with the pair kF32PairSlots rounds ahead
    __syncwarp();
    if (vt_elect_one()) {
      const long long np = pi + kF32PairSlots * n_warps;
      if (np < n_pairs) fill(sl, np, bars + slot * 8);
    }
    if (++slot == kF32PairSlots) {
      slot = 0;
      parity ^= 1u;
    }
    int obase = 0;
    Butterfly<S::NACC, 8, float>::run(acc, lane, obase);  // over the 16 lanes of the half-warp
    float m = (obase < S::NOFF) ? acc[0] : INFINITY;
#pragma unroll
    for (int o = 8; o > 0; o >>= 1) m = fminf(m, __shfl_xor_sync(0xffffffffu, m, o));
    const long long ti = 2 * pi + half;
    if (ti < n) {
      unsigned long long key = ((unsigned long long)__float_as_uint(m) << 32) | (unsigned long long)(base_index + ti);
      best = key < best ? key : best;
      if (scores != nullptr && l16 == 0) scores[ti] = m;
    }
  }
  __shared__ unsigned long long sm[kF32RingThreads / 32];
  best = warp_min_u64(best);
  if (lane == 0) sm[wid] = best;
  __syncthreads();
  if (threadIdx.x == 0) {
    unsigned long long k = sm[0];
#pragma unroll
    for (int i = 1; i < kF32RingThreads / 32; ++i) k = sm[i] < k ? sm[i] : k;
    if (k != ~0ull) atomicMin(key_out, k);
  }
}

// Circular mode (all 32 cyclic row shifts; extension).  The shift of a (stored row t, query row s) pair is
// (t - s) mod 32, which depends on the run-time row t -- but only through t mod 8 once the 32 counters are kept
// in registers and ROTATED by eight places after every eight stored rows: inside a block of eight rows the
// pair (i, s) always adds into register (i - s) mod 32, and the rotation re-labels the registers for the next
// block.  32 register MOVs per block replace 256 shared-memory read-modify-writes.
// eight stored rows (t0 .. t0+7, held in registers) against every query row; query row outermost so that only
// its eight plane words are live as (uniform-register) operands at a time.
// The warps of the CTA meet at a barrier after every four query rows (32 row pairs), so that they fetch the same
// stretch of the unrolled code together; `active` is false for a warp that has run out of groups.
constexpr int kCircSyncMask = 3;
__device__ __forceinline__ void circ_block(const uint4 (&lo)[8], const uint4 (&hi)[8], uint32_t (&cnt)[32], bool active) {
#pragma unroll
  for (int s = 0; s < 32; ++s) {
    if (active) {
#pragma unroll
      for (int i = 0; i < 8; ++i) cnt[(i - s) & 31] += lt_row(lo[i], hi[i], s);
    }
    if ((s & kCircSyncMask) == kCircSyncMask) __syncthreads();
  }
}

__global__ void __launch_bounds__(kPkThreads, 4)
    k_vt_sweep_packed_circ(const uint4* __restrict__ packed, long long n, long long base_index,
                           unsigned long long* __restrict__ key_out, uint32_t* __restrict__ scores,
                           const int* __restrict__ n_dev) {
  if (n_dev != nullptr) n = *n_dev;
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const long long n_groups = (n + 31) >> 5;
  const long long warp0 = ((long long)blockIdx.x * kPkThreads + threadIdx.x) >> 5;
  const long long n_warps = ((long long)gridDim.x * kPkThreads) >> 5;
  unsigned long long best = ~0ull;
  // every warp of the CTA makes as many rounds as its first warp; one without a group only keeps the barriers
  for (long long g = warp0; g - wid < n_groups; g += n_warps) {
    const bool active = g < n_groups;
    const uint4* gp = packed + (active ? g : 0) * kGroupU4 + lane;
    uint32_t cnt[32];
#pragma unroll
    for (int o = 0; o < 32; ++o) cnt[o] = 0;
#pragma unroll 1
    for (int c = 0; c < 4; ++c) {
      // during block c register r counts shift (r + 8c) mod 32
      uint4 lo[8], hi[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        lo[i] = ld_stream_u4(gp + ((8 * c + i) * 2 + 0) * 32);
        hi[i] = ld_stream_u4(gp + ((8 * c + i) * 2 + 1) * 32);
      }
      circ_block(lo, hi, cnt, active);
      uint32_t rot[32];
#pragma unroll
      for (int r = 0; r < 32; ++r) rot[r] = cnt[(r + 8) & 31];
#pragma unroll
      for (int r = 0; r < 32; ++r) cnt[r] = rot[r];
    }
    // four rotations by eight: register r counts shift r again
    uint32_t A = 0;
#pragma unroll
    for (int w4 = 0; w4 < 4; ++w4) {
      const uint4 v = ld_stream_u4(gp + 32 * 2 * 32 + w4 * 32);
      A += (v.x & 0xffffu) + (v.x >> 16) + (v.y & 0xffffu) + (v.y >> 16) + (v.z & 0xffffu) + (v.z >> 16) +
           (v.w & 0xffffu) + (v.w >> 16);
    }
    const uint32_t bq = c_vtq[257];
    uint32_t m = 0xffffffffu;
#pragma unroll
    for (int o = 0; o < 32; ++o) m = min(m, A + 256u * cnt[o] - bq);
    const long long ti = g * 32 + lane;
    if (active && ti < n) {
      const unsigned long long key = ((unsigned long long)m << 32) | (unsigned long long)(base_index + ti);
      best = key < best ? key : best;
      if (scores != nullptr) scores[ti] = m;
    }
  }
  __shared__ unsigned long long sm[kPkThreads / 32];
  best = warp_min_u64(best);
  if (lane == 0) sm[wid] = best;
  __syncthreads();
  if (threadIdx.x == 0) {
    unsigned long long k = sm[0];
#pragma unroll
    for (int i = 1; i < kPkThreads / 32; ++i) k = sm[i] < k ? sm[i] : k;
    if (k != ~0ull) atomicMin(key_out, k);
  }
}

extern "C" int prs_vt_sweep_f32(const float* lib, long long n, const float* query, int mode, long long base_index,
                                unsigned long long* key_out, float* scores, void* stream) {
  PRS_REQUIRE(query && key_out && n >= 0 && (lib || n == 0), "prs_vt_sweep_f32: bad argument");
  PRS_REQUIRE(mode == PRS_VT_MODE_REF || mode == PRS_VT_MODE_CIRCULAR, "prs_vt_sweep_f32: unknown mode %d", mode);
  PRS_REQUIRE(base_index >= 0 && base_index + n <= 0xffffffffLL, "prs_vt_sweep_f32: template index does not fit 32 bits");
  cudaStream_t st = (cudaStream_t)stream;
  PRS_CUDA(cudaMemsetAsync(key_out, 0xff, sizeof(unsigned long long), st));
  if (n == 0) return PRS_OK;
  if (mode == PRS_VT_MODE_REF) {
    constexpr int smem = (kF32RingThreads / 32) * kF32PairSlots * (2 * kF32ItemBytes + 8);  // 92 KB: above the default
    PRS_CUDA(cudaFuncSetAttribute(k_vt_sweep_f32_pair, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    const long long pairs = (n + 1) / 2;
    long long blocks = (pairs + (kF32RingThreads / 32) - 1) / (kF32RingThreads / 32);
    if (blocks > 148LL * kF32PairCtasPerSm) blocks = 148LL * kF32PairCtasPerSm;
    k_vt_sweep_f32_pair<<<(int)blocks, kF32RingThreads, smem, st>>>(lib, n, query, base_index, key_out, scores);
  } else {
    k_vt_sweep_f32<PRS_VT_MODE_CIRCULAR><<<sweep_grid(n), kVtThreads, 0, st>>>(lib, n, query, base_index, key_out, scores);
  }
  PRS_CUDA(cudaGetLastError());
  return PRS_OK;
}

// n: the library size the kernel uses when n_dev is NULL; n_grid: the size the grid is laid out for
static int launch_packed_sweep(const uint4* packed, long long n, long long n_grid, int mode, long long base_index,
                               unsigned long long* key_out, uint32_t* scores, const int* n_dev, cudaStream_t st) {
  const long long groups = (n_grid + 31) / 32;
  long long blocks = (groups + (kPkThreads / 32) - 1) / (kPkThreads / 32);
  if (blocks < 1) blocks = 1;
  if (mode == PRS_VT_MODE_REF) {
    constexpr int smem = (kPkThreads / 32) * kRingSlots * (kItemBytes + 8);
    static_assert(smem <= 48 * 1024, "the rings fit the default limit of dynamic shared memory");
    if (blocks > 148LL * kRingCtasPerSm) blocks = 148LL * kRingCtasPerSm;
    k_vt_sweep_packed_ref_ring<<<(int)blocks, kPkThreads, smem, st>>>(packed, n, base_index, key_out, scores, n_dev);
  } else {
    if (blocks > 148LL * 16) blocks = 148LL * 16;
    k_vt_sweep_packed_circ<<<(int)blocks, kPkThreads, 0, st>>>(packed, n, base_index, key_out, scores, n_dev);
  }
  PRS_CUDA(cudaGetLastError());
  return PRS_OK;
}

// VtqScope for callers outside this file (sharded.cu replays a graph that contains a packed sweep): the scope object
// lives from begin to end; one at a time per host thread is all the mutex allows anyway.
static thread_local VtqScope* t_ext_scope = nullptr;
int prs_vtq_begin(cudaStream_t st) {
  VtqScope* sc = new (std::nothrow) VtqScope();
  PRS_REQUIRE(sc, "out of host memory");
  int rc = sc->begin(st);
  if (rc != PRS_OK) {
    delete sc;
    return rc;
  }
  t_ext_scope = sc;
  return PRS_OK;
}
int prs_vtq_end(cudaStream_t) {
  VtqScope* sc = t_ext_scope;
  t_ext_scope = nullptr;
  if (!sc) return PRS_OK;
  int rc = sc->end();
  delete sc;
  return rc;
}

extern "C" size_t prs_vt_packed_bytes(long long n) {
  return (size_t)((n + 31) / 32) * kGroupU4 * sizeof(uint4);
}

extern "C" int prs_vt_pack_u8(const uint8_t* src, long long n, void* packed, long long first, void* stream) {
  PRS_REQUIRE(packed && n >= 0 && first >= 0 && (src || n == 0), "prs_vt_pack_u8: bad argument");
  if (n == 0) return PRS_OK;
  const long long threads = n * 32;
  k_vt_pack_u8<<<(unsigned)((threads + 255) / 256), 256, 0, (cudaStream_t)stream>>>(src, n, (uint4*)packed, first);
  PRS_CUDA(cudaGetLastError());
  return PRS_OK;
}

extern "C" int prs_vt_unpack_u8(const void* packed, long long index, uint8_t* dst, void* stream) {
  PRS_REQUIRE(packed && dst && index >= 0, "prs_vt_unpack_u8: bad argument");
  k_vt_unpack_u8<<<1, 1024, 0, (cudaStream_t)stream>>>((const uint4*)packed, index, dst);
  PRS_CUDA(cudaGetLastError());
  return PRS_OK;
}

extern "C" int prs_vt_sweep_packed_u8(const void* packed, long long n, const uint8_t* query, int mode,
                                      long long base_index, unsigned long long* key_out, uint32_t* scores,
                                      void* scratch, void* stream) {
  PRS_REQUIRE(query && key_out && scratch && n >= 0 && (packed || n == 0), "prs_vt_sweep_packed_u8: bad argument");
  PRS_REQUIRE(mode == PRS_VT_MODE_REF || mode == PRS_VT_MODE_CIRCULAR, "prs_vt_sweep_packed_u8: unknown mode %d", mode);
  PRS_REQUIRE(base_index >= 0 && base_index + n <= 0xffffffffLL,
              "prs_vt_sweep_packed_u8: template index does not fit 32 bits");
  cudaStream_t st = (cudaStream_t)stream;
  if (n == 0) {
    PRS_CUDA(cudaMemsetAsync(key_out, 0xff, sizeof(unsigned long long), st));
    return PRS_OK;
  }
  // query -> bit planes -> constant bank (stream ordered; sweeps on other streams of the device are ordered behind
  // each other through VtqScope)
  k_vt_pack_query<<<1, 32, 0, st>>>(query, (uint32_t*)scratch, key_out);
  cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
  if (st != nullptr) PRS_CUDA(cudaStreamIsCapturing(st, &cap));
  VtqScope scope;
  if (cap == cudaStreamCaptureStatusNone)  // a caller capturing its own graph orders its launches itself
    if (int rc = scope.begin(st)) return rc;
  PRS_CUDA(cudaMemcpyToSymbolAsync(c_vtq, scratch, (32 * 8 + 2) * sizeof(uint32_t), 0, cudaMemcpyDeviceToDevice, st));
  int rc = launch_packed_sweep((const uint4*)packed, n, n, mode, base_index, key_out, scores, nullptr, st);
  if (int rc2 = scope.end()) return rc != PRS_OK ? rc : rc2;
  return rc;
}

// The two halves of prs_vt_sweep_packed_u8 for a caller that replays the second one as a graph (sharded.cu): the query's
// bit planes (and the reset of the key) on the caller's stream, then constant upload + sweep from those planes.
int prs_vt_pack_query_launch(const uint8_t* query, void* scratch, unsigned long long* key, cudaStream_t st) {
  k_vt_pack_query<<<1, 32, 0, st>>>(query, (uint32_t*)scratch, key);
  PRS_CUDA(cudaGetLastError());
  return PRS_OK;
}
int prs_vt_sweep_packed_planes(const void* packed, long long n, const void* planes, int mode, long long base_index,
                               unsigned long long* key_out, cudaStream_t st) {
  if (n == 0) return PRS_OK;
  cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
  if (st != nullptr) PRS_CUDA(cudaStreamIsCapturing(st, &cap));
  VtqScope scope;
  if (cap == cudaStreamCaptureStatusNone)
    if (int rc = scope.begin(st)) return rc;
  PRS_CUDA(cudaMemcpyToSymbolAsync(c_vtq, planes, (32 * 8 + 2) * sizeof(uint32_t), 0, cudaMemcpyDeviceToDevice, st));
  int rc = launch_packed_sweep((const uint4*)packed, n, n, mode, base_index, key_out, nullptr, nullptr, st);
  if (int rc2 = scope.end()) return rc != PRS_OK ? rc : rc2;
  return rc;
}

// =============================================================================================
// One whole frame of the ROS loop (ratslam/ros_simulate.py:98-105,134-137) with a single host
// synchronisation: odometry H2D -> pose-cell update -> frame H2D -> sub-sample -> library sweep ->
// create-or-match decided ON THE DEVICE (view_templates.py:67-73; a created template is packed straight
// into slot n of the library) -> 32-byte result D2H.
struct FrameScratch {               // device scratch layout (bytes)
  static constexpr size_t kFrame = 0;                   // uint8 frame, up to 1 MiB
  static constexpr size_t kTpl = 1 << 20;               // uint8[1024] sub-sampled template
  static constexpr size_t kPlanes = kTpl + 1024;        // uint32[264] query planes
  static constexpr size_t kKey = kPlanes + 2048;        // uint64 key
  static constexpr size_t kResult = kKey + 64;          // prs_frame_result
  static constexpr size_t kOdom = kResult + 64;         // double[2]
  static constexpr size_t kBytes = kOdom + 64;
};

// Per-agent layout of the ensemble frame (prs_ens_*): B agents share the query, each has its own library, template
// count, threshold, location table and pose-cell network.  The default is the single-agent frame (B = 1, no strides).
struct VtAgents {
  int B = 1;
  long long lib_u4 = 0;                 // uint4 per agent library
  const double* threshold = nullptr;    // [B]; null: the kernel's scalar threshold
  long long* loc = nullptr;             // [B][loc_stride]: a created template's row receives the agent's arg-max
  long long loc_stride = 0;
  int* g_max = nullptr;                 // largest group count over the agents, raised by the decision (the sweep's grid)
  const int* ctr = nullptr;             // frame index within the record chunk: the agent's record is res[*ctr * B + b]
  // ensemble ticks: agent b replays recording rec_of[b], whose template is tpl + rec_of[b] * 1024; present[r] = 0 where
  // recording r has no image at this tick, and there its agents append and inject nothing
  const int* rec_of = nullptr;          // [B]; null: one template
  const uint8_t* present = nullptr;     // [R]
};

// One warp per agent (b = global warp index), lane t packs row t of a created template.
// dec (optional): a second, device-side copy of the decision (created, template_index, n_templates) for the frame's
// injection node when `res` is the pinned host record
__global__ void k_vt_decide_append(const unsigned long long* __restrict__ key, const uint8_t* __restrict__ tpl,
                                   uint4* __restrict__ packed, int n, double threshold,
                                   const long long* __restrict__ argmax, const int* __restrict__ pc_err,
                                   prs_frame_result* __restrict__ res, int* __restrict__ n_dev, int write_pc = 1,
                                   prs_frame_result* __restrict__ dec = nullptr, VtAgents ag = VtAgents()) {
  const int b = (int)((blockIdx.x * blockDim.x + threadIdx.x) >> 5), t = threadIdx.x & 31;
  if (b >= ag.B) return;  // whole warps
  if (n_dev != nullptr) n = n_dev[b];
  __syncwarp();
  if (ag.rec_of != nullptr) {
    const int r = ag.rec_of[b];
    if (!ag.present[r]) {  // the recording has ended: a "no frame" record, the library stays as it is
      if (t == 0) {
        res += (long long)*ag.ctr * ag.B + b;
        res->argmax = argmax[b];
        res->key = ~0ull;
        res->created = 0;
        res->template_index = -1;
        res->n_templates = n;
        res->pc_err = pc_err[b];
      }
      return;
    }
    tpl += (size_t)r * 1024;
  }
  const unsigned long long k = key[b];
  const unsigned score = (unsigned)(k >> 32);
  if (ag.threshold != nullptr) threshold = ag.threshold[b];
  // strict '>' (view_templates.py:67) on the caller's number: a score is an integer <= 130560, exact in a double, so a
  // negative threshold creates on every frame and a fractional or huge one means what it means to the reference
  const bool create = (n == 0) || (k == ~0ull) || ((double)score > threshold);
  if (create) {
    vt_pack_row(tpl, packed + b * ag.lib_u4, n, t);
  }
  if (t == 0) {
    res += (ag.ctr != nullptr ? (long long)*ag.ctr * ag.B : 0) + b;
    if (write_pc) res->argmax = argmax ? argmax[b] : -1;  // else the pose-cell kernel writes both fields itself
    res->key = k;
    res->created = create ? 1 : 0;
    res->template_index = create ? n : (int)(k & 0xffffffffu);
    res->n_templates = n + (create ? 1 : 0);
    if (write_pc) res->pc_err = pc_err ? pc_err[b] : 0;
    if (n_dev != nullptr) n_dev[b] = n + (create ? 1 : 0);
    if (create && ag.loc != nullptr) ag.loc[b * ag.loc_stride + n] = argmax[b];
    if (create && ag.g_max != nullptr) atomicMax(ag.g_max, (n + 32) >> 5);  // groups of n + 1 templates
    if (dec != nullptr) {
      dec->created = create ? 1 : 0;
      dec->template_index = create ? n : (int)(k & 0xffffffffu);
      dec->n_templates = n + (create ? 1 : 0);
    }
  }
}

// View-template -> pose-cell injection at the tail of a frame (ros_simulate.py:106-108): posecells[location(template)]
// += energy, where a created template's location is the arg-max its match was made with and a matched template's is
// whatever its row of the location table holds (C-order flat index x*Y*Th + y*Th + th, -1 = not a valid cell).  One
// thread does it all: one table row, one cell, one comparison.  The cached arg-max is kept current in O(1): no other
// cell changed, so with energy >= 0 the first maximum (numpy.argmax) is either the old one or the injected cell.
//   dec    : this frame's decision, device memory (never the pinned record: no read over the bus)
//   argmax : the cached arg-max of pc_work, the one the match was made with; updated in place
//   res    : the frame's record, receives PRS_ERR_INJECT_LOC (on top of pc_err, the pose-cell bits it already holds)
// The node sits on the frame's critical path and is a chain of dependent loads: the arg-max cell is read alongside the
// table row, a created template needs no row read at all, and the index arithmetic is 32-bit where the grid allows.
template <typename I>
__device__ __forceinline__ size_t pc_theta_major(I f, I X, I Y, I Th) {  // [x][y][th] flat index -> [th][x][y] offset
  const I xy = f / Th, th = f - xy * Th, x = xy / Y, y = xy - x * Y;
  return ((size_t)th * X + x) * Y + y;
}

// Ensemble frames (energies != null): one thread per agent b with its own network, table row stride, record and
// energies[b]; an energy that is not >= 0 (the ensemble's "no injection") leaves agent b alone.
template <typename T>
__global__ void k_frame_inject(T* __restrict__ state, long long* __restrict__ loc, const prs_frame_result* dec,
                               long long* __restrict__ argmax, const int* __restrict__ pc_err, prs_frame_result* res,
                               int X, int Y, int Th, T energy, const double* __restrict__ energies = nullptr,
                               VtAgents ag = VtAgents()) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= ag.B) return;
  const long long N = (long long)X * Y * Th;
  if (energies != nullptr) {
    const double e = energies[b];
    if (!(e >= 0.0)) return;
    if (ag.rec_of != nullptr && !ag.present[ag.rec_of[b]]) return;  // no frame, nothing to inject
    energy = (T)e;
    const long long r = (ag.ctr != nullptr ? (long long)*ag.ctr * ag.B : 0) + b;
    dec += r;
    res += r;
    state += b * N;
    loc += b * ag.loc_stride;
    argmax += b;
    pc_err += b;
  }
  const bool narrow = N <= 0xffffffffLL;
  auto offset = [&](long long f) {
    return narrow ? pc_theta_major<unsigned>((unsigned)f, X, Y, Th) : pc_theta_major<long long>(f, X, Y, Th);
  };
  const long long a = *argmax;
  const int ti = dec->template_index;
  const bool created = dec->created != 0;
  const bool a_ok = a >= 0 && a < N;
  const size_t oa = a_ok ? offset(a) : 0;
  const T m = state[oa];  // the arg-max's value; no other cell than the injected one changes
  long long c = a;
  if (created)
    loc[ti] = a;
  else
    c = loc[ti];
  if (c < 0 || c >= N) {  // the posecells of the frame stay as they are
    res->pc_err = pc_err[0] | PRS_ERR_INJECT_LOC;
    return;
  }
  const size_t oc = c == a ? oa : offset(c);
  const T v = (c == a ? m : state[oc]) + energy;  // k_inject's arithmetic
  state[oc] = v;
  if (c != a && (!a_ok || v > m || (v == m && c < a))) *argmax = c;
}

extern "C" size_t prs_frame_scratch_bytes(void) { return FrameScratch::kBytes; }

extern "C" int prs_frame_host(prs_pc_handle pc, void* pc_state, const void* gi, void* pc_work, const double* odom_host,
                              void* vt_packed, int n_templates, double threshold, int mode,
                              const uint8_t* frame_host, int im_rows, int im_cols, int row_lo, int row_hi, int row_step,
                              int col_lo, int col_hi, int col_step, void* scratch, prs_frame_result* result_host,
                              void* stream) {
  PRS_REQUIRE(pc && pc_state && gi && pc_work && vt_packed && frame_host && scratch && result_host,
              "prs_frame_host: null argument");
  PRS_REQUIRE((size_t)im_rows * im_cols <= (1u << 20), "prs_frame_host: frame larger than 1 MiB");
  cudaStream_t st = (cudaStream_t)stream;
  char* sc = (char*)scratch;
  uint8_t* d_frame = (uint8_t*)(sc + FrameScratch::kFrame);
  uint8_t* d_tpl = (uint8_t*)(sc + FrameScratch::kTpl);
  uint32_t* d_planes = (uint32_t*)(sc + FrameScratch::kPlanes);
  unsigned long long* d_key = (unsigned long long*)(sc + FrameScratch::kKey);
  prs_frame_result* d_res = (prs_frame_result*)(sc + FrameScratch::kResult);
  double* d_odom = (double*)(sc + FrameScratch::kOdom);
  // pc_work: device int64 argmax[1], float/double total[1] (8 bytes), int err[1]
  long long* d_argmax = (long long*)pc_work;
  void* d_total = (char*)pc_work + 8;
  int* d_err = (int*)((char*)pc_work + 16);
  int rc;
  if (odom_host) {  // ros_simulate.py:134-137: one pose-cell update with this twist
    PRS_CUDA(cudaMemcpyAsync(d_odom, odom_host, 2 * sizeof(double), cudaMemcpyHostToDevice, st));
    rc = prs_pc_step(pc, pc_state, d_odom, gi, d_argmax, d_total, d_err, st);
    if (rc != PRS_OK) return rc;
  }
  PRS_CUDA(cudaMemcpyAsync(d_frame, frame_host, (size_t)im_rows * im_cols, cudaMemcpyHostToDevice, st));
  rc = prs_vt_extract_u8(d_frame, im_rows, im_cols, row_lo, row_hi, row_step, col_lo, col_hi, col_step, d_tpl, 32, 32, st);
  if (rc != PRS_OK) return rc;
  rc = prs_vt_sweep_packed_u8(vt_packed, n_templates, d_tpl, mode, 0, d_key, nullptr, d_planes, st);
  if (rc != PRS_OK) return rc;
  k_vt_decide_append<<<1, 32, 0, st>>>(d_key, d_tpl, (uint4*)vt_packed, n_templates, threshold, d_argmax, d_err, d_res,
                                       nullptr);
  PRS_CUDA(cudaGetLastError());
  PRS_CUDA(cudaMemcpyAsync(result_host, d_res, sizeof(prs_frame_result), cudaMemcpyDeviceToHost, st));
  PRS_CUDA(cudaStreamSynchronize(st));
  return PRS_OK;
}

// =============================================================================================
// Any template shape (rows x cols) and any max_offset: one warp per template, lanes stride over the
// window's pixels.  Used when ViewTemplates is configured away from the reference's 32x32 / offset 8
// (view_templates.py:14,44); correctness path, not tuned.
template <typename T, typename ACC>
__global__ void __launch_bounds__(256)
    k_vt_sweep_any(const T* __restrict__ lib, long long n, const T* __restrict__ query, int rows, int cols, int max_offset,
                   long long base_index, unsigned long long* __restrict__ key_out, ACC* __restrict__ scores) {
  const int lane = threadIdx.x & 31;
  const long long warp0 = ((long long)blockIdx.x * 256 + threadIdx.x) >> 5;
  const long long n_warps = ((long long)gridDim.x * 256) >> 5;
  const int win = rows - 2 * max_offset;  // rows compared per offset
  unsigned long long best = ~0ull;
  for (long long ti = warp0; ti < n; ti += n_warps) {
    const T* tp = lib + ti * rows * cols;
    ACC m = 0;
    bool first = true;
    for (int o = -max_offset + 1; o < max_offset; ++o) {
      ACC s = 0;
      for (int i = lane; i < win * cols; i += 32) {
        const int r = i / cols, c = i - r * cols;
        const T a = tp[(max_offset + o + r) * cols + c], b = query[(max_offset + r) * cols + c];
        if constexpr (sizeof(T) == 1)
          s += (ACC)(uint8_t)(a - b);  // uint8 arithmetic wraps; abs() is the identity (view_templates.py:23)
        else
          s += fabsf(a - b);
      }
#pragma unroll
      for (int d = 16; d > 0; d >>= 1) s += __shfl_xor_sync(0xffffffffu, s, d);
      if (first || s < m) m = s;
      first = false;
    }
    unsigned hi;
    if constexpr (sizeof(T) == 1)
      hi = (unsigned)m;
    else
      hi = __float_as_uint(m);
    const unsigned long long key = ((unsigned long long)hi << 32) | (unsigned long long)(base_index + ti);
    best = key < best ? key : best;
    if (scores != nullptr && lane == 0) scores[ti] = m;
  }
  block_min_to_global(best, key_out);
}

template <typename T, typename ACC>
static int sweep_any(const T* lib, long long n, const T* query, int rows, int cols, int max_offset, long long base_index,
                     unsigned long long* key_out, ACC* scores, cudaStream_t st) {
  PRS_REQUIRE(query && key_out && n >= 0 && (lib || n == 0), "prs_vt_sweep_any: bad argument");
  PRS_REQUIRE(rows > 0 && cols > 0 && max_offset >= 1 && rows - 2 * max_offset >= 0,
              "prs_vt_sweep_any: %dx%d templates cannot be compared with max_offset %d", rows, cols, max_offset);
  PRS_REQUIRE(base_index >= 0 && base_index + n <= 0xffffffffLL, "prs_vt_sweep_any: template index does not fit 32 bits");
  PRS_CUDA(cudaMemsetAsync(key_out, 0xff, sizeof(unsigned long long), st));
  if (n == 0) return PRS_OK;
  k_vt_sweep_any<T, ACC><<<sweep_grid(n), 256, 0, st>>>(lib, n, query, rows, cols, max_offset, base_index, key_out, scores);
  PRS_CUDA(cudaGetLastError());
  return PRS_OK;
}

extern "C" int prs_vt_sweep_any_u8(const uint8_t* lib, long long n, const uint8_t* query, int rows, int cols,
                                   int max_offset, long long base_index, unsigned long long* key_out, uint32_t* scores,
                                   void* stream) {
  return sweep_any<uint8_t, uint32_t>(lib, n, query, rows, cols, max_offset, base_index, key_out, scores, (cudaStream_t)stream);
}

extern "C" int prs_vt_sweep_any_f32(const float* lib, long long n, const float* query, int rows, int cols, int max_offset,
                                    long long base_index, unsigned long long* key_out, float* scores, void* stream) {
  return sweep_any<float, float>(lib, n, query, rows, cols, max_offset, base_index, key_out, scores, (cudaStream_t)stream);
}


// ---------------------------------------------------------------------------------------------
// Short frame chain for replayed frames over small libraries.  With the plan's host buffers pinned (and therefore
// mapped into the device's address space) the template branch of a frame is three kernels and no copy node:
//   k_vt_frame_prepare   reads the 32x32 masked pixels straight from the pinned frame (about 2 KB cross the bus
//                        instead of the whole 64 KB frame), builds the template, its bit planes and row sums,
//                        resets the key
//   k_vt_sweep_packed_ref_small   the bit-sliced sweep with the query planes in shared memory instead of the
//                        constant bank (no cudaMemcpyToSymbol node) and one block per group of 32 templates;
//                        only used below kSmallLibrary templates
//   k_vt_decide_append   writes its 32-byte result straight into the pinned result buffer
// and the pose-cell kernel reads its two doubles of odometry from the pinned buffer as well.
constexpr int kSmallLibrary = 1 << 16;

// The query of `frame`: the template, its bit planes and row sums.  A block of 1024 threads, one per template pixel.
__device__ __forceinline__ void vt_prepare_query(const uint8_t* __restrict__ frame, int im_cols, int row_lo, int row_step,
                                                 int col_lo, int col_step, uint8_t* __restrict__ tpl,
                                                 uint32_t* __restrict__ planes, uint32_t* s_sum) {
  const int t = threadIdx.x >> 5, c = threadIdx.x & 31;  // template row, column
  const int rr = row_lo + (t / (row_step - 1)) * row_step + (t % (row_step - 1)) + 1;
  const int cc = col_lo + (c / (col_step - 1)) * col_step + (c % (col_step - 1)) + 1;
  const uint32_t px = frame[(size_t)rr * im_cols + cc];
  tpl[t * 32 + c] = (uint8_t)px;
  uint32_t mine = 0;
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    const uint32_t b = __ballot_sync(0xffffffffu, (px >> k) & 1u);
    if (c == k) mine = b;
  }
  if (c < 8) planes[t * 8 + c] = mine;
  uint32_t sum = px;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
  if (c == 0) s_sum[t] = sum;
  __syncthreads();
  if (t == 0) {
    uint32_t all = s_sum[c], mid = (c >= 8 && c < 24) ? all : 0;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      all += __shfl_xor_sync(0xffffffffu, all, o);
      mid += __shfl_xor_sync(0xffffffffu, mid, o);
    }
    if (c == 0) {
      planes[256] = mid;
      planes[257] = all;
    }
  }
}

__global__ void __launch_bounds__(1024)
    k_vt_frame_prepare(const uint8_t* __restrict__ frame, int im_cols, int row_lo, int row_step, int col_lo, int col_step,
                       uint8_t* __restrict__ tpl, uint32_t* __restrict__ planes, unsigned long long* __restrict__ key) {
  __shared__ uint32_t s_sum[32];
  if (threadIdx.x == 0) *key = ~0ull;
  vt_prepare_query(frame, im_cols, row_lo, row_step, col_lo, col_step, tpl, planes, s_sum);
}

// Ensemble ticks: block r prepares recording r's query into tpl + r * 1024 and planes + r * kQueryStride.  A recording's
// images sit contiguously in its chunk, frames[r][chunk] (bytes (r * chunk + s) * frame_bytes), but not at the tick
// index: its image at tick *ctr is slot s = slots[*ctr][r] of the chunk, and s = -1 (no image at this tick, or past
// the recording's end) clears present[r].  The blocks reset the n_keys agents' keys.
constexpr int kQueryStride = 512;  // uint32 words between two recordings' query planes (258 used)

__global__ void __launch_bounds__(1024)
    k_vt_frame_prepare_multi(const uint8_t* __restrict__ frames, int chunk, long long frame_bytes, int im_cols, int row_lo,
                             int row_step, int col_lo, int col_step, uint8_t* __restrict__ tpl,
                             uint32_t* __restrict__ planes, unsigned long long* __restrict__ key, int n_keys,
                             const int* __restrict__ ctr, uint8_t* __restrict__ present, const int* __restrict__ slots) {
  __shared__ uint32_t s_sum[32];
  const int r = blockIdx.x, R = gridDim.x, f = *ctr;
  for (int i = r * 1024 + (int)threadIdx.x; i < n_keys; i += R * 1024) key[i] = ~0ull;
  const int s = slots[(size_t)f * R + r];
  const bool here = s >= 0;
  if (threadIdx.x == 0) present[r] = here ? 1 : 0;
  if (!here) return;  // block-uniform
  vt_prepare_query(frames + ((size_t)r * chunk + s) * frame_bytes, im_cols, row_lo, row_step, col_lo, col_step,
                   tpl + (size_t)r * 1024, planes + (size_t)r * kQueryStride, s_sum);
}

__device__ __forceinline__ uint32_t lt_row_q(const uint4& lo, const uint4& hi, const uint32_t* q) {
  uint32_t lt = ~lo.x & q[0];
  lt = (~lo.y & q[1]) | (~(lo.y ^ q[1]) & lt);
  lt = (~lo.z & q[2]) | (~(lo.z ^ q[2]) & lt);
  lt = (~lo.w & q[3]) | (~(lo.w ^ q[3]) & lt);
  lt = (~hi.x & q[4]) | (~(hi.x ^ q[4]) & lt);
  lt = (~hi.y & q[5]) | (~(hi.y ^ q[5]) & lt);
  lt = (~hi.z & q[6]) | (~(hi.z ^ q[6]) & lt);
  lt = (~hi.w & q[7]) | (~(hi.w ^ q[7]) & lt);
  return (uint32_t)__popc(lt);
}

// Small libraries are latency-bound, not bandwidth-bound: with one warp per group of 32 templates the 30 stored
// rows are 30 dependent load rounds (measured: 25 us for a 30-template library).  Here a block of 16 warps shares
// one group: warp w < 15 compares rows 2w+1 and 2w+2 (one load round, 480 compares), warp 15 forms the window sums,
// and the per-offset counts meet in shared memory (integer adds: exact, order-free).
constexpr int kSmallThreads = 512;

// <false>: the single-agent frame's sweep of one library against one query.
// <true> (ensemble ticks): n_agents libraries of lib_u4 uint4 each, agent b's live count n_dev[b] and key key_out[b].
// The blocks grid-stride over (agent, group) items, G = *g_max groups per agent (the largest live group count, kept by
// the decision kernel); an item past its agent's live count is skipped, so the work follows sum_b n_b, not the
// capacity.  Agent b is compared with the query of its recording rec_of[b], qplanes + rec_of[b] * kQueryStride, and
// skipped where present[rec_of[b]] = 0.  A block reloads q only when its item's recording differs from the last one it
// loaded (the agents of a recording have contiguous indices).
template <bool kMulti>
__global__ void __launch_bounds__(kSmallThreads)
    k_vt_sweep_packed_ref_small(const uint4* __restrict__ packed, const uint32_t* __restrict__ qplanes,
                                unsigned long long* __restrict__ key_out, const int* __restrict__ n_dev,
                                int n_agents = 1, long long lib_u4 = 0, const int* __restrict__ g_max = nullptr,
                                const int* __restrict__ rec_of = nullptr, const uint8_t* __restrict__ present = nullptr) {
  __shared__ uint32_t q[32 * 8 + 8];
  __shared__ uint32_t s_cnt[15][32];
  __shared__ uint32_t s_A[15][32];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const long long G = g_max != nullptr ? (long long)*g_max : ((long long)*n_dev + 31) >> 5;
  const long long items = G * n_agents;
  if ((long long)blockIdx.x >= items) return;  // the grid is laid out for the capacity, not the live count
  if (!kMulti)
    for (int i = threadIdx.x; i < 32 * 8 + 2; i += kSmallThreads) q[i] = qplanes[i];
  [[maybe_unused]] int q_rec = -1;
  for (long long item = blockIdx.x; item < items; item += gridDim.x) {
    const int b = (int)(item / G);
    const long long g = item - b * G;
    const long long n = n_dev[b];
    if (g * 32 >= n) continue;  // block-uniform
    if (kMulti) {
      const int r = rec_of[b];
      if (!present[r]) continue;  // block-uniform: the recording has ended
      if (r != q_rec) {           // block-uniform; the last item's final barrier retired every reader of q
        for (int i = threadIdx.x; i < 32 * 8 + 2; i += kSmallThreads) q[i] = qplanes[(size_t)r * kQueryStride + i];
        q_rec = r;
      }
    }
    if (threadIdx.x < 15 * 32) s_cnt[wid][lane] = 0;
    __syncthreads();  // also publishes q on the first pass
    const uint4* gp = packed + b * lib_u4 + g * kGroupU4 + lane;
    if (wid < 15) {
      const int t0 = 2 * wid + 1;
      const uint4 lo0 = ld_stream_u4(gp + (t0 * 2 + 0) * 32), hi0 = ld_stream_u4(gp + (t0 * 2 + 1) * 32);
      const uint4 lo1 = ld_stream_u4(gp + (t0 * 2 + 2) * 32), hi1 = ld_stream_u4(gp + (t0 * 2 + 3) * 32);
#pragma unroll
      for (int o = -7; o <= 7; ++o) {
        uint32_t c = 0;
        const int s0 = t0 - o, s1 = t0 + 1 - o;  // warp-uniform
        if (s0 >= 8 && s0 <= 23) c += lt_row_q(lo0, hi0, q + s0 * 8);
        if (s1 >= 8 && s1 <= 23) c += lt_row_q(lo1, hi1, q + s1 * 8);
        if (c) atomicAdd(&s_cnt[o + 7][lane], c);
      }
    } else {
      uint32_t R[32];
#pragma unroll
      for (int w4 = 0; w4 < 4; ++w4) {
        const uint4 v = ld_stream_u4(gp + 32 * 2 * 32 + w4 * 32);
        const uint32_t ww[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          R[(w4 * 4 + j) * 2] = ww[j] & 0xffffu;
          R[(w4 * 4 + j) * 2 + 1] = ww[j] >> 16;
        }
      }
      uint32_t A = 0;
#pragma unroll
      for (int r = 1; r <= 16; ++r) A += R[r];
#pragma unroll
      for (int o = -7; o <= 7; ++o) {
        s_A[o + 7][lane] = A;
        if (o < 7) A = A - R[8 + o] + R[24 + o];
      }
    }
    __syncthreads();
    if (wid == 0) {
      const uint32_t bq = q[256];
      uint32_t m = 0xffffffffu;
#pragma unroll
      for (int o = 0; o < 15; ++o) m = min(m, s_A[o][lane] + 256u * s_cnt[o][lane] - bq);
      const long long ti = g * 32 + lane;
      unsigned long long best = ti < n ? ((unsigned long long)m << 32) | (unsigned long long)ti : ~0ull;
      best = warp_min_u64(best);
      if (lane == 0) atomicMin(key_out + b, best);
    }
    __syncthreads();
  }
}

// ---------------------------------------------------------------------------------------------
// The same frame as a CUDA graph: every pointer is fixed at creation (pinned host buffers included), the
// library size lives in device memory, so a frame is ONE graph launch + one synchronisation instead of
// eleven stream operations.  Two executables: with and without the pose-cell update (ros_simulate.py:128
// drops near-zero twists).
struct prs_frame_plan {
  prs_pc_handle pc;
  void *pc_state, *pc_work, *vt_packed, *scratch;
  const void* gi;
  double* odom_host;
  uint8_t* frame_host;
  prs_frame_result* result_host;
  double threshold;
  int mode, capacity;
  int im_rows, im_cols, row_lo, row_hi, row_step, col_lo, col_hi, col_step;
  cudaGraphExec_t exec[2];
  bool ready[2];
  int* d_n;
  int warm[2];
  cudaStream_t side;       // the pose-cell update runs here, concurrently with the template branch
  cudaEvent_t ev_fork, ev_join;
  cudaEvent_t ev_done;     // recorded behind every frame launched by prs_replay_run
  // device-side aliases of the pinned host buffers (zero-copy), null when a buffer is not pinned
  const double* odom_map;
  const uint8_t* frame_map;
  prs_frame_result* result_map;
  // prs_frame_set_inject: the location table (null = no injection) and the energy of the frame's last node
  long long* inj_loc;
  double inj_energy;
};

static int frame_enqueue(prs_frame_plan* f, bool moved, cudaStream_t st) {
  char* sc = (char*)f->scratch;
  uint8_t* d_frame = (uint8_t*)(sc + FrameScratch::kFrame);
  uint8_t* d_tpl = (uint8_t*)(sc + FrameScratch::kTpl);
  uint32_t* d_planes = (uint32_t*)(sc + FrameScratch::kPlanes);
  unsigned long long* d_key = (unsigned long long*)(sc + FrameScratch::kKey);
  prs_frame_result* d_res = (prs_frame_result*)(sc + FrameScratch::kResult);
  double* d_odom = (double*)(sc + FrameScratch::kOdom);
  long long* d_argmax = (long long*)f->pc_work;
  void* d_total = (char*)f->pc_work + 8;
  int* d_err = (int*)((char*)f->pc_work + 16);
  const bool zero_copy = f->odom_map && f->frame_map && f->result_map;
  // the short chain (see k_vt_frame_prepare): reference mode, 32x32 templates out of a step >= 2 mask, small library
  const bool short_chain = zero_copy && f->mode == PRS_VT_MODE_REF && f->capacity <= kSmallLibrary;
  int rc;
  int pc_mirrored = 0;
  if (moved) {  // fork: the pose-cell update does not depend on the frame until the decision
    PRS_CUDA(cudaEventRecord(f->ev_fork, st));
    PRS_CUDA(cudaStreamWaitEvent(f->side, f->ev_fork, 0));
    const double* od = f->odom_map;
    if (!zero_copy) {
      PRS_CUDA(cudaMemcpyAsync(d_odom, f->odom_host, 2 * sizeof(double), cudaMemcpyHostToDevice, f->side));
      od = d_odom;
    }
    // with mapped buffers the cluster kernel writes the arg-max and the error bits into the host record itself:
    // nothing on the template branch waits for the pose-cell update then
    if (zero_copy)
      rc = prs_pc_step_mirror(f->pc, f->pc_state, od, f->gi, d_argmax, d_total, d_err, &f->result_map->argmax,
                              &f->result_map->pc_err, &pc_mirrored, f->side);
    else
      rc = prs_pc_step(f->pc, f->pc_state, od, f->gi, d_argmax, d_total, d_err, f->side);
    if (rc != PRS_OK) return rc;
    PRS_CUDA(cudaEventRecord(f->ev_join, f->side));
  }
  if (short_chain) {
    rc = check_mask(f->im_rows, f->im_cols, f->row_lo, f->row_hi, f->row_step, f->col_lo, f->col_hi, f->col_step, 32, 32);
    if (rc != PRS_OK) return rc;
    k_vt_frame_prepare<<<1, 1024, 0, st>>>(f->frame_map, f->im_cols, f->row_lo, f->row_step, f->col_lo, f->col_step,
                                           d_tpl, d_planes, d_key);
    long long blocks = ((long long)f->capacity + 31) / 32;
    if (blocks > 148LL * 4) blocks = 148LL * 4;
    k_vt_sweep_packed_ref_small<false><<<(int)blocks, kSmallThreads, 0, st>>>((const uint4*)f->vt_packed, d_planes, d_key, f->d_n);
  } else {
    PRS_CUDA(cudaMemcpyAsync(d_frame, f->frame_host, (size_t)f->im_rows * f->im_cols, cudaMemcpyHostToDevice, st));
    rc = prs_vt_extract_u8(d_frame, f->im_rows, f->im_cols, f->row_lo, f->row_hi, f->row_step, f->col_lo, f->col_hi,
                           f->col_step, d_tpl, 32, 32, st);
    if (rc != PRS_OK) return rc;
    PRS_CUDA(cudaMemsetAsync(d_key, 0xff, sizeof(unsigned long long), st));
    k_vt_pack_query<<<1, 32, 0, st>>>(d_tpl, d_planes);
    PRS_CUDA(cudaMemcpyToSymbolAsync(c_vtq, d_planes, (32 * 8 + 2) * sizeof(uint32_t), 0, cudaMemcpyDeviceToDevice, st));
    // grid sized for the capacity; the kernels read the live count from device memory
    rc = launch_packed_sweep((const uint4*)f->vt_packed, 0, f->capacity, f->mode, 0, d_key, nullptr, f->d_n, st);
    if (rc != PRS_OK) return rc;
  }
  if (moved && !pc_mirrored) PRS_CUDA(cudaStreamWaitEvent(st, f->ev_join, 0));  // the decision reports the new arg-max
  prs_frame_result* rec = zero_copy ? f->result_map : d_res;
  k_vt_decide_append<<<1, 32, 0, st>>>(d_key, d_tpl, (uint4*)f->vt_packed, 0, f->threshold, d_argmax, d_err, rec, f->d_n,
                                       pc_mirrored ? 0 : 1, (zero_copy && f->inj_loc) ? d_res : nullptr);
  PRS_CUDA(cudaGetLastError());
  if (moved && pc_mirrored) PRS_CUDA(cudaStreamWaitEvent(st, f->ev_join, 0));  // join: the frame ends with both branches
  if (f->inj_loc) {  // behind both branches: the decision and the update (also the mirrored one the decision skips)
    prs_pc_plan* pc = f->pc;
    if (int rc_ = prs_pc_active_invalidate(pc, st)) return rc_;  // as prs_pc_inject: the carried lists are stale
    if (pc->dtype == PRS_F32)
      k_frame_inject<float><<<1, 32, 0, st>>>((float*)f->pc_state, f->inj_loc, d_res, d_argmax, d_err, rec, pc->X, pc->Y,
                                              pc->Th, (float)f->inj_energy);
    else
      k_frame_inject<double><<<1, 32, 0, st>>>((double*)f->pc_state, f->inj_loc, d_res, d_argmax, d_err, rec, pc->X, pc->Y,
                                               pc->Th, f->inj_energy);
    PRS_CUDA(cudaGetLastError());
  }
  if (!zero_copy)
    PRS_CUDA(cudaMemcpyAsync(f->result_host, d_res, sizeof(prs_frame_result), cudaMemcpyDeviceToHost, st));
  return PRS_OK;
}

extern "C" int prs_frame_create(prs_pc_handle pc, void* pc_state, const void* gi, void* pc_work, void* vt_packed,
                                int n_templates, int capacity, double threshold, int mode, int im_rows, int im_cols,
                                int row_lo, int row_hi, int row_step, int col_lo, int col_hi, int col_step,
                                void* scratch, double* odom_host, uint8_t* frame_host, prs_frame_result* result_host,
                                prs_frame_plan** out) {
  PRS_REQUIRE(pc && pc_state && gi && pc_work && vt_packed && scratch && odom_host && frame_host && result_host && out,
              "prs_frame_create: null argument");
  PRS_REQUIRE((size_t)im_rows * im_cols <= (1u << 20), "prs_frame_create: frame larger than 1 MiB");
  PRS_REQUIRE(capacity >= 1 && n_templates >= 0 && n_templates < capacity, "prs_frame_create: library has no free slot");
  prs_frame_plan* f = new (std::nothrow) prs_frame_plan();
  PRS_REQUIRE(f, "prs_frame_create: out of host memory");
  *f = prs_frame_plan{pc, pc_state, pc_work, vt_packed, scratch, gi, odom_host, frame_host, result_host, threshold, mode,
                      capacity, im_rows, im_cols, row_lo, row_hi, row_step, col_lo, col_hi, col_step, {nullptr, nullptr},
                      {false, false}, nullptr, {0, 0}, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
  {  // pinned buffers are mapped: kernels can read the inputs and write the result in place
    auto mapped = [](const void* p) -> void* {
      cudaPointerAttributes a;
      if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
        cudaGetLastError();
        return nullptr;
      }
      return a.type == cudaMemoryTypeHost ? a.devicePointer : nullptr;
    };
    f->odom_map = (const double*)mapped(odom_host);
    f->frame_map = (const uint8_t*)mapped(frame_host);
    f->result_map = (prs_frame_result*)mapped(result_host);
  }
  f->d_n = (int*)((char*)scratch + FrameScratch::kOdom + 32);
  cudaError_t e = cudaStreamCreateWithFlags(&f->side, cudaStreamNonBlocking);
  if (e == cudaSuccess) e = cudaEventCreateWithFlags(&f->ev_fork, cudaEventDisableTiming);
  if (e == cudaSuccess) e = cudaEventCreateWithFlags(&f->ev_join, cudaEventDisableTiming);
  if (e == cudaSuccess) e = cudaEventCreateWithFlags(&f->ev_done, cudaEventDisableTiming);
  if (e == cudaSuccess) e = cudaMemcpy(f->d_n, &n_templates, sizeof(int), cudaMemcpyHostToDevice);
  if (e != cudaSuccess) {
    prs_set_error("prs_frame_create: %s", cudaGetErrorString(e));
    delete f;
    return PRS_E_CUDA;
  }
  *out = f;
  return PRS_OK;
}

extern "C" int prs_frame_destroy(prs_frame_plan* f) {
  if (f) {
    for (int i = 0; i < 2; ++i)
      if (f->ready[i]) cudaGraphExecDestroy(f->exec[i]);
    if (f->side) cudaStreamDestroy(f->side);
    if (f->ev_fork) cudaEventDestroy(f->ev_fork);
    if (f->ev_join) cudaEventDestroy(f->ev_join);
    if (f->ev_done) cudaEventDestroy(f->ev_done);
    delete f;
  }
  return PRS_OK;
}

// The library size the plan's kernels read lives in device memory (shared by the plans built on one scratch
// buffer): a caller that appended templates outside the plan (ViewTemplates.match / create) puts the host's count back.
extern "C" int prs_frame_set_count(prs_frame_plan* f, int n_templates, void* stream) {
  PRS_REQUIRE(f && n_templates >= 0 && n_templates < f->capacity, "prs_frame_set_count: bad argument");
  PRS_CUDA(cudaMemcpyAsync(f->d_n, &n_templates, sizeof(int), cudaMemcpyHostToDevice, (cudaStream_t)stream));
  PRS_CUDA(cudaStreamSynchronize((cudaStream_t)stream));
  return PRS_OK;
}

// Turning the injection on or off, or changing its energy or table, changes the frame's last node: the captured graphs
// go, the next frame of each kind runs eagerly again and the one after it captures.
extern "C" int prs_frame_set_inject(prs_frame_plan* f, double energy, long long* loc_dev) {
  PRS_REQUIRE(f, "prs_frame_set_inject: null plan");
  PRS_REQUIRE(energy >= 0.0 && energy <= 1.7976931348623157e308,
              "prs_frame_set_inject: the energy must be finite and >= 0, got %g", energy);
  if (f->inj_loc == loc_dev && (loc_dev == nullptr || f->inj_energy == energy)) return PRS_OK;
  for (int i = 0; i < 2; ++i) {
    if (f->ready[i]) cudaGraphExecDestroy(f->exec[i]);
    f->ready[i] = false;
    f->warm[i] = 0;
  }
  f->inj_loc = loc_dev;
  f->inj_energy = energy;
  return PRS_OK;
}

// One frame.  `moved` != 0: odom_host (given at creation) holds (vtrans, vrot) and the pose cells are updated first.
// The first call of each kind runs eagerly (it also warms every lazily initialised kernel attribute), the second
// captures the graph, later ones replay it.
extern "C" int prs_frame_launch(prs_frame_plan* f, int moved, void* stream) {
  PRS_REQUIRE(f, "prs_frame_launch: null plan");
  cudaStream_t st = (cudaStream_t)stream;
  const int v = moved ? 1 : 0;
  int rc = PRS_OK;
  // the long chain sweeps through the per-device constant buffer: order the whole frame behind sweeps on other streams
  const bool uses_vtq = !(f->odom_map && f->frame_map && f->result_map && f->mode == PRS_VT_MODE_REF && f->capacity <= kSmallLibrary);
  VtqScope scope;
  if (uses_vtq)
    if (int rc0 = scope.begin(st)) return rc0;
  if (f->ready[v]) {
    PRS_CUDA(cudaGraphLaunch(f->exec[v], st));
  } else if (f->warm[v] < 1 || st == nullptr) {  // the legacy default stream cannot be captured
    ++f->warm[v];
    rc = frame_enqueue(f, moved != 0, st);
    if (rc != PRS_OK) return rc;
  } else {
    cudaGraph_t g = nullptr;
    PRS_CUDA(cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal));
    rc = frame_enqueue(f, moved != 0, st);
    cudaError_t e = cudaStreamEndCapture(st, &g);
    if (rc != PRS_OK || e != cudaSuccess) {
      if (g) cudaGraphDestroy(g);
      if (rc == PRS_OK) prs_set_error("prs_frame_launch: capture failed: %s", cudaGetErrorString(e));
      return rc != PRS_OK ? rc : PRS_E_CUDA;
    }
    PRS_CUDA(cudaGraphInstantiate(&f->exec[v], g, 0));
    cudaGraphDestroy(g);
    f->ready[v] = true;
    PRS_CUDA(cudaGraphLaunch(f->exec[v], st));
  }
  return scope.end();
}

extern "C" int prs_frame_run(prs_frame_plan* f, int moved, void* stream) {
  int rc = prs_frame_launch(f, moved, stream);
  if (rc != PRS_OK) return rc;
  PRS_CUDA(cudaStreamSynchronize((cudaStream_t)stream));
  return PRS_OK;
}

// The whole replay loop (ros_simulate.py:152-166 driven from arrays) on the host side of the C ABI: frame t is
// staged into the pinned buffers of plan t mod n_plans and launched while the earlier frames are still running;
// a plan is reused once its event has fired and its 32-byte result has been copied out.  All plans must share the
// device-side state (pose cells, library, template count, scratch) and differ only in their pinned host buffers;
// the library must have room for T more templates.
//   frames  : host uint8 [T][im_rows][im_cols] (pageable is fine: each frame is copied into the plan's pinned buffer)
//   odom    : host double [T][2] = (vtrans, vrot) as passed to PoseCellNetwork.update
//   moved   : host uint8 [T], 0 = no pose-cell update for this frame (ros_simulate.py:128)
//   results : host prs_frame_result [T]
extern "C" int prs_replay_run(prs_frame_plan* const* plans, int n_plans, const uint8_t* frames, const double* odom,
                              const uint8_t* moved, int T, prs_frame_result* results, void* stream) {
  PRS_REQUIRE(plans && n_plans >= 1 && n_plans <= 16 && T >= 0 && results, "prs_replay_run: bad argument");
  PRS_REQUIRE(T == 0 || (frames && odom && moved), "prs_replay_run: null input");
  PRS_REQUIRE(stream != nullptr, "prs_replay_run: needs a non-default stream (the frames replay as CUDA graphs)");
  for (int i = 0; i < n_plans; ++i) PRS_REQUIRE(plans[i], "prs_replay_run: null plan");
  cudaStream_t st = (cudaStream_t)stream;
  const size_t fbytes = (size_t)plans[0]->im_rows * plans[0]->im_cols;
  int rc = PRS_OK;
  int launched = 0;
  for (int t = 0; t < T; ++t) {
    prs_frame_plan* f = plans[t % n_plans];
    if (t >= n_plans) {
      PRS_CUDA(cudaEventSynchronize(f->ev_done));
      results[t - n_plans] = *f->result_host;
    }
    memcpy(f->frame_host, frames + (size_t)t * fbytes, fbytes);
    if (moved[t]) {
      f->odom_host[0] = odom[2 * t];
      f->odom_host[1] = odom[2 * t + 1];
    }
    rc = prs_frame_launch(f, moved[t] ? 1 : 0, st);
    if (rc != PRS_OK) break;
    PRS_CUDA(cudaEventRecord(f->ev_done, st));
    launched = t + 1;
  }
  // drain: the last min(n_plans, launched) frames
  for (int t = launched > n_plans ? launched - n_plans : 0; t < launched; ++t) {
    prs_frame_plan* f = plans[t % n_plans];
    if (cudaEventSynchronize(f->ev_done) != cudaSuccess) {
      prs_set_error("prs_replay_run: %s", cudaGetErrorString(cudaGetLastError()));
      return PRS_E_CUDA;
    }
    results[t] = *f->result_host;
  }
  return rc;
}

// ---------------------------------------------------------------------------------------------
// Ensemble replay: B agents, each with its own pose-cell network (the B networks of one plan), view-template library,
// threshold and injection energy; agent b replays recording rec_of[b] of R.  A recording is a stream of ticks, each an
// optional gated twist and an optional image (a frame replay is the stream in which every tick has an image), and a
// tick is ONE graph for the whole ensemble:
//   side branch  k_ens_odom_multi (each network its recording's twist, (0, 0) where that recording did not move or has
//                ended) -> [mixed: k_ens_snapshot save] -> prs_pc_step -> [mixed: k_ens_snapshot restore ->
//                prs_pc_active_invalidate] -> [activity: k_ens_activity]
//   template     k_vt_frame_prepare_multi (one block per recording) -> k_vt_sweep_packed_ref_small<true> over every
//                agent's library (grid-stride over (agent, group))
//   join         k_vt_decide_append, one warp per agent -> [k_frame_inject, one thread per agent] -> k_ens_advance (the
//                device-side tick counter)
// The restore runs before the join, so the decision and the injection of a still network see its state, arg-max and
// error bits as they were: what a skipped update leaves.  A tick where no recording moved runs no update; one where
// every recording moved needs no snapshot, so with R = 1 no tick is mixed.  A tick without an image in any recording
// is lean: the side branch's nodes run on the tick's stream itself, then k_ens_no_image writes the records and advances
// the counter -- no query, sweep, decision or injection.  Six graphs: {no update, all moved, mixed} x {image, none}.
// With the activity capture on (prs_ens_set_activity), an image tick without update runs k_ens_activity on the main
// stream before the decision; a lean tick captures nothing.
// Images, odometry, gates and image slots go to the device a chunk of ticks at a time, the records [chunk][B] come
// back a chunk at a time.
constexpr int kEnsChunk = 256;

// Device scratch of an ensemble plan (prs_ens_scratch_bytes), every part 256-byte aligned.  A chunk holds `chunk` ticks
// of each of the R recordings, as many as fit kEnsFrameBytes of images (at least one, at most kEnsChunk).  The
// per-agent snapshot of a mixed tick is empty when R = 1.
constexpr size_t kEnsFrameBytes = 256u << 20;

struct EnsScratch {
  int chunk = 0;
  size_t frames = 0, odom_chunk = 0, gate = 0, slots = 0, rec = 0, odom = 0, key = 0, tpl = 0, planes = 0, present = 0,
         still = 0, wsnap = 0, snap = 0, misc = 0, bytes = 0;
  EnsScratch() = default;
  EnsScratch(int B, int R, long long fbytes, size_t net_bytes) {
    auto up = [](size_t v) { return (v + 255) & ~(size_t)255; };
    const long long fit = (long long)(kEnsFrameBytes / ((size_t)R * fbytes));
    chunk = (int)(fit < 1 ? 1 : fit > kEnsChunk ? kEnsChunk : fit);
    const size_t snaps = R > 1 ? (size_t)B : 0;
    frames = 0;
    odom_chunk = frames + up((size_t)R * chunk * fbytes);
    gate = odom_chunk + up((size_t)chunk * R * 2 * sizeof(double));
    slots = gate + up((size_t)chunk * R);
    rec = slots + up((size_t)chunk * R * sizeof(int));
    odom = rec + up((size_t)chunk * B * sizeof(prs_frame_result));
    key = odom + up((size_t)B * 2 * sizeof(double));
    tpl = key + up((size_t)B * sizeof(unsigned long long));
    planes = tpl + up((size_t)R * 1024);
    present = planes + up((size_t)R * kQueryStride * sizeof(uint32_t));
    still = present + up((size_t)R);
    wsnap = still + up((size_t)B);
    snap = wsnap + up(snaps * 3 * sizeof(long long));
    misc = snap + up(snaps * net_bytes);  // int tick counter, int group maximum, int largest live count
    bytes = misc + 256;
  }
};

// Network b gets its recording's (vtrans, vrot) where that recording moved at this tick (bit 1 of gate[*ctr][r]), else
// (0, 0), which no pose-cell kernel rejects; still[b] = 1 marks the network whose update the mixed tick undoes.
__global__ void k_ens_odom_multi(const double* __restrict__ odom_chunk, const uint8_t* __restrict__ gate,
                                 const int* __restrict__ ctr, const int* __restrict__ rec_of, int R,
                                 double* __restrict__ odom, uint8_t* __restrict__ still, int B) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  const size_t i = (size_t)*ctr * R + rec_of[b];
  const bool mv = (gate[i] & 2) != 0;
  odom[2 * b] = mv ? odom_chunk[2 * i] : 0.0;
  odom[2 * b + 1] = mv ? odom_chunk[2 * i + 1] : 0.0;
  still[b] = mv ? 0 : 1;
}

// The mixed tick's save (kRestore = false, before prs_pc_step) and restore (after it) of every still network: its
// state slice of `words` W-words, and its pc_work slots (arg-max, total of total_bytes, err), to and from one snapshot per agent.
// Blocks of other networks return at once.
template <bool kRestore, typename W>
__global__ void k_ens_snapshot(W* __restrict__ state, W* __restrict__ snap, long long words, int per_net,
                               const uint8_t* __restrict__ still, long long* __restrict__ work,
                               long long* __restrict__ wsnap, int B, int total_bytes) {
  const int b = blockIdx.x / per_net;
  if (!still[b]) return;
  W* s = state + b * words;
  W* d = snap + b * words;
  for (long long i = (long long)(blockIdx.x % per_net) * blockDim.x + threadIdx.x; i < words;
       i += (long long)per_net * blockDim.x) {
    if (kRestore)
      s[i] = d[i];
    else
      d[i] = s[i];
  }
  if (blockIdx.x % per_net == 0 && threadIdx.x == 0) {
    int* err = (int*)(work + 2 * (size_t)B);
    int* total32 = (int*)(work + B);  // a float32 plan's totals are 4-byte elements of the 8-byte slots' region
    if (kRestore) {
      work[b] = wsnap[3 * b];
      if (total_bytes == 4)
        total32[b] = (int)wsnap[3 * b + 1];
      else
        work[B + b] = wsnap[3 * b + 1];
      err[b] = (int)wsnap[3 * b + 2];
    } else {
      wsnap[3 * b] = work[b];
      wsnap[3 * b + 1] = total_bytes == 4 ? total32[b] : work[B + b];
      wsnap[3 * b + 2] = err[b];
    }
  }
}

__global__ void k_ens_advance(int* ctr) { ++*ctr; }

// A tick without an image in any recording, in place of the decision: every agent's "no image" record -- the arg-max,
// error bits and template count as the tick's update left them, template -1, as k_vt_decide_append writes for an agent
// whose recording has no image -- then the tick counter advances.  One block, one thread per agent (strided past 1024).
__global__ void __launch_bounds__(1024)
    k_ens_no_image(const long long* __restrict__ argmax, const int* __restrict__ pc_err, const int* __restrict__ n_dev,
                   prs_frame_result* __restrict__ rec, int* __restrict__ ctr, int B) {
  prs_frame_result* row = rec + (long long)*ctr * B;
  for (int b = threadIdx.x; b < B; b += blockDim.x) {
    prs_frame_result* r = row + b;
    r->argmax = argmax[b];
    r->key = ~0ull;
    r->created = 0;
    r->template_index = -1;
    r->n_templates = n_dev[b];
    r->pc_err = pc_err[b];
  }
  __syncthreads();  // every thread has read the counter
  if (threadIdx.x == 0) ++*ctr;
}

// group maximum and largest live count of the libraries a plan starts from
__global__ void k_ens_init(const int* __restrict__ n_dev, int B, int* __restrict__ misc) {
  for (int b = threadIdx.x; b < B; b += blockDim.x) {
    atomicMax(misc + 1, (n_dev[b] + 31) >> 5);
    atomicMax(misc + 2, n_dev[b]);
  }
}

// ---------------------------------------------------------------------------------------------
// Pose-cell activity capture (prs_ens_set_activity, DESIGN.md 4.15): at every tick with an image, each agent's cells
// above a threshold in the state its match is made with -- after the tick's update (and a mixed tick's restore),
// before its injection -- as the viewers draw them (cells > 0.002).  An entry is the count of such cells and the first
// K of them in the reference's C order [x][y][th]: an int32 flat index x*Y*Th + y*Th + th and the state's value.
// Entries live in slots [chunk][B][K] indexed by the tick counter; after a run, k_ens_activity_scan and
// k_ens_activity_gather pack the kept cells of the run's ticks into one prefix, so what crosses the bus scales with the
// captured cells, not with B * K * ticks.
constexpr int kActThreads = 512;

// Buffer of the capture (prs_ens_activity_bytes), every part 256-byte aligned: counts int32 [chunk][B] (-1 = no image),
// slots int32 idx [chunk][B][K] and T val [chunk][B][K], the packed offsets int64 [chunk * B + 1] (the last one is the
// total) and the packed idx and val [chunk * B * K].
struct EnsActivity {
  size_t counts = 0, idx = 0, val = 0, off = 0, pidx = 0, pval = 0, bytes = 0;
  EnsActivity() = default;
  EnsActivity(int B, int chunk, int K, int es) {
    auto up = [](size_t v) { return (v + 255) & ~(size_t)255; };
    const size_t rows = (size_t)chunk * B, cells = rows * K;
    counts = 0;
    idx = counts + up(rows * sizeof(int));
    val = idx + up(cells * sizeof(int));
    off = val + up(cells * es);
    pidx = off + up((rows + 1) * sizeof(long long));
    pval = pidx + up(cells * sizeof(int));
    bytes = pval + up(cells * es);
  }
};

// Block-wide exclusive scan of one int per thread (blockDim a multiple of 32, at most 1024); `total` gets the sum.
__device__ __forceinline__ int act_block_scan(int v, int* total) {
  __shared__ int warp_sum[32];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = blockDim.x >> 5;
  int x = v;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const int y = __shfl_up_sync(0xffffffffu, x, d);
    if (lane >= d) x += y;
  }
  __syncthreads();  // warp_sum of an earlier call has been read
  if (lane == 31) warp_sum[w] = x;
  __syncthreads();
  if (w == 0) {
    int s = lane < nw ? warp_sum[lane] : 0;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const int y = __shfl_up_sync(0xffffffffu, s, d);
      if (lane >= d) s += y;
    }
    if (lane < nw) warp_sum[lane] = s;  // inclusive sums of the warps
  }
  __syncthreads();
  *total = warp_sum[nw - 1];
  return x - v + (w > 0 ? warp_sum[w - 1] : 0);
}

// One CTA per network.  The state is theta-major [B][Th][X][Y], so line p = x*Y + y of plane th sits at th*X*Y + p and a
// thread owns lines p0 + threadIdx.x of consecutive rounds p0: its loads are coalesced across the block, and C order is
// line-major (flat = p*Th + th), so a block scan of the per-line counts in each round gives every cell its C-order rank
// -- deterministic, no sort.  A second, cached read of the (few) lines with kept cells writes them.  An agent whose
// recording has no image at the tick gets count -1 (bit 0 of the tick's gate, as k_ens_odom_multi reads bit 1).
template <typename T>
__global__ void __launch_bounds__(kActThreads, 2)
    k_ens_activity(const T* __restrict__ state, int P, int Th, double thr, int K, const uint8_t* __restrict__ gate,
                   const int* __restrict__ ctr, const int* __restrict__ rec_of, int R, int B, int* __restrict__ counts,
                   int* __restrict__ idx, T* __restrict__ val) {
  const int b = blockIdx.x, c = *ctr;
  const size_t row = (size_t)c * B + b;
  if (!(gate[(size_t)c * R + rec_of[b]] & 1)) {
    if (threadIdx.x == 0) counts[row] = -1;
    return;
  }
  const T* s = state + (size_t)b * P * Th;
  int* out_idx = idx + row * K;
  T* out_val = val + row * K;
  int base = 0;  // cells of the earlier rounds
  for (int p0 = 0; p0 < P; p0 += blockDim.x) {
    const int p = p0 + threadIdx.x;
    int n = 0;
    if (p < P) {
#pragma unroll 6
      for (int th = 0; th < Th; ++th) n += (double)s[(size_t)th * P + p] > thr ? 1 : 0;  // independent loads in flight
    }
    int total;
    int o = base + act_block_scan(n, &total);
    if (n > 0 && o < K) {
      for (int th = 0; th < Th && o < K; ++th) {
        const T v = s[(size_t)th * P + p];
        if ((double)v > thr) {
          out_idx[o] = p * Th + th;
          out_val[o] = v;
          ++o;
        }
      }
    }
    base += total;
  }
  if (threadIdx.x == 0) counts[row] = base;
}

// After a run of n = ticks * B entries: entries of agents without an image at the tick (the lean ticks' rows are never
// written) become -1, and off[i] = sum of min(count, K) over the entries before i, off[n] the total.  One block: each
// thread a contiguous segment, a block scan of the segment sums (in 64 bits).
constexpr int kActScanThreads = 512;
__global__ void __launch_bounds__(kActScanThreads)
    k_ens_activity_scan(int* __restrict__ counts, const uint8_t* __restrict__ gate, const int* __restrict__ rec_of, int R,
                        int B, long long n, int K, long long* __restrict__ off) {
  __shared__ long long part[kActScanThreads];
  const long long per = (n + kActScanThreads - 1) / kActScanThreads;
  const long long i0 = threadIdx.x * per < n ? threadIdx.x * per : n, i1 = i0 + per < n ? i0 + per : n;
  long long t = i0 / B;
  int b = (int)(i0 - t * B);
  long long sum = 0;
  for (long long i = i0; i < i1; ++i) {
    int cnt = counts[i];
    if (!(gate[t * R + rec_of[b]] & 1)) counts[i] = cnt = -1;
    sum += cnt < 0 ? 0 : cnt < K ? cnt : K;
    if (++b == B) b = 0, ++t;
  }
  part[threadIdx.x] = sum;
  __syncthreads();
  for (int d = 1; d < kActScanThreads; d <<= 1) {
    const long long y = (int)threadIdx.x >= d ? part[threadIdx.x - d] : 0;
    __syncthreads();
    part[threadIdx.x] += y;
    __syncthreads();
  }
  long long o = part[threadIdx.x] - sum;
  for (long long i = i0; i < i1; ++i) {
    off[i] = o;
    const int cnt = counts[i];
    o += cnt < 0 ? 0 : cnt < K ? cnt : K;
  }
  if (threadIdx.x == kActScanThreads - 1) off[n] = part[threadIdx.x];
}

// One warp per entry: its min(count, K) kept cells to the packed prefix at off[i].
template <typename T>
__global__ void k_ens_activity_gather(const int* __restrict__ counts, const long long* __restrict__ off,
                                      const int* __restrict__ idx, const T* __restrict__ val, long long n, int K,
                                      int* __restrict__ pidx, T* __restrict__ pval) {
  const long long i = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (i >= n) return;
  const int cnt = counts[i];
  const int k = cnt < 0 ? 0 : cnt < K ? cnt : K;
  const long long o = off[i];
  for (int j = lane; j < k; j += 32) {
    pidx[o + j] = idx[i * K + j];
    pval[o + j] = val[i * K + j];
  }
}

struct prs_ens_plan {
  prs_pc_handle pc;
  void *pc_state, *pc_work, *libs;
  const void* gi;
  int* n_dev;
  const double* thr_dev;
  const double* energy_dev;
  long long* loc_dev;
  int B, R, capacity;
  const int* rec_of;
  long long lib_u4, fbytes, room;  // room: image ticks the libraries can still take (one template per agent and image)
  int im_cols, row_lo, row_step, col_lo, col_step;
  char* scratch;
  EnsScratch lay;
  // the tick's graphs: [v] with an image in some recording, [3 + v] without; v = 0 no recording moved, 1 every
  // recording moved, 2 mixed
  cudaGraphExec_t exec[6];
  bool ready[6];
  int warm[6];
  cudaStream_t side;
  cudaEvent_t ev_fork, ev_join;
  // prs_ens_set_activity: the capture buffer (null = no capture node), its threshold and cells per entry, and the
  // ticks of the last run, which prs_ens_activity_pack packs
  char* act = nullptr;
  double act_thr = 0.0;
  int act_k = 0, act_ticks = 0;
};

static size_t ens_net_bytes(const prs_pc_plan* pc) { return (size_t)pc->N * (pc->dtype == PRS_F32 ? 4 : 8); }

static int ens_tick_enqueue(prs_ens_plan* e, int v, bool image, cudaStream_t st) {
  char* sc = e->scratch;
  const EnsScratch& M = e->lay;
  prs_pc_plan* pc = e->pc;
  long long* d_argmax = (long long*)e->pc_work;
  void* d_total = (char*)e->pc_work + 8 * (size_t)e->B;
  int* d_err = (int*)((char*)e->pc_work + 16 * (size_t)e->B);
  int* d_ctr = (int*)(sc + M.misc);
  int* d_gmax = d_ctr + 1;
  double* d_odom = (double*)(sc + M.odom);
  unsigned long long* d_key = (unsigned long long*)(sc + M.key);
  prs_frame_result* d_rec = (prs_frame_result*)(sc + M.rec);
  const uint8_t* d_gate = (const uint8_t*)(sc + M.gate);
  uint8_t* d_present = (uint8_t*)(sc + M.present);
  uint8_t* d_still = (uint8_t*)(sc + M.still);
  const int B = e->B, R = e->R;
  const cudaStream_t side = image ? e->side : st;
  // the activity capture (image ticks only): the state the tick's match is made with, before its injection
  auto activity = [&](cudaStream_t s) {
    const EnsActivity A(B, M.chunk, e->act_k, pc->dtype == PRS_F32 ? 4 : 8);
    const int P = pc->X * pc->Y;
    const int threads = P >= kActThreads ? kActThreads : (P + 31) / 32 * 32;
    if (pc->dtype == PRS_F32)
      k_ens_activity<float><<<B, threads, 0, s>>>((const float*)e->pc_state, P, pc->Th, e->act_thr, e->act_k, d_gate,
                                                  d_ctr, e->rec_of, R, B, (int*)(e->act + A.counts),
                                                  (int*)(e->act + A.idx), (float*)(e->act + A.val));
    else
      k_ens_activity<double><<<B, threads, 0, s>>>((const double*)e->pc_state, P, pc->Th, e->act_thr, e->act_k, d_gate,
                                                   d_ctr, e->rec_of, R, B, (int*)(e->act + A.counts),
                                                   (int*)(e->act + A.idx), (double*)(e->act + A.val));
    return cudaGetLastError();
  };
  int rc;
  if (v != 0) {
    if (image) {  // fork: the pose-cell update does not depend on the images until the decision
      PRS_CUDA(cudaEventRecord(e->ev_fork, st));
      PRS_CUDA(cudaStreamWaitEvent(e->side, e->ev_fork, 0));
    }
    k_ens_odom_multi<<<(B + 255) / 256, 256, 0, side>>>((const double*)(sc + M.odom_chunk), d_gate, d_ctr, e->rec_of, R,
                                                        d_odom, d_still, B);
    PRS_CUDA(cudaGetLastError());
    const int es = pc->dtype == PRS_F32 ? 4 : 8;
    const size_t net_bytes = ens_net_bytes(pc);
    const bool wide = net_bytes % 16 == 0;
    const long long words = (long long)(net_bytes / (wide ? 16 : 4));
    const int per_net = (int)((words + 4095) / 4096);  // 256 threads x 16 words per block
    auto snapshot = [&](bool restore) {
      long long* ws = (long long*)(sc + M.wsnap);
      long long* w = (long long*)e->pc_work;
      const dim3 grid((unsigned)B * per_net);
      if (wide) {
        if (restore)
          k_ens_snapshot<true, uint4><<<grid, 256, 0, side>>>((uint4*)e->pc_state, (uint4*)(sc + M.snap), words, per_net,
                                                                 d_still, w, ws, B, es);
        else
          k_ens_snapshot<false, uint4><<<grid, 256, 0, side>>>((uint4*)e->pc_state, (uint4*)(sc + M.snap), words,
                                                                  per_net, d_still, w, ws, B, es);
      } else {
        if (restore)
          k_ens_snapshot<true, unsigned><<<grid, 256, 0, side>>>((unsigned*)e->pc_state, (unsigned*)(sc + M.snap), words,
                                                                    per_net, d_still, w, ws, B, es);
        else
          k_ens_snapshot<false, unsigned><<<grid, 256, 0, side>>>((unsigned*)e->pc_state, (unsigned*)(sc + M.snap),
                                                                     words, per_net, d_still, w, ws, B, es);
      }
      return cudaGetLastError();
    };
    if (v == 2) PRS_CUDA(snapshot(false));
    rc = prs_pc_step(pc, e->pc_state, d_odom, e->gi, d_argmax, d_total, d_err, side);
    if (rc != PRS_OK) return rc;
    if (v == 2) {
      PRS_CUDA(snapshot(true));
      if (int rc_ = prs_pc_active_invalidate(pc, side)) return rc_;  // the carried lists describe the undone update
    }
    // on the side branch, beside the sweep: only reads the state, so the active-set lists stay valid
    if (image && e->act) PRS_CUDA(activity(side));
    if (image) PRS_CUDA(cudaEventRecord(e->ev_join, e->side));
  }
  if (!image) {
    k_ens_no_image<<<1, B < 1024 ? (B + 31) / 32 * 32 : 1024, 0, st>>>(d_argmax, d_err, e->n_dev, d_rec, d_ctr, B);
    PRS_CUDA(cudaGetLastError());
    return PRS_OK;
  }
  k_vt_frame_prepare_multi<<<R, 1024, 0, st>>>((const uint8_t*)(sc + M.frames), M.chunk, e->fbytes, e->im_cols, e->row_lo,
                                               e->row_step, e->col_lo, e->col_step, (uint8_t*)(sc + M.tpl),
                                               (uint32_t*)(sc + M.planes), d_key, B, d_ctr, d_present,
                                               (const int*)(sc + M.slots));
  long long blocks = (long long)B * ((e->capacity + 31) / 32);
  if (blocks > 148LL * 4) blocks = 148LL * 4;
  // With one recording a tick with an image has it for every agent: the per-agent recording and presence checks
  // cannot fail, and they cost the latency-bound sweep a chain of dependent loads per item (6 % of the frame at B = 1024)
  const bool one = R == 1;
  if (one)
    k_vt_sweep_packed_ref_small<false><<<(int)blocks, kSmallThreads, 0, st>>>(
        (const uint4*)e->libs, (const uint32_t*)(sc + M.planes), d_key, e->n_dev, B, e->lib_u4, d_gmax);
  else
    k_vt_sweep_packed_ref_small<true><<<(int)blocks, kSmallThreads, 0, st>>>(
        (const uint4*)e->libs, (const uint32_t*)(sc + M.planes), d_key, e->n_dev, B, e->lib_u4, d_gmax, e->rec_of,
        d_present);
  if (v != 0) PRS_CUDA(cudaStreamWaitEvent(st, e->ev_join, 0));  // the decision reports the new arg-max
  if (v == 0 && e->act) PRS_CUDA(activity(st));                 // no update: the state as the last tick left it
  VtAgents ag;
  ag.B = B;
  ag.lib_u4 = e->lib_u4;
  ag.threshold = e->thr_dev;
  ag.loc = e->loc_dev;
  ag.loc_stride = e->capacity;
  ag.g_max = d_gmax;
  ag.ctr = d_ctr;
  if (!one) {
    ag.rec_of = e->rec_of;
    ag.present = d_present;
  }
  k_vt_decide_append<<<(B + 3) / 4, 128, 0, st>>>(d_key, (const uint8_t*)(sc + M.tpl), (uint4*)e->libs, 0, 0.0, d_argmax,
                                                  d_err, d_rec, e->n_dev, 1, nullptr, ag);
  PRS_CUDA(cudaGetLastError());
  if (e->energy_dev) {
    if (int rc_ = prs_pc_active_invalidate(pc, st)) return rc_;  // as prs_pc_inject: the carried lists are stale
    if (pc->dtype == PRS_F32)
      k_frame_inject<float><<<(B + 127) / 128, 128, 0, st>>>((float*)e->pc_state, e->loc_dev, d_rec, d_argmax, d_err, d_rec,
                                                             pc->X, pc->Y, pc->Th, 0.0f, e->energy_dev, ag);
    else
      k_frame_inject<double><<<(B + 127) / 128, 128, 0, st>>>((double*)e->pc_state, e->loc_dev, d_rec, d_argmax, d_err,
                                                              d_rec, pc->X, pc->Y, pc->Th, 0.0, e->energy_dev, ag);
    PRS_CUDA(cudaGetLastError());
  }
  k_ens_advance<<<1, 1, 0, st>>>(d_ctr);
  PRS_CUDA(cudaGetLastError());
  return PRS_OK;
}

// One tick: the first call of each kind runs eagerly (lazily initialised kernel attributes), the second captures the
// graph, later ones replay it.
static int ens_tick_launch(prs_ens_plan* e, int v, bool image, cudaStream_t st) {
  const int i = image ? v : 3 + v;
  if (e->ready[i]) {
    PRS_CUDA(cudaGraphLaunch(e->exec[i], st));
    return PRS_OK;
  }
  if (e->warm[i] < 1) {
    ++e->warm[i];
    return ens_tick_enqueue(e, v, image, st);
  }
  cudaGraph_t g = nullptr;
  PRS_CUDA(cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal));
  int rc = ens_tick_enqueue(e, v, image, st);
  cudaError_t err = cudaStreamEndCapture(st, &g);
  if (rc != PRS_OK || err != cudaSuccess) {
    if (g) cudaGraphDestroy(g);
    if (rc == PRS_OK) prs_set_error("prs_ens_run: capture failed: %s", cudaGetErrorString(err));
    return rc != PRS_OK ? rc : PRS_E_CUDA;
  }
  err = cudaGraphInstantiate(&e->exec[i], g, 0);
  cudaGraphDestroy(g);
  PRS_CUDA(err);
  e->ready[i] = true;
  PRS_CUDA(cudaGraphLaunch(e->exec[i], st));
  return PRS_OK;
}

extern "C" size_t prs_ens_scratch_bytes(prs_pc_handle pc, int R, int im_rows, int im_cols) {
  if (!pc || R < 1 || im_rows < 1 || im_cols < 1) return 0;
  return EnsScratch(pc->B, R, (long long)im_rows * im_cols, ens_net_bytes(pc)).bytes;
}

extern "C" int prs_ens_create(prs_pc_handle pc, void* pc_state, const void* gi, void* pc_work, void* libs, int capacity,
                              int* n_dev, const double* threshold_dev, const double* energy_dev, long long* loc_dev,
                              int R, const int* rec_of_dev, int mode, int im_rows, int im_cols, int row_lo, int row_hi,
                              int row_step, int col_lo, int col_hi, int col_step, void* scratch, prs_ens_plan** out) {
  PRS_REQUIRE(pc && pc_state && gi && pc_work && libs && n_dev && threshold_dev && loc_dev && rec_of_dev && scratch && out,
              "prs_ens_create: null argument");
  PRS_REQUIRE(R >= 1, "prs_ens_create: %d recordings", R);
  PRS_REQUIRE(mode == PRS_VT_MODE_REF, "prs_ens_create: only the reference mode (PRS_VT_MODE_REF) is supported, got %d",
              mode);
  PRS_REQUIRE(capacity >= 1 && capacity <= kSmallLibrary, "prs_ens_create: capacity %d outside [1, %d]", capacity,
              kSmallLibrary);
  PRS_REQUIRE(im_rows >= 1 && im_cols >= 1 && (size_t)im_rows * im_cols <= (1u << 20),
              "prs_ens_create: frame must be 1 byte to 1 MiB");
  if (int rc = check_mask(im_rows, im_cols, row_lo, row_hi, row_step, col_lo, col_hi, col_step, 32, 32)) return rc;
  if (int rc = prs_pc_check_device(pc, "prs_ens_create")) return rc;
  const int B = pc->B;
  const long long fbytes = (long long)im_rows * im_cols;
  prs_ens_plan* e = new (std::nothrow) prs_ens_plan{pc, pc_state, pc_work, libs, gi, n_dev, threshold_dev, energy_dev,
                                                     loc_dev, B, R, capacity, rec_of_dev,
                                                     (long long)(prs_vt_packed_bytes(capacity) / 16), fbytes, 0, im_cols,
                                                     row_lo, row_step, col_lo, col_step, (char*)scratch,
                                                     EnsScratch(B, R, fbytes, ens_net_bytes(pc)), {}, {}, {}, nullptr,
                                                     nullptr, nullptr};
  PRS_REQUIRE(e, "prs_ens_create: out of host memory");
  int* misc = (int*)(e->scratch + e->lay.misc);
  int init[3] = {0, 0, 0};
  cudaError_t err = cudaStreamCreateWithFlags(&e->side, cudaStreamNonBlocking);
  if (err == cudaSuccess) err = cudaEventCreateWithFlags(&e->ev_fork, cudaEventDisableTiming);
  if (err == cudaSuccess) err = cudaEventCreateWithFlags(&e->ev_join, cudaEventDisableTiming);
  if (err == cudaSuccess) err = cudaMemcpy(misc, init, sizeof(init), cudaMemcpyHostToDevice);
  if (err == cudaSuccess) {
    k_ens_init<<<1, 256>>>(n_dev, B, misc);
    err = cudaGetLastError();
  }
  if (err == cudaSuccess) err = cudaMemcpy(init, misc, sizeof(init), cudaMemcpyDeviceToHost);
  if (err != cudaSuccess) {
    prs_set_error("prs_ens_create: %s", cudaGetErrorString(err));
    prs_ens_destroy(e);
    return PRS_E_CUDA;
  }
  e->room = (long long)capacity - init[2];
  *out = e;
  return PRS_OK;
}

// Room counts image ticks, not templates (a run may append one per image tick); a session that feeds a plan in pieces
// recounts it from the libraries as they are after the earlier runs.
extern "C" int prs_ens_refresh_room(prs_ens_plan* e, void* stream) {
  PRS_REQUIRE(e && stream, "prs_ens_refresh_room: bad argument");
  const cudaStream_t st = (cudaStream_t)stream;
  int* misc = (int*)(e->scratch + e->lay.misc);
  int n = 0;
  PRS_CUDA(cudaMemsetAsync(misc + 2, 0, sizeof(int), st));
  k_ens_init<<<1, 256, 0, st>>>(e->n_dev, e->B, misc);  // the group maximum it raises is already at least as high
  PRS_CUDA(cudaGetLastError());
  PRS_CUDA(cudaMemcpyAsync(&n, misc + 2, sizeof(int), cudaMemcpyDeviceToHost, st));
  PRS_CUDA(cudaStreamSynchronize(st));
  e->room = (long long)e->capacity - n;
  return PRS_OK;
}

extern "C" int prs_ens_destroy(prs_ens_plan* e) {
  if (e) {
    for (int i = 0; i < 6; ++i)
      if (e->ready[i]) cudaGraphExecDestroy(e->exec[i]);
    if (e->side) cudaStreamDestroy(e->side);
    if (e->ev_fork) cudaEventDestroy(e->ev_fork);
    if (e->ev_join) cudaEventDestroy(e->ev_join);
    delete e;
  }
  return PRS_OK;
}

extern "C" int prs_ens_run(prs_ens_plan* e, const uint8_t* const* frames, const double* odom, const uint8_t* gate,
                           const int* n_images, int T, prs_frame_result* results, void* stream) {
  PRS_REQUIRE(e && T >= 0 && n_images && (T == 0 || (frames && odom && gate && results)), "prs_ens_run: bad argument");
  PRS_REQUIRE(stream != nullptr, "prs_ens_run: needs a non-default stream (the ticks replay as CUDA graphs)");
  const int R = e->R;
  // slots[t][r]: recording r's image at tick t, counted from the first image of t's chunk; -1 = none
  const EnsScratch& M = e->lay;
  PRS_REQUIRE(!e->act || T <= M.chunk, "prs_ens_run: with the activity capture on, a run takes at most %d ticks, got %d",
              M.chunk, T);
  std::vector<int> slots((size_t)T * R);
  std::vector<uint8_t> variant(T), has_image(T);
  std::vector<int> seen(R, 0), in_chunk(R, 0);
  long long image_ticks = 0;
  for (int t = 0; t < T; ++t) {
    if (t % M.chunk == 0) std::fill(in_chunk.begin(), in_chunk.end(), 0);
    bool any = false, all = true, img = false;
    for (int r = 0; r < R; ++r) {
      const uint8_t g = gate[(size_t)t * R + r];
      const bool here = (g & 1) != 0, mv = (g & 2) != 0;
      slots[(size_t)t * R + r] = here ? in_chunk[r]++ : -1;
      seen[r] += here ? 1 : 0;
      img |= here;
      any |= mv;
      all &= mv;
    }
    variant[t] = (uint8_t)(!any ? 0 : all ? 1 : 2);
    has_image[t] = img ? 1 : 0;
    image_ticks += img ? 1 : 0;
  }
  for (int r = 0; r < R; ++r)
    PRS_REQUIRE(n_images[r] == seen[r] && (seen[r] == 0 || frames[r]),
                "prs_ens_run: recording %d has %d images in its gate, n_images says %d (or no frames)", r, seen[r],
                n_images[r]);
  PRS_REQUIRE(image_ticks <= e->room,
              "prs_ens_run: %lld ticks with images do not fit the libraries (room for %lld more templates)",
              image_ticks, e->room);
  if (int rc = prs_pc_check_device(e->pc, "prs_ens_run")) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  char* ms = e->scratch;
  const size_t rec_bytes = (size_t)e->B * sizeof(prs_frame_result);
  std::vector<long long> first(R, 0);  // each recording's first image of the chunk
  int rc = PRS_OK;
  e->act_ticks = 0;
  for (int c0 = 0; c0 < T && rc == PRS_OK; c0 += M.chunk) {
    const int n = T - c0 < M.chunk ? T - c0 : M.chunk;
    long long img_ticks = 0;
    for (int t = c0; t < c0 + n; ++t) img_ticks += has_image[t];
    for (int r = 0; r < R; ++r) {
      int nr = 0;
      for (int t = c0; t < c0 + n; ++t) nr += slots[(size_t)t * R + r] >= 0 ? 1 : 0;
      if (nr > 0)
        PRS_CUDA(cudaMemcpyAsync(ms + M.frames + (size_t)r * M.chunk * e->fbytes, frames[r] + first[r] * e->fbytes,
                                 (size_t)nr * e->fbytes, cudaMemcpyHostToDevice, st));
      first[r] += nr;
    }
    PRS_CUDA(cudaMemcpyAsync(ms + M.odom_chunk, odom + (size_t)c0 * R * 2, (size_t)n * R * 2 * sizeof(double),
                             cudaMemcpyHostToDevice, st));
    PRS_CUDA(cudaMemcpyAsync(ms + M.gate, gate + (size_t)c0 * R, (size_t)n * R, cudaMemcpyHostToDevice, st));
    PRS_CUDA(cudaMemcpyAsync(ms + M.slots, slots.data() + (size_t)c0 * R, (size_t)n * R * sizeof(int),
                             cudaMemcpyHostToDevice, st));
    PRS_CUDA(cudaMemsetAsync(ms + M.misc, 0, sizeof(int), st));  // the tick counter
    int done = 0;
    for (; done < n; ++done) {
      rc = ens_tick_launch(e, variant[c0 + done], has_image[c0 + done] != 0, st);
      if (rc != PRS_OK) break;
    }
    if (done > 0)
      PRS_CUDA(cudaMemcpyAsync(results + (size_t)c0 * e->B, ms + M.rec, (size_t)done * rec_bytes, cudaMemcpyDeviceToHost,
                               st));
    e->room -= img_ticks;
    e->act_ticks = done;
  }
  const cudaError_t err = cudaStreamSynchronize(st);
  if (rc == PRS_OK && err != cudaSuccess) {
    prs_set_error("prs_ens_run: %s", cudaGetErrorString(err));
    return PRS_E_CUDA;
  }
  return rc;
}

extern "C" int prs_ens_chunk(prs_ens_plan* e) { return e ? e->lay.chunk : 0; }

extern "C" size_t prs_ens_activity_bytes(prs_ens_plan* e, int max_cells) {
  if (!e || max_cells < 0 || max_cells > e->pc->N) return 0;
  return EnsActivity(e->B, e->lay.chunk, max_cells, e->pc->dtype == PRS_F32 ? 4 : 8).bytes;
}

// Turning the capture on or off, or changing its threshold or cells per entry, adds or changes a node of the image
// ticks: the captured graphs go, as in prs_frame_set_inject.
extern "C" int prs_ens_set_activity(prs_ens_plan* e, double threshold, int max_cells, void* buffer) {
  PRS_REQUIRE(e, "prs_ens_set_activity: null plan");
  if (buffer != nullptr) {
    PRS_REQUIRE(std::isfinite(threshold), "prs_ens_set_activity: the threshold must be finite, got %g", threshold);
    PRS_REQUIRE(max_cells >= 0 && max_cells <= e->pc->N,
                "prs_ens_set_activity: max_cells %d outside [0, %lld]", max_cells, (long long)e->pc->N);
  }
  for (int i = 0; i < 6; ++i) {
    if (e->ready[i]) cudaGraphExecDestroy(e->exec[i]);
    e->ready[i] = false;
    e->warm[i] = 0;
  }
  e->act = (char*)buffer;
  e->act_thr = buffer ? threshold : 0.0;
  e->act_k = buffer ? max_cells : 0;
  e->act_ticks = 0;
  return PRS_OK;
}

extern "C" int prs_ens_activity_pack(prs_ens_plan* e, int* counts, long long* total, void* stream) {
  PRS_REQUIRE(e && e->act && counts && total && stream, "prs_ens_activity_pack: bad argument (or no capture)");
  const cudaStream_t st = (cudaStream_t)stream;
  const int es = e->pc->dtype == PRS_F32 ? 4 : 8;
  const EnsActivity A(e->B, e->lay.chunk, e->act_k, es);
  const long long n = (long long)e->act_ticks * e->B;
  char* a = e->act;
  *total = 0;
  if (n == 0) return PRS_OK;
  k_ens_activity_scan<<<1, kActScanThreads, 0, st>>>((int*)(a + A.counts), (const uint8_t*)(e->scratch + e->lay.gate), e->rec_of,
                                          e->R, e->B, n, e->act_k, (long long*)(a + A.off));
  PRS_CUDA(cudaGetLastError());
  if (e->act_k > 0) {
    const unsigned grid = (unsigned)((n * 32 + 255) / 256);
    if (es == 4)
      k_ens_activity_gather<float><<<grid, 256, 0, st>>>((const int*)(a + A.counts), (const long long*)(a + A.off),
                                                         (const int*)(a + A.idx), (const float*)(a + A.val), n, e->act_k,
                                                         (int*)(a + A.pidx), (float*)(a + A.pval));
    else
      k_ens_activity_gather<double><<<grid, 256, 0, st>>>((const int*)(a + A.counts), (const long long*)(a + A.off),
                                                          (const int*)(a + A.idx), (const double*)(a + A.val), n,
                                                          e->act_k, (int*)(a + A.pidx), (double*)(a + A.pval));
    PRS_CUDA(cudaGetLastError());
  }
  PRS_CUDA(cudaMemcpyAsync(counts, a + A.counts, (size_t)n * sizeof(int), cudaMemcpyDeviceToHost, st));
  PRS_CUDA(cudaMemcpyAsync(total, a + A.off + (size_t)n * sizeof(long long), sizeof(long long), cudaMemcpyDeviceToHost,
                           st));
  PRS_CUDA(cudaStreamSynchronize(st));
  return PRS_OK;
}

extern "C" int prs_ens_activity_copy(prs_ens_plan* e, long long n, int* idx, void* val, void* stream) {
  PRS_REQUIRE(e && e->act && n >= 0 && (n == 0 || (idx && val)) && stream, "prs_ens_activity_copy: bad argument");
  PRS_REQUIRE(n <= (long long)e->act_ticks * e->B * e->act_k, "prs_ens_activity_copy: %lld cells, the run kept at most %lld",
              n, (long long)e->act_ticks * e->B * e->act_k);
  if (n == 0) return PRS_OK;
  const cudaStream_t st = (cudaStream_t)stream;
  const int es = e->pc->dtype == PRS_F32 ? 4 : 8;
  const EnsActivity A(e->B, e->lay.chunk, e->act_k, es);
  PRS_CUDA(cudaMemcpyAsync(idx, e->act + A.pidx, (size_t)n * sizeof(int), cudaMemcpyDeviceToHost, st));
  PRS_CUDA(cudaMemcpyAsync(val, e->act + A.pval, (size_t)n * es, cudaMemcpyDeviceToHost, st));
  PRS_CUDA(cudaStreamSynchronize(st));
  return PRS_OK;
}

// ---------------------------------------------------------------------------------------------
// Agent copies inside a plan's buffers (prs_ens_copy_agents, EnsembleSession.reassign).  A row's live data: its state
// slice, its pc_work slots, n_dev, the library groups of its n templates and the first n entries of its location row.
// Slots past n are never read (the sweep masks lanes >= n) and an append writes its slot whole (vt_pack_row: all 32
// plane rows and row sums of its lane), so the destination's stale tail needs no clearing.  The stage holds K rows with
// room for the largest live count among them.
struct EnsRows {
  char* state;  // [rows][state bytes]
  long long* argmax;
  char* total;  // 8-byte slots; a float32 plan's totals are 4-byte elements of the region
  int* err;
  int* n;
  char* lib;            // [rows][lib_bytes]
  long long lib_bytes;
  long long* loc;       // [rows][loc_stride]
  long long loc_stride;
};

struct EnsCopyStage {
  size_t table = 0, state = 0, argmax = 0, total = 0, err = 0, n = 0, lib = 0, loc = 0, bytes = 0;
  int max_n = 0;
  EnsCopyStage(int K, size_t table_ints, size_t net_bytes, int max_n_) : max_n(max_n_) {
    auto up = [](size_t v) { return (v + 255) & ~(size_t)255; };
    state = up(table_ints * sizeof(int));
    argmax = state + up((size_t)K * net_bytes);
    total = argmax + up((size_t)K * 8);
    err = total + up((size_t)K * 8);
    n = err + up((size_t)K * 4);
    lib = n + up((size_t)K * 4);
    loc = lib + up((size_t)K * prs_vt_packed_bytes(max_n));
    bytes = loc + up((size_t)K * max_n * 8);
  }
  EnsRows rows(char* p) const {
    return EnsRows{p + state, (long long*)(p + argmax), p + total, (int*)(p + err), (int*)(p + n), p + lib,
                   (long long)prs_vt_packed_bytes(max_n), (long long*)(p + loc), max_n};
  }
};

// Pair m copies row src_row[m] of `src` into row dst_row[m] of `dst`: blockIdx.y strides over the pairs, the blocks
// along x share each region of a pair.  The live count is the source's n_dev, at most max_n (the stage's room).  No
// pair's destination is another pair's source within one launch.
template <typename W>
__global__ void __launch_bounds__(256)
    k_ens_copy_rows(EnsRows src, EnsRows dst, const int* __restrict__ pairs, int n_pairs, long long state_words,
                    int total_bytes, int max_n) {
  const long long i0 = (long long)blockIdx.x * blockDim.x + threadIdx.x, step = (long long)gridDim.x * blockDim.x;
  for (int m = blockIdx.y; m < n_pairs; m += gridDim.y) {
    const int s = pairs[m], d = pairs[n_pairs + m];
    const int n = min(src.n[s], max_n);
    const W* ss = (const W*)src.state + s * state_words;
    W* ds = (W*)dst.state + d * state_words;
    for (long long i = i0; i < state_words; i += step) ds[i] = ss[i];
    const long long lib_u4 = (long long)((n + 31) >> 5) * kVtGroupU4;
    const uint4* sl = (const uint4*)(src.lib + s * src.lib_bytes);
    uint4* dl = (uint4*)(dst.lib + d * dst.lib_bytes);
    for (long long i = i0; i < lib_u4; i += step) dl[i] = sl[i];
    for (long long i = i0; i < n; i += step) dst.loc[d * dst.loc_stride + i] = src.loc[s * src.loc_stride + i];
    if (blockIdx.x == 0 && threadIdx.x == 0) {
      dst.argmax[d] = src.argmax[s];
      if (total_bytes == 4)
        ((int*)dst.total)[d] = ((const int*)src.total)[s];
      else
        ((long long*)dst.total)[d] = ((const long long*)src.total)[s];
      dst.err[d] = src.err[s];
      dst.n[d] = n;
    }
  }
}

static int ens_copy_plan(const char* who, prs_ens_plan* e, int n_moves, const int* dst, const int* src,
                         const int* n_templates, AgentMoves& mv, int& max_n) {
  PRS_REQUIRE(e && (n_moves == 0 || n_templates), "%s: bad argument", who);
  if (int rc = agent_moves(who, e->B, n_moves, dst, src, mv)) return rc;
  max_n = 0;
  for (int m = 0; m < n_moves; ++m) {
    const int n = n_templates[src[m]];
    PRS_REQUIRE(n >= 0 && n <= e->capacity, "%s: row %d holds %d templates, the capacity is %d", who, src[m], n,
                e->capacity);
  }
  for (int r : mv.stage_rows) max_n = std::max(max_n, n_templates[r]);
  return PRS_OK;
}

extern "C" size_t prs_ens_copy_stage_bytes(prs_ens_plan* e, int n_moves, const int* dst, const int* src,
                                           const int* n_templates) {
  AgentMoves mv;
  int max_n = 0;
  if (ens_copy_plan("prs_ens_copy_stage_bytes", e, n_moves, dst, src, n_templates, mv, max_n)) return 0;
  return EnsCopyStage(mv.K(), mv.table().size(), ens_net_bytes(e->pc), max_n).bytes;
}

// The plan's own rows as a copy source or destination.
static EnsRows ens_plan_rows(const prs_ens_plan* e) {
  const int B = e->B;
  return EnsRows{(char*)e->pc_state, (long long*)e->pc_work, (char*)e->pc_work + 8 * (size_t)B,
                 (int*)((char*)e->pc_work + 16 * (size_t)B), e->n_dev, (char*)e->libs, e->lib_u4 * 16, e->loc_dev,
                 e->capacity};
}

// One k_ens_copy_rows launch over n_pairs pairs whose live counts are at most `bound`.
static cudaError_t ens_copy_launch(const prs_ens_plan* e, const EnsRows& from, const EnsRows& to, const int* pairs,
                                   int n_pairs, int bound, cudaStream_t st) {
  if (n_pairs == 0) return cudaSuccess;
  const size_t net_bytes = ens_net_bytes(e->pc);
  const bool wide = net_bytes % 16 == 0;
  const long long state_words = (long long)(net_bytes / (wide ? 16 : 4));
  const int es = e->pc->dtype == PRS_F32 ? 4 : 8;
  // about 16 blocks per SM over all pairs, no more along x than a pair's largest region takes
  const long long words = std::max((long long)((bound + 31) >> 5) * kVtGroupU4, state_words);
  long long gx = (148LL * 16 + n_pairs - 1) / n_pairs;
  gx = std::max(1LL, std::min(gx, (words + 1023) / 1024));
  const dim3 grid((unsigned)gx, (unsigned)std::min(n_pairs, 65535));
  if (wide)
    k_ens_copy_rows<uint4><<<grid, 256, 0, st>>>(from, to, pairs, n_pairs, state_words, es, bound);
  else
    k_ens_copy_rows<unsigned><<<grid, 256, 0, st>>>(from, to, pairs, n_pairs, state_words, es, bound);
  return cudaGetLastError();
}

extern "C" int prs_ens_copy_agents(prs_ens_plan* e, int n_moves, const int* dst, const int* src, const int* n_templates,
                                   void* stage, size_t stage_bytes, void* stream) {
  AgentMoves mv;
  int max_n = 0;
  if (int rc = ens_copy_plan("prs_ens_copy_agents", e, n_moves, dst, src, n_templates, mv, max_n)) return rc;
  if (n_moves == 0) return PRS_OK;
  const std::vector<int> table = mv.table();
  const EnsCopyStage L(mv.K(), table.size(), ens_net_bytes(e->pc), max_n);
  PRS_REQUIRE(stage && stage_bytes >= L.bytes, "prs_ens_copy_agents: the stage has %zu bytes, the moves need %zu",
              stage_bytes, L.bytes);
  if (int rc = prs_pc_check_device(e->pc, "prs_ens_copy_agents")) return rc;
  const cudaStream_t st = (cudaStream_t)stream;
  char* p = (char*)stage;
  PRS_CUDA(cudaMemcpyAsync(p, table.data(), table.size() * sizeof(int), cudaMemcpyHostToDevice, st));
  const EnsRows plan = ens_plan_rows(e), rows = L.rows(p);
  const int* d_table = (const int*)p;
  const int K = mv.K(), n_direct = (int)mv.direct.size() / 2, n_staged = (int)mv.staged.size() / 2;
  PRS_CUDA(ens_copy_launch(e, plan, rows, d_table, K, max_n, st));
  PRS_CUDA(ens_copy_launch(e, plan, plan, d_table + 2 * K, n_direct, e->capacity, st));
  PRS_CUDA(ens_copy_launch(e, rows, plan, d_table + 2 * K + 2 * n_direct, n_staged, max_n, st));
  return prs_pc_active_invalidate(e->pc, st);  // the carried lists describe the rows as they were
}

// ---------------------------------------------------------------------------------------------
// Agents carried between plans (prs_ens_export_agents / prs_ens_import_agents: a session's agents reassigned across
// devices).  The stage is EnsCopyStage's layout for K rows, its table region holding a header that describes the rows
// -- so it depends on no plan -- then the export's and the import's pair tables.
namespace {
constexpr int kEnsStageMagic = 0x50525345;  // "ESRP"
constexpr int kStageHeaderInts = 16;
struct EnsStageHeader {
  int magic, K, max_n, dtype, X, Y, Th, pad;
  long long net_bytes, bytes;
};
static_assert(sizeof(EnsStageHeader) <= kStageHeaderInts * sizeof(int), "stage header");
EnsCopyStage ens_transfer_stage(int K, size_t net_bytes, int max_n) {
  return EnsCopyStage(K, kStageHeaderInts + 4 * (size_t)K, net_bytes, max_n);
}
}  // namespace

static int ens_export_check(const char* who, prs_ens_plan* e, int n, const int* rows, const int* n_templates,
                            int& max_n) {
  PRS_REQUIRE(e && n >= 0 && (n == 0 || (rows && n_templates)), "%s: bad argument", who);
  max_n = 0;
  for (int k = 0; k < n; ++k) {
    PRS_REQUIRE(rows[k] >= 0 && rows[k] < e->B, "%s: row %d outside [0, %d)", who, rows[k], e->B);
    const int c = n_templates[rows[k]];
    PRS_REQUIRE(c >= 0 && c <= e->capacity, "%s: row %d holds %d templates, the capacity is %d", who, rows[k], c,
                e->capacity);
    max_n = std::max(max_n, c);
  }
  return PRS_OK;
}

extern "C" size_t prs_ens_export_stage_bytes(prs_ens_plan* e, int n, const int* rows, const int* n_templates) {
  int max_n = 0;
  if (ens_export_check("prs_ens_export_stage_bytes", e, n, rows, n_templates, max_n) || n == 0) return 0;
  return ens_transfer_stage(n, ens_net_bytes(e->pc), max_n).bytes;
}

extern "C" int prs_ens_export_agents(prs_ens_plan* e, int n, const int* rows, const int* n_templates, void* stage,
                                     size_t stage_bytes, void* stream) {
  int max_n = 0;
  if (int rc = ens_export_check("prs_ens_export_agents", e, n, rows, n_templates, max_n)) return rc;
  if (n == 0) return PRS_OK;
  const size_t net_bytes = ens_net_bytes(e->pc);
  const EnsCopyStage L = ens_transfer_stage(n, net_bytes, max_n);
  PRS_REQUIRE(stage && stage_bytes >= L.bytes, "prs_ens_export_agents: the stage has %zu bytes, the rows need %zu",
              stage_bytes, L.bytes);
  if (int rc = prs_pc_check_device(e->pc, "prs_ens_export_agents")) return rc;
  std::vector<int> table(kStageHeaderInts + 2 * (size_t)n, 0);
  const EnsStageHeader h{kEnsStageMagic, n, max_n, e->pc->dtype, e->pc->X, e->pc->Y, e->pc->Th, 0,
                         (long long)net_bytes, (long long)L.bytes};
  memcpy(table.data(), &h, sizeof(h));
  for (int k = 0; k < n; ++k) {  // plan row rows[k] -> stage row k (a row may be exported more than once)
    table[kStageHeaderInts + k] = rows[k];
    table[kStageHeaderInts + n + k] = k;
  }
  const cudaStream_t st = (cudaStream_t)stream;
  char* p = (char*)stage;
  PRS_CUDA(cudaMemcpyAsync(p, table.data(), table.size() * sizeof(int), cudaMemcpyHostToDevice, st));
  PRS_CUDA(ens_copy_launch(e, ens_plan_rows(e), L.rows(p), (const int*)p + kStageHeaderInts, n, max_n, st));
  return PRS_OK;
}

extern "C" int prs_ens_import_agents(prs_ens_plan* e, int n, const int* rows, const void* stage, size_t stage_bytes,
                                     void* stream) {
  PRS_REQUIRE(e && n >= 0 && (n == 0 || (rows && stage)), "prs_ens_import_agents: bad argument");
  if (n == 0) return PRS_OK;
  std::vector<int> seen(e->B, 0);
  for (int k = 0; k < n; ++k) {
    PRS_REQUIRE(rows[k] >= 0 && rows[k] < e->B && !seen[rows[k]],
                "prs_ens_import_agents: row %d outside [0, %d) or imported twice", rows[k], e->B);
    seen[rows[k]] = 1;
  }
  if (int rc = prs_pc_check_device(e->pc, "prs_ens_import_agents")) return rc;
  const cudaStream_t st = (cudaStream_t)stream;
  EnsStageHeader h;
  PRS_REQUIRE(stage_bytes >= sizeof(h), "prs_ens_import_agents: the stage has %zu bytes", stage_bytes);
  PRS_CUDA(cudaMemcpyAsync(&h, stage, sizeof(h), cudaMemcpyDeviceToHost, st));
  PRS_CUDA(cudaStreamSynchronize(st));
  const size_t net_bytes = ens_net_bytes(e->pc);
  PRS_REQUIRE(h.magic == kEnsStageMagic && h.K == n && (size_t)h.bytes <= stage_bytes,
              "prs_ens_import_agents: the stage does not hold %d exported rows", n);
  PRS_REQUIRE(h.dtype == e->pc->dtype && h.X == e->pc->X && h.Y == e->pc->Y && h.Th == e->pc->Th &&
                  (size_t)h.net_bytes == net_bytes,
              "prs_ens_import_agents: the stage holds %d x %d x %d networks of dtype %d, the plan %d x %d x %d of dtype %d",
              h.X, h.Y, h.Th, h.dtype, e->pc->X, e->pc->Y, e->pc->Th, e->pc->dtype);
  PRS_REQUIRE(h.max_n >= 0 && h.max_n <= e->capacity,
              "prs_ens_import_agents: a staged row holds %d templates, the capacity is %d", h.max_n, e->capacity);
  const EnsCopyStage L = ens_transfer_stage(n, net_bytes, h.max_n);
  std::vector<int> pairs(2 * (size_t)n);
  for (int k = 0; k < n; ++k) {  // stage row k -> plan row rows[k]
    pairs[k] = k;
    pairs[n + k] = rows[k];
  }
  char* p = (char*)stage;
  int* d_pairs = (int*)p + kStageHeaderInts + 2 * n;
  PRS_CUDA(cudaMemcpyAsync(d_pairs, pairs.data(), pairs.size() * sizeof(int), cudaMemcpyHostToDevice, st));
  PRS_CUDA(ens_copy_launch(e, L.rows(p), ens_plan_rows(e), d_pairs, n, h.max_n, st));
  // an imported row may hold more templates than any row had: the sweep's group bound and the room follow it
  k_ens_init<<<1, 256, 0, st>>>(e->n_dev, e->B, (int*)(e->scratch + e->lay.misc));
  PRS_CUDA(cudaGetLastError());
  e->room = std::min(e->room, (long long)e->capacity - h.max_n);
  return prs_pc_active_invalidate(e->pc, st);  // the carried lists describe the rows as they were
}

extern "C" int prs_stage_copy(void* dst, int dst_device, const void* src, int src_device, size_t bytes, void* stream) {
  PRS_REQUIRE((bytes == 0 || (dst && src)) && dst_device >= 0 && src_device >= 0, "prs_stage_copy: bad argument");
  if (bytes == 0) return PRS_OK;
  const cudaStream_t st = (cudaStream_t)stream;
  if (dst_device == src_device)
    PRS_CUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToDevice, st));
  else
    PRS_CUDA(cudaMemcpyPeerAsync(dst, dst_device, src, src_device, bytes, st));
  return PRS_OK;
}
