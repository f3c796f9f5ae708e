// Generic pose-cell update: any grid shape, float or double, any batch.
//
// One PoseCellNetwork.update() (ratslam/posecell_network.py:326-353) as a short
// sequence of kernels over the theta-major state [B][Th][X][Y] kept in HBM/L2:
//
//   k_plan         odometry -> integer origins, LUT filter choice, theta origin   (:252-267,249,304)
//   k_dog_theta    E,I = ge*P, gi*P along theta   \  the 7x7x7 DoG correlate of :336 (convolution.py
//   k_dog_y        E,I along y                     > :228-246) as separable E - I: kernel_3d ==
//   k_dog_x_inhib  A = aE*E - aI*I, inhibited     /  aE ge(x)ge(x)ge - aI gi(x)gi(x)gi; inhibition :339-340,
//                  + per-block partial sums                                        sum for :343
//   k_sum_final    total, 1/total                                                  (:343-345)
//   k_shift2d      per-plane shifted 7x7 correlate, * 1/total, clamp               (:273-274,300; convolution.py:320-340)
//   k_theta_final  7-tap theta correlate, clamp, per-block arg-max                 (:304-314; convolution.py:344-359)
//   k_argmax_final first maximum in the reference's C order [x][y][th]             (:317-319)
//
// The normalisation is applied after the 2-D stage instead of before it: every
// operation in between is linear or a clamp at zero, so only rounding differs.
// This path is the strict-parity (float64) implementation and the one used for
// shapes the fused SMEM-resident kernel (posecell_resident.cu) does not cover.
#include "common.cuh"

namespace {

constexpr int kThreads = 256;

// Which network a block works on.  Normally blockIdx.z (or .x) itself.  As the dense fall-back of the active-set path
// (posecell_active.cu) the grid has only kFallbackSlots entries in that dimension and walks the device-side list of flagged
// networks: a grid sized for all B networks costs 0.5 ns per block that merely finds out it has nothing to do -- 0.7 ms per
// update for 2600 networks of 50x50x10.
constexpr int kFallbackSlots = 32;
#define PRS_NET_LOOP(bz, dim)                                                                \
  const int n_work_ = only_cnt != nullptr ? *only_cnt : (int)gridDim.dim;                    \
  for (int slot_ = blockIdx.dim; slot_ < n_work_; slot_ += gridDim.dim)                      \
    if (const int bz = only_list != nullptr ? only_list[slot_] : slot_; true)

template <typename T>
__device__ __forceinline__ T fma_t(T a, T b, T c);
template <>
__device__ __forceinline__ float fma_t<float>(float a, float b, float c) { return fmaf(a, b, c); }
template <>
__device__ __forceinline__ double fma_t<double>(double a, double b, double c) { return fma(a, b, c); }

// ---------------------------------------------------------------------------
// Decisions of one path-integration step, bit-for-bit the float64 arithmetic numpy does on the host
// (explicit _rn intrinsics keep the compiler from contracting mul+sub into an FMA).
__global__ void k_plan(const double* __restrict__ odom, const double* __restrict__ cos_th,
                       const double* __restrict__ sin_th, int B, int Th, int minXY, double vtrans_scale,
                       double vrot_scale, int* __restrict__ shift, unsigned char* __restrict__ fsel,
                       int* __restrict__ ogi, int* __restrict__ err) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B * Th) return;
  prs_plan_cell(i / Th, i % Th, Th, minXY, odom, cos_th, sin_th, vtrans_scale, vrot_scale, shift, fsel, ogi, err);
}

// ---------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(kThreads) k_dog_theta(const T* __restrict__ P, T* __restrict__ E, T* __restrict__ I,
                                                        int XY, int Th, PcTables<T> tab,
                                                        const int* __restrict__ only_list, const int* __restrict__ only_cnt) {
  int p = blockIdx.x * kThreads + threadIdx.x;
  if (p >= XY) return;
  int k = blockIdx.y;
  PRS_NET_LOOP(bz, z) {
    size_t base = (size_t)bz * Th * XY;
    T e = 0, i = 0;
#pragma unroll
    for (int t = 0; t < 7; ++t) {
      int kk = wrap1(k + t - 3, Th);
      T v = P[base + (size_t)kk * XY + p];
      e = fma_t(tab.ge[t], v, e);
      i = fma_t(tab.gi[t], v, i);
    }
    size_t o = base + (size_t)k * XY + p;
    E[o] = e;
    I[o] = i;
  }
}

template <typename T>
__global__ void __launch_bounds__(kThreads) k_dog_y(const T* __restrict__ Ei, const T* __restrict__ Ii, T* __restrict__ E,
                                                    T* __restrict__ I, int X, int Y, int Th, PcTables<T> tab,
                                                    const int* __restrict__ only_list,
                                                    const int* __restrict__ only_cnt) {
  int XY = X * Y;
  int p = blockIdx.x * kThreads + threadIdx.x;
  if (p >= XY) return;
  int x = p / Y, y = p - x * Y;
  PRS_NET_LOOP(bz, z) {
    size_t row = ((size_t)bz * Th + blockIdx.y) * XY + (size_t)x * Y;
    T e = 0, i = 0;
#pragma unroll
    for (int t = 0; t < 7; ++t) {
      int yy = wrap1(y + t - 3, Y);
      e = fma_t(tab.ge[t], Ei[row + yy], e);
      i = fma_t(tab.gi[t], Ii[row + yy], i);
    }
    E[row + y] = e;
    I[row + y] = i;
  }
}

template <typename T>
__device__ __forceinline__ T block_sum(T v, T* sm) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
  int w = threadIdx.x >> 5, l = threadIdx.x & 31;
  if (l == 0) sm[w] = v;
  __syncthreads();
  if (w == 0) {
    v = l < (kThreads / 32) ? sm[l] : T(0);
#pragma unroll
    for (int o = 4; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
  }
  return v;  // valid in thread 0
}

template <typename T>
__global__ void __launch_bounds__(kThreads)
    k_dog_x_inhib(const T* __restrict__ Ei, const T* __restrict__ Ii, T* __restrict__ A, const T* __restrict__ gi, int X,
                  int Y, int Th, PcTables<T> tab, T* __restrict__ part, const int* __restrict__ only_list,
                  const int* __restrict__ only_cnt) {
  __shared__ T sm[kThreads / 32];
  int XY = X * Y;
  int p = blockIdx.x * kThreads + threadIdx.x;
  PRS_NET_LOOP(bz, z) {
    T a = 0;
    if (p < XY) {
      int x = p / Y, y = p - x * Y;
      size_t plane = ((size_t)bz * Th + blockIdx.y) * XY;
      T e = 0, i = 0;
#pragma unroll
      for (int t = 0; t < 7; ++t) {
        int xx = wrap1(x + t - 3, X);
        e = fma_t(tab.gex[t], Ei[plane + (size_t)xx * Y + y], e);
        i = fma_t(tab.gix[t], Ii[plane + (size_t)xx * Y + y], i);
      }
      a = e - i;
      const T g = gi[bz];
      a = (a < g) ? inhib_floor(g) : a - g;  // posecell_network.py:339-340
      A[plane + p] = a;
    }
    T s = block_sum(a, sm);
    if (threadIdx.x == 0) part[((size_t)bz * Th + blockIdx.y) * gridDim.x + blockIdx.x] = s;
    __syncthreads();  // sm is reused by the next network of the list
  }
}

template <typename T>
__global__ void __launch_bounds__(kThreads) k_sum_final(const T* __restrict__ part, int np, T* __restrict__ total,
                                                        T* __restrict__ inv_total, const int* __restrict__ only_list,
                                                        const int* __restrict__ only_cnt) {
  __shared__ T sm[kThreads / 32];
  PRS_NET_LOOP(bz, x) {
    const T* p = part + (size_t)bz * np;
    T s = 0;
    for (int i = threadIdx.x; i < np; i += kThreads) s += p[i];
    s = block_sum(s, sm);
    if (threadIdx.x == 0) {
      total[bz] = s;
      inv_total[bz] = (s != T(0)) ? T(1) / s : T(1);  // posecell_network.py:344-345
    }
    __syncthreads();
  }
}

template <typename T>
__global__ void __launch_bounds__(kThreads)
    k_shift2d(const T* __restrict__ A, T* __restrict__ Bp, const int* __restrict__ shift,
              const unsigned char* __restrict__ fsel, const T* __restrict__ inv_total, int X, int Y, int Th,
              PcTables<T> tab, const int* __restrict__ only_list, const int* __restrict__ only_cnt) {
  int XY = X * Y;
  int p = blockIdx.x * kThreads + threadIdx.x;
  if (p >= XY) return;
  int x = p / Y, y = p - x * Y;
  PRS_NET_LOOP(bz, z) {
    int bk = bz * Th + blockIdx.y;
    size_t plane = (size_t)bk * XY;
    int ox = shift[2 * bk], oy = shift[2 * bk + 1];
    const T* F = tab.f2d[fsel[bk]];
    int xs[7], ys[7];
    int sx = modp(x + ox - 3, X), sy = modp(y + oy - 3, Y);
#pragma unroll
    for (int t = 0; t < 7; ++t) {
      xs[t] = (sx + t) % X;
      ys[t] = (sy + t) % Y;
    }
    T acc = 0;
#pragma unroll
    for (int a = 0; a < 7; ++a) {
      const T* row = A + plane + (size_t)xs[a] * Y;
#pragma unroll
      for (int b = 0; b < 7; ++b) acc = fma_t(F[a * 7 + b], row[ys[b]], acc);
    }
    acc *= inv_total[bz];
    Bp[plane + p] = (acc < T(0)) ? T(0) : acc;  // posecell_network.py:300
  }
}

template <typename T>
__device__ __forceinline__ void amax_combine(T& v, long long& i, T v2, long long i2) {
  if (v2 > v || (v2 == v && i2 < i)) {
    v = v2;
    i = i2;
  }
}

template <typename T>
__device__ __forceinline__ void block_argmax(T& v, long long& idx, T* smv, long long* smi) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    T v2 = __shfl_down_sync(0xffffffffu, v, o);
    long long i2 = __shfl_down_sync(0xffffffffu, idx, o);
    amax_combine(v, idx, v2, i2);
  }
  int w = threadIdx.x >> 5, l = threadIdx.x & 31;
  if (l == 0) {
    smv[w] = v;
    smi[w] = idx;
  }
  __syncthreads();
  if (w == 0) {
    if (l < kThreads / 32) {
      v = smv[l];
      idx = smi[l];
    } else {
      v = -INFINITY;
      idx = 0x7fffffffffffffffLL;
    }
#pragma unroll
    for (int o = 4; o > 0; o >>= 1) {
      T v2 = __shfl_down_sync(0xffffffffu, v, o);
      long long i2 = __shfl_down_sync(0xffffffffu, idx, o);
      amax_combine(v, idx, v2, i2);
    }
  }
}

// FINAL == true : theta correlate + clamp + store + partial arg-max (update step)
// FINAL == false: partial arg-max of an existing state (get_pc_max without update)
template <typename T, bool FINAL>
__global__ void __launch_bounds__(kThreads)
    k_theta_final(const T* __restrict__ Bp, T* __restrict__ S, const int* __restrict__ ogi, int X, int Y, int Th,
                  PcTables<T> tab, T* __restrict__ part_val, long long* __restrict__ part_idx,
                  const int* __restrict__ only_list, const int* __restrict__ only_cnt) {
  __shared__ T smv[kThreads / 32];
  __shared__ long long smi[kThreads / 32];
  int XY = X * Y;
  int p = blockIdx.x * kThreads + threadIdx.x;
  int k = blockIdx.y;
  PRS_NET_LOOP(bz, z) {
    size_t base = (size_t)bz * Th * XY;
    T c = -INFINITY;
    long long idx = 0x7fffffffffffffffLL;
    if (p < XY) {
      if (FINAL) {
        const T* f = tab.f1d[ogi[bz]];
        c = 0;
#pragma unroll
        for (int t = 0; t < 7; ++t) c = fma_t(f[t], Bp[base + (size_t)wrap1(k + t - 3, Th) * XY + p], c);
        c = (c < T(0)) ? T(0) : c;  // posecell_network.py:314
        S[base + (size_t)k * XY + p] = c;
      } else {
        c = Bp[base + (size_t)k * XY + p];
      }
      idx = (long long)p * Th + k;  // reference flat index (x*Y + y)*Th + th
    }
    block_argmax(c, idx, smv, smi);
    if (threadIdx.x == 0) {
      size_t o = ((size_t)bz * Th + blockIdx.y) * gridDim.x + blockIdx.x;
      part_val[o] = c;
      part_idx[o] = idx;
    }
    __syncthreads();  // smv / smi are reused by the next network of the list
  }
}

template <typename T>
__global__ void __launch_bounds__(kThreads) k_argmax_final(const T* __restrict__ part_val,
                                                           const long long* __restrict__ part_idx, int np,
                                                           long long* __restrict__ argmax,
                                                           const int* __restrict__ only_list,
                                                           const int* __restrict__ only_cnt) {
  __shared__ T smv[kThreads / 32];
  __shared__ long long smi[kThreads / 32];
  PRS_NET_LOOP(bz, x) {
    const T* pv = part_val + (size_t)bz * np;
    const long long* pi = part_idx + (size_t)bz * np;
    T v = -INFINITY;
    long long idx = 0x7fffffffffffffffLL;
    for (int i = threadIdx.x; i < np; i += kThreads) amax_combine(v, idx, pv[i], pi[i]);
    block_argmax(v, idx, smv, smi);
    if (threadIdx.x == 0) argmax[bz] = idx;
    __syncthreads();
  }
}

template <typename T>
__global__ void k_fill(T* p, int n, T v) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) p[i] = v;
}

template <typename T>
__global__ void k_inject(T* state, size_t off, size_t stride, int count, T energy) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < count) state[off + (size_t)i * stride] += energy;
}

// xyt[b][x][y][th]  <->  state[b][th][x][y]
template <typename T, bool IMPORT>
__global__ void __launch_bounds__(kThreads) k_transpose(T* __restrict__ state, T* __restrict__ xyt, int XY, int Th) {
  int p = blockIdx.x * kThreads + threadIdx.x;
  if (p >= XY) return;
  size_t base = (size_t)blockIdx.z * Th * XY;
  int k = blockIdx.y;
  if (IMPORT)
    state[base + (size_t)k * XY + p] = xyt[base + (size_t)p * Th + k];
  else
    xyt[base + (size_t)p * Th + k] = state[base + (size_t)k * XY + p];
}

template <typename T>
int generic_step_t(prs_pc_plan* p, const PcTables<T>& tab, T* state, const double* odom, const T* gi, long long* argmax,
                   T* total, int* err, cudaStream_t st) {
  const int X = p->X, Y = p->Y, Th = p->Th, B = p->B, XY = X * Y;
  dim3 grid(p->nblk_plane, Th, B);
  const int np = Th * p->nblk_plane;
  T *s1 = (T*)p->s1, *s2 = (T*)p->s2, *s3 = (T*)p->s3, *s4 = (T*)p->s4;
  int nbt = B * Th;
  // non-null while prs_pc_step runs this path as the active-set fall-back: a small grid walks the list of flagged networks
  const int *ol = p->only_list, *oc = p->only_cnt;
  if (ol != nullptr) grid.z = B < kFallbackSlots ? B : kFallbackSlots;
  const int nb1 = ol != nullptr ? (int)grid.z : B;
  k_plan<<<(nbt + 127) / 128, 128, 0, st>>>(odom, p->cos_th, p->sin_th, B, Th, X < Y ? X : Y, p->vtrans_scale,
                                            p->vrot_scale, p->shift, p->fsel, p->ogi, err);
  k_dog_theta<T><<<grid, kThreads, 0, st>>>(state, s1, s2, XY, Th, tab, ol, oc);
  k_dog_y<T><<<grid, kThreads, 0, st>>>(s1, s2, s3, s4, X, Y, Th, tab, ol, oc);
  k_dog_x_inhib<T><<<grid, kThreads, 0, st>>>(s3, s4, s1, gi, X, Y, Th, tab, (T*)p->part_val, ol, oc);
  k_sum_final<T><<<nb1, kThreads, 0, st>>>((const T*)p->part_val, np, total, (T*)p->inv_total, ol, oc);
  k_shift2d<T><<<grid, kThreads, 0, st>>>(s1, s2, p->shift, p->fsel, (const T*)p->inv_total, X, Y, Th, tab, ol, oc);
  k_theta_final<T, true><<<grid, kThreads, 0, st>>>(s2, state, p->ogi, X, Y, Th, tab, (T*)p->part_val, p->part_idx, ol, oc);
  k_argmax_final<T><<<nb1, kThreads, 0, st>>>((const T*)p->part_val, p->part_idx, np, argmax, ol, oc);
  PRS_CUDA(cudaGetLastError());
  return PRS_OK;
}

template <typename T>
int generic_path_integration_t(prs_pc_plan* p, const PcTables<T>& tab, T* state, const double* odom, int* err,
                               cudaStream_t st) {
  const int X = p->X, Y = p->Y, Th = p->Th, B = p->B;
  dim3 grid(p->nblk_plane, Th, B);
  int nbt = B * Th;
  k_plan<<<(nbt + 127) / 128, 128, 0, st>>>(odom, p->cos_th, p->sin_th, B, Th, X < Y ? X : Y, p->vtrans_scale,
                                            p->vrot_scale, p->shift, p->fsel, p->ogi, err);
  k_fill<T><<<(B + 127) / 128, 128, 0, st>>>((T*)p->inv_total, B, T(1));
  k_shift2d<T><<<grid, kThreads, 0, st>>>(state, (T*)p->s2, p->shift, p->fsel, (const T*)p->inv_total, X, Y, Th, tab, nullptr, nullptr);
  k_theta_final<T, true><<<grid, kThreads, 0, st>>>((const T*)p->s2, state, p->ogi, X, Y, Th, tab, (T*)p->part_val,
                                                    p->part_idx, nullptr, nullptr);
  PRS_CUDA(cudaGetLastError());
  return PRS_OK;
}

}  // namespace

int prs_pc_launch_plan(prs_pc_plan* p, const double* odom, int* err, cudaStream_t st) {
  const int nbt = p->B * p->Th;
  k_plan<<<(nbt + 127) / 128, 128, 0, st>>>(odom, p->cos_th, p->sin_th, p->B, p->Th, p->X < p->Y ? p->X : p->Y,
                                            p->vtrans_scale, p->vrot_scale, p->shift, p->fsel, p->ogi, err);
  PRS_CUDA(cudaGetLastError());
  return PRS_OK;
}

int prs_pc_launch_sum_final_f32(prs_pc_plan* p, int np, float* total, cudaStream_t st) {
  k_sum_final<float><<<p->B, kThreads, 0, st>>>((const float*)p->part_val, np, total, (float*)p->inv_total, nullptr, nullptr);
  PRS_CUDA(cudaGetLastError());
  return PRS_OK;
}

int prs_pc_launch_argmax_final_f32(prs_pc_plan* p, int np, long long* argmax, cudaStream_t st) {
  k_argmax_final<float><<<p->B, kThreads, 0, st>>>((const float*)p->part_val, p->part_idx, np, argmax, nullptr, nullptr);
  PRS_CUDA(cudaGetLastError());
  return PRS_OK;
}

int prs_pc_generic_path_integration(prs_pc_plan* p, void* state, const double* odom, int* err, cudaStream_t st) {
  if (p->dtype == PRS_F32) return generic_path_integration_t<float>(p, p->tf, (float*)state, odom, err, st);
  return generic_path_integration_t<double>(p, p->td, (double*)state, odom, err, st);
}

int prs_pc_generic_step(prs_pc_plan* p, void* state, const double* odom, const void* gi, long long* argmax, void* total,
                        int* err, cudaStream_t st) {
  if (p->dtype == PRS_F32)
    return generic_step_t<float>(p, p->tf, (float*)state, odom, (const float*)gi, argmax, (float*)total, err, st);
  return generic_step_t<double>(p, p->td, (double*)state, odom, (const double*)gi, argmax, (double*)total, err, st);
}

int prs_pc_generic_argmax(prs_pc_plan* p, const void* state, long long* argmax, cudaStream_t st) {
  dim3 grid(p->nblk_plane, p->Th, p->B);
  const int np = p->Th * p->nblk_plane;
  if (p->dtype == PRS_F32) {
    k_theta_final<float, false><<<grid, kThreads, 0, st>>>((const float*)state, nullptr, nullptr, p->X, p->Y, p->Th, p->tf,
                                                           (float*)p->part_val, p->part_idx, nullptr, nullptr);
    k_argmax_final<float><<<p->B, kThreads, 0, st>>>((const float*)p->part_val, p->part_idx, np, argmax, nullptr, nullptr);
  } else {
    k_theta_final<double, false><<<grid, kThreads, 0, st>>>((const double*)state, nullptr, nullptr, p->X, p->Y, p->Th,
                                                            p->td, (double*)p->part_val, p->part_idx, nullptr, nullptr);
    k_argmax_final<double><<<p->B, kThreads, 0, st>>>((const double*)p->part_val, p->part_idx, np, argmax, nullptr, nullptr);
  }
  PRS_CUDA(cudaGetLastError());
  return PRS_OK;
}

// ---------------------------------------------------------------------------- C ABI (shape-independent parts)
extern "C" int prs_pc_inject(prs_pc_handle h, void* state, int b, int x, int y, int th, double energy, void* stream) {
  PRS_REQUIRE(h && state, "prs_pc_inject: null argument");
  PRS_REQUIRE(b < h->B && x >= 0 && x < h->X && y >= 0 && y < h->Y && th >= 0 && th < h->Th,
              "prs_pc_inject: location (%d,%d,%d) of network %d is outside the %dx%dx%d grid", x, y, th, b, h->X, h->Y,
              h->Th);
  const int first = b < 0 ? 0 : b, count = b < 0 ? h->B : 1;
  size_t off = ((size_t)first * h->Th + th) * h->X * h->Y + (size_t)x * h->Y + y;
  cudaStream_t st = (cudaStream_t)stream;
  if (int rc_ = prs_pc_active_invalidate(h, st)) return rc_;
  if (h->dtype == PRS_F32)
    k_inject<float><<<(count + 127) / 128, 128, 0, st>>>((float*)state, off, (size_t)h->N, count, (float)energy);
  else
    k_inject<double><<<(count + 127) / 128, 128, 0, st>>>((double*)state, off, (size_t)h->N, count, energy);
  PRS_CUDA(cudaGetLastError());
  return PRS_OK;
}

// Cells of network b whose activity exceeds `thr`, in the reference's C order [x][y][th] -- what both viewers
// draw (simulate.py:61 `nonzero(pc > .002)`, ratslam_viewer.py:137).  Two passes keep the order deterministic:
// per-block counts, then an exclusive scan by block 0 and a compacting pass.
template <typename T>
__global__ void __launch_bounds__(256) k_active_count(const T* __restrict__ state, int XY, int Th, double thr,
                                                      int* __restrict__ counts) {
  // one block per 256 consecutive reference-order cells; cell c = (x*Y + y)*Th + th lives at state[th*XY + x*Y + y]
  const long long c = (long long)blockIdx.x * 256 + threadIdx.x;
  const long long N = (long long)XY * Th;
  int hit = 0;
  if (c < N) {
    const int th = (int)(c % Th);
    const long long p = c / Th;
    hit = ((double)state[(size_t)th * XY + p] > thr) ? 1 : 0;
  }
  const int total = __syncthreads_count(hit);
  if (threadIdx.x == 0) counts[blockIdx.x] = total;
}

template <typename T>
__global__ void __launch_bounds__(256) k_active_write(const T* __restrict__ state, int XY, int Th, double thr,
                                                      const int* __restrict__ offsets, int max_out,
                                                      int* __restrict__ idx_out, T* __restrict__ val_out) {
  __shared__ int s_warp[8];
  const long long c = (long long)blockIdx.x * 256 + threadIdx.x;
  const long long N = (long long)XY * Th;
  T v = 0;
  int hit = 0;
  if (c < N) {
    const int th = (int)(c % Th);
    const long long p = c / Th;
    v = state[(size_t)th * XY + p];
    hit = ((double)v > thr) ? 1 : 0;
  }
  const unsigned bal = __ballot_sync(0xffffffffu, hit);
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  if (lane == 0) s_warp[w] = __popc(bal);
  __syncthreads();
  int base = offsets[blockIdx.x];
  for (int i = 0; i < w; ++i) base += s_warp[i];
  const int pos = base + __popc(bal & ((1u << lane) - 1));
  if (hit && pos < max_out) {
    idx_out[pos] = (int)c;
    val_out[pos] = v;
  }
}

__global__ void k_exclusive_scan_small(const int* __restrict__ counts, int n, int* __restrict__ offsets,
                                       int* __restrict__ total) {
  // single thread block, sequential chunks: n is (cells / 256), at most a few tens of thousands
  __shared__ int s_part[256];
  const int per = (n + 255) / 256;
  const int lo = threadIdx.x * per, hi = min(n, lo + per);
  int s = 0;
  for (int i = lo; i < hi; ++i) s += counts[i];
  s_part[threadIdx.x] = s;
  __syncthreads();
  int base = 0;
  for (int i = 0; i < threadIdx.x; ++i) base += s_part[i];
  for (int i = lo; i < hi; ++i) {
    offsets[i] = base;
    base += counts[i];
  }
  if (threadIdx.x == 255) *total = base;
}

__global__ void k_unravel_pack(const long long* __restrict__ argmax, const int* __restrict__ err, int B, int Y, int Th,
                               int4* __restrict__ out) {
  int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  const long long f = argmax[b];
  const int th = (int)(f % Th);
  const long long xy = f / Th;
  out[b] = make_int4((int)(xy / Y), (int)(xy % Y), th, err[b]);
}

int prs_pc_launch_unravel_pack(prs_pc_plan* p, const long long* argmax, const int* err, int* out, cudaStream_t st) {
  k_unravel_pack<<<(p->B + 127) / 128, 128, 0, st>>>(argmax, err, p->B, p->Y, p->Th, (int4*)out);
  PRS_CUDA(cudaGetLastError());
  return PRS_OK;
}

extern "C" int prs_pc_active_cells(prs_pc_handle h, const void* state, int b, double threshold, int max_out, int* idx_out,
                                   void* val_out, int* count_out, void* work, void* stream) {
  PRS_REQUIRE(h && state && idx_out && val_out && count_out && work, "prs_pc_active_cells: null argument");
  PRS_REQUIRE(b >= 0 && b < h->B && max_out >= 0, "prs_pc_active_cells: bad network index or capacity");
  cudaStream_t st = (cudaStream_t)stream;
  const int XY = h->X * h->Y;
  const int nblk = (int)((h->N + 255) / 256);
  int* counts = (int*)work;
  int* offsets = counts + nblk;
  if (h->dtype == PRS_F32) {
    const float* s = (const float*)state + (size_t)b * h->N;
    k_active_count<float><<<nblk, 256, 0, st>>>(s, XY, h->Th, threshold, counts);
    k_exclusive_scan_small<<<1, 256, 0, st>>>(counts, nblk, offsets, count_out);
    k_active_write<float><<<nblk, 256, 0, st>>>(s, XY, h->Th, threshold, offsets, max_out, idx_out, (float*)val_out);
  } else {
    const double* s = (const double*)state + (size_t)b * h->N;
    k_active_count<double><<<nblk, 256, 0, st>>>(s, XY, h->Th, threshold, counts);
    k_exclusive_scan_small<<<1, 256, 0, st>>>(counts, nblk, offsets, count_out);
    k_active_write<double><<<nblk, 256, 0, st>>>(s, XY, h->Th, threshold, offsets, max_out, idx_out, (double*)val_out);
  }
  PRS_CUDA(cudaGetLastError());
  return PRS_OK;
}

extern "C" size_t prs_pc_active_work_bytes(prs_pc_handle h) {
  return h ? (size_t)((h->N + 255) / 256) * 2 * sizeof(int) : 0;
}

extern "C" int prs_pc_argmax(prs_pc_handle h, const void* state, long long* argmax, void* stream) {
  PRS_REQUIRE(h && state && argmax, "prs_pc_argmax: null argument");
  return prs_pc_generic_argmax(h, state, argmax, (cudaStream_t)stream);
}

static int transpose(prs_pc_handle h, void* state, void* xyt, bool import, cudaStream_t st) {
  dim3 grid(h->nblk_plane, h->Th, h->B);
  int XY = h->X * h->Y;
  if (h->dtype == PRS_F32) {
    if (import)
      k_transpose<float, true><<<grid, kThreads, 0, st>>>((float*)state, (float*)xyt, XY, h->Th);
    else
      k_transpose<float, false><<<grid, kThreads, 0, st>>>((float*)state, (float*)xyt, XY, h->Th);
  } else {
    if (import)
      k_transpose<double, true><<<grid, kThreads, 0, st>>>((double*)state, (double*)xyt, XY, h->Th);
    else
      k_transpose<double, false><<<grid, kThreads, 0, st>>>((double*)state, (double*)xyt, XY, h->Th);
  }
  PRS_CUDA(cudaGetLastError());
  return PRS_OK;
}

extern "C" int prs_pc_import_xyt(prs_pc_handle h, void* state, const void* xyt, void* stream) {
  PRS_REQUIRE(h && state && xyt, "prs_pc_import_xyt: null argument");
  if (int rc_ = prs_pc_active_invalidate(h, (cudaStream_t)stream)) return rc_;
  return transpose(h, state, const_cast<void*>(xyt), true, (cudaStream_t)stream);
}

extern "C" int prs_pc_export_xyt(prs_pc_handle h, const void* state, void* xyt, void* stream) {
  PRS_REQUIRE(h && state && xyt, "prs_pc_export_xyt: null argument");
  return transpose(h, const_cast<void*>(state), xyt, false, (cudaStream_t)stream);
}
