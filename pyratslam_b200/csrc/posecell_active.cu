// Active-set pose-cell update (opt-in: PRS_OPT_ACTIVE_SET; reported separately from the dense kernels, SURVEY.md 8d).
//
// The attractor dynamics of ratslam/posecell_network.py:326-353 keep the activity in a compact packet: the global
// inhibition (:339-340) is an absolute threshold on a state that is renormalised to sum 1 (:343-345), so after one
// update a 21x21x36 network holds 30...80 non-zero cells out of 15 876 and a 256x256x72 one a few hundred out of
// 4.7 million.  The dense kernels of this library cost the same whatever the state holds; this path does the same
// arithmetic only where it can be non-zero, and stays exact for ANY state:
//
//   k_pc_scan    streams the state once (16-byte loads, the only pass over all cells) and appends the flat index of every
//                non-zero cell to the network's active list (capacity `cap`; an overflowing network is handled densely);
//   k_pc_active  one CTA per network.  The lists give per-axis occupancy bitmasks S_x, S_y, S_th; every later support is
//                a PRODUCT OF PER-AXIS SETS (which also covers several packets and packets that straddle the periodic
//                border, with no bounding-box arithmetic): G = S dilated by the 3-cell reach of the DoG, the support
//                of the inhibited result inside G, its image under each plane's 7x7 filter and integer origin
//                (convolution.py:320-340), and the 3-plane reach of the theta filter.  The stages -- theta, y, x passes of
//                the separable DoG, inhibition and sum, 7x7 stage, theta stage with 1/total, clamp, arg-max -- run on
//                compressed sub-grids indexed by positions in those sets, in shared memory, tap for tap in the order of
//                the generic kernels (posecell_generic.cu) with the taps that fall outside a set skipped: such a tap
//                multiplies an exact zero, so the result is the dense one.  The state is then updated IN PLACE: the old
//                active cells are zeroed and the new non-zero cells written; everything else is zero and stays zero.
//   fallback     a network whose compressed grids do not fit the first launch's arena goes to a second launch with a big
//                one; a network whose list overflowed, that does not fit there either, or whose global inhibition is
//                negative (then the zero cells do not stay zero) is flagged and appended to a work list; the plan's dense
//                kernels then run for the flagged networks only.  Inside the graph prs_pc_step replays, the second
//                launch and the dense kernels are the body of a conditional node that this kernel raises
//                (cudaGraphSetConditional) only when it defers or flags a network.
//
// Measured (B200): 1.6-2.1x the dense kernels on 4096 x 21x21x36 float32, 3.4-4.7x on the float64 and 50x50x10 ensembles,
// 1.7-1.8x on one 256x256x72 network (DESIGN.md 4.8); the scan runs at the HBM roof, k_pc_active at 61 % issue utilisation
// with 19 k warp instructions per network.
//
// PRS_OPT_ACTIVE_SET = 2 additionally keeps the list k_pc_active wrote (the new non-zero cells) as the next update's
// input: k_pc_scan then returns at once for that network and an update no longer reads the state at all.  Every
// library call that writes the state invalidates the lists; a caller that writes it by other means must call
// prs_pc_invalidate_active.
#include "common.cuh"

namespace {

constexpr int kMaxDim = 256;        // per-axis bitmasks
constexpr int kScanT = 256;

__device__ __forceinline__ float fma_t(float a, float b, float c) { return fmaf(a, b, c); }
__device__ __forceinline__ double fma_t(double a, double b, double c) { return fma(a, b, c); }

__device__ __forceinline__ bool nz(float v) { return (__float_as_uint(v) & 0x7fffffffu) != 0u; }  // -0.0 counts as zero
__device__ __forceinline__ bool nz(double v) { return ((unsigned long long)__double_as_longlong(v) << 1) != 0ull; }

// ---------------------------------------------------------------------------------------------- scan
__device__ __forceinline__ void scan_hit(int* cnt, int* idx, int cap, long long local) {
  const int pos = atomicAdd(cnt, 1);
  if (pos < cap) idx[pos] = (int)local;
}

template <typename T>
struct V16;
template <>
struct V16<float> {
  using V = float4;
  static constexpr int n = 4;
};
template <>
struct V16<double> {
  using V = double2;
  static constexpr int n = 2;
};
__device__ __forceinline__ void unpack(const float4& v, float* o) { o[0] = v.x, o[1] = v.y, o[2] = v.z, o[3] = v.w; }
__device__ __forceinline__ void unpack(const double2& v, double* o) { o[0] = v.x, o[1] = v.y; }
__device__ __forceinline__ bool any_nz(const float4& v) {
  return ((__float_as_uint(v.x) | __float_as_uint(v.y) | __float_as_uint(v.z) | __float_as_uint(v.w)) & 0x7fffffffu) != 0u;
}
__device__ __forceinline__ bool any_nz(const double2& v) {
  return (((unsigned long long)__double_as_longlong(v.x) | (unsigned long long)__double_as_longlong(v.y)) << 1) != 0ull;
}

// grid (chunks, B).  VEC: N * sizeof(T) is a multiple of 16 and the state is 16-byte aligned.
template <typename T, bool VEC>
__global__ void __launch_bounds__(kScanT) k_pc_scan(const T* __restrict__ state, long long N, int per_chunk,
                                                    int* __restrict__ al_cnt, int* __restrict__ al_idx, int cap,
                                                    const int* __restrict__ al_valid, int* __restrict__ dense_cnt) {
  const int b = blockIdx.y;
  if (blockIdx.x == 0 && b == 0 && threadIdx.x == 0) dense_cnt[0] = dense_cnt[1] = 0;  // k_pc_active counts from 0
  if (al_valid[b]) return;  // the list k_pc_active left is current
  const T* src = state + (size_t)b * N;
  int* cnt = al_cnt + b;
  int* idx = al_idx + (size_t)b * cap;
  if (VEC) {
    using V = typename V16<T>::V;
    constexpr int n = V16<T>::n;
    const long long nv = N / n;
    const long long lo = (long long)blockIdx.x * per_chunk;  // in vectors
    long long hi = lo + per_chunk;
    hi = hi < nv ? hi : nv;
    const V* s = reinterpret_cast<const V*>(src);
    for (long long i0 = lo + threadIdx.x; i0 < hi; i0 += 4 * kScanT) {
      V v[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const long long i = i0 + (long long)u * kScanT;
        if (i < hi) v[u] = __ldcs(s + i);
      }
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const long long i = i0 + (long long)u * kScanT;
        if (i < hi && any_nz(v[u])) {
          T e[n];
          unpack(v[u], e);
#pragma unroll
          for (int q = 0; q < n; ++q)
            if (nz(e[q])) scan_hit(cnt, idx, cap, i * n + q);
        }
      }
    }
  } else {
    const long long lo = (long long)blockIdx.x * per_chunk;
    long long hi = lo + per_chunk;
    hi = hi < N ? hi : N;
    for (long long i = lo + threadIdx.x; i < hi; i += kScanT)
      if (nz(src[i])) scan_hit(cnt, idx, cap, i);
  }
}

// ---------------------------------------------------------------------------------------------- active-set update
template <int MAXD>
struct AxisSet {   // a subset of an axis' coordinates: sorted list and coordinate -> position (-1 = not a member)
  unsigned char list[MAXD];
  short pos[MAXD];
};

__device__ __forceinline__ bool test_bit(const unsigned* m, int c) { return (m[c >> 5] >> (c & 31)) & 1u; }

// One warp turns a finished mask (bits >= n are clear) into the sorted list and the position table; returns the size.
template <int MAXD>
__device__ __noinline__ int set_from_mask(const unsigned* mask, int n, AxisSet<MAXD>* s, int lane) {
  int off = 0;
#pragma unroll 1
  for (int w = 0; w * 32 < n; ++w) {
    const unsigned m = mask[w];
    const int c = w * 32 + lane;
    const bool in = (m >> lane) & 1u;
    const int p = off + __popc(m & ((1u << lane) - 1u));
    if (c < n) s->pos[c] = in ? (short)p : (short)-1;
    if (in) s->list[p] = (unsigned char)c;
    off += __popc(m);
  }
  return off;
}

// The whole block derives a mask: bit c = pred(c) for c < n (the caller separates this from its readers by a barrier).
template <typename P>
__device__ __forceinline__ void derive_mask(int n, unsigned* mask, P pred) {
#pragma unroll 1
  for (int c0 = 0; c0 < n; c0 += blockDim.x) {
    const int c = c0 + threadIdx.x;
    const unsigned w = __ballot_sync(0xffffffffu, c < n && pred(c));
    if ((threadIdx.x & 31) == 0 && c < n) mask[c >> 5] = w;
  }
}

// any member within 3 cells (periodic), n >= 3.  Seven independent bit tests (no short-circuit: the kernel is bound by the
// latency of dependent steps), one copy of the code.
__device__ __noinline__ bool dilated(const unsigned* m, int c, int n) {
  unsigned b = 0;
  int q = c - 3;
  q += q < 0 ? n : 0;
#pragma unroll
  for (int d = 0; d < 7; ++d) {
    b |= (m[q >> 5] >> (q & 31));
    q = q + 1 == n ? 0 : q + 1;
  }
  return b & 1u;
}

// One periodic line of a 7-tap correlate on a compressed axis.  Outputs live at the n positions of the DILATED set G of
// that axis, inputs at the positions of the set S it was dilated from; spos[g] = position in S of G's member g, or -1.
// The neighbours of G-position g are the G-positions g-3 .. g+3 taken cyclically: inside a run of consecutive coordinates
// that is literally true, and a step across the end of a run lands on the first / last three members of the neighbouring
// run, which are not in S (a run of G begins exactly three cells before a member of S) -- the input there is the same
// zero the true neighbour (outside G, or such a fringe cell itself) holds.  So a chunk of CH consecutive outputs of a line
// is a register window of CH + 6 inputs: no coordinate arithmetic and no table look-up per tap.  A work item is one
// (line, chunk): the kernel is bound by the latency of a CTA's dependent steps, so the chunks of a line go to different
// threads rather than one after the other.
template <typename W, int CH, typename LD, typename EM>
__device__ __forceinline__ void window_chunk(const short* __restrict__ spos, int n, int g0, W zero, LD ld, EM emit) {
  W win[CH + 6];
  int q = g0 - 3;
  while (q < 0) q += n;  // at most three rounds (n >= 1): no integer division in the hot loops
#pragma unroll
  for (int j = 0; j < CH + 6; ++j) {
    const int s = spos[q];
    win[j] = zero;
    if (s >= 0) win[j] = ld(s);
    q = q + 1 == n ? 0 : q + 1;
  }
#pragma unroll
  for (int jj = 0; jj < CH; ++jj)
    if (g0 + jj < n) emit(g0 + jj, &win[jj]);
}

__device__ __noinline__ void plan_cell_noinline(int k, int Th, int minXY, const double* odom, const double* cos_th,
                                                const double* sin_th, double vts, double vrs, int* shift,
                                                unsigned char* fsel, int* ogi, int* err) {
  prs_plan_cell(0, k, Th, minXY, odom, cos_th, sin_th, vts, vrs, shift, fsel, ogi, err);
}

template <typename T>
struct Pr {
  T e, i;
};

template <typename T>
struct ActArgs {
  T* state;
  const double* odom;
  const T* gi;
  long long* argmax;
  T* total;
  int* err;
  const double *cos_th, *sin_th;
  double vtrans_scale, vrot_scale;
  int X, Y, Th, B;
  int *al_cnt, *al_idx, *al_valid;
  int cap, track;
  int *dense_flag, *dense_list, *dense_cnt;
  // work items: every network (wl == nullptr) or the *wl_cnt networks listed in wl (second tier)
  const int *wl, *wl_cnt;
  // where a network whose compressed grids do not fit this launch's arena goes: the second tier's list (first tier of
  // two), else the dense list
  int *over_list, *over_cnt;
  unsigned long long cond;  // conditional handle of the graph this launch is a node of (0: none): raised with the first flag
  int cap0, cap1;  // elements of T in the two regions of the dynamic shared-memory arena
  PcTables<T> tab;
};

constexpr int kActMaxT = 256;
// outputs per register window of the WIDE kernels in float32 (half as many in float64): 1-D passes, 7x7 stage
constexpr int kActCh = 12;
constexpr int kActCh2 = 8;

// l / n for 0 <= l < 2^21, n > 0, inv = 1.0f / n: (l + 0.5) / n is never within float rounding of an integer there
__device__ __forceinline__ int fdiv(int l, float inv) { return __float2int_rz((__int2float_rn(l) + 0.5f) * inv); }

// MAXD: upper bound of the three grid dimensions (64 for ensembles of small grids: 4 KB of static shared memory per CTA
// instead of 15 KB, so that more networks are in flight per SM)
// WIDE: register windows that cover a whole line of a typical packet (fewer work items: fewer instructions, the choice for
// thousands of networks) or windows of four outputs (more items in flight: lower latency, the choice for a few networks).
template <typename T, int MAXD, bool WIDE>
__global__ void __launch_bounds__(kActMaxT, 4) k_pc_active(const __grid_constant__ ActArgs<T> a) {
  // Outputs per register window.  A work item costs ~100 instructions before its first FMA (window positions, predicated
  // loads, line decode), so a window covers the whole line of a typical packet (11 outputs) where the registers allow it.
  constexpr int CH = !WIDE ? 4 : (sizeof(T) == 4 ? kActCh : kActCh / 2);      // 1-D passes
  constexpr int CH2 = !WIDE ? 4 : (sizeof(T) == 4 ? kActCh2 : kActCh2 / 2);   // 7x7 stage (accumulators + two windows)
  constexpr int MW = MAXD / 32;
  using Set = AxisSet<MAXD>;
  extern __shared__ __align__(16) unsigned char arena_raw[];
  // sets: 0..2 S_x, S_y, S_th (later SA_x, SA_y, SA_th: the support of the inhibited result); 3..5 G_x, G_y, G_th (S dilated
  // by the reach of the DoG); 6, 7 DA_x, DA_y (SA dilated by the reach of the 7x7 filter); 8, 9 B_x, B_y (DA displaced by
  // the active planes' integer origins); 10 D_th (SA_th dilated by the reach of the theta filter)
  __shared__ Set s_set[11];
  // position in a dilated set -> position in the set it was dilated from: G -> S (x, y, theta), DA -> SA (x, y), D_th -> SA_th
  __shared__ short s_spos[6][MAXD];
  __shared__ short s_a2g[2][MAXD];      // SA_x / SA_y position -> G_x / G_y position (where A stores that row / column)
  __shared__ int s_om[2][MAXD];         // integer origin of active plane s (position in SA_th), reduced modulo X / Y
  __shared__ unsigned s_mS[3][MW], s_mG[3][MW], s_mA[3][MW], s_mD[3][MW], s_mB[2][MW];
  __shared__ int s_n[16];
  __shared__ int s_shift[2 * MAXD];
  __shared__ unsigned char s_fsel[MAXD];
  __shared__ T s_F[2][49];
  __shared__ int s_ogi, s_newcnt;
  __shared__ T s_red[kActMaxT / 32];
  __shared__ int s_redi[kActMaxT / 32];
  __shared__ T s_total;

  const int tid = threadIdx.x, nt = blockDim.x, lane = tid & 31, wid = tid >> 5, nw = nt >> 5;
  if (a.wl_cnt != nullptr && (int)blockIdx.x >= *a.wl_cnt) return;
  const int b = a.wl != nullptr ? a.wl[blockIdx.x] : (int)blockIdx.x;
  const int X = a.X, Y = a.Y, Th = a.Th, XY = X * Y;
  T* st = a.state + (size_t)b * ((size_t)XY * Th);
  T* R0 = reinterpret_cast<T*>(arena_raw);
  T* R1 = R0 + a.cap0;
  const int cap0 = a.cap0, cap1 = a.cap1;
  const int n_act = a.al_cnt[b];
  const int* lidx = a.al_idx + (size_t)b * a.cap;
  const T g_inh = a.gi[b];

  // the update's decisions (posecell_network.py:252-267,304), the arithmetic of every other path
#pragma unroll 1
  for (int k = tid; k < Th; k += nt)
    plan_cell_noinline(k, Th, X < Y ? X : Y, a.odom + 2 * (size_t)b, a.cos_th, a.sin_th, a.vtrans_scale, a.vrot_scale,
                       s_shift, s_fsel, &s_ogi, a.err + b);
#pragma unroll 1
  for (int i = tid; i < 3 * MW; i += nt)
    (&s_mS[0][0])[i] = 0u, (&s_mG[0][0])[i] = 0u, (&s_mA[0][0])[i] = 0u, (&s_mD[0][0])[i] = 0u;
#pragma unroll 1
  for (int i = tid; i < 2 * MW; i += nt) (&s_mB[0][0])[i] = 0u;
#pragma unroll 1
  for (int i = tid; i < 98; i += nt) (&s_F[0][0])[i] = a.tab.f2d[i / 49][i % 49];
  if (tid == 0) s_newcnt = 0;
  __syncthreads();

  auto go_dense = [&]() {
    if (tid == 0) {
      a.dense_flag[b] = 1;
      a.dense_list[atomicAdd(a.dense_cnt, 1)] = b;
      if (a.cond != 0ull) cudaGraphSetConditional((cudaGraphConditionalHandle)a.cond, 1u);  // the dense fall-back runs
      a.al_cnt[b] = 0;
      a.al_valid[b] = 0;
    }
  };
  auto overflow = [&]() {  // the compressed grids do not fit this launch's arena
    if (a.over_list == nullptr)
      go_dense();
    else if (tid == 0) {
      a.over_list[atomicAdd(a.over_cnt, 1)] = b;  // the list and its count stay as they are for the second tier
      if (a.cond != 0ull) cudaGraphSetConditional((cudaGraphConditionalHandle)a.cond, 1u);  // ... which is in the body
    }
  };
  if (n_act > a.cap || !(g_inh >= T(0))) {
    go_dense();
    return;
  }

  int best_i = 0;
  T best_v = T(0), tot = T(0);
  int nBX = 0, nBY = 0, nDK = 0;
  bool alive = false, zeroed = false;
  Set *Gx = &s_set[3], *Gy = &s_set[4], *Gk = &s_set[5], *SAx = &s_set[0], *SAy = &s_set[1], *SAk = &s_set[2],
      *DAx = &s_set[6], *DAy = &s_set[7], *BXs = &s_set[8], *BYs = &s_set[9], *DK = &s_set[10];
  if (n_act > 0) {
    // ---- occupancy of the three axes, their dilations, the sets
#pragma unroll 1
    for (int e = tid; e < n_act; e += nt) {
      const int f = lidx[e];
      const int k = f / XY, r = f - k * XY, x = r / Y, y = r - x * Y;
      atomicOr(&s_mS[0][x >> 5], 1u << (x & 31));
      atomicOr(&s_mS[1][y >> 5], 1u << (y & 31));
      atomicOr(&s_mS[2][k >> 5], 1u << (k & 31));
    }
    __syncthreads();
    derive_mask(X, s_mG[0], [&](int c) { return dilated(s_mS[0], c, X); });
    derive_mask(Y, s_mG[1], [&](int c) { return dilated(s_mS[1], c, Y); });
    derive_mask(Th, s_mG[2], [&](int c) { return dilated(s_mS[2], c, Th); });
    __syncthreads();
#pragma unroll 1
    for (int q = wid; q < 6; q += nw) {
      const int ax = q % 3, n = ax == 0 ? X : (ax == 1 ? Y : Th);
      const int c = set_from_mask(q < 3 ? s_mS[ax] : s_mG[ax], n, &s_set[q], lane);
      if (lane == 0) s_n[q] = c;
    }
    __syncthreads();
    const int nSx = s_n[0], nSy = s_n[1], nSk = s_n[2], nGx = s_n[3], nGy = s_n[4], nGk = s_n[5];
#pragma unroll 1
    for (int ax = 0; ax < 3; ++ax)
#pragma unroll 1
      for (int g = tid; g < s_n[3 + ax]; g += nt) s_spos[ax][g] = s_set[ax].pos[s_set[3 + ax].list[g]];
    const long long nXc = (long long)nSx * nSy * nSk, nP1 = (long long)nSx * nSy * nGk, nP2 = (long long)nSx * nGy * nGk,
                    nA = (long long)nGx * nGy * nGk;
    if (nXc > cap0 || 2 * nP2 > cap0 || 2 * nP1 > cap1 || nA > cap1) {
      overflow();
      return;
    }
    // ---- compact input Xc[i][j][s] (R0), positions in S_x, S_y, S_th
    T* Xc = R0;
#pragma unroll 1
    for (int c = tid; c < (int)nXc; c += nt) Xc[c] = T(0);
    __syncthreads();
#pragma unroll 1
    for (int e = tid; e < n_act; e += nt) {
      const int f = lidx[e];
      const int k = f / XY, r = f - k * XY, x = r / Y, y = r - x * Y;
      Xc[(s_set[0].pos[x] * nSy + s_set[1].pos[y]) * nSk + s_set[2].pos[k]] = st[f];
    }
    __syncthreads();
    // ---- theta pass (k_dog_theta), one thread per (i, j) line: P1[i][j][g] pairs (R1)
    Pr<T>* P1 = reinterpret_cast<Pr<T>*>(R1);
    const int chK = (nGk + CH - 1) / CH, chY = (nGy + CH - 1) / CH, chX = (nGx + CH - 1) / CH;
    const float inv_nGk = 1.0f / (float)nGk;
#pragma unroll 1
    for (int it = tid; it < nSx * nSy * chK; it += nt) {
      const int c = chK == 1 ? 0 : it / (nSx * nSy), l = it - c * (nSx * nSy), g0 = c * CH;
      const T* in = Xc + l * nSk;
      Pr<T>* out = P1 + l * nGk;
      window_chunk<T, CH>(
          s_spos[2], nGk, g0, T(0), [&](int s) { return in[s]; },
          [&](int g, const T* w) {
            T e = 0, i = 0;
#pragma unroll
            for (int t = 0; t < 7; ++t) e = fma_t(a.tab.ge[t], w[t], e), i = fma_t(a.tab.gi[t], w[t], i);
            out[g] = Pr<T>{e, i};
          });
    }
    __syncthreads();
    // ---- y pass (k_dog_y), one thread per (i, g) line: P2[i][gy][g] pairs (R0)
    Pr<T>* P2 = reinterpret_cast<Pr<T>*>(R0);
#pragma unroll 1
    for (int it = tid; it < nSx * nGk * chY; it += nt) {
      const int c = chY == 1 ? 0 : it / (nSx * nGk), l = it - c * (nSx * nGk), g0 = c * CH;
      const int i0 = fdiv(l, inv_nGk), g = l - i0 * nGk;
      const Pr<T>* in = P1 + i0 * nSy * nGk + g;
      Pr<T>* out = P2 + i0 * nGy * nGk + g;
      window_chunk<Pr<T>, CH>(
          s_spos[1], nGy, g0, Pr<T>{T(0), T(0)}, [&](int s) { return in[s * nGk]; },
          [&](int gy, const Pr<T>* w) {
            T e = 0, i = 0;
#pragma unroll
            for (int t = 0; t < 7; ++t) e = fma_t(a.tab.ge[t], w[t].e, e), i = fma_t(a.tab.gi[t], w[t].i, i);
            out[gy * nGk] = Pr<T>{e, i};
          });
    }
    __syncthreads();
    // ---- x pass, inhibition (posecell_network.py:339-340), sum (:343) (k_dog_x_inhib), one thread per (gy, g) line:
    //      A[gx][gy][g] (R1); the axes' occupancy of the result
    T* A = R1;
    T psum = T(0);
    const int lineA = nGy * nGk;
#pragma unroll 1
    for (int it = tid; it < lineA * chX; it += nt) {
      const int c = chX == 1 ? 0 : it / lineA, l = it - c * lineA, g0 = c * CH;
      const Pr<T>* in = P2 + l;
      T* out = A + l;
      bool any = false;
      window_chunk<Pr<T>, CH>(
          s_spos[0], nGx, g0, Pr<T>{T(0), T(0)}, [&](int s) { return in[s * lineA]; },
          [&](int gx, const Pr<T>* w) {
            T e = 0, i = 0;
#pragma unroll
            for (int t = 0; t < 7; ++t) e = fma_t(a.tab.gex[t], w[t].e, e), i = fma_t(a.tab.gix[t], w[t].i, i);
            T v = e - i;
            v = (v < g_inh) ? T(0) : v - g_inh;
            out[gx * lineA] = v;
            psum += v;
            if (nz(v)) {
              const int x = Gx->list[gx];
              atomicOr(&s_mA[0][x >> 5], 1u << (x & 31));
              any = true;
            }
          });
      if (any) {
        const int gy = fdiv(l, inv_nGk), g = l - gy * nGk;
        const int y = Gy->list[gy], k = Gk->list[g];
        atomicOr(&s_mA[1][y >> 5], 1u << (y & 31));
        atomicOr(&s_mA[2][k >> 5], 1u << (k & 31));
      }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) psum += __shfl_down_sync(0xffffffffu, psum, o);
    if (lane == 0) s_red[wid] = psum;
    __syncthreads();
    if (tid == 0) {
      T s = T(0);
#pragma unroll 1
      for (int w = 0; w < nw; ++w) s += s_red[w];  // fixed order
      s_total = s;
    }
    // ---- support SA of the inhibited result; its dilations by the reach of the 7x7 filter (x, y) and of the theta filter
    derive_mask(X, s_mD[0], [&](int c) { return dilated(s_mA[0], c, X); });
    derive_mask(Y, s_mD[1], [&](int c) { return dilated(s_mA[1], c, Y); });
    derive_mask(Th, s_mD[2], [&](int c) { return dilated(s_mA[2], c, Th); });
    __syncthreads();
    tot = s_total;
    alive = tot != T(0);
    if (alive) {
      const T inv = T(1) / tot;  // posecell_network.py:344-345
#pragma unroll 1
      for (int q = wid; q < 6; q += nw) {  // SA_x, SA_y, SA_th (slots 0..2), DA_x, DA_y (6, 7), D_th (10)
        const int ax = q % 3, n = ax == 0 ? X : (ax == 1 ? Y : Th);
        const int slot = q < 3 ? q : (q < 5 ? q + 3 : 10);
        const int c = set_from_mask(q < 3 ? s_mA[ax] : s_mD[ax], n, &s_set[slot], lane);
        if (lane == 0) s_n[6 + q] = c;
      }
      __syncthreads();
      const int nSAx = s_n[6], nSAy = s_n[7], nSAk = s_n[8], nDAx = s_n[9], nDAy = s_n[10];
      nDK = s_n[11];
#pragma unroll 1
      for (int s = tid; s < nSAk; s += nt) {
        const int k = SAk->list[s];
        s_om[0][s] = modp(s_shift[2 * k], X);
        s_om[1][s] = modp(s_shift[2 * k + 1], Y);
      }
#pragma unroll 1
      for (int g = tid; g < nDAx; g += nt) s_spos[3][g] = SAx->pos[DAx->list[g]];
#pragma unroll 1
      for (int g = tid; g < nDAy; g += nt) s_spos[4][g] = SAy->pos[DAy->list[g]];
#pragma unroll 1
      for (int g = tid; g < nDK; g += nt) s_spos[5][g] = SAk->pos[DK->list[g]];
#pragma unroll 1
      for (int g = tid; g < nSAx; g += nt) s_a2g[0][g] = Gx->pos[SAx->list[g]];
#pragma unroll 1
      for (int g = tid; g < nSAy; g += nt) s_a2g[1][g] = Gy->pos[SAy->list[g]];
      __syncthreads();
      // where the result of the 7x7 stage can be non-zero: cell x of plane k reads rows x + ox_k - 3 .. + 3
      // (convolution.py:329-331), i.e. x + ox_k must be in DA_x for one of the active planes
      derive_mask(X, s_mB[0], [&](int c) {
        bool in = false;
#pragma unroll 1
        for (int s = 0; s < nSAk; ++s) {
          int q = c + s_om[0][s];
          q -= q >= X ? X : 0;
          in = in || test_bit(s_mD[0], q);
        }
        return in;
      });
      derive_mask(Y, s_mB[1], [&](int c) {
        bool in = false;
#pragma unroll 1
        for (int s = 0; s < nSAk; ++s) {
          int q = c + s_om[1][s];
          q -= q >= Y ? Y : 0;
          in = in || test_bit(s_mD[1], q);
        }
        return in;
      });
      __syncthreads();
#pragma unroll 1
      for (int q = wid; q < 2; q += nw) {
        const int c = set_from_mask(s_mB[q], q == 0 ? X : Y, &s_set[8 + q], lane);
        if (lane == 0) s_n[12 + q] = c;
      }
      __syncthreads();
      nBX = s_n[12], nBY = s_n[13];
      if ((long long)nDAx * nDAy * nSAk > cap0) {
        overflow();
        return;
      }
      // From here on the update is carried out: the old active cells go to zero now, the theta stage below -- behind the
      // barrier that follows the 7x7 stage -- writes the new non-zero cells into the state as it produces them.
#pragma unroll 1
      for (int e = tid; e < n_act; e += nt) st[lidx[e]] = T(0);
      zeroed = true;
      // ---- 7x7 stage (k_shift2d) in each active plane's own frame -- B'[jx][jy][s] (R0) holds the value of the cell whose
      //      read window is centred on DA_x[jx], DA_y[jy]; the plane's integer origin is applied by the theta stage's
      //      gather.  One thread per (jx, s) line along y: the seven source rows and the window's columns are looked up
      //      once, then it is register windows and FMAs (rows and columns outside SA hold zeros: skipped / zero).
      T* Bc = R0;
      const int chB = (nDAy + CH2 - 1) / CH2, nLB = nDAx * nSAk;
      const float inv_nSAk = 1.0f / (float)nSAk, inv_nBY = 1.0f / (float)s_n[13];
#pragma unroll 1
      for (int it = tid; it < nLB * chB; it += nt) {
        const int cb = chB == 1 ? 0 : it / nLB, l = it - cb * nLB, g0 = cb * CH2;
        const int jx = fdiv(l, inv_nSAk), s = l - jx * nSAk, k = SAk->list[s];
        const T* F = s_F[s_fsel[k]];
        const int gk = Gk->pos[k];
        int q0 = jx - 3;
        while (q0 < 0) q0 += nDAx;
        {
          int col[CH2 + 6];
          int q = g0 - 3;
          while (q < 0) q += nDAy;
#pragma unroll
          for (int j = 0; j < CH2 + 6; ++j) {
            const int sa = s_spos[4][q];
            col[j] = sa >= 0 ? s_a2g[1][sa] * nGk : -1;
            q = q + 1 == nDAy ? 0 : q + 1;
          }
          T acc[CH2];
#pragma unroll
          for (int jj = 0; jj < CH2; ++jj) acc[jj] = T(0);
          int qx = q0;
#pragma unroll
          for (int u = 0; u < 7; ++u) {
            const int sa = s_spos[3][qx];
            qx = qx + 1 == nDAx ? 0 : qx + 1;
            if (sa < 0) continue;
            const T* row = A + s_a2g[0][sa] * lineA + gk;
            T fr[7];
#pragma unroll
            for (int t = 0; t < 7; ++t) fr[t] = F[u * 7 + t];
            T w[CH2 + 6];
#pragma unroll
            for (int j = 0; j < CH2 + 6; ++j) {
              w[j] = T(0);
              if (col[j] >= 0) w[j] = row[col[j]];
            }
#pragma unroll
            for (int jj = 0; jj < CH2; ++jj)
#pragma unroll
              for (int t = 0; t < 7; ++t) acc[jj] = fma_t(fr[t], w[jj + t], acc[jj]);
          }
#pragma unroll
          for (int jj = 0; jj < CH2; ++jj)
            if (g0 + jj < nDAy) {
              const T v = acc[jj] * inv;
              Bc[(jx * nDAy + g0 + jj) * nSAk + s] = (v < T(0)) ? T(0) : v;  // posecell_network.py:300
            }
        }
      }
      __syncthreads();
      // ---- theta stage (k_theta_final), clamp (:314), arg-max candidates, one thread per (x, y) line, written straight into the state
      T ft[7];
#pragma unroll
      for (int t = 0; t < 7; ++t) ft[t] = a.tab.f1d[s_ogi][t];
      int* nidx = a.al_idx + (size_t)b * a.cap;
      const int chD = (nDK + CH - 1) / CH, nLD = nBX * nBY;
#pragma unroll 1
      for (int it = tid; it < nLD * chD; it += nt) {
        const int cd = chD == 1 ? 0 : it / nLD, l = it - cd * nLD, g0 = cd * CH;
        const int jx = fdiv(l, inv_nBY), jy = l - jx * nBY, x = BXs->list[jx], y = BYs->list[jy];
        const int ref0 = (x * Y + y) * Th;  // numpy.argmax order (:317-319)
        T* out = st + x * Y + y;
        window_chunk<T, CH>(
            s_spos[5], nDK, g0, T(0),
            [&](int s) {  // plane SA_th[s] at (x, y): the 7x7 result whose window is centred on (x + ox, y + oy)
              int cx = x + s_om[0][s], cy = y + s_om[1][s];
              cx -= cx >= X ? X : 0;
              cy -= cy >= Y ? Y : 0;
              const int px = DAx->pos[cx], py = DAy->pos[cy];
              return (px >= 0 && py >= 0) ? Bc[(px * nDAy + py) * nSAk + s] : T(0);
            },
            [&](int dk, const T* w) {
              T v = 0;
#pragma unroll
              for (int t = 0; t < 7; ++t) v = fma_t(ft[t], w[t], v);
              if (v > T(0)) {  // clamp (:314): everything else stays the zero it is
                const int k = DK->list[dk];
                out[k * XY] = v;
                if (a.track) {
                  const int pos = atomicAdd(&s_newcnt, 1);
                  if (pos < a.cap) nidx[pos] = k * XY + x * Y + y;
                }
                const int ref = ref0 + k;
                if (v > best_v || (v == best_v && ref < best_i)) best_v = v, best_i = ref;
              }
            });
      }
    }
  }
  // ---- arg-max: first maximum in reference order; every cell outside D is zero, and so is cell 0 when nothing is positive
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const T v2 = __shfl_down_sync(0xffffffffu, best_v, o);
    const int i2 = __shfl_down_sync(0xffffffffu, best_i, o);
    if (v2 > best_v || (v2 == best_v && i2 < best_i)) best_v = v2, best_i = i2;
  }
  __syncthreads();
  if (lane == 0) s_red[wid] = best_v, s_redi[wid] = best_i;
  if (!zeroed)  // a network that died in this update (nothing survived the inhibition): its old cells go to zero
#pragma unroll 1
    for (int e = tid; e < n_act; e += nt) st[lidx[e]] = T(0);
  __syncthreads();
  if (tid == 0) {
    T v = s_red[0];
    int i = s_redi[0];
#pragma unroll 1
    for (int w = 1; w < nw; ++w)
      if (s_red[w] > v || (s_red[w] == v && s_redi[w] < i)) v = s_red[w], i = s_redi[w];
    a.argmax[b] = v > T(0) ? (long long)i : 0;
    a.total[b] = tot;
    a.dense_flag[b] = 0;
    const bool keep = a.track && s_newcnt <= a.cap;
    a.al_cnt[b] = keep ? s_newcnt : 0;
    a.al_valid[b] = keep ? 1 : 0;
  }
}

template <typename T>
int active_launch(prs_pc_plan* p, T* state, const double* odom, const T* gi, long long* argmax, T* total, int* err,
                  const PcTables<T>& tab, int part, cudaStream_t st) {
  const long long N = p->N;
  if (part == 0) {
  const bool vec = (N * (long long)sizeof(T)) % 16 == 0 && ((uintptr_t)state % 16) == 0;
  // scan: chunks of a network so that the grid fills the machine; a chunk is a multiple of what one pass of a CTA covers
  const long long units = vec ? N / V16<T>::n : N;
  const long long pass = (long long)kScanT * (vec ? 4 : 1);
  long long want_ctas = 148LL * 8;
  long long chunks = (want_ctas + p->B - 1) / p->B;
  const long long max_chunks = (units + pass - 1) / pass;
  if (chunks > max_chunks) chunks = max_chunks;
  if (chunks < 1) chunks = 1;
  long long per = (units + chunks - 1) / chunks;
  per = (per + pass - 1) / pass * pass;
  chunks = (units + per - 1) / per;
  dim3 sgrid((unsigned)chunks, (unsigned)p->B);
  if (vec)
    k_pc_scan<T, true><<<sgrid, kScanT, 0, st>>>(state, N, (int)per, p->al_cnt, p->al_idx, p->al_cap, p->al_valid,
                                                 p->dense_cnt);
  else
    k_pc_scan<T, false><<<sgrid, kScanT, 0, st>>>(state, N, (int)per, p->al_cnt, p->al_idx, p->al_cap, p->al_valid,
                                                  p->dense_cnt);
  }
  ActArgs<T> a;
  a.state = state, a.odom = odom, a.gi = gi, a.argmax = argmax, a.total = total, a.err = err;
  a.cos_th = p->cos_th, a.sin_th = p->sin_th, a.vtrans_scale = p->vtrans_scale, a.vrot_scale = p->vrot_scale;
  a.X = p->X, a.Y = p->Y, a.Th = p->Th, a.B = p->B;
  a.al_cnt = p->al_cnt, a.al_idx = p->al_idx, a.al_valid = p->al_valid, a.cap = p->al_cap;
  a.track = p->opt_active == 2 ? 1 : 0;
  a.dense_flag = p->dense_flag, a.dense_list = p->dense_list, a.dense_cnt = p->dense_cnt;
  a.tab = tab;
  a.cond = p->act_cond;
  const int maxd = p->X > p->Y ? (p->X > p->Th ? p->X : p->Th) : (p->Y > p->Th ? p->Y : p->Th);
  // Two tiers for plans of many networks: part 0 launches every network with a small arena (the typical packet; the kernel
  // is bound by the latency of a CTA's dependent phases, so networks in flight per SM are what counts), part 1 the
  // networks whose compressed grids did not fit, with a big arena, before anything is left to the dense kernels.  Plans
  // of a few networks have one tier (part 0, big arena).  Regions: 40 % for {Xc, P2, B'}, 60 % for {P1, A}.
  const bool two = p->act_arena1 > 0;
  if (part == 1 && !two) return PRS_OK;
  {
    const int tier = two ? part : 1;
    const int arena = tier == 0 ? p->act_arena1 : p->act_arena;
    const int elems = arena / (int)sizeof(T);
    a.cap0 = (elems * 2 / 5) & ~3, a.cap1 = elems - a.cap0;
    const bool first_of_two = tier == 0;
    a.wl = tier == 1 && two ? p->big_list : nullptr;
    a.wl_cnt = a.wl != nullptr ? p->dense_cnt + 1 : nullptr;
    a.over_list = first_of_two ? p->big_list : nullptr;
    a.over_cnt = first_of_two ? p->dense_cnt + 1 : nullptr;
    const bool wide = p->B > 2 * 148;  // (a few hundred small networks: all CTAs resident at once, latency is what counts)
    if (maxd <= 64 && wide)
      k_pc_active<T, 64, true><<<p->B, p->act_threads, arena, st>>>(a);
    else if (maxd <= 64)
      k_pc_active<T, 64, false><<<p->B, p->act_threads, arena, st>>>(a);
    else if (wide)
      k_pc_active<T, kMaxDim, true><<<p->B, p->act_threads, arena, st>>>(a);
    else
      k_pc_active<T, kMaxDim, false><<<p->B, p->act_threads, arena, st>>>(a);
  }
  PRS_CUDA(cudaGetLastError());
  return PRS_OK;
}

}  // namespace

int prs_pc_active_supported(const prs_pc_plan* p) {
  return p->X <= kMaxDim && p->Y <= kMaxDim && p->Th <= kMaxDim && p->X >= 3 && p->Y >= 3 && p->Th >= 3;
}

// Buffers and launch shape of the active-set path (made when the option is first switched on).
int prs_pc_active_prepare(prs_pc_plan* p) {
  if (p->al_cnt) return PRS_OK;
  PRS_REQUIRE(prs_pc_active_supported(p), "active-set path: every grid dimension must be in [3, %d]", kMaxDim);
  // a few large networks: one big CTA each with most of an SM's shared memory; many networks: several CTAs per SM
  const int maxd0 = p->X > p->Y ? (p->X > p->Th ? p->X : p->Th) : (p->Y > p->Th ? p->Y : p->Th);
  const bool few = p->B <= 16 || (maxd0 > 64 && p->B <= 2 * 148);  // big CTAs only where a network can need the room
  // (measured, 4096 networks of 21x21x36: first tier of 20 KB 0.158 ms per update; of 12 KB 0.192 ms: too many networks
  // run twice; of 48 KB 0.20 ms: too few in flight)
  const int threads = few ? 256 : 128, arena = few ? 160 * 1024 : 72 * 1024, arena1 = few ? 0 : 20 * 1024;
  const int cap = few ? 8192 : 512;
  p->act_threads = threads, p->act_arena = arena, p->act_arena1 = arena1, p->al_cap = cap;
  PRS_CUDA(cudaFuncSetAttribute(k_pc_active<float, 64, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
  PRS_CUDA(cudaFuncSetAttribute(k_pc_active<double, 64, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
  PRS_CUDA(cudaFuncSetAttribute(k_pc_active<float, kMaxDim, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
  PRS_CUDA(cudaFuncSetAttribute(k_pc_active<double, kMaxDim, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
  PRS_CUDA(cudaFuncSetAttribute(k_pc_active<float, 64, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
  PRS_CUDA(cudaFuncSetAttribute(k_pc_active<double, 64, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
  PRS_CUDA(cudaFuncSetAttribute(k_pc_active<float, kMaxDim, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
  PRS_CUDA(cudaFuncSetAttribute(k_pc_active<double, kMaxDim, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
  const size_t B = (size_t)p->B;
  PRS_CUDA(cudaMalloc(&p->al_idx, B * cap * sizeof(int)));
  PRS_CUDA(cudaMalloc(&p->al_valid, B * sizeof(int)));
  PRS_CUDA(cudaMalloc(&p->dense_flag, B * sizeof(int)));
  PRS_CUDA(cudaMalloc(&p->dense_list, B * sizeof(int)));
  PRS_CUDA(cudaMalloc(&p->big_list, B * sizeof(int)));
  PRS_CUDA(cudaMalloc(&p->dense_cnt, 2 * sizeof(int)));  // [0] dense networks, [1] second-tier networks
  PRS_CUDA(cudaMalloc(&p->al_cnt, B * sizeof(int)));
  PRS_CUDA(cudaMemset(p->al_cnt, 0, B * sizeof(int)));
  PRS_CUDA(cudaMemset(p->al_valid, 0, B * sizeof(int)));
  PRS_CUDA(cudaMemset(p->dense_flag, 0, B * sizeof(int)));
  PRS_CUDA(cudaMemset(p->dense_cnt, 0, 2 * sizeof(int)));
  return PRS_OK;
}

int prs_pc_active_invalidate(prs_pc_plan* p, cudaStream_t st) {
  if (!p->al_cnt) return PRS_OK;
  PRS_CUDA(cudaMemsetAsync(p->al_cnt, 0, (size_t)p->B * sizeof(int), st));
  PRS_CUDA(cudaMemsetAsync(p->al_valid, 0, (size_t)p->B * sizeof(int), st));
  return PRS_OK;
}

// scan + active-set update of every network; the flagged ones are left to the caller's dense kernels
int prs_pc_active_step(prs_pc_plan* p, void* state, const double* odom, const void* gi, long long* argmax, void* total,
                       int* err, int part, cudaStream_t st) {
  if (p->dtype == PRS_F32)
    return active_launch<float>(p, (float*)state, odom, (const float*)gi, argmax, (float*)total, err, p->tf, part, st);
  return active_launch<double>(p, (double*)state, odom, (const double*)gi, argmax, (double*)total, err, p->td, part, st);
}
