// Tiled pose-cell update for large grids (float32), e.g. BASELINE config 3: one 256x256x72 network.
//
// The state of such a grid (18.9 MB) lives in L2, not in one SM's shared memory, so the update
// (ratslam/posecell_network.py:326-353) is four tiled kernels that stream it through L2 once each:
//
//   k_tl_theta      theta pass of the separable DoG: one thread per (x,y) line, a 7-register window slides
//                   along theta, every cell is read once;            P -> (E,I) float2        12 B / cell
//   k_tl_yx         y pass then x pass on a 32x32 tile (+3 halo) in shared memory, packed FFMA2 on (E,I),
//                   A = aE*E - aI*I, inhibition (:339-340), per-tile partial sums (:343)      8.5 + 4 B / cell
//   k_tl_2d         7x7 correlate (:273-274, convolution.py:320-340) on a 64x32 tile whose halo load is
//                   displaced by the plane's integer origin (the shift is free), 2x4 outputs per thread,
//                   rows arrive by LDS.128; * 1/total, clamp (:300)                            5.3 + 4 B / cell
//   k_tl_theta_fin  shifted 7-tap theta pass (convolution.py:344-359), clamp (:314), block arg-max  8 B / cell
//
// Four launches per update: the decisions (k_plan's arithmetic) run inside k_tl_theta, the grid-wide sum of
// k_tl_yx's tile sums is formed by one block of the 7x7 kernel, and the arg-max is finished by the last block of
// k_tl_theta_fin to retire (an atomicInc counter that wraps back to zero; partials are added in a fixed order).
// k_tl_2d_pair takes the place of k_tl_2d when there are enough plane pairs to fill the chip.  Any X, Y, Th >= 3
// (edge tiles are masked, halos wrap by modulo); chosen by the plan for float32 grids of at least 1024 cells per
// plane that the fused SMEM-resident kernel does not cover.
#include "common.cuh"

namespace {

constexpr int kT = 256;

// v in [-n, 2n): one conditional add/sub instead of an integer division (the kernels below are issue bound)
__device__ __forceinline__ int wrap_near(int v, int n) {
  v += v < 0 ? n : 0;
  v -= v >= n ? n : 0;
  return v;
}

// ------------------------------------------------------------------------------------------------
constexpr int kTK = 8;  // theta cells per thread in the two theta kernels (7-register window + 8 new loads)

struct PlanArgs {  // what prs_plan_cell needs; the theta kernel runs it for its network in one of its blocks
  const double *odom, *cos_th, *sin_th;
  double vtrans_scale, vrot_scale;
  int* shift;
  unsigned char* fsel;
  int *ogi, *err;
  int minXY;
};

// A filter coefficient read from the kernel parameters is a constant-bank operand; ptxas re-materialises
// it with one LDCU/UMOV per use, which costs an issue slot each time in these issue-bound kernels.  Passing
// the value through an empty asm pins it in an ordinary register for the rest of the kernel.
__device__ __forceinline__ float pin(float v) {
  asm volatile("" : "+f"(v));
  return v;
}

// Block-level combine without a barrier: every warp publishes its partial result in shared memory and bumps a
// shared counter; only the warp that arrives last goes on (the others are done and free their issue slots --
// a __syncthreads here made every warp wait for the slowest memory access of the block).  *cnt must have been
// zeroed before a barrier that every warp has passed.
__device__ __forceinline__ bool last_warp_of_block(unsigned* cnt, int nwarps) {
  unsigned old = 0;
  if ((threadIdx.x & 31) == 0) {
    asm volatile("fence.acq_rel.cta;" ::: "memory");  // __threadfence_block() is the sequentially-consistent flavour
    old = atomicAdd(cnt, 1u);
  }
  old = __shfl_sync(0xffffffffu, old, 0);
  if (old != (unsigned)(nwarps - 1)) return false;
  asm volatile("fence.acq_rel.cta;" ::: "memory");
  return true;
}

template <int V>
struct Vec;
template <>
struct Vec<1> {
  using F = float;
  using F2 = float2;
};
template <>
struct Vec<4> {
  using F = float4;
  using F2 = float4;  // two (E,I) pairs
};
template <int V>
__device__ __forceinline__ void ldv(const float* p, float* out);
template <>
__device__ __forceinline__ void ldv<1>(const float* p, float* out) {
  out[0] = *p;
}
template <>
__device__ __forceinline__ void ldv<4>(const float* p, float* out) {
  const float4 v = *reinterpret_cast<const float4*>(p);
  out[0] = v.x, out[1] = v.y, out[2] = v.z, out[3] = v.w;
}
template <>
__device__ __forceinline__ void ldv<2>(const float* p, float* out) {
  const float2 v = *reinterpret_cast<const float2*>(p);
  out[0] = v.x, out[1] = v.y;
}

// The 7 + kTK - 1 planes a chunk of kTK theta cells reads.  `inner` (block-uniform) = no periodic wrap and no
// ragged end in this chunk: plane addresses are then one pointer plus multiples of the plane stride.
template <int V, int TK>
__device__ __forceinline__ void load_window(const float* base, int k_lo, int XY, int Th, bool inner,
                                            float (&w)[TK + 6][V]) {
  if (inner) {
    const float* q = base + (size_t)(k_lo - 3) * XY;
#pragma unroll
    for (int j = 0; j < TK + 6; ++j) {
      ldv<V>(q, w[j]);
      q += XY;
    }
  } else {
    const bool near = Th >= TK + 3;  // k_lo - 3 + j stays within [-Th, 2 Th)
#pragma unroll
    for (int j = 0; j < TK + 6; ++j) {
      const int kq = near ? wrap_near(k_lo - 3 + j, Th) : modp(k_lo - 3 + j, Th);
      ldv<V>(base + (size_t)kq * XY, w[j]);
    }
  }
}

// V = cells per thread along the (x,y) line index p: 2 when X*Y is even (64-bit loads, and the two (E,I) pairs
// leave as one 128-bit store, so that a warp writes whole 32-byte sectors), else 1.  TK = theta cells per thread.
template <int V, int TK>
__global__ void __launch_bounds__(kT) k_tl_theta(const float* __restrict__ P, float2* __restrict__ EI, int XY, int Th,
                                                 PcTables<float> tab, PlanArgs pa) {
  if (blockIdx.x == 0 && blockIdx.z == 0) {  // decisions of this update, needed from k_tl_2d on
    for (int k = threadIdx.x; k < Th; k += kT)
      prs_plan_cell(blockIdx.y, k, Th, pa.minXY, pa.odom, pa.cos_th, pa.sin_th, pa.vtrans_scale, pa.vrot_scale, pa.shift,
                    pa.fsel, pa.ogi, pa.err);
  }
  const int p = (blockIdx.x * kT + threadIdx.x) * V;
  if (p >= XY) return;
  const size_t base = (size_t)blockIdx.y * Th * XY + p;
  const int k_lo = blockIdx.z * TK;
  const bool inner = k_lo >= 3 && k_lo + TK + 3 <= Th;
  const float e0 = pin(tab.ge[3]), e1 = pin(tab.ge[2]), e2 = pin(tab.ge[1]), e3 = pin(tab.ge[0]);
  const float i0 = pin(tab.gi[3]), i1 = pin(tab.gi[2]), i2 = pin(tab.gi[1]), i3 = pin(tab.gi[0]);
  float w[TK + 6][V];  // planes k_lo-3 .. k_lo+TK+2, all loads issued before the first use
  load_window<V, TK>(P + base, k_lo, XY, Th, inner, w);
  float2* q = EI + base + (size_t)k_lo * XY;
#pragma unroll
  for (int kk = 0; kk < TK; ++kk) {
    if (inner || k_lo + kk < Th) {
      float2 o[V];
#pragma unroll
      for (int v = 0; v < V; ++v) {
        const float s1 = w[kk + 2][v] + w[kk + 4][v], s2 = w[kk + 1][v] + w[kk + 5][v], s3 = w[kk][v] + w[kk + 6][v];
        o[v].x = fmaf(e0, w[kk + 3][v], fmaf(e1, s1, fmaf(e2, s2, e3 * s3)));
        o[v].y = fmaf(i0, w[kk + 3][v], fmaf(i1, s1, fmaf(i2, s2, i3 * s3)));
      }
      if (V == 2)
        *reinterpret_cast<float4*>(q) = make_float4(o[0].x, o[0].y, o[V - 1].x, o[V - 1].y);
      else
        q[0] = o[0];
    }
    q += XY;
  }
}

// ------------------------------------------------------------------------------------------------
constexpr int kYXx = 64, kYXy = 32;      // outputs per tile (x rows, y columns)
constexpr int kYXrows = kYXx + 6;        // 70 halo rows
constexpr int kYXcols = kYXy + 6;        // 38 halo columns
constexpr int kInStride = kYXcols + 1;   // 39: odd, so that lanes walking down rows hit distinct banks
constexpr int kMidStride = kYXy + 1;     // 33
constexpr int kTyx = 288;                // 9 warps: 4 x 70 = 280 y-pass items, 8 x 32 = 256 x-pass items

__global__ void __launch_bounds__(kTyx) k_tl_yx(const float2* __restrict__ EI, float* __restrict__ A,
                                                const float* __restrict__ gi, int X, int Y, int Th, TlPairs tp,
                                                float* __restrict__ part) {
  constexpr int kT = kTyx;
  __shared__ float2 s_in[kYXrows * kInStride];
  __shared__ unsigned s_cnt;
  __shared__ float2 s_mid[kYXrows * kMidStride];
  __shared__ float s_red[(kT + 31) / 32];
  const int XY = X * Y;
  const int x0 = blockIdx.x * kYXx, y0 = blockIdx.y * kYXy;
  const int plane = blockIdx.z;  // b * Th + k
  const float2* src = EI + (size_t)plane * XY;
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  if (tid == 0) s_cnt = 0;
  // halo tile: one warp per row, lanes walk along y
  {
    constexpr int NW = kT / 32;
    constexpr int NR = (kYXrows + NW - 1) / NW;
    float2 va[NR], vb[NR];
    if (x0 >= 3 && x0 - 3 + kYXrows <= X && y0 >= 3 && y0 - 3 + kYXcols <= Y) {  // interior tile: no periodic wrap
      const float2* q = src + (size_t)(x0 - 3 + wid) * Y + (y0 - 3 + lane);
#pragma unroll
      for (int i = 0; i < NR; ++i) {
        if (wid + i * NW < kYXrows) {
          va[i] = q[0];
          if (lane + 32 < kYXcols) vb[i] = q[32];
        }
        q += (size_t)NW * Y;
      }
    } else {  // periodic wrap: column offsets once per thread, one conditional subtract per row, 32-bit indices
      const int gy0 = modp(y0 - 3, Y);
      int gya = gy0 + lane, gyb = gy0 + lane + 32;
      gya = gya >= Y ? gya % Y : gya;
      gyb = gyb >= Y ? gyb % Y : gyb;
      const bool xnear = X >= kYXrows;
      int gx = xnear ? wrap_near(x0 - 3 + wid, X) : modp(x0 - 3 + wid, X);
      const float2* pa = src + gya;
      const float2* pb = src + gyb;
      if (xnear) {  // (block-uniform; as a select inside one loop the integer division ran for every row, taken or not)
#pragma unroll
        for (int i = 0; i < NR; ++i) {
          if (wid + i * NW < kYXrows) {
            const unsigned rb = (unsigned)(gx * Y);
            va[i] = pa[rb];
            if (lane + 32 < kYXcols) vb[i] = pb[rb];
          }
          gx += NW;
          gx -= gx >= X ? X : 0;
        }
      } else {
#pragma unroll
        for (int i = 0; i < NR; ++i) {
          if (wid + i * NW < kYXrows) {
            const unsigned rb = (unsigned)(gx * Y);
            va[i] = pa[rb];
            if (lane + 32 < kYXcols) vb[i] = pb[rb];
          }
          gx = (gx + NW) % X;
        }
      }
    }
    float2* d = s_in + wid * kInStride + lane;
#pragma unroll
    for (int i = 0; i < NR; ++i) {
      if (wid + i * NW < kYXrows) {
        d[i * NW * kInStride] = va[i];
        if (lane + 32 < kYXcols) d[i * NW * kInStride + 32] = vb[i];
      }
    }
  }
  __syncthreads();
  // y pass: item = (segment of 8 outputs, halo row); lanes walk down the rows (280 of 288 threads busy)
  if (tid < 4 * kYXrows) {
    const int seg = tid / kYXrows, r = tid - seg * kYXrows;
    const float2* sp = s_in + r * kInStride + seg * 8;
    float2 in[14];
#pragma unroll
    for (int j = 0; j < 14; ++j) in[j] = sp[j];
    float2* mp = s_mid + r * kMidStride + seg * 8;
#pragma unroll
    for (int jj = 0; jj < 8; ++jj) {
      float2 acc = make_float2(0.f, 0.f);
#pragma unroll
      for (int t = 0; t < 7; ++t) acc = __ffma2_rn(in[jj + t], tp.ty[t], acc);
      mp[jj] = acc;
    }
  }
  __syncthreads();
  // x pass: item = (segment of 8 outputs, column); lanes walk along y (256 of 288 threads busy)
  float psum = 0.f;
  if (tid < (kYXx / 8) * kYXy) {
    const int seg = wid, y = lane;
    const float2* sp = s_mid + seg * 8 * kMidStride + y;
    float2 in[14];
#pragma unroll
    for (int j = 0; j < 14; ++j) in[j] = sp[j * kMidStride];
    const float g = gi[plane / Th], g_lo = inhib_floor(g);
    const int gy = y0 + y, gx0 = x0 + seg * 8;
    float* Ap = A + (size_t)plane * XY;
    float a[8];
#pragma unroll
    for (int jj = 0; jj < 8; ++jj) {
      float2 acc = make_float2(0.f, 0.f);
#pragma unroll
      for (int t = 0; t < 7; ++t) acc = __ffma2_rn(in[jj + t], tp.tx[t], acc);
      const float d = (acc.x - acc.y) - g;
      a[jj] = d < 0.f ? g_lo : d;  // posecell_network.py:339-340: (a < gi) ? max(-gi, 0) : a - gi
    }
    // rows of this segment inside the grid (0 when the column is outside): one compare per element masks the edges
    const int nv = gy < Y ? X - gx0 : 0;
    float* q = Ap + (unsigned)(gx0 * Y + gy);
#pragma unroll
    for (int jj = 0; jj < 8; ++jj) {
      if (jj < nv) {
        q[(unsigned)(jj * Y)] = a[jj];
        psum += a[jj];
      }
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) psum += __shfl_xor_sync(0xffffffffu, psum, o);
  if (lane == 0) s_red[wid] = psum;
  if (!last_warp_of_block(&s_cnt, kT / 32)) return;
  // the last warp of the block adds the warp sums in a fixed order and publishes the tile's partial sum; the
  // grid-wide total is formed by every block of the next kernel (tile_total), so that no block of this one waits
  // for a grid-scope fence and an atomic before it can retire
  if (lane == 0) {
    float sum = 0.f;
#pragma unroll
    for (int w = 0; w < kT / 32; ++w) sum += s_red[w];
    const int ntiles = gridDim.x * gridDim.y, b = plane / Th, k = plane - b * Th;
    part[(size_t)b * Th * ntiles + (size_t)k * ntiles + blockIdx.y * gridDim.x + blockIdx.x] = sum;
  }
}

// Grid-wide sum of the previous kernel's per-tile partial sums (posecell_network.py:343), formed by ONE block per
// network -- the first block of the 7x7 kernel, as a side job after its own tile -- in a fixed order.  The 7x7
// stage itself does not need the total: it is a positive scale factor, max(s*v, 0) = s*max(v, 0), and the theta
// pass after it is linear, so 1/total is applied by the last kernel.  No block ever waits for a fence or an atomic.
__device__ __forceinline__ void block_tile_total(const float* __restrict__ part, int np, float* __restrict__ total,
                                                 float* __restrict__ inv_total, float* s_w) {
  float acc = 0.f;
  for (int i0 = threadIdx.x; i0 < np; i0 += kT * 4) {  // four independent loads in flight per thread
    float v[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) v[u] = i0 + kT * u < np ? part[i0 + kT * u] : 0.f;
#pragma unroll
    for (int u = 0; u < 4; ++u) acc += v[u];
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  __syncthreads();  // s_w may alias shared memory the tile stage has just read
  if ((threadIdx.x & 31) == 0) s_w[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    float t = 0.f;
#pragma unroll
    for (int w = 0; w < kT / 32; ++w) t += s_w[w];
    *total = t;
    *inv_total = (t != 0.f) ? 1.f / t : 1.f;  // posecell_network.py:344-345
  }
}


// ------------------------------------------------------------------------------------------------
constexpr int k2X = 64, k2Y = 32;          // outputs per tile
constexpr int k2XH = k2X + 6, k2YH = k2Y + 6;
constexpr int k2Stride = 40;               // floats per halo row, a multiple of 4 for LDS.128

__global__ void __launch_bounds__(kT) k_tl_2d(const float* __restrict__ A, float* __restrict__ Bp,
                                              const int* __restrict__ shift, const unsigned char* __restrict__ fsel,
                                              const float* __restrict__ part, int np, float* __restrict__ total,
                                              float* __restrict__ inv_total, int X, int Y, int Th,
                                              PcTables<float> tab) {
  __shared__ __align__(16) float s_a[k2XH * k2Stride];
  const int XY = X * Y;
  const int x0 = blockIdx.x * k2X, y0 = blockIdx.y * k2Y;
  const int plane = blockIdx.z;
  const float* src = A + (size_t)plane * XY;
  const int tid = threadIdx.x;
  // the plane's integer origin displaces the tile that is loaded (convolution.py:329-331)
  const int gx0 = modp(x0 + shift[2 * plane] - 3, X), gy0 = modp(y0 + shift[2 * plane + 1] - 3, Y);
  {
    const int lane = tid & 31, wid = tid >> 5;
    int gya = gy0 + lane, gyb = gy0 + lane + 32;
    gya = gya >= Y ? gya % Y : gya;
    gyb = gyb >= Y ? gyb % Y : gyb;
    constexpr int NR = (k2XH + kT / 32 - 1) / (kT / 32);
    const bool xnear = X >= k2XH;
    float va[NR], vb[NR];
#pragma unroll
    for (int i = 0; i < NR; ++i) {
      const int r = wid + i * (kT / 32);
      if (r < k2XH) {
        int gx = gx0 + r;
        gx = xnear ? (gx >= X ? gx - X : gx) : gx % X;
        const float* row = src + gx * Y;
        va[i] = row[gya];
        if (lane + 32 < k2YH) vb[i] = row[gyb];
      }
    }
#pragma unroll
    for (int i = 0; i < NR; ++i) {
      const int r = wid + i * (kT / 32);
      if (r < k2XH) {
        s_a[r * k2Stride + lane] = va[i];
        if (lane + 32 < k2YH) s_a[r * k2Stride + lane + 32] = vb[i];
      }
    }
  }
  float F[49];
  {
    const float* f = tab.f2d[fsel[plane]];
#pragma unroll
    for (int i = 0; i < 49; ++i) F[i] = f[i];
  }
  __syncthreads();
  const int xb = tid >> 3, yb = tid & 7;
  const int x = 2 * xb, y = 4 * yb;
  float acc[2][4];
#pragma unroll
  for (int d = 0; d < 2; ++d)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[d][j] = 0.f;
#pragma unroll
  for (int rr = 0; rr < 8; ++rr) {
    const float4* rp = reinterpret_cast<const float4*>(s_a + (x + rr) * k2Stride + y);
    const float4 v0 = rp[0], v1 = rp[1], v2 = rp[2];
    const float in[12] = {v0.x, v0.y, v0.z, v0.w, v1.x, v1.y, v1.z, v1.w, v2.x, v2.y, v2.z, v2.w};
    if (rr <= 6) {
#pragma unroll
      for (int j = 0; j < 4; ++j)
#pragma unroll
        for (int q = 0; q < 7; ++q) acc[0][j] = fmaf(in[j + q], F[rr * 7 + q], acc[0][j]);
    }
    if (rr >= 1) {
#pragma unroll
      for (int j = 0; j < 4; ++j)
#pragma unroll
        for (int q = 0; q < 7; ++q) acc[1][j] = fmaf(in[j + q], F[(rr - 1) * 7 + q], acc[1][j]);
    }
  }
  const int gy = y0 + y;
#pragma unroll
  for (int d = 0; d < 2; ++d) {
    const int gx = x0 + x + d;
    if (gx >= X) continue;
    float o[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) o[j] = fmaxf(acc[d][j], 0.f);  // posecell_network.py:300 (1/total: see block_tile_total)
    float* dst = Bp + (size_t)plane * XY + (size_t)gx * Y + gy;
    if ((Y & 3) == 0 && gy + 3 < Y) {
      *reinterpret_cast<float4*>(dst) = make_float4(o[0], o[1], o[2], o[3]);
    } else {
#pragma unroll
      for (int j = 0; j < 4; ++j)
        if (gy + j < Y) dst[j] = o[j];
    }
  }
  if (np > 0 && blockIdx.x == 0 && blockIdx.y == 0 && plane % Th == 0)  // side job of one block per network
    block_tile_total(part + (size_t)(plane / Th) * np, np, total + plane / Th, inv_total + plane / Th, s_a);
}

// ------------------------------------------------------------------------------------------------
// The same 7x7 stage on TWO adjacent theta planes at once with packed FFMA2 (the kernel above is bound by
// instruction issue: 49 FFMA per cell).  The two planes' tiles -- each displaced by its own origin -- are
// interleaved as float2 in shared memory; the coefficient pairs (F_k0[a][q], F_k1[a][q]) come from the constant
// bank as uniform-register operands of the FFMA2 (no registers, no shared-memory traffic).
// A thread owns a patch of 2 rows x 4 columns of outputs: 8 halo rows of 10 float2 feed 392 FFMA2.
// The eight lanes of a quarter warp read windows that start 4 float2 apart; 16-byte unit u of a row is
// therefore stored at u ^ ((u >> 3) & 1), which spreads the eight units {h, h + 2, ...} over all eight
// 16-byte bank groups: conflict-free LDS.128 (the unswizzled 2 x 4 patch needed 7.75 wavefronts per LDS.128
// and was bound by the shared-memory pipe).
constexpr int k2pX = 64;                                   // output rows per tile
constexpr int k2pW = 4;                                    // output columns per thread
constexpr int k2pY = 8 * k2pW;                             // output columns per tile
constexpr int k2pXH = k2pX + 6, k2pYH = k2pY + 6;          // halo tile
constexpr int k2pUnits = ((k2pYH + 1) / 2 + 7) / 8 * 8;    // 16-byte units per row, a multiple of 8
constexpr int k2pStride = 2 * k2pUnits;                    // float2 per halo row
constexpr int k2pNH = (k2pW + 6) / 2;                      // LDS.128 per window row
constexpr int k2pNC = (k2pYH + 31) / 32;                   // columns per lane in the fill
__device__ __forceinline__ int swz2p(int u) { return u ^ ((u >> 3) & 1); }

__global__ void __launch_bounds__(kT, 4)
    k_tl_2d_pair(const float* __restrict__ A, float* __restrict__ Bp, const int* __restrict__ shift,
                 const unsigned char* __restrict__ fsel, const float* __restrict__ part, int np,
                 float* __restrict__ total, float* __restrict__ inv_total, int X, int Y, int Th, int NPh, TlPairs tp) {
  __shared__ __align__(16) float2 s_a[k2pXH * k2pStride];
  const int XY = X * Y;
  const int x0 = blockIdx.x * k2pX, y0 = blockIdx.y * k2pY;
  const int b = blockIdx.z / NPh, kp = blockIdx.z - b * NPh;
  const int k0 = 2 * kp, k1 = (2 * kp + 1 < Th) ? 2 * kp + 1 : 2 * kp;
  const int pl0 = b * Th + k0, pl1 = b * Th + k1;
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const int combo = fsel[pl0] * 2 + fsel[pl1];  // block-uniform: the coefficient pairs come from the constant bank
  {
    // each plane's integer origin displaces the tile that is loaded (convolution.py:329-331); one warp per halo
    // row, lanes along y (columns lane, lane + 32, ...)
    constexpr int NW = kT / 32;
    constexpr int NR = (k2pXH + NW - 1) / NW;
    constexpr int NC = k2pNC;
    const bool xnear = X >= k2pXH;
    int dcol[NC];  // where this lane's columns land in the swizzled row
#pragma unroll
    for (int c = 0; c < NC; ++c) {
      const int col = lane + 32 * c;
      dcol[c] = swz2p(col >> 1) * 2 + (col & 1);
    }
    float v[2][NR][NC];
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int pl = h == 0 ? pl0 : pl1;
      const float* src = A + (size_t)pl * XY;
      const int gx0 = modp(x0 + shift[2 * pl] - 3, X), gy0 = modp(y0 + shift[2 * pl + 1] - 3, Y);
      if (gy0 + k2pYH <= Y && xnear) {  // no wrap along y (block-uniform): one row pointer, immediate column offsets
#pragma unroll
        for (int i = 0; i < NR; ++i) {
          const int r = wid + i * NW;
          if (r < k2pXH) {
            int gx = gx0 + r;
            gx -= gx >= X ? X : 0;
            const float* q = src + (size_t)gx * Y + (gy0 + lane);
#pragma unroll
            for (int c = 0; c < NC; ++c)
              if (32 * c + 32 <= k2pYH || lane + 32 * c < k2pYH) v[h][i][c] = q[32 * c];
          }
        }
      } else {
        int gy[NC];
#pragma unroll
        for (int c = 0; c < NC; ++c) {
          gy[c] = gy0 + lane + 32 * c;
          gy[c] = gy[c] >= Y ? gy[c] % Y : gy[c];
        }
#pragma unroll
        for (int i = 0; i < NR; ++i) {
          const int r = wid + i * NW;
          if (r < k2pXH) {
            int gx = gx0 + r;
            gx = xnear ? (gx >= X ? gx - X : gx) : gx % X;
            const int rb = gx * Y;
#pragma unroll
            for (int c = 0; c < NC; ++c)
              if (32 * c + 32 <= k2pYH || lane + 32 * c < k2pYH) v[h][i][c] = src[rb + gy[c]];
          }
        }
      }
    }
#pragma unroll
    for (int i = 0; i < NR; ++i) {
      const int r = wid + i * NW;
      if (r < k2pXH) {
        float2* d = s_a + r * k2pStride;
#pragma unroll
        for (int c = 0; c < NC; ++c)
          if (32 * c + 32 <= k2pYH || lane + 32 * c < k2pYH) d[dcol[c]] = make_float2(v[0][i][c], v[1][i][c]);
      }
    }
  }
  __syncthreads();
  const int xb = tid >> 3, yb = tid & 7;
  const int x = 2 * xb, y = k2pW * yb;
  // the 16-byte units of this thread's window, as pointers into row x (rows add immediates)
  const float4* rp[k2pNH];
#pragma unroll
  for (int h = 0; h < k2pNH; ++h)
    rp[h] = reinterpret_cast<const float4*>(s_a + x * k2pStride) + swz2p((k2pW / 2) * yb + h);
  float2 acc[2][k2pW];
#pragma unroll
  for (int d = 0; d < 2; ++d)
#pragma unroll
    for (int j = 0; j < k2pW; ++j) acc[d][j] = make_float2(0.f, 0.f);
#pragma unroll
  for (int rr = 0; rr < 8; ++rr) {
    float2 in[2 * k2pNH];
#pragma unroll
    for (int h = 0; h < k2pNH; ++h) {
      const float4 v = rp[h][rr * (k2pStride / 2)];
      in[2 * h] = make_float2(v.x, v.y);
      in[2 * h + 1] = make_float2(v.z, v.w);
    }
    if (rr <= 6) {
#pragma unroll
      for (int j = 0; j < k2pW; ++j)
#pragma unroll
        for (int q = 0; q < 7; ++q) acc[0][j] = __ffma2_rn(in[j + q], tp.f2p[combo][rr][q], acc[0][j]);
    }
    if (rr >= 1) {
#pragma unroll
      for (int j = 0; j < k2pW; ++j)
#pragma unroll
        for (int q = 0; q < 7; ++q) acc[1][j] = __ffma2_rn(in[j + q], tp.f2p[combo][rr - 1][q], acc[1][j]);
    }
  }
  const int gy = y0 + y;
  const bool vec = (Y & 3) == 0 && gy + k2pW - 1 < Y;
#pragma unroll
  for (int d = 0; d < 2; ++d) {
    const int gx = x0 + x + d;
    if (gx >= X) continue;
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      if (h == 1 && k1 == k0) continue;  // odd Th: the last pair has one plane
      float o[k2pW];
#pragma unroll
      for (int j = 0; j < k2pW; ++j) o[j] = fmaxf(h == 0 ? acc[d][j].x : acc[d][j].y, 0.f);  // posecell_network.py:300 (1/total: see block_tile_total)
      float* dst = Bp + (size_t)(h == 0 ? pl0 : pl1) * XY + gx * Y + gy;
      if (vec) {
#pragma unroll
        for (int j = 0; j < k2pW; j += 4) reinterpret_cast<float4*>(dst)[j / 4] = make_float4(o[j], o[j + 1], o[j + 2], o[j + 3]);
      } else {
#pragma unroll
        for (int j = 0; j < k2pW; ++j)
          if (gy + j < Y) dst[j] = o[j];
      }
    }
  }
  if (np > 0 && blockIdx.x == 0 && blockIdx.y == 0 && kp == 0)  // side job of one block per network
    block_tile_total(part + (size_t)b * np, np, total + b, inv_total + b, reinterpret_cast<float*>(s_a));
}

// ------------------------------------------------------------------------------------------------
template <int V, int TK, int MINB>
__global__ void __launch_bounds__(kT, MINB) k_tl_theta_fin(const float* __restrict__ Bp, float* __restrict__ S,
                                                     const int* __restrict__ ogi, const float* __restrict__ inv_total,
                                                     int XY, int Th, PcTables<float> tab,
                                                     float* __restrict__ part_val, long long* __restrict__ part_idx,
                                                     unsigned* __restrict__ done_ctr, long long* __restrict__ argmax) {
  __shared__ float s_v[kT / 32];
  __shared__ int s_i[kT / 32];
  __shared__ unsigned s_cnt;
  if (threadIdx.x == 0) s_cnt = 0;
  __syncthreads();  // the only barrier, before any memory latency has been incurred
  const int p = (blockIdx.x * kT + threadIdx.x) * V;
  const int k_lo = blockIdx.z * TK;
  // values are >= 0 after the clamp, so their bit patterns order like the values.  Per line (p + v) the best value
  // and its theta are tracked with a strict '>' (theta ascending: the lowest theta of a tie stays).
  float bestv[V];
  int bestk[V];
#pragma unroll
  for (int v = 0; v < V; ++v) bestv[v] = -1.f, bestk[v] = 0;
  const bool live = p < XY;
  if (live) {
    const size_t base = (size_t)blockIdx.y * Th * XY + p;
    const bool inner = k_lo >= 3 && k_lo + TK + 3 <= Th;
    const float* f = tab.f1d[ogi[blockIdx.y]];
    const float inv = inv_total[blockIdx.y];  // 1/total of the normalisation (posecell_network.py:344-345), folded into the taps
    const float f0 = pin(f[0] * inv), f1 = pin(f[1] * inv), f2 = pin(f[2] * inv), f3 = pin(f[3] * inv),
                f4 = pin(f[4] * inv), f5 = pin(f[5] * inv), f6 = pin(f[6] * inv);
    float w[TK + 6][V];
    load_window<V, TK>(Bp + base, k_lo, XY, Th, inner, w);
    float* q = S + base + (size_t)k_lo * XY;
#pragma unroll
    for (int kk = 0; kk < TK; ++kk) {
      if (inner || k_lo + kk < Th) {
        float c[V];
#pragma unroll
        for (int v = 0; v < V; ++v) {
          const float r = fmaf(f0, w[kk][v], fmaf(f1, w[kk + 1][v], fmaf(f2, w[kk + 2][v], fmaf(f3, w[kk + 3][v],
                          fmaf(f4, w[kk + 4][v], fmaf(f5, w[kk + 5][v], f6 * w[kk + 6][v]))))));
          c[v] = fmaxf(r, 0.f);  // posecell_network.py:314
          if (c[v] > bestv[v]) bestv[v] = c[v], bestk[v] = kk;
        }
        if (V == 4)
          *reinterpret_cast<float4*>(q) = make_float4(c[0], c[1 % V], c[2 % V], c[3 % V]);
        else if (V == 2)
          *reinterpret_cast<float2*>(q) = make_float2(c[0], c[1 % V]);
        else
          q[0] = c[0];
      }
      q += XY;
    }
  }
  // block arg-max (numpy.argmax: first maximum in [x][y][th] order): lines ascending with a strict '>', then
  // REDUX.MAX on the bits and REDUX.MIN on the flat index among the lanes that hold the warp's maximum
  {
    float best = bestv[0];
    int ib = p * Th + k_lo + bestk[0];
#pragma unroll
    for (int v = 1; v < V; ++v)
      if (bestv[v] > best) best = bestv[v], ib = (p + v) * Th + k_lo + bestk[v];
    const unsigned vb = (live && best >= 0.f) ? __float_as_uint(best) : 0u;
    const unsigned wmax = __reduce_max_sync(0xffffffffu, vb);
    if (!(live && best >= 0.f && vb == wmax)) ib = 0x7fffffff;  // the plan guarantees X*Y*Th < 2^31
    const int widx = __reduce_min_sync(0xffffffffu, ib);
    if ((threadIdx.x & 31) == 0) {
      s_v[threadIdx.x >> 5] = __uint_as_float(wmax);
      s_i[threadIdx.x >> 5] = widx;
    }
  }
  if (!last_warp_of_block(&s_cnt, kT / 32)) return;
  // last warp of the block: best (value, lowest index) of the block; in the last block of this network, of the grid
  const int lane = threadIdx.x & 31;
  const int nslots = gridDim.x * gridDim.z;
  float bv = lane < kT / 32 ? s_v[lane] : -1.f;
  long long bi = lane < kT / 32 ? (long long)s_i[lane] : 0x7fffffffffffffffLL;
  auto warp_best = [&]() {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const float v2 = __shfl_xor_sync(0xffffffffu, bv, o);
      const long long i2 = __shfl_xor_sync(0xffffffffu, bi, o);
      if (v2 > bv || (v2 == bv && i2 < bi)) {
        bv = v2;
        bi = i2;
      }
    }
  };
  warp_best();
  int last = 0;
  if (lane == 0) {
    const size_t slot = (size_t)blockIdx.y * nslots + (size_t)blockIdx.z * gridDim.x + blockIdx.x;
    part_val[slot] = bv;
    part_idx[slot] = bi;
    __threadfence();
    last = (atomicInc(&done_ctr[blockIdx.y], (unsigned)(nslots - 1)) == (unsigned)(nslots - 1)) ? 1 : 0;
  }
  last = __shfl_sync(0xffffffffu, last, 0);
  if (last) {
    __threadfence();
    // One warp is left: batches of eight independent L2 loads per lane (a plain loop over volatile pointers costs
    // one L2 round trip per iteration, at the very end of the kernel where nothing hides it).
    const float* pv = part_val + (size_t)blockIdx.y * nslots;
    const long long* pi = part_idx + (size_t)blockIdx.y * nslots;
    bv = -1.f;
    bi = 0x7fffffffffffffffLL;
    for (int i0 = lane; i0 < nslots; i0 += 32 * 8) {
      float v[8];
      long long ix[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        const int i = i0 + 32 * u;
        v[u] = i < nslots ? __ldcg(pv + i) : -1.f;
        ix[u] = i < nslots ? __ldcg(pi + i) : 0x7fffffffffffffffLL;
      }
#pragma unroll
      for (int u = 0; u < 8; ++u)
        if (v[u] > bv || (v[u] == bv && ix[u] < bi)) {
          bv = v[u];
          bi = ix[u];
        }
    }
    warp_best();
    if (lane == 0) argmax[blockIdx.y] = bi;
  }
}

}  // namespace

int prs_pc_tiled_supported(const prs_pc_plan* p) {
  if (p->dtype != PRS_F32) return 0;
  if ((long long)p->B * p->Th > 65535) return 0;  // gridDim.z of the tile kernels
  return (p->X * p->Y >= 1024) ? 1 : 0;
}

int prs_pc_tiled_step(prs_pc_plan* p, float* state, const double* odom, const float* gi, long long* argmax, float* total,
                      int* err, cudaStream_t st) {
  const int X = p->X, Y = p->Y, Th = p->Th, B = p->B, XY = X * Y;
  float2* EI = (float2*)p->s1;  // s1|s2 are contiguous: 2*B*N floats
  float* A = (float*)p->s3;
  float* Bp = (float*)p->s4;
  const int nchunk = (Th + kTK - 1) / kTK;
  const PlanArgs pa{odom, p->cos_th, p->sin_th, p->vtrans_scale, p->vrot_scale, p->shift, p->fsel, p->ogi, err,
                    X < Y ? X : Y};
  const int V = (XY % 2 == 0) ? 2 : 1;
  const int nline = (XY / V + kT - 1) / kT;
  if (Th >= 36 && Th % 12 == 0) {  // longer chunks re-read fewer planes: (12 + 6) / 12 loads per cell
    const dim3 g(nline, B, Th / 12);
    if (V == 2)
      k_tl_theta<2, 12><<<g, kT, 0, st>>>(state, EI, XY, Th, p->tf, pa);
    else
      k_tl_theta<1, 12><<<g, kT, 0, st>>>(state, EI, XY, Th, p->tf, pa);
  } else {
    const dim3 g(nline, B, nchunk);
    if (V == 2)
      k_tl_theta<2, kTK><<<g, kT, 0, st>>>(state, EI, XY, Th, p->tf, pa);
    else
      k_tl_theta<1, kTK><<<g, kT, 0, st>>>(state, EI, XY, Th, p->tf, pa);
  }
  const dim3 g2((X + kYXx - 1) / kYXx, (Y + kYXy - 1) / kYXy, B * Th);
  k_tl_yx<<<g2, kTyx, 0, st>>>(EI, A, gi, X, Y, Th, p->tl, (float*)p->part_val);
  const int np = Th * (int)(g2.x * g2.y);
  const int NPh = (Th + 1) / 2;
  const dim3 g3p((X + k2pX - 1) / k2pX, (Y + k2pY - 1) / k2pY, B * NPh);
  if ((long long)g3p.x * g3p.y * g3p.z >= 2 * 148) {  // enough plane pairs to fill the chip: packed FFMA2 variant
    k_tl_2d_pair<<<g3p, kT, 0, st>>>(A, Bp, p->shift, p->fsel, (const float*)p->part_val, np, total, (float*)p->inv_total, X, Y, Th, NPh, p->tl);
  } else {
    const dim3 g3((X + k2X - 1) / k2X, (Y + k2Y - 1) / k2Y, B * Th);
    k_tl_2d<<<g3, kT, 0, st>>>(A, Bp, p->shift, p->fsel, (const float*)p->part_val, np, total, (float*)p->inv_total, X, Y, Th, p->tf);
  }
  // cells x planes per thread of the shifted theta pass: 4 x 8 where X*Y allows, else 2 x 12, else 1 x 8
#define PRS_FIN(V_, TK_, MB_)                                                                                      \
  k_tl_theta_fin<V_, TK_, MB_><<<dim3((XY / V_ + kT - 1) / kT, B, (Th + TK_ - 1) / TK_), kT, 0, st>>>(              \
      Bp, state, p->ogi, (const float*)p->inv_total, XY, Th, p->tf, (float*)p->part_val, p->part_idx, p->done_ctr, \
      argmax)
  if (XY % 4 == 0)
    PRS_FIN(4, 8, 4);
  else if (XY % 2 == 0)
    PRS_FIN(2, 12, 5);
  else
    PRS_FIN(1, 8, 1);
#undef PRS_FIN
  PRS_CUDA(cudaGetLastError());
  return PRS_OK;
}
