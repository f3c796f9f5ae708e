// One pose-cell network spread over a thread-block cluster (float32, sm_100a): a low-latency path for a single
// reference-size network -- simulate.py's 50x50x10 and the ROS node's 21x21x36 -- and for ensembles too small
// to fill the chip with one CTA per network (the automatic choice while B * C <= 148 CTAs).
//
// A network update (ratslam/posecell_network.py:326-353) on ONE SM is bound by that SM's FP32 issue rate
// (98 FMA per cell: 14 us for 21x21x36, the fused resident kernel); as four grid-wide launches it is bound by
// launch and dependency latency (21 us for 50x50x10, the tiled path).  Here the C CTAs of a cluster (C = the largest
// divisor of Th that is <= 8) each own P = Th / C consecutive theta planes, keep every intermediate in their own
// shared memory, and exchange only what the two theta passes need:
//
//   load     P + 6 state planes (own planes + 3 periodic neighbours each side) global -> SMEM
//   1 theta  separable DoG along theta                                   s_in  -> s_ei  (E, I) pairs, y halo
//   2 y      7-tap pass, packed FFMA2 on (E, I)                          s_ei  -> s_mid, x halo
//   3 x      7-tap pass, A = aE*E - aI*I inhibited (inhib_floor), CTA partial sum; stored moved by the plane's integer
//            origin (convolution.py:320-340) with periodic halos         s_mid -> s_a
//   4 7x7    wrap-free correlate with the plane's LUT filter, clamp      s_a   -> s_b
//   -- cluster barrier: partial sums and s_b become visible to the other CTAs --
//   5 theta  shifted 7-tap pass (convolution.py:344-359) over own + neighbours' planes (DSMEM reads), 1/total folded
//            into the taps, clamp, -> global state; per-CTA arg-max candidate
//   -- cluster barrier -- CTA 0 picks the network's arg-max (numpy.argmax order) and writes total.
//
// Shapes are run-time values (strided item loops, ragged segments are masked); P is a template parameter so that
// the theta windows live in registers.
#include <cooperative_groups.h>

#include <mutex>

#include "common.cuh"

namespace cg = cooperative_groups;

namespace {

constexpr int kNT = 512;

// n / d for 0 <= n < 2^16 and 1 <= d < 2^16 with one multiply-high (m = floor(2^32 / d) + 1); the item loops below
// would otherwise spend more issue slots on index arithmetic than on their FMAs.
struct FastDiv {
  unsigned m;
  int d;
  FastDiv() : m(0), d(1) {}
  explicit FastDiv(int d_) : m((unsigned)(0x100000000ULL / (unsigned)d_) + 1u), d(d_) {}  // on the host, once per launch
  __device__ __forceinline__ int div(int n) const { return (int)__umulhi((unsigned)n, m); }
};

__device__ __forceinline__ unsigned smem_u32(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void st_shared_f32(unsigned addr, float v) {
  asm volatile("st.shared.f32 [%0], %1;" ::"r"(addr), "f"(v) : "memory");
}

struct ClLayout {  // element counts / strides of the shared-memory arrays, identical on host and device
  int X, Y, XY, P;
  int nsy, nsx;     // 8-wide segments along y and x
  int SE;           // s_ei row stride (float2): 8*nsy + 6 columns, odd
  int SM;           // s_mid row stride (float2): Y, odd
  int RM;           // s_mid rows per plane: 8*nsx + 6
  int SA;           // s_a row stride (float): 8*nsy + 6, odd
  int RA;           // s_a rows per plane: 2*ceil(X/2) + 6
  size_t off_in, off_ei, off_mid, off_a, off_b, off_misc, bytes;
  __host__ __device__ ClLayout(int X_, int Y_, int P_) {
    X = X_, Y = Y_, XY = X_ * Y_, P = P_;
    nsy = (Y + 7) / 8, nsx = (X + 7) / 8;
    SE = (8 * nsy + 6) | 1;
    SM = Y | 1;
    RM = 8 * nsx + 6;
    SA = (8 * nsy + 6) | 1;
    RA = 2 * ((X + 1) / 2) + 6;
    size_t o = 0;
    off_in = o, o += ((size_t)(P + 6) * XY * 4 + 15) / 16 * 16;
    off_ei = o, o += ((size_t)P * X * SE * 8 + 15) / 16 * 16;
    off_mid = o, o += ((size_t)P * RM * SM * 8 + 15) / 16 * 16;
    off_a = o, o += ((size_t)P * RA * SA * 4 + 15) / 16 * 16;
    off_b = o, o += ((size_t)P * XY * 4 + 15) / 16 * 16;
    off_misc = o, o += 2048;
    bytes = o;
  }
};

struct ClMisc {          // the small per-CTA block at off_misc
  int4 plan[9];          // (ox mod X, oy mod Y, fsel, -) of the CTA's planes
  union {
    float f2d[2][49];    // LUT filters (P odd: scalar 7x7 stage)
    float2 f2p[4][49];   // (F_p, F_{p+1}) coefficient pairs of the CTA's plane pairs (P even: packed 7x7 stage)
  };
  float red[kNT / 32];
  unsigned redv[kNT / 32];
  int redi[kNT / 32];
  float part;            // this CTA's partial sum (read by the others after the first cluster barrier)
  float best_v;          // this CTA's arg-max candidate (read by CTA 0 after the second)
  int best_i;
  int og;                // index into f1d
  int err;               // PRS_ERR_* bits of this CTA's planes (read by CTA 0 after the second cluster barrier)
};
static_assert(sizeof(ClMisc) <= 2048, "misc block must fit its slot");

struct ClArgs {
  float* state;
  const double* odom;
  const float* gi;
  long long* argmax;
  float* total;
  int* err;
  const double *cos_th, *sin_th;
  double vtrans_scale, vrot_scale;
  int X, Y, Th;
  int err_store;  // 1: err[b] is overwritten with this update's bits (no pre-zeroed buffer needed); 0: OR-ed into it
  long long* argmax2;  // optional second destination of the arg-max and the error bits (e.g. a pinned, mapped host
  int* err2;           // result record: the frame graph then needs no kernel behind this one to publish them)
  FastDiv dY, dX, dRows, dNsx, dNxp, dRows2;  // Y, X, P*X, ceil(X/8), ceil(X/2), (P/2)*X
};

template <int P>
__global__ void __launch_bounds__(kNT, 1) k_pc_cluster(ClArgs a, PcTables<float> tab, TlPairs tp) {
  cg::cluster_group cluster = cg::this_cluster();
  const int C = (int)cluster.num_blocks();
  const int rank = (int)cluster.block_rank();
  const int b = blockIdx.x / C;
  const int X = a.X, Y = a.Y, Th = a.Th, XY = X * Y;
  const ClLayout L(X, Y, P);  // constants of the launch: folded by the compiler into a few multiplies
  extern __shared__ __align__(16) unsigned char smem[];
  float* s_in = reinterpret_cast<float*>(smem + L.off_in);
  float2* s_ei = reinterpret_cast<float2*>(smem + L.off_ei);
  float2* s_mid = reinterpret_cast<float2*>(smem + L.off_mid);
  float* s_a = reinterpret_cast<float*>(smem + L.off_a);
  float* s_b = reinterpret_cast<float*>(smem + L.off_b);
  ClMisc* m = reinterpret_cast<ClMisc*>(smem + L.off_misc);
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const int k0 = rank * P;
  float* gst = a.state + (size_t)b * Th * XY;

  // ---- decisions of this update for the CTA's planes, float64 exactly as numpy computes them on the host
  //      (posecell_network.py:252-267,249,304); LUT filters into shared memory
  if (wid == 0) {
    int e = 0;
    if (tid < P) {
      const int k = k0 + tid;
      const double* od = a.odom + (size_t)b * 2;
      const double vt = __ddiv_rn(od[0], a.vtrans_scale);
      const double ex = __dmul_rn(vt, a.cos_th[k]);
      const double ey = __dmul_rn(vt, a.sin_th[k]);
      const double oxd = rint(ex), oyd = rint(ey);  // numpy.around: half to even
      const int key = (int)__dmul_rn(__dsub_rn(ex, oxd), 10.0);
      m->plan[tid] = make_int4(modp((int)oxd, X), modp((int)oyd, Y), key < 0 ? 1 : 0, 0);
      e = key >= 5 ? PRS_ERR_LUT_KEY : 0;
      if (tid == 0) {
        if (!(3.0 + ceil(fabs(vt)) <= (double)(X < Y ? X : Y))) e |= PRS_ERR_RADIUS;
        const double og = floor(__dadd_rn(__ddiv_rn(od[1], a.vrot_scale), 0.5));
        if (!(fabs(og) <= 64.0)) e |= PRS_ERR_THETA;
        const int ogc = og < -(double)PRS_OG_RANGE ? -PRS_OG_RANGE : (og > (double)PRS_OG_RANGE ? PRS_OG_RANGE : (int)og);
        m->og = ogc + PRS_OG_RANGE;
      }
    }
    e = (int)__reduce_or_sync(0xffffffffu, (unsigned)e);
    if (tid == 0) m->err = e;
  }
  if (P % 2 != 0)
    for (int i = tid; i < 98; i += kNT) m->f2d[i / 49][i % 49] = tab.f2d[i / 49][i % 49];

  // ---- load the P + 6 planes this CTA's theta pass reads: all of a thread's loads are issued before the first
  //      store (one memory round trip per 512 elements of a plane, not one per plane)
  {
    const float* srcp[P + 6];
#pragma unroll
    for (int j = 0; j < P + 6; ++j) srcp[j] = gst + (size_t)wrap1(k0 - 3 + j, Th) * XY;  // Th >= 3
    if ((XY & 3) == 0) {
      const int n4 = XY >> 2;
      for (int i = tid; i < n4; i += kNT) {
        float4 v[P + 6];
#pragma unroll
        for (int j = 0; j < P + 6; ++j) v[j] = reinterpret_cast<const float4*>(srcp[j])[i];
#pragma unroll
        for (int j = 0; j < P + 6; ++j) reinterpret_cast<float4*>(s_in + j * XY)[i] = v[j];
      }
    } else {
      for (int i = tid; i < XY; i += kNT) {
        float v[P + 6];
#pragma unroll
        for (int j = 0; j < P + 6; ++j) v[j] = srcp[j][i];
#pragma unroll
        for (int j = 0; j < P + 6; ++j) s_in[j * XY + i] = v[j];
      }
    }
  }
  __syncthreads();
  if (P % 2 == 0) {  // coefficient pairs of the plane pairs (the plan is visible after the barrier)
    for (int i = tid; i < (P / 2) * 49; i += kNT) {
      const int pp = i / 49, t = i - pp * 49;
      m->f2p[pp % 4][t] = make_float2(tab.f2d[m->plan[2 * pp].z][t], tab.f2d[m->plan[2 * pp + 1].z][t]);
    }
  }
  const FastDiv dY = a.dY, dX = a.dX;

  // ---- 1. theta pass of the separable DoG: one cell per item, window of P + 6 planes in registers
  {
    const float e0 = tab.ge[3], e1 = tab.ge[2], e2 = tab.ge[1], e3 = tab.ge[0];
    const float i0 = tab.gi[3], i1 = tab.gi[2], i2 = tab.gi[1], i3 = tab.gi[0];
    for (int c = tid; c < XY; c += kNT) {
      const int x = dY.div(c), y = c - x * Y;
      float w[P + 6];
#pragma unroll
      for (int j = 0; j < P + 6; ++j) w[j] = s_in[j * XY + c];
      const int hal = y < 3 ? Y : (y >= Y - 3 ? -Y : 0);  // periodic image of this column inside the y halo
#pragma unroll
      for (int p = 0; p < P; ++p) {
        const float s1 = w[p + 2] + w[p + 4], s2 = w[p + 1] + w[p + 5], s3 = w[p] + w[p + 6];
        const float e = fmaf(e0, w[p + 3], fmaf(e1, s1, fmaf(e2, s2, e3 * s3)));
        const float i = fmaf(i0, w[p + 3], fmaf(i1, s1, fmaf(i2, s2, i3 * s3)));
        float2* row = s_ei + (p * X + x) * L.SE;
        row[y + 3] = make_float2(e, i);
        if (hal != 0) row[y + 3 + hal] = make_float2(e, i);
      }
    }
  }
  __syncthreads();

  // ---- 2. y pass: item = (row of a plane, 8-output segment); lanes walk down the rows (odd row stride)
  {
    const int rows = P * X;
    const FastDiv dR = a.dRows;
    for (int it = tid; it < rows * L.nsy; it += kNT) {
      const int seg = dR.div(it), r = it - seg * rows;
      const int p = dX.div(r), x = r - p * X;
      const float2* sp = s_ei + r * L.SE + seg * 8;
      float2 in[14];
#pragma unroll
      for (int j = 0; j < 14; ++j) in[j] = sp[j];
      float2* mp = s_mid + (p * L.RM + x + 3) * L.SM + seg * 8;
      const int hal = x < 3 ? X : (x >= X - 3 ? -X : 0);
#pragma unroll
      for (int jj = 0; jj < 8; ++jj) {
        float2 acc = make_float2(0.f, 0.f);
#pragma unroll
        for (int t = 0; t < 7; ++t) acc = __ffma2_rn(in[jj + t], tp.ty[t], acc);
        if (seg * 8 + jj < Y) {
          mp[jj] = acc;
          if (hal != 0) mp[hal * L.SM + jj] = acc;
        }
      }
    }
  }
  __syncthreads();

  // ---- 3. x pass + inhibition (posecell_network.py:339-340) + partial sum (:343); the result is stored moved by
  //         the plane's integer origin, with 3 periodic halo rows and columns, so that stage 4 never wraps
  {
    float psum = 0.f;
    const float g = a.gi[b], g_lo = inhib_floor(g);
    const FastDiv dS = a.dNsx;
    for (int it = tid; it < P * L.nsx * Y; it += kNT) {
      const int t2 = dY.div(it), y = it - t2 * Y;
      const int p = dS.div(t2), seg = t2 - p * L.nsx;
      const float2* sp = s_mid + (p * L.RM + seg * 8) * L.SM + y;
      float2 in[14];
#pragma unroll
      for (int j = 0; j < 14; ++j) in[j] = sp[j * L.SM];
      const int4 pl = m->plan[p];
      int yd = y - pl.y;
      yd += yd < 0 ? Y : 0;
      const int yh = yd < 3 ? Y : (yd >= Y - 3 ? -Y : 0);
      // s_a: planes 2q, 2q+1 interleaved as float2 when P is even (stage 4 then runs packed FFMA2 on the pair)
      constexpr int ES = (P % 2 == 0) ? 2 : 1;
      float* ap = (P % 2 == 0) ? s_a + (p >> 1) * (L.RA * L.SA * 2) + (p & 1) : s_a + p * (L.RA * L.SA);
      int xd = seg * 8 - pl.x;  // destination row of output 0; rows advance with a periodic wrap
      xd += xd < 0 ? X : 0;
      // byte address in shared memory, advanced incrementally (left to itself the compiler re-derives the closed
      // form -- some 30 integer instructions -- for every one of the 8 outputs)
      unsigned sa = smem_u32(ap) + 4u * (unsigned)(((xd + 3) * L.SA + yd + 3) * ES);
      const int rstepb = 4 * L.SA * ES, yoffb = 4 * yh * ES, Xb = X * rstepb;
#pragma unroll
      for (int jj = 0; jj < 8; ++jj) {
        float2 acc = make_float2(0.f, 0.f);
#pragma unroll
        for (int t = 0; t < 7; ++t) acc = __ffma2_rn(in[jj + t], tp.tx[t], acc);
        if (seg * 8 + jj < X) {
          const float d = (acc.x - acc.y) - g;
          const float v = d < 0.f ? g_lo : d;  // (a < gi) ? max(-gi, 0) : a - gi, see inhib_floor
          psum += v;
          const int xoffb = xd < 3 ? Xb : (xd >= X - 3 ? -Xb : 0);
          st_shared_f32(sa, v);
          if (yh != 0) st_shared_f32(sa + yoffb, v);
          if (xoffb != 0) {
            st_shared_f32(sa + xoffb, v);
            if (yh != 0) st_shared_f32(sa + xoffb + yoffb, v);
          }
        }
        ++xd;
        sa += rstepb;
        if (xd == X) xd = 0, sa -= Xb;
        asm volatile("" : "+r"(sa), "+r"(xd));
      }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) psum += __shfl_xor_sync(0xffffffffu, psum, o);
    if (lane == 0) m->red[wid] = psum;
  }
  __syncthreads();
  if (tid == 0) {
    float s = 0.f;
#pragma unroll
    for (int w = 0; w < kNT / 32; ++w) s += m->red[w];
    m->part = s;
  }

  // ---- 4. 7x7 correlate (posecell_network.py:273-274) of 2 rows x 8 columns per item, clamp (:300); with an even
  //         number of planes two planes go through it at once as float2 (packed FFMA2, coefficient pairs)
  if (P % 2 == 0) {  // item = (plane pair, row, 8 columns): a short critical path matters more here than reuse
    const int rows = (P / 2) * X;
    const FastDiv dR = a.dRows2;
    for (int it = tid; it < rows * L.nsy; it += kNT) {
      const int seg = dR.div(it), r = it - seg * rows;
      const int pp = dX.div(r), x = r - pp * X;
      const float2* F = m->f2p[pp % 4];
      const float2* ap = reinterpret_cast<const float2*>(s_a) + (pp * L.RA + x) * L.SA + seg * 8;
      float2 acc[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) acc[j] = make_float2(0.f, 0.f);
#pragma unroll
      for (int rr = 0; rr < 7; ++rr) {
        float2 in[14];
#pragma unroll
        for (int j = 0; j < 14; ++j) in[j] = ap[rr * L.SA + j];
#pragma unroll
        for (int q = 0; q < 7; ++q) {
          const float2 f = F[rr * 7 + q];
#pragma unroll
          for (int j = 0; j < 8; ++j) acc[j] = __ffma2_rn(in[j + q], f, acc[j]);
        }
      }
      float* o0 = s_b + (2 * pp) * XY + x * Y + seg * 8;
#pragma unroll
      for (int j = 0; j < 8; ++j)
        if (seg * 8 + j < Y) {
          o0[j] = fmaxf(acc[j].x, 0.f);
          o0[XY + j] = fmaxf(acc[j].y, 0.f);
        }
    }
  } else
  {
    const int nxp = (X + 1) / 2;
    const int rows = P * nxp;
    for (int it = tid; it < rows * L.nsy; it += kNT) {
      const int seg = it / rows, r = it - seg * rows;
      const int p = r / nxp, x = 2 * (r - p * nxp);
      const float* F = m->f2d[m->plan[p].z];
      const float* ap = s_a + (p * L.RA + x) * L.SA + seg * 8;
      float acc[2][8];
#pragma unroll
      for (int d = 0; d < 2; ++d)
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[d][j] = 0.f;
#pragma unroll
      for (int rr = 0; rr < 8; ++rr) {
        float in[14];
#pragma unroll
        for (int j = 0; j < 14; ++j) in[j] = ap[rr * L.SA + j];
        if (rr <= 6) {
#pragma unroll
          for (int q = 0; q < 7; ++q) {
            const float f = F[rr * 7 + q];
#pragma unroll
            for (int j = 0; j < 8; ++j) acc[0][j] = fmaf(in[j + q], f, acc[0][j]);
          }
        }
        if (rr >= 1) {
#pragma unroll
          for (int q = 0; q < 7; ++q) {
            const float f = F[(rr - 1) * 7 + q];
#pragma unroll
            for (int j = 0; j < 8; ++j) acc[1][j] = fmaf(in[j + q], f, acc[1][j]);
          }
        }
      }
#pragma unroll
      for (int d = 0; d < 2; ++d) {
        if (x + d < X) {
          float* o = s_b + p * XY + (x + d) * Y + seg * 8;
#pragma unroll
          for (int j = 0; j < 8; ++j)
            if (seg * 8 + j < Y) o[j] = fmaxf(acc[d][j], 0.f);
        }
      }
    }
  }
  cluster.sync();  // every CTA's s_b and partial sum are complete and visible cluster-wide

  // ---- total and 1/total (posecell_network.py:343-345), the same fixed order in every CTA
  float tot = 0.f;
  for (int r = 0; r < C; ++r) tot += cluster.map_shared_rank(&m->part, r)[0];
  const float inv = (tot != 0.f) ? 1.f / tot : 1.f;

  // ---- 5. shifted theta pass (convolution.py:344-359), clamp (:314), -> global.  The window's planes -- own ones
  //         and three neighbours each side, which live in other CTAs (DSMEM) -- are first gathered into s_in.
  {
    const float* srcp[P + 6];  // plane k0 - 3 + j lives in CTA ((k mod Th) / P) at local index (k mod Th) % P
#pragma unroll
    for (int j = 0; j < P + 6; ++j) {
      const int k = wrap1(k0 - 3 + j, Th);
      const int owner = k / P;
      srcp[j] = (owner == rank ? s_b : cluster.map_shared_rank(s_b, owner)) + (k - owner * P) * XY;
    }
    if ((XY & 3) == 0) {
      for (int i = tid; i < (XY >> 2); i += kNT) {
        float4 v[P + 6];
#pragma unroll
        for (int j = 0; j < P + 6; ++j) v[j] = reinterpret_cast<const float4*>(srcp[j])[i];
#pragma unroll
        for (int j = 0; j < P + 6; ++j) reinterpret_cast<float4*>(s_in + j * XY)[i] = v[j];
      }
    } else {
      for (int i = tid; i < XY; i += kNT) {
        float v[P + 6];
#pragma unroll
        for (int j = 0; j < P + 6; ++j) v[j] = srcp[j][i];
#pragma unroll
        for (int j = 0; j < P + 6; ++j) s_in[j * XY + i] = v[j];
      }
    }
  }
  __syncthreads();
  float best = -1.f;
  int bidx = 0x7fffffff;
  {
    const float* f1 = tab.f1d[m->og];
    float fc[7];
#pragma unroll
    for (int t = 0; t < 7; ++t) fc[t] = f1[t] * inv;
    for (int c = tid; c < XY; c += kNT) {
      float w[P + 6];
#pragma unroll
      for (int j = 0; j < P + 6; ++j) w[j] = s_in[j * XY + c];
      const int flat0 = c * Th + k0;  // [x][y][th] order: c = x * Y + y
      float* gp = gst + (size_t)k0 * XY + c;
#pragma unroll
      for (int p = 0; p < P; ++p) {
        float r = fc[6] * w[p + 6];
#pragma unroll
        for (int t = 5; t >= 0; --t) r = fmaf(fc[t], w[p + t], r);
        r = fmaxf(r, 0.f);
        gp[(size_t)p * XY] = r;
        if (r > best) best = r, bidx = flat0 + p;  // a thread's cells come in ascending flat order
      }
    }
  }
  // CTA arg-max (numpy.argmax: first maximum in [x][y][th] order): values are >= 0, bit patterns order like values
  {
    const unsigned vb = best >= 0.f ? __float_as_uint(best) : 0u;
    const unsigned wmax = __reduce_max_sync(0xffffffffu, vb);
    const int widx = __reduce_min_sync(0xffffffffu, (best >= 0.f && vb == wmax) ? bidx : 0x7fffffff);
    if (lane == 0) m->redv[wid] = wmax, m->redi[wid] = widx;
    __syncthreads();
    if (wid == 0) {
      const unsigned v = lane < kNT / 32 ? m->redv[lane] : 0u;
      const int ix = lane < kNT / 32 ? m->redi[lane] : 0x7fffffff;
      const unsigned bmax = __reduce_max_sync(0xffffffffu, v);
      const int bi = __reduce_min_sync(0xffffffffu, v == bmax ? ix : 0x7fffffff);
      if (lane == 0) m->best_v = __uint_as_float(bmax), m->best_i = bi;
    }
  }
  cluster.sync();  // candidates visible; nobody reads another CTA's s_b any more
  if (rank == 0 && tid == 0) {
    float bv = -1.f;
    int bi = 0x7fffffff;
    for (int r = 0; r < C; ++r) {
      const float v = cluster.map_shared_rank(&m->best_v, r)[0];
      const int ix = cluster.map_shared_rank(&m->best_i, r)[0];
      if (v > bv || (v == bv && ix < bi)) bv = v, bi = ix;
    }
    a.argmax[b] = bi;
    a.total[b] = tot;
    int e = 0;
    for (int r = 0; r < C; ++r) e |= cluster.map_shared_rank(&m->err, r)[0];
    if (a.err_store)
      a.err[b] = e;
    else if (e)
      atomicOr(a.err + b, e);
    if (a.argmax2 != nullptr) {
      a.argmax2[b] = bi;
      a.err2[b] = e;
    }
  }
  cluster.sync();  // CTA 0 has read every candidate: shared memory may go away
}

template <int P>
cudaLaunchConfig_t make_config(const prs_pc_plan* p, int C, size_t smem, cudaStream_t st, cudaLaunchAttribute* attr) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(p->B * C, 1, 1);
  cfg.blockDim = dim3(kNT, 1, 1);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = C;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  return cfg;
}

// Can a cluster of C CTAs with this much shared memory be co-scheduled on the current device?  Sets the function
// attributes the launch needs (shared-memory opt-in; non-portable cluster sizes above 8) as a side effect.
template <int P>
int cluster_fits(const prs_pc_plan* p, int C) {  // the number of clusters of C CTAs the device runs at once (0: none)
  const ClLayout L(p->X, p->Y, P);
  if (L.bytes > (size_t)227 * 1024) return 0;
  auto kern = k_pc_cluster<P>;
  static size_t smem_set[64] = {};  // the opt-in limit is only ever raised: other plans may need the larger value
  static std::mutex mu;
  std::lock_guard<std::mutex> lk(mu);
  if (p->device < 0 || p->device >= 64) return 0;
  const size_t want = L.bytes > smem_set[p->device] ? L.bytes : smem_set[p->device];
  if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)want) != cudaSuccess ||
      (C > 8 && cudaFuncSetAttribute(kern, cudaFuncAttributeNonPortableClusterSizeAllowed, 1) != cudaSuccess)) {
    (void)cudaGetLastError();
    return 0;
  }
  smem_set[p->device] = want;
  cudaLaunchAttribute attr[1];
  cudaLaunchConfig_t cfg = make_config<P>(p, C, L.bytes, nullptr, attr);
  cfg.gridDim = dim3(C, 1, 1);
  int n = 0;
  if (cudaOccupancyMaxActiveClusters(&n, kern, &cfg) != cudaSuccess) {
    (void)cudaGetLastError();
    return 0;
  }
  return n;
}

template <int P>
int launch(prs_pc_plan* p, int C, const ClArgs& args, cudaStream_t st) {
  const ClLayout L(p->X, p->Y, P);
  cudaLaunchAttribute attr[1];
  cudaLaunchConfig_t cfg = make_config<P>(p, C, L.bytes, st, attr);
  PRS_CUDA(cudaLaunchKernelEx(&cfg, k_pc_cluster<P>, args, p->tf, p->tl));
  return PRS_OK;
}

int fits_dispatch(const prs_pc_plan* p, int C, int P) {
  switch (P) {
    case 1: return cluster_fits<1>(p, C);
    case 2: return cluster_fits<2>(p, C);
    case 3: return cluster_fits<3>(p, C);
    case 4: return cluster_fits<4>(p, C);
    case 5: return cluster_fits<5>(p, C);
    case 6: return cluster_fits<6>(p, C);
    case 7: return cluster_fits<7>(p, C);
    case 8: return cluster_fits<8>(p, C);
    case 9: return cluster_fits<9>(p, C);
  }
  return 0;
}

}  // namespace

// Plan-time choice of the cluster size C (a divisor of Th, up to 16; sizes above 8 are "non-portable" and are only
// taken if the occupancy query confirms them on this device; a CTA holds P = Th / C <= 9 planes within the
// shared-memory limit).  More CTAs mean less work on each one's critical path -- measured for ONE 21x21x36 network:
// 9.9 us (C = 9), 10.3 (C = 12), 11.4 (C = 6), 13.6 (C = 4) -- but only while all B clusters run at once: the device
// co-schedules about 12 clusters of 9, 16 of 6, 24 of 4 (cudaOccupancyMaxActiveClusters), and a second wave doubles the
// time (profiles/r2_b_sweep.txt).  So: the largest C whose clusters all fit at once for this B; an even P (the packed
// two-plane 7x7 stage) is preferred over a slightly larger C with an odd P.  *one_wave tells whether the chosen C runs
// the B networks in a single wave.  Returns C, or 0 if the path does not apply to this plan.
int prs_pc_cluster_choose(const prs_pc_plan* p, int* one_wave) {
  if (one_wave) *one_wave = 0;
  if (p->dtype != PRS_F32) return 0;
  if (p->X < 7 || p->Y < 7) return 0;  // a halo of 3 must be a single periodic image
  if ((long long)p->X * p->Y >= 65536) return 0;  // FastDiv range
  int cand[16], nact[16], nc = 0;
  for (int C = 16; C >= 2; --C) {
    if (p->Th % C != 0) continue;
    const int P = p->Th / C;
    if (P > 9) break;
    const int n = fits_dispatch(p, C, P);
    if (n >= 1) cand[nc] = C, nact[nc] = n, ++nc;
  }
  if (nc == 0) return 0;
  int pick = -1;
  for (int i = 0; i < nc && pick < 0; ++i)
    if (p->B <= nact[i]) pick = i;
  if (pick < 0) return cand[0];  // more networks than any cluster size runs at once: not the automatic choice anyway
  if (one_wave) *one_wave = 1;
  const int P = p->Th / cand[pick];
  if ((P & 1) && pick + 1 < nc && p->B <= nact[pick + 1] && ((p->Th / cand[pick + 1]) & 1) == 0 &&
      10 * cand[pick + 1] >= 7 * cand[pick])
    ++pick;
  return cand[pick];
}

int prs_pc_cluster_step(prs_pc_plan* p, float* state, const double* odom, const float* gi, long long* argmax,
                        float* total, int* err, int err_store, cudaStream_t st, long long* argmax2, int* err2) {
  const int C = p->cluster_C;
  PRS_REQUIRE(C >= 2, "cluster path not available for this plan");
  const int P = p->Th / C;
  ClArgs args{state, odom, gi, argmax, total, err, p->cos_th, p->sin_th, p->vtrans_scale, p->vrot_scale,
              p->X, p->Y, p->Th, err_store, argmax2, err2};
  const int nxp = (p->X + 1) / 2;
  args.dY = FastDiv(p->Y);
  args.dX = FastDiv(p->X);
  args.dRows = FastDiv(P * p->X);
  args.dNsx = FastDiv((p->X + 7) / 8);
  args.dNxp = FastDiv(nxp);
  args.dRows2 = FastDiv(P >= 2 ? (P / 2) * p->X : 1);
  switch (P) {
    case 1: return launch<1>(p, C, args, st);
    case 2: return launch<2>(p, C, args, st);
    case 3: return launch<3>(p, C, args, st);
    case 4: return launch<4>(p, C, args, st);
    case 5: return launch<5>(p, C, args, st);
    case 6: return launch<6>(p, C, args, st);
    case 7: return launch<7>(p, C, args, st);
    case 8: return launch<8>(p, C, args, st);
    case 9: return launch<9>(p, C, args, st);
  }
  prs_set_error("cluster path not available for this plan");
  return PRS_E_INVALID;
}
