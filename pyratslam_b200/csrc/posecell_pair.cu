// Fused, SMEM-resident pose-cell update with ONE NETWORK PER 2-CTA CLUSTER (sm_100a), float32 and float64.
//
// The whole PoseCellNetwork.update() (ratslam/posecell_network.py:326-353) -- 7x7x7 DoG correlate, global
// inhibition, normalisation, per-heading shifted 7x7 correlate, 7-tap theta correlate, arg-max -- runs with the
// state in shared memory between the stages, as in posecell_resident.cu; HBM sees one read and one write of the
// state per update (8 B per cell in float32, 16 B in float64).  What is different: the network is split in two theta
// halves over the two CTAs of a thread-block cluster.  A half needs 77 KB of shared memory (float32) instead of the
// 213 KB of the one-CTA kernel, so TWO networks' worth of CTAs are resident on every SM: while one CTA sits in one of
// the short, latency-bound stages (theta / y / x passes, reductions, barriers) the other one keeps the FP32 pipe busy
// with its 7x7 stage.  (Round 1's one-CTA kernel ran 14 warps per SM at 52 % FMA-pipe activity with 16 % of its
// samples waiting at barriers.)  The same halving is what makes a float64 network fit at all (145 KB per CTA).
//
// Theta halves.  With T planes, MID = T/2 and H = T/2 planes per CTA, CTA r owns the window of H consecutive planes
// that is centred on CC = MID (r = 0) or plane 0 (r = 1): local plane l = 0..H-1 is global plane (CC - H/2 + l) mod T.
// cos((k - MID) 2pi/T) is even about both centres, so inside a window the planes CC + q and CC - q (local H/2 +- q)
// have the same cosine: the same integer x origin (posecell_network.py:252-267) and the same LUT filter.  They are
// processed as one float2 "plane pair" q = 1..H/2-1 by the packed FFMA2 stages, exactly like the mirror pairs of
// the one-CTA kernel; pair 0 is (centre, edge) = (local H/2, local 0), whose x origins differ: the edge plane is
// stored rotated by the difference in stage 1 (every stage up to the 2-D one is a periodic correlate and commutes
// with that translation).
//
// Stages of one CTA (X*Y = 441 lines of a 21x21x36 network, NQ = 9 plane pairs):
//   1 theta pass   thread = (x,y) line: H + 6 planes from global memory (the 3-plane halos of the window are simply
//                  read as well: 24 of 36 planes per CTA, the overlap comes from L2) -> (E, I) pairs      11 op / cell
//   2 y pass       thread = (plane, x) line, in place, FFMA2 on (E, I)                                    7 FFMA2 / cell
//   3 x pass       thread = (pair, y) column of both planes, A = aE*E - aI*I inhibited (inhib_floor), partial sum;
//                  written with 3 periodic halo rows as the float2 pair tensor A2                          7 FFMA2 / cell
//   4 7x7 stage    thread = (pair, x) row, FFMA2 over the pair, result row stored at x - ox                24.5 FFMA2 / cell
//   -- cluster barrier: B2 and the partial sums are visible to the peer --
//   5 theta pass   thread = (x,y) line: own H planes from B2, 3 + 3 halo planes from the PEER's B2 through
//                  distributed shared memory, 1/total folded into the taps, clamp, -> global, arg-max    3.5 FFMA2 / cell
//   -- cluster barrier: the peer has read my B2; CTA 1's arg-max candidate has reached CTA 0 --
// The grid is persistent: as many clusters as are co-resident (2 CTAs per SM in float32) stride over the networks.
#include <cooperative_groups.h>

#include <mutex>

#include "common.cuh"

namespace cg = cooperative_groups;

namespace {

template <typename R>
struct Vec2;
template <>
struct Vec2<float> {
  using type = float2;
};
template <>
struct Vec2<double> {
  using type = double2;
};

__device__ __forceinline__ float2 fma2(float2 a, float2 b, float2 c) { return __ffma2_rn(a, b, c); }
__device__ __forceinline__ double2 fma2(double2 a, double2 b, double2 c) {
  return make_double2(fma(a.x, b.x, c.x), fma(a.y, b.y, c.y));
}
__device__ __forceinline__ float2 add2(float2 a, float2 b) { return __fadd2_rn(a, b); }
__device__ __forceinline__ double2 add2(double2 a, double2 b) { return make_double2(a.x + b.x, a.y + b.y); }
__device__ __forceinline__ float2 mk2(float a, float b) { return make_float2(a, b); }
__device__ __forceinline__ double2 mk2(double a, double b) { return make_double2(a, b); }
__device__ __forceinline__ float max0(float v) { return fmaxf(v, 0.f); }
__device__ __forceinline__ double max0(double v) { return fmax(v, 0.0); }
// bit patterns of non-negative values order like the values
__device__ __forceinline__ unsigned long long val_bits(float v) { return (unsigned long long)__float_as_uint(v); }
__device__ __forceinline__ unsigned long long val_bits(double v) { return (unsigned long long)__double_as_longlong(v); }

template <int X, int Y, int T, typename R>
struct PairLayout {
  using R2 = typename Vec2<R>::type;
  static constexpr int XY = X * Y;
  static constexpr int H = T / 2;    // planes per CTA
  static constexpr int LC = H / 2;   // local index of the window's centre plane
  static constexpr int NQ = H / 2;   // plane pairs per CTA: (centre, edge) and LC - 1 mirror pairs
  // A2 plane: X + 6 rows (3 periodic halo rows each side: stage 4 never wraps an index); the plane stride is padded
  // until PS == X*Y (mod 16), which keeps the warp-wide 64-bit loads of stage 4 conflict free (see posecell_resident.cu)
  static constexpr int kPSraw = (X + 6) * Y;
  static constexpr int PS = kPSraw + ((XY % 16) - (kPSraw % 16) + 16) % 16;
  static constexpr int kPlanInts = 4 * T + 4;  // int4 (ox, oy, -, fsel)[T], misc[4]
  static constexpr size_t kElems = (size_t)(NQ * PS + NQ * XY > H * XY ? NQ * PS + NQ * XY : H * XY);
  static constexpr size_t kBufOff = 0;                                       // R2[kElems]: (E, I), later A2 | B2
  static constexpr size_t kTabOff = (sizeof(R2) * kElems + 15) / 16 * 16;    // PcTables<R>
  static constexpr size_t kPairOff = (kTabOff + sizeof(PcTables<R>) + 15) / 16 * 16;  // R2[4][7][8] paired 2-D coefficients
  static constexpr size_t kCfOff = kPairOff + 4 * 7 * 8 * sizeof(R2);        // R2[7] (ge, gi), R2[7] (gex, gix)
  static constexpr size_t kPlanOff = kCfOff + 14 * sizeof(R2);               // two plans (double buffered)
  static constexpr size_t kRedOff = (kPlanOff + 2 * kPlanInts * 4 + 15) / 16 * 16;
  // reduction scratch: u64 wmax[32]; R wsum[32]; R part[2]; u64 peer_val; int peer_flat; int best_flat; int err
  static constexpr size_t kBytes = kRedOff + 32 * 8 + 32 * sizeof(R) + 2 * sizeof(R) + 8 + 4 + 4 + 16;
};

// Decisions of one update for theta plane k, float64 exactly as numpy computes them on the host
// (posecell_network.py:252-267,249,304).  plan[k] = (ox mod X, oy mod Y, -, LUT filter).
template <int X, int Y, int T>
__device__ __forceinline__ void pair_plan_plane(int k, const double* __restrict__ od, const double* __restrict__ cos_th,
                                                const double* __restrict__ sin_th, double vtrans_scale,
                                                double vrot_scale, int* plan, int* err_b) {
  const double vt = __ddiv_rn(od[0], vtrans_scale);
  const double ex = __dmul_rn(vt, cos_th[k]);
  const double ey = __dmul_rn(vt, sin_th[k]);
  const double oxd = rint(ex), oyd = rint(ey);  // numpy.around: half to even
  const int key = (int)__dmul_rn(__dsub_rn(ex, oxd), 10.0);
  const int ox = modp((int)oxd, X), oy = modp((int)oyd, Y);
  reinterpret_cast<int4*>(plan)[k] = make_int4(ox, oy, 0, key < 0 ? 1 : 0);
  int e = key >= 5 ? PRS_ERR_LUT_KEY : 0;
  if (k == 0) {
    if (!(3.0 + ceil(fabs(vt)) <= (double)(X < Y ? X : Y))) e |= PRS_ERR_RADIUS;
    const double og = floor(__dadd_rn(__ddiv_rn(od[1], vrot_scale), 0.5));
    if (!(fabs(og) <= 64.0)) e |= PRS_ERR_THETA;
    const int ogc = og < -(double)PRS_OG_RANGE ? -PRS_OG_RANGE : (og > (double)PRS_OG_RANGE ? PRS_OG_RANGE : (int)og);
    plan[4 * T] = ogc + PRS_OG_RANGE;
  }
  if (e && err_b != nullptr) atomicOr(err_b, e);
}

template <int X, int Y, int T, int NT, typename R>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(NT, sizeof(R) == 4 ? 2 : 1)
    k_pc_pair(R* state, const double* __restrict__ odom, int n_steps, const R* __restrict__ gi,
              long long* __restrict__ argmax, R* __restrict__ total, int* __restrict__ err,
              const double* __restrict__ cos_th, const double* __restrict__ sin_th, double vtrans_scale,
              double vrot_scale, int B, const __grid_constant__ PcTables<R> tabp) {
  using L = PairLayout<X, Y, T, R>;
  using R2 = typename L::R2;
  constexpr int XY = L::XY, H = L::H, LC = L::LC, NQ = L::NQ, PS = L::PS, MID = T / 2;
  constexpr int NW = NT / 32;
  constexpr int kPlanT0 = NT - 64;  // the threads that prepare the next update's plan during stage 4
  static_assert(X >= 7 && Y >= 7, "the pair kernel needs X, Y >= 7");
  static_assert(T % 4 == 0 && T >= 16 && T <= 64, "theta halves of an even number of planes, at least 8 each");
  static_assert(NT % 32 == 0 && kPlanT0 >= NQ * X && NQ * Y <= NT, "one work item per thread in stages 3 and 4");
  cg::cluster_group cluster = cg::this_cluster();
  const int rank = (int)cluster.block_rank();
  const int cid = (int)(blockIdx.x >> 1), ncl = (int)(gridDim.x >> 1);
  const int CC = rank == 0 ? MID : 0;     // centre plane of my window
  const int P0 = (CC - LC + T) % T;       // global plane of local plane 0 (the edge plane)
  extern __shared__ __align__(128) unsigned char smem[];
  R2* buf2 = reinterpret_cast<R2*>(smem + L::kBufOff);
  R2* A2 = buf2;            // [NQ][X+6 rows][Y], plane stride PS
  R2* B2 = buf2 + NQ * PS;  // [NQ][X][Y]
  const PcTables<R>* tab = reinterpret_cast<const PcTables<R>*>(smem + L::kTabOff);
  R2* s_f2p = reinterpret_cast<R2*>(smem + L::kPairOff);  // [(fs0*2+fs1)*7 + a][8]
  R2* s_cf_ty = reinterpret_cast<R2*>(smem + L::kCfOff);
  R2* s_cf_x = s_cf_ty + 7;
  int* s_plan = reinterpret_cast<int*>(smem + L::kPlanOff);
  unsigned long long* s_wmax = reinterpret_cast<unsigned long long*>(smem + L::kRedOff);
  R* s_wsum = reinterpret_cast<R*>(smem + L::kRedOff + 32 * 8);
  R* s_part = s_wsum + 32;  // [2]: partial sums of CTA 0 and CTA 1 (each CTA holds both after the cluster barrier)
  unsigned long long* s_peer_val = reinterpret_cast<unsigned long long*>(smem + L::kRedOff + 32 * 8 + 34 * sizeof(R));
  int* s_peer_flat = reinterpret_cast<int*>(s_peer_val + 1);
  int* s_best_flat = s_peer_flat + 1;
  const int tid = threadIdx.x;
  const int wid = tid >> 5, lane = tid & 31;
  // the peer's view of the arrays it reads from / writes to me
  const R2* peerB2 = cluster.map_shared_rank(B2, rank ^ 1);
  R* peer_part = cluster.map_shared_rank(s_part, rank ^ 1);
  unsigned long long* peer_peer_val = cluster.map_shared_rank(s_peer_val, rank ^ 1);
  int* peer_peer_flat = cluster.map_shared_rank(s_peer_flat, rank ^ 1);
  int* err_dst = rank == 0 ? err : nullptr;  // both CTAs see the same odometry: one of them reports

  // ---- one-time set-up: tables, coefficient pairs, first plan
  for (int i = tid; i < (int)(sizeof(PcTables<R>) / sizeof(R)); i += NT)
    reinterpret_cast<R*>(smem + L::kTabOff)[i] = reinterpret_cast<const R*>(&tabp)[i];
  if (tid < 7) {
    s_cf_ty[tid] = mk2(tabp.ge[tid], tabp.gi[tid]);
    s_cf_x[tid] = mk2(tabp.gex[tid], tabp.gix[tid]);
  }
  for (int i = tid; i < 4 * 7 * 8; i += NT) {
    const int q = i & 7, a = (i >> 3) % 7, combo = i / 56;
    s_f2p[i] = q < 7 ? mk2(tabp.f2d[combo >> 1][a * 7 + q], tabp.f2d[combo & 1][a * 7 + q]) : mk2((R)0, (R)0);
  }
  if (tid >= kPlanT0 && tid < kPlanT0 + T && cid < B && n_steps > 0)
    pair_plan_plane<X, Y, T>(tid - kPlanT0, odom + (size_t)cid * 2, cos_th, sin_th, vtrans_scale, vrot_scale, s_plan,
                             err_dst ? err_dst + cid : nullptr);
  if (tid == 0) *s_best_flat = 0x7fffffff;
  cluster.sync();  // both CTAs of the cluster are running (DSMEM may be touched) and the set-up is visible
  int slot = 0;

  for (int b = cid; b < B; b += ncl) {
    R* gst = state + (size_t)b * (XY * T);
    const R g_inh = gi[b], g_lo = inhib_floor(g_inh);
    for (int step = 0; step < n_steps; ++step) {
      const int* plan = s_plan + slot * L::kPlanInts;
      const int4* plan4 = reinterpret_cast<const int4*>(plan);

      // ---- 1. theta pass of the separable DoG: global -> (E, I) pairs of my H planes.  The state is read with
      //      ld.global.cg: on later steps half of it was written by the peer CTA (another SM's L1 would be stale).
      {
        const R e0 = tab->ge[3], e1 = tab->ge[2], e2 = tab->ge[1], e3 = tab->ge[0];
        const R i0 = tab->gi[3], i1 = tab->gi[2], i2 = tab->gi[1], i3 = tab->gi[0];
        // pair 0 = (centre, edge): stage 4 applies the x origin of the pair's first plane to both, so the edge plane
        // is stored rotated by the difference of the two origins
        const int rot = (plan4[P0].x - plan4[CC].x) * Y;
        constexpr int IT1 = (XY + NT - 1) / NT;
#pragma unroll 1
        for (int it = 0; it < IT1; ++it) {
          const int p = tid + it * NT;
          if (p < XY) {
            R in[H + 6];
            int k = P0 - 3 + T;
            k -= k >= T ? T : 0;
#pragma unroll
            for (int l = 0; l < H + 6; ++l) {
              in[l] = __ldcg(gst + k * XY + p);
              k = k + 1 == T ? 0 : k + 1;
            }
            int pe = p - rot;
            pe += pe < 0 ? XY : 0;
            pe -= pe >= XY ? XY : 0;
#pragma unroll
            for (int l = 0; l < H; ++l) {
              const R c = in[l + 3];
              const R s1 = in[l + 4] + in[l + 2];
              const R s2 = in[l + 5] + in[l + 1];
              const R s3 = in[l + 6] + in[l];
              const R e = fma(e0, c, fma(e1, s1, fma(e2, s2, e3 * s3)));
              const R i = fma(i0, c, fma(i1, s1, fma(i2, s2, i3 * s3)));
              buf2[l == 0 ? pe : l * XY + p] = mk2(e, i);
            }
          }
        }
      }
      __syncthreads();

      // ---- 2. y pass, in place on each (plane, x) line
      {
        R2 cf[7];
#pragma unroll
        for (int t = 0; t < 7; ++t) cf[t] = s_cf_ty[t];
        constexpr int IT2 = (H * X + NT - 1) / NT;
#pragma unroll 1
        for (int it = 0; it < IT2; ++it) {
          const int ln = tid + it * NT;
          if (ln < H * X) {
            R2* line = buf2 + ln * Y;
            R2 in[Y];
#pragma unroll
            for (int y = 0; y < Y; ++y) in[y] = line[y];
#pragma unroll
            for (int y = 0; y < Y; ++y) {
              R2 acc = mk2((R)0, (R)0);
#pragma unroll
              for (int t = 0; t < 7; ++t) acc = fma2(in[(y + t + Y - 3) % Y], cf[t], acc);
              line[y] = acc;
            }
          }
        }
      }
      __syncthreads();

      // ---- 3. x pass + global inhibition (posecell_network.py:339-340) + sum (:343): a thread takes the same y
      //      column of BOTH planes of a pair; the column it READS is y + oy of the plane (the y part of the origin)
      R2 keep[X];
      R psum = (R)0;
      const int q3 = tid / Y, y3 = tid - q3 * Y;
      if (tid < NQ * Y) {
        R2 cf[7];
#pragma unroll
        for (int t = 0; t < 7; ++t) cf[t] = s_cf_x[t];
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          const int l = h == 0 ? LC + q3 : (q3 == 0 ? 0 : LC - q3);
          int k = P0 + l;
          k -= k >= T ? T : 0;
          int ys = y3 + plan4[k].y;
          ys -= ys >= Y ? Y : 0;
          const R2* col = buf2 + l * XY + ys;
          R2 in[X];
#pragma unroll
          for (int x = 0; x < X; ++x) in[x] = col[x * Y];
#pragma unroll
          for (int x = 0; x < X; ++x) {
            R2 acc = mk2(-g_inh, (R)0);  // the inhibition rides in the accumulator
#pragma unroll
            for (int t = 0; t < 7; ++t) acc = fma2(in[(x + t + X - 3) % X], cf[t], acc);
            const R d = acc.x - acc.y;
            const R a = d < (R)0 ? g_lo : d;  // (a < gi) ? max(-gi, 0) : a - gi (posecell_network.py:339-340)
            if (h == 0)
              keep[x].x = a;
            else
              keep[x].y = a;
          }
        }
        R2 ps2 = keep[0];
#pragma unroll
        for (int x = 1; x < X; ++x) ps2 = add2(ps2, keep[x]);
        psum = ps2.x + ps2.y;
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) psum += __shfl_xor_sync(0xffffffffu, psum, o);
      if (lane == 0) s_wsum[wid] = psum;
      __syncthreads();  // every (E, I) pair has been consumed: the bytes become A2 / B2
      if (tid < NQ * Y) {
        R2* dst = A2 + q3 * PS + y3;  // row r of the halo layout is grid row r - 3
#pragma unroll
        for (int x = 0; x < X; ++x) {
          dst[(x + 3) * Y] = keep[x];
          if (x < 3) dst[(x + 3 + X) * Y] = keep[x];
          if (x >= X - 3) dst[(x + 3 - X) * Y] = keep[x];
        }
      }
      if (wid == 0) {
        R sacc = lane < NW ? s_wsum[lane] : (R)0;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) sacc += __shfl_xor_sync(0xffffffffu, sacc, o);
        if (lane == 0) {  // my half's sum, to me and to the peer (visible after the cluster barrier behind stage 4)
          s_part[rank] = sacc;
          peer_part[rank] = sacc;
        }
      }
      __syncthreads();  // publishes A2

      // ---- 4. 7x7 periodic correlate of both planes of a pair at once (posecell_network.py:273-274,300);
      //      meanwhile two otherwise idle warps prepare the plan of the next update.
      const bool last_step = (step + 1 == n_steps);
      const int nb = last_step ? b + ncl : b;
      const int nstep = last_step ? 0 : step + 1;
      if (tid >= kPlanT0) {
        if (tid < kPlanT0 + T && nb < B)
          pair_plan_plane<X, Y, T>(tid - kPlanT0, odom + ((size_t)nstep * B + nb) * 2, cos_th, sin_th, vtrans_scale,
                                   vrot_scale, s_plan + (slot ^ 1) * L::kPlanInts, err_dst ? err_dst + nb : nullptr);
      } else if (tid < NQ * X) {
        const int q = tid / X, x = tid - q * X;
        int kA = P0 + LC + q, kB = q == 0 ? P0 : P0 + LC - q;
        kA -= kA >= T ? T : 0;
        kB -= kB >= T ? T : 0;
        const int fsA = plan4[kA].w, fsB = plan4[kB].w;
        const R2* ctab = s_f2p + (fsA * 2 + fsB) * 56;
        const R2* rows = A2 + q * PS + x * Y;  // halo layout: tap row a of output row x is row x + a
        R2 acc[Y];
#pragma unroll
        for (int j = 0; j < Y; ++j) acc[j] = mk2((R)0, (R)0);
#pragma unroll
        for (int a = 0; a < 7; ++a) {
          R2 row[Y];
#pragma unroll
          for (int j = 0; j < Y; ++j) row[j] = rows[a * Y + j];
          R2 cf[7];
#pragma unroll
          for (int c = 0; c < 7; ++c) cf[c] = ctab[a * 8 + c];
#pragma unroll
          for (int j = 0; j < Y; ++j) {
#pragma unroll
            for (int c = 0; c < 7; ++c) acc[j] = fma2(row[(j + c + Y - 3) % Y], cf[c], acc[j]);
          }
        }
        // x origin of the pair: the row computed from rows x-3..x+3 is row x - ox of the result
        int xs = x - plan4[kA].x;
        xs += xs < 0 ? X : 0;
        R2* o = B2 + q * XY + xs * Y;
#pragma unroll
        for (int j = 0; j < Y; ++j)  // posecell_network.py:300; 1/total is applied by stage 5
          o[j] = mk2(max0(acc[j].x), max0(acc[j].y));
      }
      cluster.sync();  // B2 and the partial sums of both halves are complete and visible to both CTAs

      // ---- 5. theta pass (convolution.py:344-359), clamp (:314), -> global, maximum.
      //      V(j) = (plane LC+j, plane LC-j) for any j: pin[j] inside the window, the halves swapped for j < 0, the
      //      centre twice for j = 0, and (peer's planes) beyond the window's ends.  Output pair m = sum_u V(m+u) *
      //      (f[3+u], f[3-u]): the second half of a mirror pair takes the taps in reverse.
      // posecell_network.py:344-345: the normalisation is a positive scale and the 7x7 stage is followed by a clamp
      // at zero and a linear pass, so 1/total is folded into the seven taps here.
      const R tot = s_part[0] + s_part[1];
      const R inv = (tot != (R)0) ? (R)1 / tot : (R)1;
      R best_v = (R)-1;
      int best_flat = 0x7fffffff;
      {
        R fc[7];
        const R* f1 = tab->f1d[plan[4 * T]];
#pragma unroll
        for (int t = 0; t < 7; ++t) fc[t] = f1[t] * inv;
        R2 cf2[7];
#pragma unroll
        for (int u = -3; u <= 3; ++u) cf2[u + 3] = mk2(fc[3 + u], fc[3 - u]);
        constexpr int IT5 = (XY + NT - 1) / NT;
#pragma unroll 1
        for (int it = 0; it < IT5; ++it) {
          const int p = tid + it * NT;
          if (p < XY) {
            R2 pin[NQ];
#pragma unroll
            for (int q = 0; q < NQ; ++q) pin[q] = B2[q * XY + p];
            // the peer's planes next to my window: lo[t] = local plane t - 3 (its last three planes: the first halves
            // of its pairs LC-3..LC-1), hi[t] = local plane H + t (its edge plane and the second halves of its
            // last two pairs)
            R lo[3], hi[3];
#pragma unroll
            for (int t = 0; t < 3; ++t) lo[t] = peerB2[(LC - 3 + t) * XY + p].x;
            hi[0] = peerB2[p].y;
            hi[1] = peerB2[(LC - 1) * XY + p].y;
            hi[2] = peerB2[(LC - 2) * XY + p].y;
            R2 out[NQ];
#pragma unroll
            for (int m = 1; m < NQ; ++m) {
              R2 acc = mk2((R)0, (R)0);
#pragma unroll
              for (int u = -3; u <= 3; ++u) {
                const int j = m + u;
                R2 v;
                if (j >= 1 && j <= NQ - 1)
                  v = pin[j];
                else if (j == 0)
                  v = mk2(pin[0].x, pin[0].x);                       // the centre plane on both sides
                else if (j < 0)
                  v = mk2(pin[-j].y, pin[-j].x);                     // crossed the centre: halves swap
                else if (j == NQ)
                  v = mk2(hi[0], pin[0].y);                          // (local H, local 0 = my edge plane)
                else
                  v = mk2(hi[j - NQ], lo[3 - (j - NQ)]);             // (local H + d, local -d), d = j - NQ
                acc = fma2(v, cf2[u + 3], acc);
              }
              out[m] = mk2(max0(acc.x), max0(acc.y));
            }
            {  // pair 0 = (centre, edge)
              R a = (R)0, c = (R)0;
#pragma unroll
              for (int u = -3; u <= 3; ++u) {
                const R va = u > 0 ? pin[u].x : (u < 0 ? pin[-u].y : pin[0].x);          // local LC + u
                const R vc = u > 0 ? pin[LC - u].y : (u < 0 ? lo[3 + u] : pin[0].y);     // local u
                a = fma(fc[3 + u], va, a);
                c = fma(fc[3 + u], vc, c);
              }
              out[0] = mk2(max0(a), max0(c));
            }
            // store: local plane LC + m <- out[m].x, LC - m <- out[m].y, LC <- out[0].x, 0 <- out[0].y
            R vmax = out[0].x > out[0].y ? out[0].x : out[0].y;
#pragma unroll
            for (int m = 0; m < NQ; ++m) {
              int kx = P0 + LC + m, ky = m == 0 ? P0 : P0 + LC - m;
              kx -= kx >= T ? T : 0;
              ky -= ky >= T ? T : 0;
              gst[kx * XY + p] = out[m].x;
              gst[ky * XY + p] = out[m].y;
              vmax = out[m].x > vmax ? out[m].x : vmax;
              vmax = out[m].y > vmax ? out[m].y : vmax;
            }
            if (vmax > best_v) {  // numpy.argmax: first maximum in [x][y][th] order; p grows with `it`
              int kb = T;
#pragma unroll
              for (int m = 0; m < NQ; ++m) {
                int kx = P0 + LC + m, ky = m == 0 ? P0 : P0 + LC - m;
                kx -= kx >= T ? T : 0;
                ky -= ky >= T ? T : 0;
                if (out[m].x == vmax && kx < kb) kb = kx;
                if (out[m].y == vmax && ky < kb) kb = ky;
              }
              best_v = vmax;
              best_flat = p * T + kb;
            }
          }
        }
      }
      // arg-max of my half: maximum of the value bits over the block, then the lowest flat index among its holders
      const unsigned long long vb = best_v >= (R)0 ? val_bits(best_v) : 0ull;
      unsigned long long wm = vb;
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        const unsigned long long other = __shfl_xor_sync(0xffffffffu, wm, o);
        wm = other > wm ? other : wm;
      }
      if (lane == 0) s_wmax[wid] = wm;
      __syncthreads();
      unsigned long long gm = lane < NW ? s_wmax[lane] : 0ull;
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        const unsigned long long other = __shfl_xor_sync(0xffffffffu, gm, o);
        gm = other > gm ? other : gm;
      }
      if (best_flat != 0x7fffffff && vb == gm) atomicMin(s_best_flat, best_flat);
      __syncthreads();
      if (tid == 0 && rank == 1) {  // my candidate goes to CTA 0
        *peer_peer_val = gm;
        *peer_peer_flat = *s_best_flat;
      }
      cluster.sync();  // the peer has read my B2 (stage 1 of the next update may overwrite it); candidates exchanged;
                       // the state in global memory is consistent for the next update
      if (tid == 0) {
        if (rank == 0) {
          const unsigned long long pv = *s_peer_val;
          const int pf = *s_peer_flat, mf = *s_best_flat;
          const int flat = pv > gm ? pf : (pv < gm ? mf : (pf < mf ? pf : mf));
          argmax[(size_t)step * B + b] = (long long)flat;
          total[(size_t)step * B + b] = tot;
        }
        *s_best_flat = 0x7fffffff;  // next written by the winners behind the next update's first block barrier
      }
      slot ^= 1;
    }
  }
  cluster.sync();  // no CTA leaves while its peer could still address its shared memory
}

struct PairState {
  std::mutex mu;
  bool configured[64] = {};
  int clusters[64] = {};
};

// Once per device and kernel (S belongs to one kernel): allow the kernel its dynamic shared memory, and find how many
// of its 2-CTA clusters fit on the device at once (half the SMs if the occupancy query fails).  The count, capped at
// B, goes to *ncl.
template <typename K>
int pair_clusters(PairState& S, K kern, int nt, size_t smem, int dev, int B, int* ncl) {
  PRS_REQUIRE(dev >= 0 && dev < 64, "pair path: device index %d out of range", dev);
  std::lock_guard<std::mutex> lk(S.mu);
  if (!S.configured[dev]) {
    PRS_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(2 * 148, 1, 1);
    cfg.blockDim = dim3(nt, 1, 1);
    cfg.dynamicSmemBytes = smem;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = 2;
    at[0].val.clusterDim.y = 1;
    at[0].val.clusterDim.z = 1;
    cfg.attrs = at;
    cfg.numAttrs = 1;
    int n = 0;
    if (cudaOccupancyMaxActiveClusters(&n, kern, &cfg) != cudaSuccess || n < 1) {
      (void)cudaGetLastError();
      int nsm = 0;
      PRS_CUDA(cudaDeviceGetAttribute(&nsm, cudaDevAttrMultiProcessorCount, dev));
      n = nsm / 2 > 0 ? nsm / 2 : 1;
    }
    S.clusters[dev] = n;
    S.configured[dev] = true;
  }
  *ncl = B < S.clusters[dev] ? B : S.clusters[dev];
  return PRS_OK;
}

template <int X, int Y, int T, int NT, typename R>
int pair_launch(prs_pc_plan* p, R* state, const double* odom, int n_steps, const R* gi, long long* argmax, R* total,
                int* err, const PcTables<R>& tab, cudaStream_t st) {
  using L = PairLayout<X, Y, T, R>;
  auto kern = k_pc_pair<X, Y, T, NT, R>;
  static PairState S;
  int ncl = 0;
  if (int rc_ = pair_clusters(S, kern, NT, L::kBytes, p->device, p->B, &ncl)) return rc_;
  kern<<<2 * ncl, NT, L::kBytes, st>>>(state, odom, n_steps, gi, argmax, total, err, p->cos_th, p->sin_th,
                                       p->vtrans_scale, p->vrot_scale, p->B, tab);
  PRS_CUDA(cudaGetLastError());
  return PRS_OK;
}


// =============================================================================================
// The same fused update for grids whose lines do not fit a thread's registers (simulate.py's 50x50x10,
// ratslam/simulate.py:9): k_pc_pair_seg.  One network per 2-CTA cluster as above, but
//   * the y and x passes and the 7x7 stage work on SEGMENTS of a line (25 / 25 / 17 outputs plus a 6-cell halo);
//   * the y pass goes from one (E, I) buffer to a second one (segments of a line are owned by different threads, so it
//     cannot run in place), the x pass from there into A2, which has a periodic halo in x AND y (no index wraps in the
//     7x7 stage); the two buffers (2 x 100 KB for 50x50x10) and A2 | B2 share the CTA's shared memory;
//   * a half may hold an ODD number of planes (Th = 10: five): the window is then centre +- LC with no edge plane and
//     pair 0 is the centre plane alone;
//   * one CTA per SM (205 KB of shared memory), the decisions of an update are evaluated at its start.
template <int X, int Y, int T>
struct SegLayout {
  static constexpr int XY = X * Y;
  static constexpr int H = T / 2;
  static constexpr bool kEdge = (H % 2 == 0);
  static constexpr int LC = kEdge ? H / 2 : (H - 1) / 2;
  static constexpr int NM = kEdge ? LC - 1 : LC;   // mirror pairs (LC + q, LC - q), q = 1..NM
  static constexpr int NQ = NM + 1;                // + pair 0 = (centre, edge or nothing)
  static constexpr int YS = Y + 6;                 // A2 row stride: 3 periodic halo columns each side
  static constexpr int PS = (X + 6) * YS;          // A2 plane stride: 3 periodic halo rows each side
  static constexpr int kElems = 2 * H * XY;        // float2: two (E, I) buffers; A2 | B2 alias them
  static_assert(NQ * PS <= H * XY, "A2 must not reach into the second (E, I) buffer the x pass reads");
  static_assert(NQ * PS + NQ * XY <= kElems, "A2 | B2 must fit the two (E, I) buffers");
  static constexpr int kPlanInts = 4 * T + 4;
  static constexpr size_t kTabOff = (size_t)8 * kElems;
  static constexpr size_t kPairOff = (kTabOff + sizeof(PcTables<float>) + 15) / 16 * 16;
  static constexpr size_t kCfOff = kPairOff + 4 * 7 * 8 * 8;
  static constexpr size_t kPlanOff = kCfOff + 14 * 8;
  static constexpr size_t kRedOff = (kPlanOff + kPlanInts * 4 + 15) / 16 * 16;
  static constexpr size_t kBytes = kRedOff + 32 * 8 + 32 * 4 + 2 * 4 + 8 + 4 + 4 + 16;
};

template <int X, int Y, int T, int NT>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(NT, 1)
    k_pc_pair_seg(float* state, const double* __restrict__ odom, int n_steps, const float* __restrict__ gi,
                  long long* __restrict__ argmax, float* __restrict__ total, int* __restrict__ err,
                  const double* __restrict__ cos_th, const double* __restrict__ sin_th, double vtrans_scale,
                  double vrot_scale, int B, const __grid_constant__ PcTables<float> tabp) {
  using L = SegLayout<X, Y, T>;
  constexpr int XY = L::XY, H = L::H, LC = L::LC, NM = L::NM, NQ = L::NQ, YS = L::YS, PS = L::PS, MID = T / 2;
  constexpr bool kEdge = L::kEdge;
  constexpr int NW = NT / 32;
  constexpr int NSY = (Y + 24) / 25, SY = (Y + NSY - 1) / NSY;    // y-pass segments (<= 25 outputs)
  constexpr int NSX = (X + 24) / 25, SX = (X + NSX - 1) / NSX;    // x-pass segments
  constexpr int NS4 = (Y + 16) / 17, S4 = (Y + NS4 - 1) / NS4;    // 7x7 row segments (<= 17 outputs)
  static_assert(X >= 7 && Y >= 7 && T % 2 == 0 && H >= 5 && T <= NT, "shape not supported by the segmented pair kernel");
  cg::cluster_group cluster = cg::this_cluster();
  const int rank = (int)cluster.block_rank();
  const int cid = (int)(blockIdx.x >> 1), ncl = (int)(gridDim.x >> 1);
  const int CC = rank == 0 ? MID : 0;
  const int P0 = (CC - LC + T) % T;
  extern __shared__ __align__(128) unsigned char smem[];
  float2* bufA = reinterpret_cast<float2*>(smem);     // (E, I) after the theta pass, [H][X][Y]
  float2* bufB = bufA + H * XY;                       // ... after the y pass
  float2* A2 = bufA;                                  // [NQ][X + 6][Y + 6]
  float2* B2 = bufA + NQ * PS;                        // [NQ][X][Y]
  const PcTables<float>* tab = reinterpret_cast<const PcTables<float>*>(smem + L::kTabOff);
  float2* s_f2p = reinterpret_cast<float2*>(smem + L::kPairOff);
  float2* s_cf_ty = reinterpret_cast<float2*>(smem + L::kCfOff);
  float2* s_cf_x = s_cf_ty + 7;
  int* s_plan = reinterpret_cast<int*>(smem + L::kPlanOff);
  unsigned long long* s_wmax = reinterpret_cast<unsigned long long*>(smem + L::kRedOff);
  float* s_wsum = reinterpret_cast<float*>(smem + L::kRedOff + 32 * 8);
  float* s_part = s_wsum + 32;
  unsigned long long* s_peer_val = reinterpret_cast<unsigned long long*>(smem + L::kRedOff + 32 * 8 + 34 * 4);
  int* s_peer_flat = reinterpret_cast<int*>(s_peer_val + 1);
  int* s_best_flat = s_peer_flat + 1;
  const int tid = threadIdx.x, wid = tid >> 5, lane = tid & 31;
  const float2* peerB2 = cluster.map_shared_rank(B2, rank ^ 1);
  float* peer_part = cluster.map_shared_rank(s_part, rank ^ 1);
  unsigned long long* peer_peer_val = cluster.map_shared_rank(s_peer_val, rank ^ 1);
  int* peer_peer_flat = cluster.map_shared_rank(s_peer_flat, rank ^ 1);
  int* err_dst = rank == 0 ? err : nullptr;

  for (int i = tid; i < (int)(sizeof(PcTables<float>) / 4); i += NT)
    reinterpret_cast<float*>(smem + L::kTabOff)[i] = reinterpret_cast<const float*>(&tabp)[i];
  if (tid < 7) {
    s_cf_ty[tid] = make_float2(tabp.ge[tid], tabp.gi[tid]);
    s_cf_x[tid] = make_float2(tabp.gex[tid], tabp.gix[tid]);
  }
  for (int i = tid; i < 4 * 7 * 8; i += NT) {
    const int q = i & 7, a = (i >> 3) % 7, combo = i / 56;
    s_f2p[i] = q < 7 ? make_float2(tabp.f2d[combo >> 1][a * 7 + q], tabp.f2d[combo & 1][a * 7 + q]) : make_float2(0.f, 0.f);
  }
  if (tid == 0) *s_best_flat = 0x7fffffff;
  cluster.sync();
  const int4* plan4 = reinterpret_cast<const int4*>(s_plan);
  // global plane of local plane l, and the local planes of pair q
  auto gplane = [&](int l) {
    int k = P0 + l;
    return k >= T ? k - T : k;
  };

  for (int b = cid; b < B; b += ncl) {
    float* gst = state + (size_t)b * (XY * T);
    const float g_inh = gi[b], g_lo = inhib_floor(g_inh);
    for (int step = 0; step < n_steps; ++step) {
      // ---- 0. the decisions of this update (posecell_network.py:252-267,249,304), float64 as numpy computes them
      if (tid < T)
        pair_plan_plane<X, Y, T>(tid, odom + ((size_t)step * B + b) * 2, cos_th, sin_th, vtrans_scale, vrot_scale, s_plan,
                                 err_dst ? err_dst + b : nullptr);
      __syncthreads();

      // ---- 1. theta pass: global -> (E, I) pairs of my H planes
      {
        const float e0 = tab->ge[3], e1 = tab->ge[2], e2 = tab->ge[1], e3 = tab->ge[0];
        const float i0 = tab->gi[3], i1 = tab->gi[2], i2 = tab->gi[1], i3 = tab->gi[0];
        const int rot = kEdge ? (plan4[P0].x - plan4[CC].x) * Y : 0;  // the edge plane is stored rotated (see above)
#pragma unroll 1
        for (int p = tid; p < XY; p += NT) {
          float in[H + 6];
          int k = P0 - 3 + T;
          k -= k >= T ? T : 0;
#pragma unroll
          for (int l = 0; l < H + 6; ++l) {
            in[l] = __ldcg(gst + k * XY + p);
            k = k + 1 == T ? 0 : k + 1;
          }
          int pe = p - rot;
          pe += pe < 0 ? XY : 0;
          pe -= pe >= XY ? XY : 0;
#pragma unroll
          for (int l = 0; l < H; ++l) {
            const float c = in[l + 3];
            const float s1 = in[l + 4] + in[l + 2], s2 = in[l + 5] + in[l + 1], s3 = in[l + 6] + in[l];
            bufA[(kEdge && l == 0) ? pe : l * XY + p] =
                make_float2(fmaf(e0, c, fmaf(e1, s1, fmaf(e2, s2, e3 * s3))), fmaf(i0, c, fmaf(i1, s1, fmaf(i2, s2, i3 * s3))));
          }
        }
      }
      __syncthreads();

      // ---- 2. y pass, bufA -> bufB; item = (line, segment)
      {
        float2 cf[7];
#pragma unroll
        for (int t = 0; t < 7; ++t) cf[t] = s_cf_ty[t];
#pragma unroll 1
        for (int it = tid; it < H * X * NSY; it += NT) {
          const int ln = it / NSY, sg = it - ln * NSY;
          const int y0 = sg * SY;
          const float2* line = bufA + ln * Y;
          float2 in[SY + 6];
#pragma unroll
          for (int t = 0; t < SY + 6; ++t) {
            int y = y0 - 3 + t;
            y += y < 0 ? Y : 0;
            y -= y >= Y ? Y : 0;
            in[t] = line[y];
          }
          float2* o = bufB + ln * Y + y0;
#pragma unroll
          for (int j = 0; j < SY; ++j) {
            float2 acc = make_float2(0.f, 0.f);
#pragma unroll
            for (int t = 0; t < 7; ++t) acc = __ffma2_rn(in[j + t], cf[t], acc);
            if (y0 + j < Y) o[j] = acc;
          }
        }
      }
      __syncthreads();

      // ---- 3. x pass + inhibition + sum, bufB -> A2 (periodic halo in x and y); item = (pair, y, segment)
      float psum = 0.f;
      {
        float2 cf[7];
#pragma unroll
        for (int t = 0; t < 7; ++t) cf[t] = s_cf_x[t];
#pragma unroll 1
        for (int it = tid; it < NQ * Y * NSX; it += NT) {
          const int sg = it % NSX, qy = it / NSX;
          const int q = qy / Y, y = qy - q * Y;
          const int x0 = sg * SX;
          float2 keep[SX];
#pragma unroll
          for (int h = 0; h < 2; ++h) {
            if (h == 1 && q == 0 && !kEdge) {
#pragma unroll
              for (int j = 0; j < SX; ++j) keep[j].y = 0.f;
              continue;
            }
            const int l = h == 0 ? LC + q : (q == 0 ? 0 : LC - q);
            int ys = y + plan4[gplane(l)].y;   // the y part of the plane's origin: the column that is READ
            ys -= ys >= Y ? Y : 0;
            const float2* col = bufB + l * XY + ys;
            float2 in[SX + 6];
#pragma unroll
            for (int t = 0; t < SX + 6; ++t) {
              int x = x0 - 3 + t;
              x += x < 0 ? X : 0;
              x -= x >= X ? X : 0;
              in[t] = col[x * Y];
            }
#pragma unroll
            for (int j = 0; j < SX; ++j) {
              float2 acc = make_float2(-g_inh, 0.f);
#pragma unroll
              for (int t = 0; t < 7; ++t) acc = __ffma2_rn(in[j + t], cf[t], acc);
              const float d = acc.x - acc.y;
              const float a = d < 0.f ? g_lo : d;  // posecell_network.py:339-340, see inhib_floor
              if (h == 0)
                keep[j].x = a;
              else
                keep[j].y = a;
            }
          }
          // A2[q][x + 3][y + 3] and its periodic images
          const int cy = y + 3;
          const int cy2 = y < 3 ? cy + Y : (y >= Y - 3 ? cy - Y : -1);
          float2* dst = A2 + q * PS;
#pragma unroll
          for (int j = 0; j < SX; ++j) {
            const int x = x0 + j;
            if (x < X) {
              psum += keep[j].x + keep[j].y;
              const int rx = x + 3;
              const int rx2 = x < 3 ? rx + X : (x >= X - 3 ? rx - X : -1);
              dst[rx * YS + cy] = keep[j];
              if (cy2 >= 0) dst[rx * YS + cy2] = keep[j];
              if (rx2 >= 0) {
                dst[rx2 * YS + cy] = keep[j];
                if (cy2 >= 0) dst[rx2 * YS + cy2] = keep[j];
              }
            }
          }
        }
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) psum += __shfl_xor_sync(0xffffffffu, psum, o);
      if (lane == 0) s_wsum[wid] = psum;
      __syncthreads();
      if (wid == 0) {
        float sacc = lane < NW ? s_wsum[lane] : 0.f;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) sacc += __shfl_xor_sync(0xffffffffu, sacc, o);
        if (lane == 0) {
          s_part[rank] = sacc;
          peer_part[rank] = sacc;
        }
      }

      // ---- 4. 7x7 correlate of both planes of a pair (posecell_network.py:273-274,300); item = (pair, x, segment)
#pragma unroll 1
      for (int it = tid; it < NQ * X * NS4; it += NT) {
        const int sg = it % NS4, qx = it / NS4;
        const int q = qx / X, x = qx - q * X;
        const int y0 = sg * S4;
        const int kA = gplane(LC + q), kB = gplane(q == 0 ? 0 : LC - q);
        const int fsA = plan4[kA].w, fsB = (q == 0 && !kEdge) ? 0 : plan4[kB].w;
        const float2* ctab = s_f2p + (fsA * 2 + fsB) * 56;
        const float2* rows = A2 + q * PS + x * YS + y0;  // halo layout: tap (a, c) of output (x, y0 + j) is [x + a][y0 + j + c]
        float2 acc[S4];
#pragma unroll
        for (int j = 0; j < S4; ++j) acc[j] = make_float2(0.f, 0.f);
#pragma unroll
        for (int a = 0; a < 7; ++a) {
          float2 row[S4 + 6];
#pragma unroll
          for (int j = 0; j < S4 + 6; ++j) row[j] = (y0 + j < Y + 6) ? rows[a * YS + j] : make_float2(0.f, 0.f);
          float2 cf[7];
#pragma unroll
          for (int c = 0; c < 7; ++c) cf[c] = ctab[a * 8 + c];
#pragma unroll
          for (int j = 0; j < S4; ++j)
#pragma unroll
            for (int c = 0; c < 7; ++c) acc[j] = __ffma2_rn(row[j + c], cf[c], acc[j]);
        }
        int xs = x - plan4[kA].x;  // the x part of the pair's origin, applied to the row that is stored
        xs += xs < 0 ? X : 0;
        float2* o = B2 + q * XY + xs * Y + y0;
#pragma unroll
        for (int j = 0; j < S4; ++j)
          if (y0 + j < Y) o[j] = make_float2(fmaxf(acc[j].x, 0.f), fmaxf(acc[j].y, 0.f));
      }
      cluster.sync();  // B2 and the partial sums of both halves are complete and visible to both CTAs

      // ---- 5. theta pass (convolution.py:344-359), clamp (:314), -> global, maximum.  V(j) = (local LC + j, local LC - j).
      const float tot = s_part[0] + s_part[1];
      const float inv = (tot != 0.f) ? 1.f / tot : 1.f;
      float best_v = -1.f;
      int best_flat = 0x7fffffff;
      {
        float fc[7];
        const float* f1 = tab->f1d[s_plan[4 * T]];
#pragma unroll
        for (int t = 0; t < 7; ++t) fc[t] = f1[t] * inv;
        float2 cf2[7];
#pragma unroll
        for (int u = -3; u <= 3; ++u) cf2[u + 3] = make_float2(fc[3 + u], fc[3 - u]);
#pragma unroll 1
        for (int p = tid; p < XY; p += NT) {
          float2 pin[NQ];
#pragma unroll
          for (int q = 0; q < NQ; ++q) pin[q] = B2[q * XY + p];
          // the peer's planes next to my window: lo[t] = my local t - 3 = its local H - 3 + t, hi[t] = my local H + t =
          // its local t.  Its local l is pair |l - LC|: first half (.x) above its centre, second half (.y) below,
          // and its edge plane (local 0 when H is even) is pair 0's second half.
          auto peer_val = [&](int l) -> float {            // the peer's local plane l (compile-time l)
            if (l == LC) return peerB2[p].x;
            if (kEdge && l == 0) return peerB2[p].y;
            return l > LC ? peerB2[(l - LC) * XY + p].x : peerB2[(LC - l) * XY + p].y;
          };
          float lo[3], hi[3];
#pragma unroll
          for (int t = 0; t < 3; ++t) {
            lo[t] = peer_val(H - 3 + t);
            hi[t] = peer_val(t);
          }
          // value of my local plane l (may lie outside 0..H-1 by up to 3)
          auto plane_val = [&](int l) -> float {
            if (l < 0) return lo[3 + l];
            if (l >= H) return hi[l - H];
            if (l == LC) return pin[0].x;
            if (kEdge && l == 0) return pin[0].y;
            return l > LC ? pin[l - LC].x : pin[LC - l].y;
          };
          float2 out[NQ];
#pragma unroll
          for (int m = 1; m <= NM; ++m) {
            float2 acc = make_float2(0.f, 0.f);
#pragma unroll
            for (int u = -3; u <= 3; ++u)
              acc = __ffma2_rn(make_float2(plane_val(LC + m + u), plane_val(LC - m - u)), cf2[u + 3], acc);
            out[m] = make_float2(fmaxf(acc.x, 0.f), fmaxf(acc.y, 0.f));
          }
          {
            float a = 0.f, c = 0.f;
#pragma unroll
            for (int u = -3; u <= 3; ++u) {
              a = fmaf(fc[3 + u], plane_val(LC + u), a);
              if (kEdge) c = fmaf(fc[3 + u], plane_val(u), c);
            }
            out[0] = make_float2(fmaxf(a, 0.f), fmaxf(c, 0.f));
          }
          float vmax = out[0].x;
          int kb = T;
#pragma unroll
          for (int m = 0; m < NQ; ++m) {
            const int kx = gplane(LC + m);
            gst[kx * XY + p] = out[m].x;
            vmax = out[m].x > vmax ? out[m].x : vmax;
            if (m > 0 || kEdge) {
              const int ky = gplane(m == 0 ? 0 : LC - m);
              gst[ky * XY + p] = out[m].y;
              vmax = out[m].y > vmax ? out[m].y : vmax;
            }
          }
          if (vmax > best_v) {  // numpy.argmax: first maximum in [x][y][th] order; p grows along the loop
#pragma unroll
            for (int m = 0; m < NQ; ++m) {
              const int kx = gplane(LC + m);
              if (out[m].x == vmax && kx < kb) kb = kx;
              if (m > 0 || kEdge) {
                const int ky = gplane(m == 0 ? 0 : LC - m);
                if (out[m].y == vmax && ky < kb) kb = ky;
              }
            }
            best_v = vmax;
            best_flat = p * T + kb;
          }
        }
      }
      const unsigned long long vb = best_v >= 0.f ? val_bits(best_v) : 0ull;
      unsigned long long wm = vb;
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        const unsigned long long other = __shfl_xor_sync(0xffffffffu, wm, o);
        wm = other > wm ? other : wm;
      }
      if (lane == 0) s_wmax[wid] = wm;
      __syncthreads();
      unsigned long long gm = lane < NW ? s_wmax[lane] : 0ull;
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        const unsigned long long other = __shfl_xor_sync(0xffffffffu, gm, o);
        gm = other > gm ? other : gm;
      }
      if (best_flat != 0x7fffffff && vb == gm) atomicMin(s_best_flat, best_flat);
      __syncthreads();
      if (tid == 0 && rank == 1) {
        *peer_peer_val = gm;
        *peer_peer_flat = *s_best_flat;
      }
      cluster.sync();  // the peer has read my B2; candidates exchanged; the state in global memory is consistent
      if (tid == 0) {
        if (rank == 0) {
          const unsigned long long pv = *s_peer_val;
          const int pf = *s_peer_flat, mf = *s_best_flat;
          const int flat = pv > gm ? pf : (pv < gm ? mf : (pf < mf ? pf : mf));
          argmax[(size_t)step * B + b] = (long long)flat;
          total[(size_t)step * B + b] = tot;
        }
        *s_best_flat = 0x7fffffff;
      }
    }
  }
  cluster.sync();
}

template <int X, int Y, int T, int NT>
int pair_seg_launch(prs_pc_plan* p, float* state, const double* odom, int n_steps, const float* gi, long long* argmax,
                    float* total, int* err, cudaStream_t st) {
  using L = SegLayout<X, Y, T>;
  auto kern = k_pc_pair_seg<X, Y, T, NT>;
  static PairState S;
  int ncl = 0;
  if (int rc_ = pair_clusters(S, kern, NT, L::kBytes, p->device, p->B, &ncl)) return rc_;
  kern<<<2 * ncl, NT, L::kBytes, st>>>(state, odom, n_steps, gi, argmax, total, err, p->cos_th, p->sin_th, p->vtrans_scale,
                                       p->vrot_scale, p->B, p->tf);
  PRS_CUDA(cudaGetLastError());
  return PRS_OK;
}

}  // namespace

// The kernel applies ONE x origin per mirror pair: around(vt * cos) must be the same for both planes, which holds
// when the host's cosine table is bitwise even about MID and about plane 0 (numpy's cos is).
int prs_pc_pair_supported(const prs_pc_plan* p) {
  const bool ros = p->X == 21 && p->Y == 21 && p->Th == 36;                       // ros_simulate.py:31
  const bool sim = p->X == 50 && p->Y == 50 && p->Th == 10 && p->dtype == PRS_F32;  // simulate.py:9 (segmented kernel)
  if (!ros && !sim) return 0;
  const int T = p->Th, mid = T / 2;
  for (int m = 1; m < mid; ++m)
    if (p->h_cos[mid + m] != p->h_cos[mid - m]) return 0;   // covers both windows: plane T - m is plane mid + (mid - m)
  return 1;
}

int prs_pc_pair_step(prs_pc_plan* p, void* state, const double* odom, int T, const void* gi, long long* argmax,
                     void* total, int* err, cudaStream_t st) {
  if (p->X == 21 && p->Y == 21 && p->Th == 36) {
    if (p->dtype == PRS_F32)
      return pair_launch<21, 21, 36, 256, float>(p, (float*)state, odom, T, (const float*)gi, argmax, (float*)total, err,
                                                 p->tf, st);
    return pair_launch<21, 21, 36, 256, double>(p, (double*)state, odom, T, (const double*)gi, argmax, (double*)total,
                                                err, p->td, st);
  }
  if (p->X == 50 && p->Y == 50 && p->Th == 10 && p->dtype == PRS_F32) {
    // 512 threads: measured for 2600 networks, 0.855 ms (256 threads, 178 registers), 0.791 ms (384), 0.768 ms (512,
    // 120 registers) -- one CTA per SM, so more warps win
    return pair_seg_launch<50, 50, 10, 512>(p, (float*)state, odom, T, (const float*)gi, argmax, (float*)total, err, st);
  }
  prs_set_error("pair path not available for this plan");
  return PRS_E_INVALID;
}
