// Fused, SMEM-resident pose-cell update for reference-size networks (float32, sm_100a).
//
// One CTA owns one network at a time and performs the whole PoseCellNetwork.update()
// (ratslam/posecell_network.py:326-353) -- 7x7x7 DoG correlate, global inhibition, normalisation,
// per-heading shifted 7x7 correlate, 7-tap theta correlate, arg-max -- with the state held in shared
// memory between the stages; HBM sees one read and one write of the state per update (8 B / cell).
// The grid is persistent: min(B, #SM) CTAs stride over the B networks of an ensemble, and the next
// network's state is fetched by a TMA bulk copy (cp.async.bulk -> mbarrier) while the current one
// is being computed.
//
// Shared memory (N = X*Y*Th cells, NP = ceil(Th/2) plane pairs):
//   stage[N] float        the next network's state as it lies in HBM, theta-major [th][x][y]   4N bytes
//   buf2[N]  float2       (E, I) pairs of the separable DoG, [th][x][y]                        8N bytes
//     after the x pass the same bytes are reused as two plane-pair-interleaved tensors
//       A2[NP][x+halo][y] float2 = (A'[mid+m], A'[mid-m])  inhibited activity; each plane already moved by the y part
//                                                   of its integer origin, 3 periodic halo rows each side
//       B2[NP][x][y] float2 = (B[mid+m], B[mid-m])    after the 2-D correlate
//     Plane pairs are MIRROR pairs about mid = Th/2 (pair 0 is (mid, 0)): cos((k-mid)*2pi/Th) is the same for
//     both, hence the same x origin -- stage 4 applies it once per thread as the first row it reads -- and the
//     same LUT filter (a variant of stage 4 that adds the tap rows sharing
//     coefficients first -- 4 or 5 row groups instead of 7 -- was measured and was NOT faster: the stage is bound
//     by the sum of its shared-memory and FMA time, not by the FMA count).
// Stages (a __syncthreads between each):
//   1 theta pass   thread = one (x,y) line of Th cells in registers, stage -> buf2         11 op / cell
//   2 y pass       thread = one (th,x) line, in place, packed FFMA2 on (E,I)               7 FFMA2 / cell
//   3 x pass       thread = one (th,y) line, A = aE*E - aI*I, inhibit, block sum; the column it READS is
//                  y + oy of its plane (the y part of the integer origin: one wrap per thread)
//   4 7x7 stage    thread = one x-row of a plane PAIR starting at row x + ox (the x part), packed
//                  FFMA2 over the pair, rows and coefficient pairs arrive by LDS.64 / LDS.128   24.5 FFMA2 / cell
//   5 theta pass   thread = one (x,y) line, packed over the plane pair, clamp, arg-max, -> global   3.5 FFMA2 / cell
// The FMA-heavy stages use the sm_100 packed instruction (fma.rn.f32x2, SASS FFMA2): same FP32 pipe
// rate as scalar FFMA (measured, bench_tools/microbench.cu) for half the issue slots, which is what
// lets the shared-memory loads issue alongside.
#include <stdlib.h>

#include <mutex>

#include "common.cuh"

#ifndef PRS_RESIDENT_S3FOLD
#define PRS_RESIDENT_S3FOLD 1
#endif
#ifndef PRS_RESIDENT_DEFER1
#define PRS_RESIDENT_DEFER1 35
#endif

namespace {

template <int X, int Y, int T>
struct ResLayout {
  static constexpr int XY = X * Y;
  static constexpr int N = XY * T;
  static constexpr int NP = (T + 1) / 2;
  // A2 plane: X+6 rows (3 periodic halo rows on each side, so stage 4 never wraps an index).  The plane
  // stride is padded until PS == X*Y (mod 16): then the float2 slot read by item (kp, x) is
  // Y*(kp*X + x) + const (mod 16) -- an odd stride across the whole warp, i.e. no bank conflicts.
  static constexpr int kPSraw = (X + 6) * Y;
  static constexpr int PS = kPSraw + ((XY % 16) - (kPSraw % 16) + 16) % 16;
  static constexpr int kPlanInts = 4 * T + 4;                              // int4 (ox, oy, ox*Y+oy, fsel)[T], misc[4]
  static constexpr size_t kStageOff = 0;                                   // float[N]
  static constexpr size_t kBufOff = ((size_t)4 * N + 15) / 16 * 16;        // float2[max(N, NP*PS + NP*XY)]
  static constexpr size_t kBufBytes = (size_t)8 * (NP * PS + NP * XY > N ? NP * PS + NP * XY : N);
  static constexpr size_t kTabOff = (kBufOff + kBufBytes + 15) / 16 * 16;  // PcTables<float>, 1 KiB slot
  static constexpr size_t kPairOff = kTabOff + 1024;                       // float2[4][7][8] paired 2-D coefficients
  static constexpr size_t kCfOff = kPairOff + 4 * 7 * 8 * 8;               // float2[7] (ge,gi), float2[7] (gex,gix)
  static constexpr size_t kPlanOff = kCfOff + 16 * 8;                      // two plans (double buffered)
  static constexpr size_t kRedOff = (kPlanOff + 2 * kPlanInts * 4 + 15) / 16 * 16;  // int[32], float[32], float[4]
  static constexpr size_t kBarOff = kRedOff + 32 * 4 + 32 * 4 + 16;        // mbarrier (8 bytes)
  static constexpr size_t kBytes = kBarOff + 16;
};
static_assert(sizeof(PcTables<float>) <= 1024, "tables must fit their shared-memory slot");

__device__ __forceinline__ float2 ffma2(float2 a, float2 b, float2 c) { return __ffma2_rn(a, b, c); }

// ---- mbarrier / TMA bulk copy (global -> shared), PTX ISA "cp.async.bulk"
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(void* bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(void* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(void* bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "WAIT_%=:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@!p bra WAIT_%=;\n"
      "}\n" ::"r"(smem_u32(bar)),
      "r"(parity)
      : "memory");
}
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, void* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_u32(dst)),
               "l"(src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// ---- update n+1 of an ensemble may start while update n still runs (programmatic dependent launch): what orders them is
//      one sequence number per network, released when the network's state of launch n is in global memory and acquired
//      before launch n+1 fetches it.
__device__ __forceinline__ unsigned ld_acquire_gpu_u32(const unsigned* p) {
  unsigned v;
  asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_release_gpu_u32(unsigned* p, unsigned v) {
  asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ void wait_network(const unsigned* net_seq, int b, unsigned seq) {
  if (seq == 0u) return;
  const unsigned want = seq - 1u;
  if (ld_acquire_gpu_u32(net_seq + b) < want) {
    unsigned long long t0, t1;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
    while (ld_acquire_gpu_u32(net_seq + b) < want) {
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
      if (t1 - t0 > 2000000000ull) __trap();  // two seconds: a broken launch order, not a slow predecessor
    }
  }
  asm volatile("fence.proxy.async;" ::: "memory");  // the bulk copy that follows reads what another CTA's stores wrote
}

// Decisions of one update for theta plane k, float64 exactly as numpy computes them on the host
// (posecell_network.py:252-267,249,304).  plan[k] = (ox mod X, oy mod Y, ox*Y + oy, LUT filter).
template <int X, int Y, int T>
__device__ __forceinline__ void plan_plane(int k, const double* __restrict__ od, const double* __restrict__ cos_th,
                                           const double* __restrict__ sin_th, double vtrans_scale, double vrot_scale,
                                           int* plan, int* err_b, int* err_s) {
  const double vt = __ddiv_rn(od[0], vtrans_scale);
  const double ex = __dmul_rn(vt, cos_th[k]);
  const double ey = __dmul_rn(vt, sin_th[k]);
  const double oxd = rint(ex), oyd = rint(ey);  // numpy.around: half to even
  const int key = (int)__dmul_rn(__dsub_rn(ex, oxd), 10.0);
  const int ox = modp((int)oxd, X), oy = modp((int)oyd, Y);
  reinterpret_cast<int4*>(plan)[k] = make_int4(ox, oy, ox * Y + oy, key < 0 ? 1 : 0);
  int e = key >= 5 ? PRS_ERR_LUT_KEY : 0;
  if (k == 0) {
    if (!(3.0 + ceil(fabs(vt)) <= (double)(X < Y ? X : Y))) e |= PRS_ERR_RADIUS;
    const double og = floor(__dadd_rn(__ddiv_rn(od[1], vrot_scale), 0.5));
    if (!(fabs(og) <= 64.0)) e |= PRS_ERR_THETA;
    const int ogc = og < -(double)PRS_OG_RANGE ? -PRS_OG_RANGE : (og > (double)PRS_OG_RANGE ? PRS_OG_RANGE : (int)og);
    plan[4 * T] = ogc + PRS_OG_RANGE;
  }
  if (e) {
    atomicOr(err_b, e);
    atomicOr(err_s, e);  // the CTA's own copy: what the packed result reports (err_b may be re-zeroed by the next launch)
  }
}

// Optional in-kernel stage timing (profiling builds of this file only: -DPRS_RESIDENT_TIMING).  Thread 0 of
// CTA 0 accumulates the cycles between consecutive barriers into timing[0..6].
#ifdef PRS_RESIDENT_TIMING
__device__ unsigned long long g_stage_cycles[8];
#define PRS_STAMP(i)                                                   \
  do {                                                                 \
    if (blockIdx.x == 0 && threadIdx.x == 0) {                         \
      const long long now_ = clock64();                                \
      if ((i) > 0) g_stage_cycles[(i)-1] += now_ - stamp_;             \
      else if (stamp_) g_stage_cycles[6] += now_ - stamp_;             \
      stamp_ = now_;                                                   \
    }                                                                  \
  } while (0)
#else
#define PRS_STAMP(i) \
  do {               \
  } while (0)
#endif

// LIST: the work items are the *wl_cnt networks listed in wl (the dense fall-back of the active-set path) instead of all B
// networks; a separate instantiation, so that the plain kernel pays nothing for the indirection.
template <int X, int Y, int T, int NT, bool LIST>
__global__ void __launch_bounds__(NT, 1)
    k_pc_resident(float* state, const double* __restrict__ odom, int n_steps, const float* __restrict__ gi,
                  long long* __restrict__ argmax, float* __restrict__ total, int* __restrict__ err,
                  const double* __restrict__ cos_th, const double* __restrict__ sin_th, double vtrans_scale,
                  double vrot_scale, int B, const PcTables<float>* __restrict__ tab_g, int ablate,
                  const int* __restrict__ wl, const int* __restrict__ wl_cnt, unsigned* __restrict__ net_seq, unsigned seq,
                  int4* __restrict__ xyze, unsigned* __restrict__ done_ctr, unsigned* __restrict__ done_host,
                  unsigned done_val) {
  using L = ResLayout<X, Y, T>;
  constexpr int XY = L::XY, N = L::N, NP = L::NP, PS = L::PS;
  constexpr int kPlanT0 = NT - 64;  // the threads that prepare the next update's plan during stage 4
  static_assert(X >= 7 && Y >= 7 && T >= 3, "resident kernel needs X, Y >= 7");
  static_assert((N * 4) % 16 == 0, "bulk copies move multiples of 16 bytes");
  static_assert(kPlanT0 >= NP * X && T <= 64, "the planning threads must be idle in stage 4");
  static_assert(NP * X <= NT && NP * Y <= NT && XY <= NT, "one work item per thread in stages 1, 3, 4, 5");
  static_assert(T % 2 == 0 && T >= 8, "mirror plane pairs need an even number of theta planes");
  // planes of the previous network's deferred result written during stage 1; the rest go out at the head of
  // stage 2 (the LSU queue, "stall_lg", is what stage 1 waits for once its index arithmetic is gone)
  constexpr int kDefer1 = PRS_RESIDENT_DEFER1 < T ? PRS_RESIDENT_DEFER1 : T;
  constexpr int MID = T / 2;  // posecell_network.py:257: mid = floor(Th / 2); pair m = (MID + m, MID - m), pair 0 = (MID, 0)
  constexpr int NW = (NT + 31) / 32;
  extern __shared__ __align__(128) unsigned char smem[];
  float* stage = reinterpret_cast<float*>(smem + L::kStageOff);
  float2* buf2 = reinterpret_cast<float2*>(smem + L::kBufOff);
  float2* A2 = buf2;            // [NP][X+6 rows][Y], plane stride PS
  float2* B2 = buf2 + NP * PS;  // [NP][X][Y]
  const PcTables<float>* tab = reinterpret_cast<const PcTables<float>*>(smem + L::kTabOff);
  float2* s_f2p = reinterpret_cast<float2*>(smem + L::kPairOff);  // [(fs0*2+fs1)*7 + a][8]
  float2* s_cf_ty = reinterpret_cast<float2*>(smem + L::kCfOff);
  float2* s_cf_x = s_cf_ty + 7;
  int* s_plan = reinterpret_cast<int*>(smem + L::kPlanOff);
  int* red_i = reinterpret_cast<int*>(smem + L::kRedOff);  // [0..NW) warp maxima, [30], [31] the two arg-max slots
  float* red_f = reinterpret_cast<float*>(smem + L::kRedOff + 32 * 4);
  float* s_val = red_f + 32;
  unsigned long long* bar = reinterpret_cast<unsigned long long*>(smem + L::kBarOff);
  const int tid = threadIdx.x;
  const int wid = tid >> 5, lane = tid & 31;
  // Work items: the B networks, or -- as the dense fallback of the active-set path (posecell_active.cu) -- the *wl_cnt
  // networks listed in wl.
  const int nW = LIST ? *wl_cnt : B;
  if ((int)blockIdx.x >= nW) return;
  auto net = [&](int wi) { return LIST ? wl[wi] : wi; };
  // seq != 0: this launch is number `seq` of the plan's chain of overlappable launches.  The next one may be scheduled as
  // soon as SMs are free (the CTAs of a ragged last wave leave 80 of 148 SMs idle for a whole network otherwise); it
  // waits per network, not per grid.
  if (seq != 0u) asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  // xyze != nullptr (single-update launches of the host API): the result also leaves as (x, y, th, err) per network --
  // get_pc_max's unravelling (posecell_network.py:318) -- which saves the host API a kernel between two updates
  auto publish = [&](size_t off, int pslot, float tot_) {
    const int flat = red_i[30 + pslot];
    argmax[off] = (long long)flat;
    total[off] = tot_;
    if (xyze != nullptr) {
      const int xy = flat / T, th = flat - xy * T, x = xy / Y;
      xyze[off] = make_int4(x, xy - x * Y, th, red_i[28 + pslot]);
    }
  };

  // ---- one-time set-up: first prefetch and the first plan's odometry (possibly a read over PCIe) are under way while the
  //      tables and coefficient pairs are copied; then the first plan
  if (tid == NT - 1) {
    mbar_init(bar, 1);
    fence_proxy_async();
    wait_network(net_seq, net(blockIdx.x), seq);
    mbar_expect_tx(bar, N * 4);
    bulk_g2s(stage, state + (size_t)net(blockIdx.x) * N, N * 4, bar);
    err[net(blockIdx.x)] = 0;  // the kernel owns err[b]: zeroed before the network's first plan ORs its bits in
    red_i[28] = red_i[29] = 0;  // error bits of the two plan slots, as the packed result reports them
  }
  double od0[2] = {0.0, 0.0};
  const bool planner = tid >= kPlanT0 && tid < kPlanT0 + T && n_steps > 0;
  if (planner) {
    const double* od = odom + (size_t)net(blockIdx.x) * 2;
    od0[0] = od[0], od0[1] = od[1];
  }
  for (int i = tid; i < (int)(sizeof(PcTables<float>) / 4); i += NT)
    reinterpret_cast<float*>(smem + L::kTabOff)[i] = reinterpret_cast<const float*>(tab_g)[i];
  if (tid < 7) {
    s_cf_ty[tid] = make_float2(tab_g->ge[tid], tab_g->gi[tid]);
    s_cf_x[tid] = make_float2(tab_g->gex[tid], tab_g->gix[tid]);
  }
  for (int i = tid; i < 4 * 7 * 8; i += NT) {
    const int q = i & 7, a = (i >> 3) % 7, combo = i / 56;
    s_f2p[i] = q < 7 ? make_float2(tab_g->f2d[combo >> 1][a * 7 + q], tab_g->f2d[combo & 1][a * 7 + q])
                     : make_float2(0.f, 0.f);
  }
  __syncthreads();
  if (planner)
    plan_plane<X, Y, T>(tid - kPlanT0, od0, cos_th, sin_th, vtrans_scale, vrot_scale, s_plan, err + net(blockIdx.x),
                        red_i + 28);
  __syncthreads();
  uint32_t parity = 0;
  int slot = 0;
  // Results of stage 5 are written to global memory lazily: when the CTA moves on to another network, the
  // 36 stores per thread are interleaved with the next network's stage 1 instead of bursting at the end of
  // stage 5 (measured: the burst stalls on the LSU queue, "stall_lg"; -4.7 % per update).  Staging them in the
  // consumed lines of the TMA buffer and writing them with one cp.async.bulk store was also measured: not faster
  // (stage 1 is bound by issue slots and registers, not by the store path).
  float2 out[NP];
  float* st_gst = nullptr;  // where the deferred results go, nullptr if none are pending
  bool pend_valid = false;
  int pend_slot = 0;
  size_t pend_off = 0;
  float pend_tot = 0.f;
#ifdef PRS_RESIDENT_TIMING
  long long stamp_ = 0;
#endif

  for (int wi = blockIdx.x; wi < nW; wi += gridDim.x) {
    const int b = net(wi);
    float* gst = state + (size_t)b * N;
    const float g_inh = gi[b], g_lo = inhib_floor(g_inh);
    for (int step = 0; step < n_steps; ++step) {
      const int* plan = s_plan + slot * L::kPlanInts;
      const int4* plan4 = reinterpret_cast<const int4*>(plan);
      PRS_STAMP(0);

      // ---- 1. theta pass of the separable DoG: stage (or global on later steps) -> (E, I) pairs.
      //      The integer origin the reference adds to its read index in the 2-D stage (convolution.py:320-340)
      //      is a translation of the whole plane, and every stage up to the 2-D one is a periodic correlate that
      //      commutes with it.  It is applied where it is free: the y part when stage 3 chooses the column a
      //      thread reads (one wrap per thread), the x part when stage 4 chooses its first row (one wrap per
      //      thread) -- not here, where it cost a plan load and six integer instructions per cell.
      if (step == 0) {
        mbar_wait(bar, parity);
        parity ^= 1;
      }
      if (!(ablate & 1) && tid < XY) {
        const float e0 = tab->ge[3], e1 = tab->ge[2], e2 = tab->ge[1], e3 = tab->ge[0];
        const float i0 = tab->gi[3], i1 = tab->gi[2], i2 = tab->gi[1], i3 = tab->gi[0];
        const int p = tid;
        // Plane 0 shares pair 0 with plane MID, whose x origin is the opposite one (cos(-pi) = -cos(0)); stage 4
        // applies the origin of a pair's first plane to both, so plane 0 is stored rotated by the difference.
        int p0 = p - (plan4[0].x - plan4[MID].x) * Y;
        p0 += p0 < 0 ? XY : 0;
        p0 -= p0 >= XY ? XY : 0;
        float in[T];
        if (step == 0) {
#pragma unroll
          for (int k = 0; k < T; ++k) in[k] = stage[k * XY + p];
        } else {
#pragma unroll
          for (int k = 0; k < T; ++k) in[k] = gst[k * XY + p];
        }
#pragma unroll
        for (int k = 0; k < T; ++k) {
          const float c = in[k];
          const float s1 = in[(k + 1) % T] + in[(k + T - 1) % T];
          const float s2 = in[(k + 2) % T] + in[(k + T - 2) % T];
          const float s3 = in[(k + 3) % T] + in[(k + T - 3) % T];
          const float e = fmaf(e0, c, fmaf(e1, s1, fmaf(e2, s2, e3 * s3)));
          const float i = fmaf(i0, c, fmaf(i1, s1, fmaf(i2, s2, i3 * s3)));
          buf2[k == 0 ? p0 : k * XY + p] = make_float2(e, i);
          if (st_gst != nullptr && k < kDefer1) {  // the previous network's plane k (mirror pair layout of out[])
            const float v = k == 0 ? out[0].y : (k < MID ? out[MID - k].y : (k == MID ? out[0].x : out[k - MID].x));
            st_gst[k * XY + p] = v;
          }
        }
        if (kDefer1 == T) st_gst = nullptr;
      }
      __syncthreads();
      PRS_STAMP(1);
      if (tid == 0 && pend_valid)  // every winner of the previous update has done its atomicMin by now
        publish(pend_off, pend_slot, pend_tot);
      pend_valid = false;
      // (the staging buffer is free again from here on; the next network is fetched by an idle thread of stage 4: code
      // at this spot -- even code that does not run -- costs the y pass 3 % of the update, measured)

      // ---- 2. y pass, in place on each (theta, x) line; the remaining deferred result planes leave here
      if (kDefer1 < T && st_gst != nullptr) {
        if (tid < XY) {
#pragma unroll
          for (int k = kDefer1; k < T; ++k) {
            const float v = k == 0 ? out[0].y : (k < MID ? out[MID - k].y : (k == MID ? out[0].x : out[k - MID].x));
            st_gst[k * XY + tid] = v;
          }
        }
        st_gst = nullptr;
      }
      if (!(ablate & 2)) {
        float2 cf[7];
#pragma unroll
        for (int t = 0; t < 7; ++t) cf[t] = s_cf_ty[t];
        constexpr int IT2 = (T * X + NT - 1) / NT;
#pragma unroll
        for (int it = 0; it < IT2; ++it) {
          const int ln = tid + it * NT;
          if (ln < T * X) {
            float2* line = buf2 + ln * Y;
            float2 in[Y];
#pragma unroll
            for (int y = 0; y < Y; ++y) in[y] = line[y];
#pragma unroll
            for (int y = 0; y < Y; ++y) {
              float2 acc = make_float2(0.f, 0.f);
#pragma unroll
              for (int t = 0; t < 7; ++t) acc = ffma2(in[(y + t + Y - 3) % Y], cf[t], acc);
              line[y] = acc;
            }
          }
        }
      }
      __syncthreads();
      PRS_STAMP(2);
      // the previous network's deferred stores are behind the barrier above: its state is complete (no variable of its
      // own for this -- the kernel's hot stages use every register they can get)
      if (tid == 0 && seq != 0u && step == 0 && wi != (int)blockIdx.x) {
        __threadfence();
        st_release_gpu_u32(net_seq + net(wi - (int)gridDim.x), seq);
      }

      // ---- 3. x pass + global inhibition (posecell_network.py:339-340) + sum (:343).
      //      A thread takes the same (y) column of BOTH planes of a mirror pair, so that the result is
      //      written as one float2 per cell.  Items are enumerated y-fastest (measured: a plane-fastest
      //      enumeration costs 2x shared-memory wavefronts on these 64-bit accesses).
      float2 keep[X];
      float psum = 0.f;
#pragma unroll
      for (int x = 0; x < X; ++x) keep[x] = make_float2(0.f, 0.f);
      const int kp3 = tid / Y, y3 = tid - kp3 * Y;  // y fastest: a warp reads contiguous float2 runs
      if (!(ablate & 4) && tid < NP * Y) {
        float2 cf[7];
#pragma unroll
        for (int t = 0; t < 7; ++t) cf[t] = s_cf_x[t];
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          const int k = h == 0 ? MID + kp3 : (kp3 == 0 ? 0 : MID - kp3);
          {
            // y origin of plane k: output column y3 is computed from input column y3 + oy_k (one wrap per thread)
            int ys = y3 + plan4[k].y;
            ys -= ys >= Y ? Y : 0;
            const float2* col = buf2 + k * XY + ys;
            float2 in[X];
#pragma unroll
            for (int x = 0; x < X; ++x) in[x] = col[x * Y];
#pragma unroll
            for (int x = 0; x < X; ++x) {
#if PRS_RESIDENT_S3FOLD
              float2 acc = make_float2(-g_inh, 0.f);  // the inhibition rides in the accumulator: one FADD less per cell
#pragma unroll
              for (int t = 0; t < 7; ++t) acc = ffma2(in[(x + t + X - 3) % X], cf[t], acc);
              const float a = fmaxf(acc.x - acc.y, 0.f);  // (a < gi) ? 0 : a - gi; gi < 0: see below the loop
#else
              float2 acc = make_float2(0.f, 0.f);
#pragma unroll
              for (int t = 0; t < 7; ++t) acc = ffma2(in[(x + t + X - 3) % X], cf[t], acc);
              const float d = (acc.x - acc.y) - g_inh;
              const float a = d < 0.f ? g_lo : d;  // (a < gi) ? max(-gi, 0) : a - gi (inhib_floor)
#endif
              if (h == 0)
                keep[x].x = a;
              else
                keep[x].y = a;
#if !PRS_RESIDENT_S3FOLD
              psum += a;
#endif
            }
          }
        }
#if PRS_RESIDENT_S3FOLD
        // gi < 0 only (a uniform branch): the cells the max above clamped end at -gi, not at 0 (inhib_floor).  A cell with
        // d == 0 exactly sits on the threshold within the rounding of the folded sum and goes with the cells below it.
        // For gi >= 0 the clamp is the whole inhibition, one FMNMX per cell.
        if (g_lo != 0.f) {
#pragma unroll
          for (int x = 0; x < X; ++x) {
            keep[x].x = keep[x].x == 0.f ? g_lo : keep[x].x;
            keep[x].y = keep[x].y == 0.f ? g_lo : keep[x].y;
          }
        }
        float2 ps2 = keep[0];  // both planes of the pair at once (add.f32x2)
#pragma unroll
        for (int x = 1; x < X; ++x) ps2 = __fadd2_rn(ps2, keep[x]);
        psum = ps2.x + ps2.y;
#endif
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) psum += __shfl_xor_sync(0xffffffffu, psum, o);
      if (lane == 0) red_f[wid] = psum;
      __syncthreads();  // every (E, I) pair has been consumed: the bytes become A2 / B2
      PRS_STAMP(3);
      if (!(ablate & 8) && tid < NP * Y) {
        float2* dst = A2 + kp3 * PS + y3;  // row r of the halo layout is grid row r - 3
#pragma unroll
        for (int x = 0; x < X; ++x) {
          dst[(x + 3) * Y] = keep[x];
          if (x < 3) dst[(x + 3 + X) * Y] = keep[x];
          if (x >= X - 3) dst[(x + 3 - X) * Y] = keep[x];
        }
      }
      if (wid == 0) {
        float sacc = lane < (NT + 31) / 32 ? red_f[lane] : 0.f;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) sacc += __shfl_xor_sync(0xffffffffu, sacc, o);
        if (lane == 0) s_val[0] = sacc;
      }
      // the error bits of the next plan start from zero, a barrier ahead of stage 4 where it is made: the shared-memory
      // copy of its slot, and err[] of the next network when that plan is its first (the previous launch ORed its own bits
      // into err[] before it finished the network this CTA is working on, so this store comes after them)
      if (tid == NT - 1) {
        red_i[28 + (slot ^ 1)] = 0;
        if (step == 0 && wi + (int)gridDim.x < nW) err[net(wi + (int)gridDim.x)] = 0;
      }
      __syncthreads();  // publishes A2 and the total
      PRS_STAMP(4);
      // posecell_network.py:344-345.  The normalisation is a positive scale: max(s*v, 0) = s*max(v, 0) and the
      // theta pass is linear, so stage 4 runs un-normalised and 1/total is folded into stage 5's seven taps.
      const float tot = s_val[0];
      const float inv = (tot != 0.f) ? 1.f / tot : 1.f;

      // ---- 4. 7x7 periodic correlate of both planes of a pair at once (posecell_network.py:273-274,300);
      //      meanwhile two otherwise idle warps prepare the plan of the next update.
      const bool last_step = (step + 1 == n_steps);
      const int nwi = last_step ? wi + (int)gridDim.x : wi;
      const int nb = nwi < nW ? net(nwi) : 0;
      const int nstep = last_step ? 0 : step + 1;
      if (tid >= kPlanT0) {
        if (tid < kPlanT0 + T && nwi < nW)
          plan_plane<X, Y, T>(tid - kPlanT0, odom + ((size_t)nstep * B + nb) * 2, cos_th, sin_th, vtrans_scale,
                              vrot_scale, s_plan + (slot ^ 1) * L::kPlanInts, err + nb, red_i + 28 + (slot ^ 1));
        // The staging buffer has been free since stage 1: an otherwise idle thread fetches the next network while this
        // one is computed -- after it has seen that network's state of the previous launch complete.
        if (tid == NT - 1 && step == 0 && wi + (int)gridDim.x < nW) {
          const int fb = net(wi + (int)gridDim.x);
          fence_proxy_async();
          wait_network(net_seq, fb, seq);
          mbar_expect_tx(bar, N * 4);
          bulk_g2s(stage, state + (size_t)fb * N, N * 4, bar);
        }
      } else if (!(ablate & 16) && tid < NP * X) {
        const int kp = tid / X, x = tid - kp * X;
        const int fsA = plan4[MID + kp].w, fsB = plan4[kp == 0 ? 0 : MID - kp].w;
        const float2* ctab = s_f2p + (fsA * 2 + fsB) * 56;
        const float2* rows = A2 + kp * PS + x * Y;  // halo layout: tap row a of output row x is row x + a
        float2 acc[Y];
#pragma unroll
        for (int j = 0; j < Y; ++j) acc[j] = make_float2(0.f, 0.f);
#pragma unroll
        for (int a = 0; a < 7; ++a) {
          float2 row[Y];
#pragma unroll
          for (int j = 0; j < Y; ++j) row[j] = rows[a * Y + j];
          const float4* cp = reinterpret_cast<const float4*>(ctab + a * 8);
          const float4 c01 = cp[0], c23 = cp[1], c45 = cp[2], c6x = cp[3];
          const float2 cf[7] = {make_float2(c01.x, c01.y), make_float2(c01.z, c01.w), make_float2(c23.x, c23.y),
                                make_float2(c23.z, c23.w), make_float2(c45.x, c45.y), make_float2(c45.z, c45.w),
                                make_float2(c6x.x, c6x.y)};
#pragma unroll
          for (int j = 0; j < Y; ++j) {
#pragma unroll
            for (int q = 0; q < 7; ++q) acc[j] = ffma2(row[(j + q + Y - 3) % Y], cf[q], acc[j]);
          }
        }
        // x origin of the pair (mirror planes have the same cosine, hence the same origin; pair 0: see stage 1):
        // the row computed from rows x-3..x+3 is row x - ox of the result.  Applied to the 21 stores rather than to
        // the 175 loads, whose conflict-free bank pattern a rotated row index would break.
        int xs = x - plan4[MID + kp].x;
        xs += xs < 0 ? X : 0;
        float2* o = B2 + kp * XY + xs * Y;
#pragma unroll
        for (int j = 0; j < Y; ++j)  // posecell_network.py:300; 1/total is applied by stage 5 (see there)
          o[j] = make_float2(fmaxf(acc[j].x, 0.f), fmaxf(acc[j].y, 0.f));
      }
      __syncthreads();
      PRS_STAMP(5);

      // ---- 5. theta pass (convolution.py:344-359), clamp (:314), registers -> global, maximum.
      //      For the mirror pair m = (MID+m, MID-m) the tap at offset u reads planes MID+(m+u) and MID-(m-u):
      //      the same pair m+u for both halves when the second half takes the taps in reverse, i.e.
      //      acc += pair(m+u) * (f[3+u], f[3-u]).  Pairs that fall off either end are swapped or pair 0.
      float vmax = 0.f;
      if (!(ablate & 32) && tid < XY) {
        const int p = tid;
        float fc[7];
        const float* f1 = tab->f1d[plan[4 * T]];
#pragma unroll
        for (int t = 0; t < 7; ++t) fc[t] = f1[t] * inv;
        float2 pin[NP];
#pragma unroll
        for (int kk = 0; kk < NP; ++kk) pin[kk] = B2[kk * XY + p];
        float2 cf2[7];
#pragma unroll
        for (int u = -3; u <= 3; ++u) cf2[u + 3] = make_float2(fc[3 + u], fc[3 - u]);
#pragma unroll
        for (int m = 1; m < NP; ++m) {
          float2 acc = make_float2(0.f, 0.f);
#pragma unroll
          for (int u = -3; u <= 3; ++u) {
            const int j = m + u;
            float2 v;
            if (j >= 1 && j <= NP - 1)
              v = pin[j];
            else if (j == 0)
              v = make_float2(pin[0].x, pin[0].x);                    // plane MID on both sides
            else if (j == NP)
              v = make_float2(pin[0].y, pin[0].y);                    // plane 0 == plane T on both sides
            else if (j < 0)
              v = make_float2(pin[-j].y, pin[-j].x);                  // crossed the middle: halves swap
            else
              v = make_float2(pin[2 * NP - j].y, pin[2 * NP - j].x);  // crossed plane 0: halves swap
            acc = ffma2(v, cf2[u + 3], acc);
          }
          out[m] = make_float2(fmaxf(acc.x, 0.f), fmaxf(acc.y, 0.f));
        }
        {  // pair 0 = (MID, 0)
          float a = 0.f, c = 0.f;
#pragma unroll
          for (int u = -3; u <= 3; ++u) {
            const float va = u > 0 ? pin[u].x : (u < 0 ? pin[-u].y : pin[0].x);
            const float vc = u > 0 ? pin[NP - u].y : (u < 0 ? pin[NP + u].x : pin[0].y);
            a = fmaf(fc[3 + u], va, a);
            c = fmaf(fc[3 + u], vc, c);
          }
          out[0] = make_float2(fmaxf(a, 0.f), fmaxf(c, 0.f));
        }
        vmax = fmaxf(out[0].x, out[0].y);
#pragma unroll
        for (int m = 1; m < NP; ++m) vmax = fmaxf(vmax, fmaxf(out[m].x, out[m].y));
        if (step + 1 < n_steps) {  // the next update of this network reads the state back from global memory
          gst[MID * XY + p] = out[0].x;
          gst[p] = out[0].y;
#pragma unroll
          for (int m = 1; m < NP; ++m) {
            gst[(MID + m) * XY + p] = out[m].x;
            gst[(MID - m) * XY + p] = out[m].y;
          }
        } else {
          st_gst = gst;  // deferred into the next network's stage 1 (or the kernel's epilogue)
        }
      }
      // arg-max (numpy.argmax: first maximum in [x][y][th] order).  Values are >= 0, so their bit patterns order
      // like the values: one REDUX per warp, one per block; then only the thread(s) holding the maximum look
      // for its lowest theta and race with atomicMin on the flat index.
      const unsigned vbits = __float_as_uint(vmax);
      const unsigned wmax = __reduce_max_sync(0xffffffffu, vbits);
      if (lane == 0) red_i[wid] = (int)wmax;
      if (tid == 0) red_i[30 + slot] = 0x7fffffff;
      __syncthreads();  // the state in global memory and every SMEM slot are consistent for the next update
      PRS_STAMP(6);
      {
        const unsigned gmax = __reduce_max_sync(0xffffffffu, lane < NW ? (unsigned)red_i[lane] : 0u);
        if (tid < XY && vbits == gmax) {
          int kbest = T;
#pragma unroll
          for (int k = T - 1; k >= 0; --k) {  // descending, so the lowest matching theta is what remains
            const float v = k == 0 ? out[0].y : (k < MID ? out[MID - k].y : (k == MID ? out[0].x : out[k - MID].x));
            if (v == vmax) kbest = k;
          }
          atomicMin(&red_i[30 + slot], tid * T + kbest);
        }
      }
      // the result of this update is complete after the next barrier; thread 0 publishes it there
      pend_valid = true;
      pend_slot = slot;
      pend_off = (size_t)step * B + b;
      pend_tot = tot;
      slot ^= 1;
    }
  }
  if (st_gst != nullptr && tid < XY) {
    st_gst[MID * XY + tid] = out[0].x;
    st_gst[tid] = out[0].y;
#pragma unroll
    for (int m = 1; m < NP; ++m) {
      st_gst[(MID + m) * XY + tid] = out[m].x;
      st_gst[(MID - m) * XY + tid] = out[m].y;
    }
  }
  __syncthreads();
  if (tid == 0 && pend_valid) publish(pend_off, pend_slot, pend_tot);
  if (tid == 0 && seq != 0u && n_steps > 0) {  // the last network of this CTA
    const int last_wi = (int)blockIdx.x + ((nW - 1 - (int)blockIdx.x) / (int)gridDim.x) * (int)gridDim.x;
    __threadfence();
    st_release_gpu_u32(net_seq + net(last_wi), seq);
  }
  // The zero-copy host API polls one word of pinned memory instead of an event (an event between two launches would
  // keep them from overlapping): the last CTA of the launch to get here stores the launch's number, behind the records.
  if (tid == 0 && done_host != nullptr) {
    __threadfence_system();
    if (atomicAdd(done_ctr, 1u) == gridDim.x - 1u) {
      atomicExch(done_ctr, 0u);
      __threadfence_system();
      asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(done_host), "r"(done_val) : "memory");
    }
  }
}

template <int X, int Y, int T, int NT>
int launch(prs_pc_plan* p, float* state, const double* odom, int n_steps, const float* gi, long long* argmax,
           float* total, int* err, cudaStream_t st) {
  using L = ResLayout<X, Y, T>;
  auto kern = k_pc_resident<X, Y, T, NT, false>;
  auto kern_list = k_pc_resident<X, Y, T, NT, true>;
  static bool configured[64] = {};  // function attributes are per device
  static int nsm_of[64] = {};
  const int dev = p->device;
  PRS_REQUIRE(dev >= 0 && dev < 64, "resident path: device index %d out of range", dev);
  {
    static std::mutex mu;  // two host threads may make their first call at the same time
    std::lock_guard<std::mutex> lk(mu);
    if (!configured[dev]) {
      PRS_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)L::kBytes));
      PRS_CUDA(cudaFuncSetAttribute(kern_list, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)L::kBytes));
      PRS_CUDA(cudaDeviceGetAttribute(&nsm_of[dev], cudaDevAttrMultiProcessorCount, dev));
      configured[dev] = true;
    }
  }
  const int nsm = nsm_of[dev];
  // (as the active-set fallback the work-list length is only known on the device: CTAs without work return at once)
  const int grid = p->B < nsm ? p->B : nsm;
  // PRS_RESIDENT_ABLATE (profiling only): bit i skips stage i+1 to attribute time; results are then meaningless
  static int ablate = [] {
    const char* e = getenv("PRS_RESIDENT_ABLATE");
    return e ? atoi(e) : 0;
  }();
  // Overlappable launches (programmatic dependent launch + per-network sequence numbers): whole-ensemble launches on a
  // stream that is not being captured.  PRS_RESIDENT_PDL=0 switches it off (profiling).
  static const bool pdl_on = [] {
    const char* e = getenv("PRS_RESIDENT_PDL");
    return !(e && atoi(e) == 0);
  }();
  cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
  if (st != nullptr) PRS_CUDA(cudaStreamIsCapturing(st, &cap));
  const bool pdl = pdl_on && p->only_list == nullptr && cap == cudaStreamCaptureStatusNone && p->net_seq != nullptr;
  bool launched = false;
  if (pdl) {
    const unsigned seq = p->res_seq + 1u;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(grid), cfg.blockDim = dim3(NT), cfg.dynamicSmemBytes = L::kBytes, cfg.stream = st;
    cudaLaunchAttribute at;
    at.id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at.val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = &at, cfg.numAttrs = 1;
    const cudaError_t le = cudaLaunchKernelEx(
        &cfg, kern, state, odom, n_steps, gi, argmax, total, err, (const double*)p->cos_th, (const double*)p->sin_th,
        p->vtrans_scale, p->vrot_scale, p->B, (const PcTables<float>*)p->tab_dev, ablate, (const int*)nullptr,
        (const int*)nullptr, p->net_seq, seq, (int4*)(n_steps == 1 ? p->res_xyze : nullptr), p->res_done_ctr,
        p->res_done_host, p->res_done_val);
    if (le == cudaSuccess) {
      p->res_seq = seq;
      launched = true;
    } else {  // a driver that refuses the attribute: plain launches from now on (the chain of sequence numbers ends here)
      (void)cudaGetLastError();
      cudaFree(p->net_seq);
      p->net_seq = nullptr;
    }
  }
  if (launched) {
    // (launched above, overlappable)
  } else if (p->only_list != nullptr) {
    kern_list<<<grid, NT, L::kBytes, st>>>(state, odom, n_steps, gi, argmax, total, err, p->cos_th, p->sin_th,
                                           p->vtrans_scale, p->vrot_scale, p->B, (const PcTables<float>*)p->tab_dev, ablate,
                                           p->only_list, p->only_cnt, nullptr, 0u, nullptr, nullptr, nullptr, 0u);
  } else {
    kern<<<grid, NT, L::kBytes, st>>>(state, odom, n_steps, gi, argmax, total, err, p->cos_th, p->sin_th, p->vtrans_scale,
                                      p->vrot_scale, p->B, (const PcTables<float>*)p->tab_dev, ablate, nullptr, nullptr,
                                      nullptr, 0u, (int4*)(n_steps == 1 ? p->res_xyze : nullptr), p->res_done_ctr,
                                      p->res_done_host, p->res_done_val);
  }
  PRS_CUDA(cudaGetLastError());
  return PRS_OK;
}

}  // namespace

#ifdef PRS_RESIDENT_TIMING
extern "C" __attribute__((visibility("default"))) int prs_debug_stage_cycles(unsigned long long* out8, int reset) {
  PRS_CUDA(cudaDeviceSynchronize());
  PRS_CUDA(cudaMemcpyFromSymbol(out8, g_stage_cycles, 8 * sizeof(unsigned long long)));
  if (reset) {
    unsigned long long z[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    PRS_CUDA(cudaMemcpyToSymbol(g_stage_cycles, z, sizeof(z)));
  }
  return PRS_OK;
}
#endif

int prs_pc_resident_supported(const prs_pc_plan* p) {
  if (p->dtype != PRS_F32) return 0;
  if (!(p->X == 21 && p->Y == 21 && p->Th == 36)) return 0;
  // The kernel applies ONE x origin per mirror pair (MID+m, MID-m), m >= 1: around(vt * cos) must be the same for
  // both planes, which holds when the host's cosine table is bitwise even about MID (numpy's cos is).
  const int mid = p->Th / 2;
  for (int m = 1; m < mid; ++m)
    if (p->h_cos[mid + m] != p->h_cos[mid - m]) return 0;
  return 1;
}

int prs_pc_resident_step(prs_pc_plan* p, void* state, const double* odom, int T, const void* gi, long long* argmax,
                         void* total, int* err, cudaStream_t st) {
  if (p->X == 21 && p->Y == 21 && p->Th == 36) {
    // PRS_RESIDENT_NT selects the CTA size (tuning knob; the default is the measured best)
    static int nt = [] {
      const char* e = getenv("PRS_RESIDENT_NT");
      return e ? atoi(e) : 448;
    }();
    if (nt == 512)
      return launch<21, 21, 36, 512>(p, (float*)state, odom, T, (const float*)gi, argmax, (float*)total, err, st);
    return launch<21, 21, 36, 448>(p, (float*)state, odom, T, (const float*)gi, argmax, (float*)total, err, st);
  }
  prs_set_error("resident path not available for this plan");
  return PRS_E_INVALID;
}
