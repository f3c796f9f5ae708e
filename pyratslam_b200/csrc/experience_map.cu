// Linked experience maps of an ensemble on the device (prs_em_*, include/pyratslam_b200.h).
//
// The per-frame update of pyratslam_b200/experience_map.py (ExperienceMap.update with linked=True: _find, _add_link,
// _create_linked, _set_current) for B agents over T recorded frames.  Each agent is a serial chain of T dependent
// steps, so one thread runs one agent and the agents run in parallel; small blocks spread them over the SMs.
//
// Every decision -- create an experience, close a loop, do nothing, add a link or find it already there -- depends only
// on integer cells, template tags and the IEEE-exact sqrt(d2) <= delta_pc test, so it is bit-identical to the host.
// The double arithmetic is written with __dadd_rn / __dsub_rn / __dmul_rn / __ddiv_rn, which nvcc does not contract
// into FMAs (Python does none), so clip_rad_180, signed_delta_rad and every heading sum are bit-identical as well.
// Only cos, sin, atan2 and hypot may differ from glibc's by an ulp or two: they reach the positions, the link lengths
// and the link headings, never a decision.
#include <math.h>
#include <string.h>

#include "agent_moves.cuh"
#include "common.cuh"

namespace {

constexpr int kEmBlock = 32;                    // one warp per block: B = 1024 agents spread over 32 SMs
constexpr double kPi = 3.141592653589793;       // math.pi
constexpr double kTwoPi = 6.283185307179586;    // 2 * math.pi (exact)

// experience_map.py:clip_rad_180
__device__ __forceinline__ double clip_rad_180(double a) {
  if (a > kPi) return __dsub_rn(a, __dmul_rn(ceil(__ddiv_rn(a, kTwoPi)), kTwoPi));
  if (a <= -kPi) return __dadd_rn(a, __dmul_rn(ceil(__ddiv_rn(fabs(a), kTwoPi)), kTwoPi));
  return a;
}

// experience_map.py:signed_delta_rad
__device__ __forceinline__ double signed_delta_rad(double a, double b) {
  const double d = __dsub_rn(clip_rad_180(b), clip_rad_180(a));
  if (d > kPi) return __dsub_rn(d, kTwoPi);
  if (d <= -kPi) return __dadd_rn(d, kTwoPi);
  return d;
}

// The workspace: structure-of-arrays, element [i][b] at i * B + b, each array at a multiple of 256 bytes, in the
// order of the header's documentation (Python views the same offsets).
struct EmLayout {
  size_t exp_x, exp_y, exp_th, link_d, link_heading, link_facing, rel, exp_cell, exp_tag, exp_next, out_head, link_from,
      link_to, link_next, vt_head, counts, bytes;
  EmLayout(int B, int T, int N) {
    size_t off = 0;
    auto take = [&](size_t rows, size_t elem) {
      const size_t o = off;
      off += (rows * B * elem + 255) / 256 * 256;
      return o;
    };
    exp_x = take(T, 8), exp_y = take(T, 8), exp_th = take(T, 8);
    link_d = take(T, 8), link_heading = take(T, 8), link_facing = take(T, 8);
    rel = take(3, 8);
    exp_cell = take(T, 8);
    exp_tag = take(T, 4), exp_next = take(T, 4), out_head = take(T, 4);
    link_from = take(T, 4), link_to = take(T, 4), link_next = take(T, 4);
    vt_head = take(N, 4);
    counts = take(4, 4);
    bytes = off;
  }
};

struct EmWork {
  double *exp_x, *exp_y, *exp_th, *link_d, *link_heading, *link_facing, *rel;
  long long* exp_cell;
  int *exp_tag, *exp_next, *out_head, *link_from, *link_to, *link_next, *vt_head, *counts;
};

// kResume = false: T frames from an empty map (prs_em_linked_run).  kResume = true (prs_em_linked_resume_run): the map
// the workspace holds -- counts, rel and the current experience's pose -- continues over T more frames; the workspace has
// E rows for the experiences and links and N template heads, and a moved frame that finds no room for one more of each,
// or a tag at or beyond N, sets *err and stops the agent instead of writing past them.
template <bool kResume>
__global__ void __launch_bounds__(kEmBlock)
    k_em_linked(int B, int T, int N, const long long* __restrict__ argmax, const int* __restrict__ tag,
                const double* __restrict__ tw, const uint8_t* __restrict__ moved, int X, int Y, int Th,
                double delta_pc, EmWork w, int* __restrict__ n_exp_out, int* __restrict__ exp_id_out,
                double* __restrict__ em_xy_out, int R = 1, const int* __restrict__ rec_of = nullptr, int E = 0,
                int* __restrict__ err = nullptr) {
  // rec_of (several recordings): agent b follows recording r = rec_of[b] of tw[T][R][2] and moved[T][R]
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  const int r = rec_of != nullptr ? rec_of[b] : 0;
  if (rec_of == nullptr) R = 1;
  const size_t sB = (size_t)B;
  if (!kResume)
    for (int v = 0; v < N; ++v) w.vt_head[v * sB + b] = -1;
  int n_exp = 0, n_links = 0, cur = -1, n_loop = 0;
  double rel_x = 0.0, rel_y = 0.0, rel_th = 0.0;
  double cur_x = 0.0, cur_y = 0.0, cur_th = 0.0;   // the current experience's pose, kept in registers
  if (kResume) {
    n_exp = w.counts[b], n_links = w.counts[sB + b], cur = w.counts[2 * sB + b], n_loop = w.counts[3 * sB + b];
    rel_x = w.rel[b], rel_y = w.rel[sB + b], rel_th = w.rel[2 * sB + b];
    if (cur >= 0) cur_x = w.exp_x[cur * sB + b], cur_y = w.exp_y[cur * sB + b], cur_th = w.exp_th[cur * sB + b];
  }
  const int YTh = Y * Th;

  // _add_link(current, to) without the duplicate check, with the agent's rel_* at this point
  auto link = [&](int to) {
    const size_t l = n_links * sB + b;
    w.link_from[l] = cur;
    w.link_to[l] = to;
    w.link_d[l] = hypot(rel_x, rel_y);
    w.link_heading[l] = signed_delta_rad(cur_th, atan2(rel_y, rel_x));
    w.link_facing[l] = signed_delta_rad(cur_th, rel_th);
    w.link_next[l] = w.out_head[cur * sB + b];
    w.out_head[cur * sB + b] = n_links;
    ++n_links;
  };
  // _set_current
  auto set_current = [&](int e, double x, double y, double th) {
    cur = e, cur_x = x, cur_y = y, cur_th = th;
    rel_x = 0.0, rel_y = 0.0, rel_th = th;
  };

  for (int t = 0; t < T; ++t) {
    const size_t tb = t * sB + b;
    const size_t tr = (size_t)t * R + r;
    if (moved[tr]) {
      if (kResume && (n_exp >= E || n_links >= E || tag[tb] >= N)) {
        atomicOr(err, 1);
        break;
      }
      // update(): the odometry since the current experience
      const double vtrans = tw[2 * tr], vrot = tw[2 * tr + 1];
      rel_th = clip_rad_180(__dadd_rn(rel_th, vrot));
      rel_x = __dadd_rn(rel_x, __dmul_rn(vtrans, cos(rel_th)));
      rel_y = __dadd_rn(rel_y, __dmul_rn(vtrans, sin(rel_th)));
      const long long cell = argmax[tb];
      const int px = (int)(cell / YTh), py = (int)(cell / Th % Y), pt = (int)(cell % Th);
      const int vt = (unsigned)tag[tb] < (unsigned)N ? tag[tb] : -1;   // any tag outside [0, N): no view template
      // _find: the nearest experience created with this view template within delta_pc cells (wrapped per axis);
      // (distance, id) order, so the lowest id wins a tie whatever the order of the walk
      int match = -1;
      double best = 0.0;
      if (vt >= 0 && cur >= 0) {
        for (int e = w.vt_head[vt * sB + b]; e >= 0; e = w.exp_next[e * sB + b]) {
          const long long c = w.exp_cell[e * sB + b];
          int dx = abs((int)(c / YTh) - px) % X, dy = abs((int)(c / Th % Y) - py) % Y, dt = abs((int)(c % Th) - pt) % Th;
          dx = min(dx, X - dx), dy = min(dy, Y - dy), dt = min(dt, Th - dt);
          const double d = sqrt((double)(dx * dx + dy * dy + dt * dt));
          if (d <= delta_pc && (match < 0 || d < best || (d == best && e < match))) match = e, best = d;
        }
      }
      if (match < 0) {
        // _create_linked: a new experience at the current one's position plus the odometry since, linked from it
        const int e = n_exp++;
        const size_t eb = e * sB + b;
        const double x = __dadd_rn(cur >= 0 ? cur_x : 0.0, rel_x), y = __dadd_rn(cur >= 0 ? cur_y : 0.0, rel_y);
        const double th = clip_rad_180(rel_th);
        w.exp_x[eb] = x, w.exp_y[eb] = y, w.exp_th[eb] = th;
        w.exp_cell[eb] = cell;
        w.exp_tag[eb] = vt;
        w.out_head[eb] = -1;
        if (vt >= 0) {
          w.exp_next[eb] = w.vt_head[vt * sB + b];
          w.vt_head[vt * sB + b] = e;
        } else {
          w.exp_next[eb] = -1;
        }
        if (cur >= 0) link(e);          // e is new: no link current -> e exists yet
        set_current(e, x, y, th);
      } else if (match != cur) {
        // a loop closure: link current -> match unless that pair is linked already, then move to match
        bool linked = false;
        for (int l = w.out_head[cur * sB + b]; l >= 0 && !linked; l = w.link_next[l * sB + b])
          linked = w.link_to[l * sB + b] == match;
        if (!linked) link(match);
        ++n_loop;
        const size_t mb = match * sB + b;
        set_current(match, w.exp_x[mb], w.exp_y[mb], w.exp_th[mb]);
      }
    }
    n_exp_out[tb] = n_exp;
    exp_id_out[tb] = cur;
    em_xy_out[2 * tb] = cur >= 0 ? cur_x : 0.0;
    em_xy_out[2 * tb + 1] = cur >= 0 ? cur_y : 0.0;
  }
  w.rel[b] = rel_x, w.rel[sB + b] = rel_y, w.rel[2 * sB + b] = rel_th;
  w.counts[b] = n_exp, w.counts[sB + b] = n_links, w.counts[2 * sB + b] = cur, w.counts[3 * sB + b] = n_loop;
}

}  // namespace

extern "C" size_t prs_em_work_bytes(int B, int T, int n_templates) {
  if (B < 1 || T < 0 || n_templates < 0) return 0;
  return EmLayout(B, T, n_templates).bytes;
}

static EmWork em_work(void* work, const EmLayout& L) {
  char* p = (char*)work;
  return EmWork{(double*)(p + L.exp_x),     (double*)(p + L.exp_y),       (double*)(p + L.exp_th),
                (double*)(p + L.link_d),    (double*)(p + L.link_heading), (double*)(p + L.link_facing),
                (double*)(p + L.rel),       (long long*)(p + L.exp_cell), (int*)(p + L.exp_tag),
                (int*)(p + L.exp_next),     (int*)(p + L.out_head),      (int*)(p + L.link_from),
                (int*)(p + L.link_to),      (int*)(p + L.link_next),     (int*)(p + L.vt_head),
                (int*)(p + L.counts)};
}

static int em_linked_launch(const char* who, int B, int T, int n_templates, const long long* argmax, const int* tag,
                            int R, const double* tw, const uint8_t* moved, const int* rec_of, int X, int Y, int Th,
                            double delta_pc, void* work, int* n_exp, int* exp_id, double* em_xy, void* stream) {
  PRS_REQUIRE(B >= 1 && T >= 0 && n_templates >= 0 && R >= 1, "%s: bad size B=%d T=%d n_templates=%d R=%d", who, B, T,
              n_templates, R);
  PRS_REQUIRE(X >= 1 && Y >= 1 && Th >= 1 && (long long)X * Y * Th <= (1LL << 30), "%s: bad grid %d x %d x %d", who, X, Y,
              Th);
  PRS_REQUIRE(work && (T == 0 || (argmax && tag && tw && moved && n_exp && exp_id && em_xy)), "%s: null argument", who);
  const EmWork w = em_work(work, EmLayout(B, T, n_templates));
  k_em_linked<false><<<(B + kEmBlock - 1) / kEmBlock, kEmBlock, 0, (cudaStream_t)stream>>>(
      B, T, n_templates, argmax, tag, tw, moved, X, Y, Th, delta_pc, w, n_exp, exp_id, em_xy, R, rec_of);
  PRS_CUDA(cudaGetLastError());
  return PRS_OK;
}

extern "C" int prs_em_linked_run(int B, int T, int n_templates, const long long* argmax, const int* tag, const double* tw,
                                 const uint8_t* moved, int X, int Y, int Th, double delta_pc, void* work, int* n_exp,
                                 int* exp_id, double* em_xy, void* stream) {
  return em_linked_launch("prs_em_linked_run", B, T, n_templates, argmax, tag, 1, tw, moved, nullptr, X, Y, Th, delta_pc,
                          work, n_exp, exp_id, em_xy, stream);
}

extern "C" int prs_em_linked_multi_run(int B, int T, int n_templates, const long long* argmax, const int* tag, int R,
                                       const double* tw, const uint8_t* moved, const int* rec_of, int X, int Y, int Th,
                                       double delta_pc, void* work, int* n_exp, int* exp_id, double* em_xy,
                                       void* stream) {
  PRS_REQUIRE(rec_of != nullptr || T == 0, "prs_em_linked_multi_run: null rec_of");
  return em_linked_launch("prs_em_linked_multi_run", B, T, n_templates, argmax, tag, R, tw, moved, rec_of, X, Y, Th,
                          delta_pc, work, n_exp, exp_id, em_xy, stream);
}

// ---------------------------------------------------------------------------------------------
// Sessions: a map workspace that lives across calls (prs_em_session_*, prs_em_linked_resume_run).  The layout is
// EmLayout(B, E, N) -- E rows of experiences and links, N template heads -- followed by one int32 error word.

extern "C" size_t prs_em_session_bytes(int B, int E, int N) {
  if (B < 1 || E < 0 || N < 0) return 0;
  return EmLayout(B, E, N).bytes + 256;
}

extern "C" int prs_em_session_init(int B, int E, int N, void* work, void* stream) {
  PRS_REQUIRE(B >= 1 && E >= 0 && N >= 0 && work, "prs_em_session_init: bad argument B=%d E=%d N=%d", B, E, N);
  const EmLayout L(B, E, N);
  char* p = (char*)work;
  const cudaStream_t st = (cudaStream_t)stream;
  const size_t sB = (size_t)B;
  PRS_CUDA(cudaMemsetAsync(p + L.vt_head, 0xFF, (size_t)N * sB * 4, st));          // -1: no experience yet
  PRS_CUDA(cudaMemsetAsync(p + L.rel, 0, 3 * sB * 8, st));
  PRS_CUDA(cudaMemsetAsync(p + L.counts, 0, 4 * sB * 4, st));
  PRS_CUDA(cudaMemsetAsync(p + L.counts + 2 * sB * 4, 0xFF, sB * 4, st));        // current experience: none
  PRS_CUDA(cudaMemsetAsync(p + L.bytes, 0, 4, st));                                // the error word
  return PRS_OK;
}

extern "C" int prs_em_session_grow(int B, int E0, int N0, int E1, int N1, const void* src, void* dst, void* stream) {
  PRS_REQUIRE(B >= 1 && E0 >= 0 && N0 >= 0 && E1 >= E0 && N1 >= N0 && src && dst && src != dst,
              "prs_em_session_grow: bad argument B=%d E %d -> %d N %d -> %d", B, E0, E1, N0, N1);
  const EmLayout A(B, E0, N0), Z(B, E1, N1);
  const char* s = (const char*)src;
  char* d = (char*)dst;
  const cudaStream_t st = (cudaStream_t)stream;
  const size_t sB = (size_t)B;
  // element [i][b] is at i * B + b in both layouts, so each array's old rows are one contiguous prefix
  const struct { size_t from, to, bytes; } arrays[] = {
      {A.exp_x, Z.exp_x, E0 * sB * 8},         {A.exp_y, Z.exp_y, E0 * sB * 8},
      {A.exp_th, Z.exp_th, E0 * sB * 8},       {A.link_d, Z.link_d, E0 * sB * 8},
      {A.link_heading, Z.link_heading, E0 * sB * 8}, {A.link_facing, Z.link_facing, E0 * sB * 8},
      {A.rel, Z.rel, 3 * sB * 8},              {A.exp_cell, Z.exp_cell, E0 * sB * 8},
      {A.exp_tag, Z.exp_tag, E0 * sB * 4},     {A.exp_next, Z.exp_next, E0 * sB * 4},
      {A.out_head, Z.out_head, E0 * sB * 4},   {A.link_from, Z.link_from, E0 * sB * 4},
      {A.link_to, Z.link_to, E0 * sB * 4},     {A.link_next, Z.link_next, E0 * sB * 4},
      {A.vt_head, Z.vt_head, N0 * sB * 4},     {A.counts, Z.counts, 4 * sB * 4},
      {A.bytes, Z.bytes, 4}};
  for (const auto& a : arrays)
    if (a.bytes) PRS_CUDA(cudaMemcpyAsync(d + a.to, s + a.from, a.bytes, cudaMemcpyDeviceToDevice, st));
  if (N1 > N0) PRS_CUDA(cudaMemsetAsync(d + Z.vt_head + N0 * sB * 4, 0xFF, (size_t)(N1 - N0) * sB * 4, st));
  return PRS_OK;
}

extern "C" int prs_em_linked_resume_run(int B, int T, int E, int N, const long long* argmax, const int* tag, int R,
                                        const double* tw, const uint8_t* moved, const int* rec_of, int X, int Y, int Th,
                                        double delta_pc, void* work, int* n_exp, int* exp_id, double* em_xy,
                                        void* stream) {
  PRS_REQUIRE(B >= 1 && T >= 0 && E >= 0 && N >= 0 && R >= 1 && (R == 1 || rec_of || T == 0),
              "prs_em_linked_resume_run: bad size B=%d T=%d E=%d N=%d R=%d (rec_of is needed for R > 1)", B, T, E, N, R);
  PRS_REQUIRE(X >= 1 && Y >= 1 && Th >= 1 && (long long)X * Y * Th <= (1LL << 30),
              "prs_em_linked_resume_run: bad grid %d x %d x %d", X, Y, Th);
  PRS_REQUIRE(work && (T == 0 || (argmax && tag && tw && moved && n_exp && exp_id && em_xy)),
              "prs_em_linked_resume_run: null argument");
  if (T == 0) return PRS_OK;
  const EmLayout L(B, E, N);
  k_em_linked<true><<<(B + kEmBlock - 1) / kEmBlock, kEmBlock, 0, (cudaStream_t)stream>>>(
      B, T, N, argmax, tag, tw, moved, X, Y, Th, delta_pc, em_work(work, L), n_exp, exp_id, em_xy, R, rec_of, E,
      (int*)((char*)work + L.bytes));
  PRS_CUDA(cudaGetLastError());
  return PRS_OK;
}

// ---------------------------------------------------------------------------------------------
// Agent copies inside a session workspace (prs_em_session_copy_agents, EnsembleSession.reassign): column d receives
// column s's experiences and links below its counts, all N rows of vt_head, rel and counts.  Rows at or past the counts
// are never read -- every list (vt_head, exp_next, out_head, link_next) points below them and a new experience or link
// writes its row whole -- so the destination's stale rows need no clearing.  The stage is a workspace of K columns with
// `rows` rows, the most experiences or links any gathered column holds.
namespace {

// array a of a workspace: 0-6 the experience arrays, 7-12 the link arrays, 13 vt_head, 14 rel, 15 counts
__device__ __forceinline__ char* em_array(const EmWork& w, int a, int& es) {
  es = 8;
  switch (a) {
    case 0: return (char*)w.exp_x;
    case 1: return (char*)w.exp_y;
    case 2: return (char*)w.exp_th;
    case 3: return (char*)w.exp_cell;
    case 4: es = 4; return (char*)w.exp_tag;
    case 5: es = 4; return (char*)w.exp_next;
    case 6: es = 4; return (char*)w.out_head;
    case 7: return (char*)w.link_d;
    case 8: return (char*)w.link_heading;
    case 9: return (char*)w.link_facing;
    case 10: es = 4; return (char*)w.link_from;
    case 11: es = 4; return (char*)w.link_to;
    case 12: es = 4; return (char*)w.link_next;
    case 13: es = 4; return (char*)w.vt_head;
    case 14: return (char*)w.rel;
    default: es = 4; return (char*)w.counts;
  }
}

// Pair p copies column pairs[p] of `src` (src_cols columns) into column pairs[n_pairs + p] of `dst` (dst_cols
// columns); thread (row j, pair p), pairs fastest, so a row's neighbouring destinations are written together.  Row j
// runs over 7 x `rows` experience rows, 6 x `rows` link rows, N vt_head rows, 3 rel and 4 count rows; rows at or past
// the source's counts return at once.  No pair's destination is another pair's source within one launch.
__global__ void __launch_bounds__(256)
    k_em_copy_cols(EmWork src, int src_cols, EmWork dst, int dst_cols, const int* __restrict__ pairs, int n_pairs,
                   int rows, int N) {
  const long long total = ((long long)13 * rows + N + 7) * n_pairs;
  for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
       idx += (long long)gridDim.x * blockDim.x) {
    const int p = (int)(idx % n_pairs);
    long long j = idx / n_pairs;
    const int s = pairs[p], d = pairs[n_pairs + p];
    int a, i;
    if (j < 13LL * rows) {
      a = (int)(j / rows), i = (int)(j % rows);
      if (i >= src.counts[(a < 7 ? 0 : 1) * (size_t)src_cols + s]) continue;
    } else if ((j -= 13LL * rows) < N) {
      a = 13, i = (int)j;
    } else if ((j -= N) < 3) {
      a = 14, i = (int)j;
    } else {
      a = 15, i = (int)j - 3;
    }
    int es;
    const char* from = em_array(src, a, es);
    char* to = em_array(dst, a, es);
    const size_t si = (size_t)i * src_cols + s, di = (size_t)i * dst_cols + d;
    if (es == 8)
      ((long long*)to)[di] = ((const long long*)from)[si];
    else
      ((int*)to)[di] = ((const int*)from)[si];
  }
}

}  // namespace

static int em_copy_plan(const char* who, int B, int E, int N, int n_moves, const int* dst, const int* src,
                        const int* n_rows, AgentMoves& mv, int& rows) {
  PRS_REQUIRE(B >= 1 && E >= 0 && N >= 0 && (n_moves == 0 || n_rows), "%s: bad argument B=%d E=%d N=%d", who, B, E, N);
  if (int rc = agent_moves(who, B, n_moves, dst, src, mv)) return rc;
  for (int m = 0; m < n_moves; ++m)
    PRS_REQUIRE(n_rows[src[m]] >= 0 && n_rows[src[m]] <= E, "%s: column %d uses %d rows, the workspace has %d", who,
                src[m], n_rows[src[m]], E);
  rows = 0;
  for (int r : mv.stage_rows) rows = std::max(rows, n_rows[r]);
  return PRS_OK;
}

static size_t em_copy_stage_offset(const AgentMoves& mv) {
  return (mv.table().size() * sizeof(int) + 255) / 256 * 256;
}

extern "C" size_t prs_em_session_copy_stage_bytes(int B, int E, int N, int n_moves, const int* dst, const int* src,
                                                  const int* n_rows) {
  AgentMoves mv;
  int rows = 0;
  if (em_copy_plan("prs_em_session_copy_stage_bytes", B, E, N, n_moves, dst, src, n_rows, mv, rows)) return 0;
  return em_copy_stage_offset(mv) + (mv.K() ? EmLayout(mv.K(), rows, N).bytes : 0);
}

extern "C" int prs_em_session_copy_agents(int B, int E, int N, void* work, int n_moves, const int* dst, const int* src,
                                          const int* n_rows, void* stage, size_t stage_bytes, void* stream) {
  AgentMoves mv;
  int rows = 0;
  if (int rc = em_copy_plan("prs_em_session_copy_agents", B, E, N, n_moves, dst, src, n_rows, mv, rows)) return rc;
  if (n_moves == 0) return PRS_OK;
  const std::vector<int> table = mv.table();
  const int K = mv.K();
  const size_t off = em_copy_stage_offset(mv);
  const size_t need = off + (K ? EmLayout(K, rows, N).bytes : 0);
  PRS_REQUIRE(work && stage && stage_bytes >= need, "prs_em_session_copy_agents: the stage has %zu bytes, the moves need %zu",
              stage_bytes, need);
  const cudaStream_t st = (cudaStream_t)stream;
  char* p = (char*)stage;
  PRS_CUDA(cudaMemcpyAsync(p, table.data(), table.size() * sizeof(int), cudaMemcpyHostToDevice, st));
  const EmWork w = em_work(work, EmLayout(B, E, N));
  const EmWork sw = em_work(p + off, EmLayout(K, rows, N));
  int direct_rows = 0;
  for (size_t m = 0; m < mv.direct.size() / 2; ++m) direct_rows = std::max(direct_rows, n_rows[mv.direct[m]]);
  auto launch = [&](const EmWork& from, int from_cols, const EmWork& to, int to_cols, const int* pairs, int n_pairs,
                    int bound) {
    if (n_pairs == 0) return cudaSuccess;
    const long long total = ((long long)13 * bound + N + 7) * n_pairs;
    const long long blocks = std::min((total + 255) / 256, 148LL * 16);
    k_em_copy_cols<<<(unsigned)blocks, 256, 0, st>>>(from, from_cols, to, to_cols, pairs, n_pairs, bound, N);
    return cudaGetLastError();
  };
  const int* d_table = (const int*)p;
  const int n_direct = (int)mv.direct.size() / 2, n_staged = (int)mv.staged.size() / 2;
  PRS_CUDA(launch(w, B, sw, K, d_table, K, rows));
  PRS_CUDA(launch(w, B, w, B, d_table + 2 * K, n_direct, direct_rows));
  PRS_CUDA(launch(sw, K, w, B, d_table + 2 * K + 2 * n_direct, n_staged, rows));
  return PRS_OK;
}

// ---------------------------------------------------------------------------------------------
// Columns carried between workspaces (prs_em_session_export_agents / prs_em_session_import_agents: a session's agents
// reassigned across devices).  The stage is a header, the export's and the import's pair tables, then a workspace of K
// columns with `rows` experience and link rows and the exporting workspace's N vt_head rows.  The header describes the
// columns, so the stage depends on no workspace.
namespace {

constexpr int kEmStageMagic = 0x50524d45;  // "EMRP"
constexpr int kEmHeaderInts = 8;
struct EmStageHeader {
  int magic, K, rows, N;
  long long bytes;
};

size_t em_transfer_offset(int K) { return ((kEmHeaderInts + 4 * (size_t)K) * sizeof(int) + 255) / 256 * 256; }

// vt_head rows [n0, N) of the listed columns set to -1: a column that received fewer template heads than its workspace
// holds keeps none of its own.
__global__ void __launch_bounds__(256) k_em_clear_heads(int* vt_head, int B, int n0, int N, const int* cols, int n_cols) {
  const long long total = (long long)(N - n0) * n_cols;
  for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
       idx += (long long)gridDim.x * blockDim.x) {
    const int c = (int)(idx % n_cols);
    const long long i = n0 + idx / n_cols;
    vt_head[i * B + cols[c]] = -1;
  }
}

}  // namespace

static int em_export_check(const char* who, int B, int E, int N, int n, const int* cols, const int* n_rows, int& rows) {
  PRS_REQUIRE(B >= 1 && E >= 0 && N >= 0 && n >= 0 && (n == 0 || (cols && n_rows)), "%s: bad argument B=%d E=%d N=%d",
              who, B, E, N);
  rows = 0;
  for (int k = 0; k < n; ++k) {
    PRS_REQUIRE(cols[k] >= 0 && cols[k] < B, "%s: column %d outside [0, %d)", who, cols[k], B);
    PRS_REQUIRE(n_rows[cols[k]] >= 0 && n_rows[cols[k]] <= E, "%s: column %d uses %d rows, the workspace has %d", who,
                cols[k], n_rows[cols[k]], E);
    rows = std::max(rows, n_rows[cols[k]]);
  }
  return PRS_OK;
}

extern "C" size_t prs_em_session_export_stage_bytes(int B, int E, int N, int n, const int* cols, const int* n_rows) {
  int rows = 0;
  if (em_export_check("prs_em_session_export_stage_bytes", B, E, N, n, cols, n_rows, rows) || n == 0) return 0;
  return em_transfer_offset(n) + EmLayout(n, rows, N).bytes;
}

extern "C" int prs_em_session_export_agents(int B, int E, int N, const void* work, int n, const int* cols,
                                            const int* n_rows, void* stage, size_t stage_bytes, void* stream) {
  int rows = 0;
  if (int rc = em_export_check("prs_em_session_export_agents", B, E, N, n, cols, n_rows, rows)) return rc;
  if (n == 0) return PRS_OK;
  const size_t off = em_transfer_offset(n), need = off + EmLayout(n, rows, N).bytes;
  PRS_REQUIRE(work && stage && stage_bytes >= need,
              "prs_em_session_export_agents: the stage has %zu bytes, the columns need %zu", stage_bytes, need);
  std::vector<int> table(kEmHeaderInts + 2 * (size_t)n, 0);
  const EmStageHeader h{kEmStageMagic, n, rows, N, (long long)need};
  memcpy(table.data(), &h, sizeof(h));
  for (int k = 0; k < n; ++k) {  // workspace column cols[k] -> stage column k (a column may be exported more than once)
    table[kEmHeaderInts + k] = cols[k];
    table[kEmHeaderInts + n + k] = k;
  }
  const cudaStream_t st = (cudaStream_t)stream;
  char* p = (char*)stage;
  PRS_CUDA(cudaMemcpyAsync(p, table.data(), table.size() * sizeof(int), cudaMemcpyHostToDevice, st));
  const long long total = ((long long)13 * rows + N + 7) * n;
  const long long blocks = std::min((total + 255) / 256, 148LL * 16);
  k_em_copy_cols<<<(unsigned)blocks, 256, 0, st>>>(em_work((void*)work, EmLayout(B, E, N)), B,
                                                   em_work(p + off, EmLayout(n, rows, N)), n,
                                                   (const int*)p + kEmHeaderInts, n, rows, N);
  PRS_CUDA(cudaGetLastError());
  return PRS_OK;
}

extern "C" int prs_em_session_import_agents(int B, int E, int N, void* work, int n, const int* cols, const void* stage,
                                            size_t stage_bytes, void* stream) {
  PRS_REQUIRE(B >= 1 && E >= 0 && N >= 0 && n >= 0 && (n == 0 || (cols && work && stage)),
              "prs_em_session_import_agents: bad argument B=%d E=%d N=%d", B, E, N);
  if (n == 0) return PRS_OK;
  std::vector<int> seen(B, 0);
  for (int k = 0; k < n; ++k) {
    PRS_REQUIRE(cols[k] >= 0 && cols[k] < B && !seen[cols[k]],
                "prs_em_session_import_agents: column %d outside [0, %d) or imported twice", cols[k], B);
    seen[cols[k]] = 1;
  }
  const cudaStream_t st = (cudaStream_t)stream;
  EmStageHeader h;
  PRS_REQUIRE(stage_bytes >= sizeof(h), "prs_em_session_import_agents: the stage has %zu bytes", stage_bytes);
  PRS_CUDA(cudaMemcpyAsync(&h, stage, sizeof(h), cudaMemcpyDeviceToHost, st));
  PRS_CUDA(cudaStreamSynchronize(st));
  PRS_REQUIRE(h.magic == kEmStageMagic && h.K == n && (size_t)h.bytes <= stage_bytes,
              "prs_em_session_import_agents: the stage does not hold %d exported columns", n);
  PRS_REQUIRE(h.rows >= 0 && h.rows <= E && h.N >= 0 && h.N <= N,
              "prs_em_session_import_agents: the stage holds %d rows and %d template heads, the workspace %d and %d",
              h.rows, h.N, E, N);
  std::vector<int> pairs(2 * (size_t)n);
  for (int k = 0; k < n; ++k) {  // stage column k -> workspace column cols[k]
    pairs[k] = k;
    pairs[n + k] = cols[k];
  }
  char* p = (char*)stage;
  int* d_pairs = (int*)p + kEmHeaderInts + 2 * n;
  PRS_CUDA(cudaMemcpyAsync(d_pairs, pairs.data(), pairs.size() * sizeof(int), cudaMemcpyHostToDevice, st));
  const EmWork w = em_work(work, EmLayout(B, E, N));
  const long long total = ((long long)13 * h.rows + h.N + 7) * n;
  const long long blocks = std::min((total + 255) / 256, 148LL * 16);
  k_em_copy_cols<<<(unsigned)blocks, 256, 0, st>>>(em_work(p + em_transfer_offset(n), EmLayout(n, h.rows, h.N)), n, w,
                                                   B, d_pairs, n, h.rows, h.N);
  PRS_CUDA(cudaGetLastError());
  if (N > h.N) {
    const long long cells = (long long)(N - h.N) * n;
    k_em_clear_heads<<<(unsigned)std::min((cells + 255) / 256, 148LL * 16), 256, 0, st>>>(w.vt_head, B, h.N, N,
                                                                                        d_pairs + n, n);
    PRS_CUDA(cudaGetLastError());
  }
  return PRS_OK;
}
