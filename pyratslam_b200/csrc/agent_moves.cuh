// Agent copies of an ensemble session (prs_ens_copy_agents, prs_em_session_copy_agents): move m makes agent row dst[m]
// an exact copy of row src[m] as it was before the call.  A source that some move overwrites is read before it is
// written: those rows alone are gathered into a stage first, and their moves read the stage.
#pragma once
#include <algorithm>
#include <vector>

#include "common.cuh"

struct AgentMoves {
  // pair lists, each [src][dst] of its count: gather (staged row -> stage row k), direct (row -> row) and staged
  // (stage row k -> row); direct and staged pairs are sorted by destination, so neighbouring threads write neighbours
  std::vector<int> gather, direct, staged;
  std::vector<int> stage_rows;  // the rows gathered, stage row k holds stage_rows[k]
  int K() const { return (int)stage_rows.size(); }
  // one host array of every list, in the order gather, direct, staged: what the device's pair table holds
  std::vector<int> table() const {
    std::vector<int> t(gather);
    t.insert(t.end(), direct.begin(), direct.end());
    t.insert(t.end(), staged.begin(), staged.end());
    return t;
  }
};

// Validates the moves (dst distinct, src != dst, both in [0, B)) and plans them; PRS_E_INVALID otherwise.
static inline int agent_moves(const char* who, int B, int n, const int* dst, const int* src, AgentMoves& mv) {
  PRS_REQUIRE(B >= 1 && n >= 0 && n <= B && (n == 0 || (dst && src)), "%s: bad argument B=%d n_moves=%d", who, B, n);
  std::vector<int> is_dst(B, 0), slot(B, -1);
  for (int m = 0; m < n; ++m) {
    PRS_REQUIRE(dst[m] >= 0 && dst[m] < B && src[m] >= 0 && src[m] < B && dst[m] != src[m],
                "%s: move %d (%d <- %d) outside [0, %d) or onto itself", who, m, dst[m], src[m], B);
    PRS_REQUIRE(!is_dst[dst[m]], "%s: row %d is the destination of two moves", who, dst[m]);
    is_dst[dst[m]] = 1;
  }
  std::vector<int> order(n);
  for (int m = 0; m < n; ++m) order[m] = m;
  std::sort(order.begin(), order.end(), [&](int a, int b) { return dst[a] < dst[b]; });
  std::vector<int> ds, dd, ss, sd;
  for (int m : order) {
    const int s = src[m];
    if (!is_dst[s]) {
      ds.push_back(s);
      dd.push_back(dst[m]);
      continue;
    }
    if (slot[s] < 0) {
      slot[s] = (int)mv.stage_rows.size();
      mv.stage_rows.push_back(s);
    }
    ss.push_back(slot[s]);
    sd.push_back(dst[m]);
  }
  mv.gather = mv.stage_rows;
  for (int k = 0; k < mv.K(); ++k) mv.gather.push_back(k);
  mv.direct = ds;
  mv.direct.insert(mv.direct.end(), dd.begin(), dd.end());
  mv.staged = ss;
  mv.staged.insert(mv.staged.end(), sd.begin(), sd.end());
  return PRS_OK;
}
