// Which times the solution of one forward call holds (src/layers/neural_ode.jl:102-116), where each of them goes, and
// t1 of the local regulariser.  Pure host logic: libLRNDE.so builds the plan once per forward call and keeps it in the
// tape; liblrnde_hostcheck.so re-exports it so that the CPU suite can compare it with the oracle.
#pragma once
#include <algorithm>
#include <cmath>
#include <vector>

#include "../../include/lrnde.h"

struct SavePlan {
  std::vector<float> times;  // the full saved solution (t1 included where :unbiased appends it)
  std::vector<int> out;      // output block of each time, -1 = dropped (_CorrectedDESolution, last_only)
  float t1 = 0.0f;           // start of the regulariser step
  int nout = 0;              // output blocks the call returns

  // the output blocks whose time, clamped to t_end (the last accepted time), equals t
  std::vector<int> blocks_at(float t, float t_end) const {
    std::vector<int> r;
    for (size_t i = 0; i < times.size(); ++i)
      if (out[i] >= 0 && std::min(times[i], t_end) == t) r.push_back(out[i]);
    return r;
  }
  // the saved times, clamped to t_end, strictly inside (t_start, t_end): descending and unique
  std::vector<float> interior_stops(float t_start, float t_end) const {
    std::vector<float> r;
    for (float s : times) {
      const float sc = std::min(s, t_end);
      if (sc > t_start && sc < t_end && std::find(r.begin(), r.end(), sc) == r.end()) r.push_back(sc);
    }
    std::sort(r.begin(), r.end(), [](float a, float b) { return a > b; });
    return r;
  }
};

// fts: the accepted times of the solve, fts[0] = t0
static inline SavePlan lr_save_plan(const lrnde_opts& o, const std::vector<float>& fts) {
  SavePlan p;
  std::vector<float>& times = p.times;
  std::vector<int>& out = p.out;
  p.t1 = o.t1;
  const int mode = o.reg_mode;
  if (o.nsave > 0) {
    for (int i = 0; i < o.nsave; ++i) times.push_back(o.saveat[i]);
    if (o.save_start && std::find(times.begin(), times.end(), o.t0) == times.end()) times.insert(times.begin(), o.t0);
    for (size_t i = 0; i < times.size(); ++i) out.push_back((int)i);
    if (mode == LRNDE_REG_UNBIASED) { times.push_back(p.t1); out.push_back(-1); }
  } else if (o.nsave == 0 && mode != LRNDE_REG_BIASED) {
    // solve(...; saveat = [t1, t2] / [t2], save_start) : the reference splats save_start into solve (neural_ode.jl:51)
    if (o.save_start) { times.push_back(o.t0); out.push_back(0); }
    if (mode == LRNDE_REG_UNBIASED) { times.push_back(p.t1); out.push_back((int)out.size()); }
    times.push_back(o.t2);
    out.push_back((int)out.size());
  } else {  // every accepted step (saveat = [] of the :biased path, or nsave == -1)
    const int start = o.save_start ? 0 : 1;
    for (int n = start; n < (int)fts.size(); ++n) { times.push_back(fts[n]); out.push_back(n - start); }
  }
  if (mode == LRNDE_REG_BIASED) {  // t1 = rand(rng, sol.t[1:end-1])   (neural_ode.jl:92)
    const int ncand = (int)times.size() - 1;
    if (ncand > 0) {
      const int idx = std::min(ncand - 1, std::max(0, (int)std::floor(o.u01 * (float)ncand)));
      p.t1 = times[idx];
    } else p.t1 = o.t0;
  }
  if (o.last_only) {   // fused diffeqsol_to_array (src/utils.jl:37): only sol.u[end] leaves the library
    int last = -1, mx = -1;
    for (size_t i = 0; i < out.size(); ++i)
      if (out[i] > mx) { mx = out[i]; last = (int)i; }
    for (size_t i = 0; i < out.size(); ++i) out[i] = ((int)i == last) ? 0 : -1;
  }
  for (int v : out) p.nout = std::max(p.nout, v + 1);
  return p;
}
