// ref_path.h -- the reference's hard-coded 85-row left-turn path (agents/base_agent.py:118-154), built on the host from
// the policy step dt.  Shared by the library (mpc_create builds one table per handle) and the test-only host harness
// (tests/hostsim), so that the CPU tests check the very function the library uses.
//
// The rows are accumulated with v * dt steps in the reference's operation order, in FP64, so the table is bit-identical
// to the numpy oracle's reference_states(dt).  The products are stored through volatile doubles: no fused multiply-add
// may change the rounding, whatever the host compiler's contraction setting.
#pragma once
#include <math.h>

#include "mpc_core.cuh"

namespace mpcb {

static_assert(40 + 20 + 25 == kNRef, "the path has 85 rows");

// out[j] = (x, y, v, heading) of row j
inline void build_reference_path(double dt, double (*out)[4]) {
  const double pi = 3.141592653589793;
  double x = 2.0, y = 50.0, h = -pi / 2;
  const double v = 10.0;
  int j = 0;
  for (int i = 0; i < 40; ++i, ++j) {                    // straight, heading -pi/2: x += 0, y += v * dt * sin(h)
    volatile double d = v * dt;
    volatile double dy = d * sin(h);
    y = y + dy;
    out[j][0] = x; out[j][1] = y; out[j][2] = v; out[j][3] = h;
  }
  const double step = (pi / 2) / 20;
  for (int i = 0; i < 20; ++i, ++j) {                    // turn: heading decremented BEFORE each move
    h = h - step;
    volatile double d = v * dt;
    volatile double dx = d * cos(h);
    volatile double dy = d * sin(h);
    x = x + dx;
    y = y + dy;
    out[j][0] = x; out[j][1] = y; out[j][2] = v; out[j][3] = h;
  }
  for (int i = 0; i < 25; ++i, ++j) {                    // straight, heading -pi: x += v * dt * cos(h), y += 0
    volatile double d = v * dt;
    volatile double dx = d * cos(h);
    x = x + dx;
    out[j][0] = x; out[j][1] = y; out[j][2] = v; out[j][3] = h;
  }
}

}  // namespace mpcb
