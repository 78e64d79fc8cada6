// mpc_prepare.cu -- observation parsing, collision prediction, latch, reference-speed regeneration.
// COMPILED WITH -fmad=false: everything that decides a flag or an index is FP64 with the same
// un-fused operation order as the numpy oracle, so flags and indices are bit-exact.
//
// Replaces (reference file:line):
//   Agent._parse_obs                      agents/base_agent.py:81-116
//   nearest reference row                 agents/pure_mpc.py:106-109, 566-570
//   predict_ego_future_positions          agents/pure_mpc.py:459-527
//   predict_future_positions              agents/pure_mpc.py:529-550
//   _check_collision (latch + detection)  agents/pure_mpc.py:552-676
//   update_reference_states               agents/pure_mpc.py:678-724
//
// Mapping: 8 (or 16) lanes per environment; lane m owns other-vehicle m.  The ego's predicted
// polyline (<= 31 FP64 points) is built cooperatively into shared memory, each lane then tests
// its vehicle's straight 31-point track against it.  Flags / earliest conflict row are combined
// with sub-warp shuffles, lane 0 of the group updates the latch and writes the solve descriptor.
#include "mpc_internal.h"

namespace mpcb {

constexpr int kPred = 30;            // PREDICTION_HORIZON, agents/pure_mpc.py:554
constexpr int kTimeThreshold = 30;   // TIME_THRESHOLD,     agents/pure_mpc.py:555
constexpr int kSafetyBuffer = 5;     // SAFETY_BUFFER_POINTS, agents/pure_mpc.py:681
constexpr int kMemorySteps = 10;     // collision_memory_steps, agents/pure_mpc.py:39
constexpr double kMaxAccPred = 3.5;  // Vehicle.max_acceleration, agents/utils.py:39
constexpr double kPi = 3.141592653589793;

__device__ __forceinline__ double norm2(double dx, double dy) { return sqrt(dx * dx + dy * dy); }
// argmin over distances compares the squared norms: sqrt is monotone, so the first minimum is the same index
// unless two squared distances differ by less than the sqrt's rounding (~1 ulp) -- and FP64 sqrt is a
// ~20-instruction software sequence that used to dominate this kernel
__device__ __forceinline__ double dist2(double dx, double dy) { return dx * dx + dy * dy; }
__device__ __forceinline__ double orient(double ax, double ay, double bx, double by, double cx, double cy) {
  return (bx - ax) * (cy - ay) - (by - ay) * (cx - ax);
}

#ifndef MPC_PREP_MIN_BLOCKS
#define MPC_PREP_MIN_BLOCKS 3      // 80 registers, 3 blocks per SM: 0.453 -> 0.431 ms per 65536 environments
#endif

template <int LPP>
__global__ void __launch_bounds__(256, MPC_PREP_MIN_BLOCKS)
k_prepare(const PrepareParams P) {
  constexpr int PPB = 256 / LPP;                      // environments per block
  __shared__ double s_ex[PPB][kPred + 1];
  __shared__ double s_ey[PPB][kPred + 1];
  // the handle's path table (built from its dt) is indexed per lane (ego_index + idx, strided argmin): staged once per
  // block into shared memory, where divergent reads cost nothing extra
  __shared__ double s_ref[kNRef][4];
  __shared__ double s_seg[kNRef - 1];
  for (int i = threadIdx.x; i < kNRef * 4; i += blockDim.x) (&s_ref[0][0])[i] = __ldg(P.ref + i);
  for (int i = threadIdx.x; i < kNRef - 1; i += blockDim.x) s_seg[i] = __ldg(P.seg + i);
  __syncthreads();
  const int g = threadIdx.x / LPP;                    // group inside the block
  const int l = threadIdx.x % LPP;                    // lane inside the group
  const int gi = blockIdx.x * PPB + g;
  const bool live = gi < P.count;
  const int b = P.first + gi;
  const int bb = P.first + (live ? gi : P.count - 1); // dead groups shadow the last env (no stores)
  const unsigned gmask = (LPP == 32) ? 0xffffffffu : (((1u << LPP) - 1u) << ((threadIdx.x % 32) / LPP * LPP));
  const float* ob = P.obs + (size_t)bb * P.V * 8;

  // ---- _parse_obs: ego row, number of present others --------------------------------------
  const double ex = ob[1], ey = ob[2];
  const double evx = ob[3], evy = ob[4];
  double eth = ob[5];
  // base_agent.py:156-170 wraps by repeated +-2pi.  Same arithmetic for any heading a simulator can
  // produce; the loop is bounded so that a non-finite or absurd heading cannot hang the kernel
  // (the reference would spin forever on inf).
  for (int it = 0; it < 64 && eth > kPi; ++it) eth -= 2 * kPi;
  for (int it = 0; it < 64 && eth < -kPi; ++it) eth += 2 * kPi;
  if (!(eth >= -kPi && eth <= kPi)) eth = 0.0;        // inf / nan / |heading| > 400 rad: defined value, status flags the solve
  const double ev = norm2(evx, evy);                  // agents/utils.py:36
  int present = 0;
  for (int r = 0; r < P.V; ++r) present += (ob[r * 8] == 1.0f) ? 1 : 0;
  int n_obs = present - 1;
  n_obs = n_obs < 0 ? 0 : (n_obs > P.M ? P.M : n_obs);

  // ---- nearest reference row: global argmin, first minimum wins ---------------------------
  double bd = 1e300;
  int bj = 0;
  for (int j = l; j < kNRef; j += LPP) {
    double d = dist2(ex - s_ref[j][0], ey - s_ref[j][1]);
    if (d < bd) { bd = d; bj = j; }
  }
#pragma unroll
  for (int o = LPP / 2; o > 0; o >>= 1) {
    double od = __shfl_xor_sync(gmask, bd, o, LPP);
    int oj = __shfl_xor_sync(gmask, bj, o, LPP);
    if (od < bd || (od == bd && oj < bj)) { bd = od; bj = oj; }
  }
  const int ego_index = bj;

  // ---- this lane's other vehicle ---------------------------------------------------------------
  const bool has_veh = l < n_obs;
  double ox = 0, oy = 0, incx = 0, incy = 0;
  float tinx = 0.f, tiny = 0.f;                        // float32 increments of the collision-check track
  if (has_veh) {
    const float* r = ob + (size_t)(l + 1) * 8;
    ox = r[1]; oy = r[2];
    const double sp = norm2((double)r[3], (double)r[4]);
    const double hd = r[5];                            // NOT wrapped, base_agent.py:112
    const double sd = sp * P.dt;                       // speed * dt * (cos, sin), base_agent.py:172-174
    const double ch = cos(hd), sh = sin(hd);
    incx = sd * ch;
    incy = sd * sh;
    // predict_future_positions (agents/pure_mpc.py:543-550) runs in float32 under the reference's pinned numpy 2.1.2:
    // float32 position + float32(speed) * float32(dt) * float32(cos, sin), see oracle predict_other_polyline
    const float sdf = (float)sp * (float)P.dt;
    tinx = sdf * (float)ch;
    tiny = sdf * (float)sh;
  }

  // ---- latch (agents/pure_mpc.py:558-563) -----------------------------------------------------
  int mem = 0, memo = -1;
  int is_col = 0;
  if (P.collision_check) {
    mem = P.latch.collision_memory[bb];
    memo = P.latch.memo_conflict[bb];
    is_col = P.latch.is_collide[bb];
    if (P.reset_mask && P.reset_mask[bb]) { mem = 0; memo = -1; is_col = 0; }
  }
  const bool latched = P.collision_check && mem > 0 && memo >= 0;
  int my_flag = 0, my_cidx = -1, my_deg = 0;
  double my_qx = 0.0, my_qy = 0.0;
  int cmin = -1;
  int stop_index = -1;
  bool aborted = false;

  if (P.collision_check && !latched) {
    // ---- ego polyline: arc length along the reference from ego_index -------------------------
    const int len = kNRef - ego_index;                 // points of reference_trajectory[start:]
    int n_valid = 0;                                   // how many of t = 1..30 produce a point
    if (len >= 2) {
      const double vref = s_ref[ego_index][2];
      // each lane owns the points t = 1 + l, 1 + l + LPP, ...; the speed ramp, the travelled distance and the
      // arc-length walk are all monotone in t, so they continue from the lane's previous point (same
      // sequential sums as the reference, evaluated once)
      double cur = ev, dist = 0.0;
      int t_done = 0;
      int idx = 0;
      double cum = 0.0, prev = 0.0;
      for (int t = 1 + l; t <= kPred; t += LPP) {
        for (int i = t_done + 1; i <= t; ++i) {
          if (cur < vref) { double nv = cur + kMaxAccPred * P.dt; cur = nv < vref ? nv : vref; }
          else cur = vref;
          dist += cur * P.dt;
        }
        t_done = t;
        // left searchsorted over cum[0..len-1], cum[0] = 0, cum[i] = cum[i-1] + seg[start+i-1]
        while (idx < len && cum < dist) {
          ++idx;
          if (idx >= len) break;
          prev = cum;
          cum = cum + s_seg[ego_index + idx - 1];
        }
        if (idx >= len) continue;                       // past the end of the path: no point
        double px, py;
        if (idx == 0) { px = s_ref[ego_index][0]; py = s_ref[ego_index][1]; }
        else {
          double alpha = (cum != prev) ? (dist - prev) / (cum - prev) : 1.0;
          alpha = alpha < 0.0 ? 0.0 : (alpha > 1.0 ? 1.0 : alpha);
          const double ax = s_ref[ego_index + idx - 1][0], ay = s_ref[ego_index + idx - 1][1];
          px = ax + alpha * (s_ref[ego_index + idx][0] - ax);
          py = ay + alpha * (s_ref[ego_index + idx][1] - ay);
        }
        s_ex[g][t] = px; s_ey[g][t] = py;
        ++n_valid;
      }
    }
    if (l == 0) { s_ex[g][0] = ex; s_ey[g][0] = ey; }
#pragma unroll
    for (int o = LPP / 2; o > 0; o >>= 1) n_valid += __shfl_xor_sync(gmask, n_valid, o, LPP);
    __syncwarp(gmask);
    const int ne = 1 + n_valid;                        // valid t form a prefix (dist is increasing)
    aborted = (len < 2) || (ne <= 1);                  // LineString of one point / 30 identical points
    if (aborted) my_deg = 1;

    if (!aborted && has_veh) {
      // ---- intersections of the ego polyline with this vehicle's straight 31-point track ------
      // The 31 track points are float32 running sums (see above).  They are NOT kept in an array: a per-thread array is
      // local memory, and 496 B x 0.5 M threads of it were 90 % of this kernel's DRAM writes (247 MB per launch,
      // profiles/r02_k_prepare_ncu_full.json vs 19 MB of outputs).  FP32 adds are free here (the kernel is FP64-bound),
      // so every use walks the sum again from the observed position.
      const float ox_f = (float)ox, oy_f = (float)oy;    // exact: the observation is float32
      float ex_f = ox_f, ey_f = oy_f;
#pragma unroll 1
      for (int t = 1; t <= kPred; ++t) { ex_f = ex_f + tinx; ey_f = ey_f + tiny; }
      const double O0x = ox, O0y = oy, OEx = ex_f, OEy = ey_f;   // track ends
      bool have = false;
      double qx = 0, qy = 0;
      const double tlen = fabs(OEx - O0x) + fabs(OEy - O0y);
      // nearest-time test of a candidate point (agents/pure_mpc.py:641-649), first minimum wins.  ONE call site (the
      // candidate loop below) and rolled loops: inlined at five sites with both 31-point loops unrolled this lambda made
      // the kernel 8 k instructions, four times the instruction cache.  The nearest TRACK point is searched in a window
      // of four indices around the projection of the candidate onto the track (the track is straight and its points are
      // float32 running sums, i.e. equally spaced to ~1e-5 of the spacing, so the squared distance is convex in the
      // index); slow tracks (spacing below a millimetre) take the full scan.
      const double trk2 = (OEx - O0x) * (OEx - O0x) + (OEy - O0y) * (OEy - O0y);
      auto time_test = [&](double cx, double cy) -> bool {
        int te = 0, to = 0;
        double bde = 1e300, bdo = 1e300;
#pragma unroll 1
        for (int t = 0; t < ne; ++t) { double d = dist2(s_ex[g][t] - cx, s_ey[g][t] - cy); if (d < bde) { bde = d; te = t; } }
        int t_lo = 0, t_hi = kPred;
        if (trk2 > 1e-3) {                                 // 30 steps of more than a millimetre
          const double proj = ((cx - O0x) * (OEx - O0x) + (cy - O0y) * (OEy - O0y)) / trk2 * kPred;
          const int tc = proj < 0.0 ? 0 : (proj > (double)kPred ? kPred : (int)proj);
          t_lo = tc - 1 < 0 ? 0 : tc - 1;
          t_hi = tc + 2 > kPred ? kPred : tc + 2;
        }
        float wx = ox_f, wy = oy_f;
#pragma unroll 1
        for (int t = 0; t < t_lo; ++t) { wx = wx + tinx; wy = wy + tiny; }
#pragma unroll 1
        for (int t = t_lo; t <= t_hi; ++t) {
          double d = dist2((double)wx - cx, (double)wy - cy);
          if (d < bdo) { bdo = d; to = t; }
          wx = wx + tinx; wy = wy + tiny;
        }
        int dtm = te - to; dtm = dtm < 0 ? -dtm : dtm;
        return dtm < kTimeThreshold;
      };
      // collinear overlaps (the same-lane case: the lane centre x = 2.0 is the path's own x): GEOS returns a LineString
      // per connected overlap and the reference takes its middle coordinate (agents/pure_mpc.py:618-622, :628-633)
      constexpr int kMaxPieces = 4, kMaxPts = 8;
      double plo[kMaxPieces], phi[kMaxPieces];
      int psg[kMaxPieces], npieces = 0;
      double ptx[kMaxPts], pty[kMaxPts];
      int npts = 0;
      const bool axx = fabs(OEx - O0x) >= fabs(OEy - O0y);   // scalar coordinate along the track: dominant axis
      const double o_a = axx ? O0x : O0y, o_b = axx ? OEx : OEy;
      const double olo = fmin(o_a, o_b), ohi = fmax(o_a, o_b);
      auto add_point = [&](double cx, double cy) {        // every intersection point; tested after the scan
        if (npts < kMaxPts) { ptx[npts] = cx; pty[npts] = cy; ++npts; } else my_deg = 1;
      };
      for (int i = 0; i + 1 < ne; ++i) {
        const double p1x = s_ex[g][i], p1y = s_ey[g][i], p2x = s_ex[g][i + 1], p2y = s_ey[g][i + 1];
        // orientation of track ends about the ego segment is affine in t: locate the sign change
        const double e0 = orient(p1x, p1y, p2x, p2y, O0x, O0y);
        const double e30 = orient(p1x, p1y, p2x, p2y, OEx, OEy);
        const double sc = (fabs(p2x - p1x) + fabs(p2y - p1y) + 1e-300) * (tlen + 1e-300);
        const double tol = 1e-7 * sc;
        if ((e0 > tol && e30 > tol) || (e0 < -tol && e30 < -tol)) continue;
        // ... and the ego segment must straddle the track's line (most segments whose LINE the track crosses are
        // nowhere near the track itself): same conservative band, the exact predicate below decides the rest
        const double f1 = orient(O0x, O0y, OEx, OEy, p1x, p1y);
        const double f2 = orient(O0x, O0y, OEx, OEy, p2x, p2y);
        if ((f1 > tol && f2 > tol) || (f1 < -tol && f2 < -tol)) continue;
        if (e0 == 0.0 && e30 == 0.0 && ohi > olo) {
          // candidate for "this ego segment lies on the track's line": the oracle asks for all four orientations of
          // every segment pair to be exactly zero
          bool allzero = true;
          float ax_ = ox_f, ay_ = oy_f;
#pragma unroll 1
          for (int j = 0; j < kPred && allzero; ++j) {
            const float bx_ = ax_ + tinx, by_ = ay_ + tiny;
            const double u1x = ax_, u1y = ay_, u2x = bx_, u2y = by_;
            allzero = orient(u1x, u1y, u2x, u2y, p1x, p1y) == 0.0 && orient(u1x, u1y, u2x, u2y, p2x, p2y) == 0.0 &&
                      orient(p1x, p1y, p2x, p2y, u1x, u1y) == 0.0 && orient(p1x, p1y, p2x, p2y, u2x, u2y) == 0.0;
            ax_ = bx_; ay_ = by_;
          }
          const double a = axx ? p1x : p1y, b = axx ? p2x : p2y;
          if (allzero && a != b) {
            const double lo = fmax(fmin(a, b), olo), hi = fmin(fmax(a, b), ohi);
            if (hi > lo) {
              if (npieces > 0 && (plo[npieces - 1] == hi || phi[npieces - 1] == lo)) {
                plo[npieces - 1] = fmin(plo[npieces - 1], lo); phi[npieces - 1] = fmax(phi[npieces - 1], hi);
              } else if (npieces < kMaxPieces) {
                plo[npieces] = lo; phi[npieces] = hi; psg[npieces] = b > a ? 1 : -1; ++npieces;
              } else {
                my_deg = 1;
              }
            }
            continue;                                     // handled as an overlap
          }
        }
        int jlo = 0, jhi = kPred - 1;
        const double de = e30 - e0;
        if (fabs(de) > tol) {
          double js = -e0 / de * kPred;
          int jc = (int)floor(js);
          jlo = jc - 1 < 0 ? 0 : jc - 1;
          jhi = jc + 1 > kPred - 1 ? kPred - 1 : jc + 1;
          if (jlo > kPred - 1 || jhi < 0) continue;
        }
        float wx = ox_f, wy = oy_f;                        // walk to the first point of the window
#pragma unroll 1
        for (int t = 0; t < jlo; ++t) { wx = wx + tinx; wy = wy + tiny; }
#pragma unroll 1
        for (int j = jlo; j <= jhi; ++j) {
          const float nx_ = wx + tinx, ny_ = wy + tiny;
          const double q1x = wx, q1y = wy, q2x = nx_, q2y = ny_;
          wx = nx_; wy = ny_;
          const double d1 = orient(q1x, q1y, q2x, q2y, p1x, p1y);
          const double d2 = orient(q1x, q1y, q2x, q2y, p2x, p2y);
          const double d3 = orient(p1x, p1y, p2x, p2y, q1x, q1y);
          const double d4 = orient(p1x, p1y, p2x, p2y, q2x, q2y);
          const double s2 = (fabs(p2x - p1x) + fabs(p2y - p1y) + 1e-300) * (fabs(q2x - q1x) + fabs(q2y - q1y) + 1e-300) + 1e-300;
          const double eps = 1e-9 * s2;
          const bool proper = (d1 * d2 < 0) && (d3 * d4 < 0);
          if (!proper) {
            if (fabs(d1) <= eps || fabs(d2) <= eps || fabs(d3) <= eps || fabs(d4) <= eps) {
              const bool box = fmin(p1x, p2x) <= fmax(q1x, q2x) + 1e-9 && fmin(q1x, q2x) <= fmax(p1x, p2x) + 1e-9 &&
                               fmin(p1y, p2y) <= fmax(q1y, q2y) + 1e-9 && fmin(q1y, q2y) <= fmax(p1y, p2y) + 1e-9;
              if (box) {
                // exact touches (orientation exactly zero, the endpoint inside the other segment's box) are genuine
                // intersection points; near zero but not zero: robust and plain predicates may differ
                auto on_seg = [](double px, double py, double sx, double sy, double ex_, double ey_) {
                  return fmin(sx, ex_) <= px && px <= fmax(sx, ex_) && fmin(sy, ey_) <= py && py <= fmax(sy, ey_);
                };
                if (d1 == 0.0 && on_seg(p1x, p1y, q1x, q1y, q2x, q2y)) add_point(p1x, p1y);
                if (d2 == 0.0 && on_seg(p2x, p2y, q1x, q1y, q2x, q2y)) add_point(p2x, p2y);
                if (d3 == 0.0 && on_seg(q1x, q1y, p1x, p1y, p2x, p2y)) add_point(q1x, q1y);
                if (d4 == 0.0 && on_seg(q2x, q2y, p1x, p1y, p2x, p2y)) add_point(q2x, q2y);
                if ((d1 != 0.0 && fabs(d1) <= eps) || (d2 != 0.0 && fabs(d2) <= eps) || (d3 != 0.0 && fabs(d3) <= eps) || (d4 != 0.0 && fabs(d4) <= eps)) my_deg = 1;
              }
            }
            continue;
          }
          const double tt = d1 / (d1 - d2);
          add_point(p1x + tt * (p2x - p1x), p1y + tt * (p2y - p1y));
        }
      }
      // ---- candidates in the reference's visiting order, then ONE nearest-time loop --------------------------------
      bool ordered = false;                               // overlaps: first passing candidate wins; points: lexicographic minimum
      if (npieces > 0) {
        // isolated points that are not part of an overlap make the result a GeometryCollection, for which the
        // reference's dispatch has no branch: no candidate at all
        bool mixed = false;
        for (int k = 0; k < npts; ++k) {
          const double c = axx ? ptx[k] : pty[k];
          bool inside = false;
          for (int q = 0; q < npieces; ++q) inside = inside || (plo[q] <= c && c <= phi[q]);
          if (!inside || orient(O0x, O0y, OEx, OEy, ptx[k], pty[k]) != 0.0) mixed = true;
        }
        npts = 0;
        ordered = true;
#pragma unroll 1
        for (int q = 0; q < npieces && !mixed; ++q) {
          // merged vertices of both polylines inside the overlap, ordered along the ego polyline (stable: ego vertices
          // first), one per position; the reference takes coords[len // 2]
          double key[2 * (kPred + 1)], vx[2 * (kPred + 1)], vy[2 * (kPred + 1)];
          int n = 0;
          auto insert = [&](double px, double py) {
            const double c = axx ? px : py;
            if (!(plo[q] <= c && c <= phi[q])) return;
            const double kk = psg[q] * c;
            int pos = n;
            while (pos > 0 && key[pos - 1] > kk) --pos;   // after the entries with an equal key (stable)
            for (int m = n; m > pos; --m) { key[m] = key[m - 1]; vx[m] = vx[m - 1]; vy[m] = vy[m - 1]; }
            key[pos] = kk; vx[pos] = px; vy[pos] = py; ++n;
          };
#pragma unroll 1
          for (int t = 0; t < ne; ++t)
            if (orient(O0x, O0y, OEx, OEy, s_ex[g][t], s_ey[g][t]) == 0.0) insert(s_ex[g][t], s_ey[g][t]);
          float wx = ox_f, wy = oy_f;
#pragma unroll 1
          for (int t = 0; t <= kPred; ++t) { insert((double)wx, (double)wy); wx = wx + tinx; wy = wy + tiny; }
          int m = 0;                                      // drop repeated positions (keep the first)
          for (int k = 0; k < n; ++k)
            if (k == 0 || key[k] != key[m - 1]) { key[m] = key[k]; vx[m] = vx[k]; vy[m] = vy[k]; ++m; }
          if (m > 0 && npts < kMaxPts) { ptx[npts] = vx[m / 2]; pty[npts] = vy[m / 2]; ++npts; }
        }
      }
#pragma unroll 1
      for (int k = 0; k < npts; ++k) {
        if (ordered && have) break;
        const double cx = ptx[k], cy = pty[k];
        if (!time_test(cx, cy)) continue;
        // isolated points are visited in lexicographic (x, y) order: keep the smallest passing one
        if (!have || (!ordered && (cx < qx || (cx == qx && cy < qy)))) { have = true; qx = cx; qy = cy; }
      }
      if (have) {
        my_flag = 1;
        my_qx = qx; my_qy = qy;
        double bdr = 1e300;
#pragma unroll 1
        for (int j = 0; j < kNRef; ++j) { double d = dist2(s_ref[j][0] - qx, s_ref[j][1] - qy); if (d < bdr) { bdr = d; my_cidx = j; } }
      }
    }
  }

  // ---- combine over the group --------------------------------------------------------------------
  int any_flag = my_flag, any_deg = my_deg;
  int min_c = my_flag ? my_cidx : 1 << 30;
#pragma unroll
  for (int o = LPP / 2; o > 0; o >>= 1) {
    any_flag |= __shfl_xor_sync(gmask, any_flag, o, LPP);
    any_deg |= __shfl_xor_sync(gmask, any_deg, o, LPP);
    int oc = __shfl_xor_sync(gmask, min_c, o, LPP);
    min_c = oc < min_c ? oc : min_c;
  }

  if (P.collision_check) {
    if (latched) {                                      // pure_mpc.py:558-563
      is_col = 1; mem -= 1; cmin = memo;
    } else if (!aborted) {                              // pure_mpc.py:660-676
      is_col = any_flag;
      if (is_col) { mem = kMemorySteps; memo = min_c; cmin = min_c; }
      else if (mem > 0) { mem -= 1; is_col = 1; cmin = -1; }
      else { memo = -1; }
    }                                                    // aborted: early return, state left as it was
  } else {
    is_col = 0;
  }

  // ---- outputs.  The SoA planes are strided by the batch, so a group writing its own environment's element would touch
  // 4 (16) bytes per plane per warp: the values of the block's PPB environments are staged in shared memory and each
  // plane is then written as one run of PPB consecutive elements (full 32-byte sectors).
  constexpr int kFloatRows = 10, kIntRows = 6;          // s0 x4, w x3, vr_a, vr_slope, vr_b | ego_index, vr_n, n_obs, mem, memo, stop
  __shared__ float s_oobs[MPC_MAX_OBSTACLES * 4][PPB];
  __shared__ float s_of[kFloatRows][PPB];
  __shared__ int s_oi[kIntRows][PPB];
  __shared__ uint8_t s_ou[2][PPB];                      // is_collide, degenerate
  // ---- per-vehicle outputs ([B][M] layouts: a warp already writes consecutive elements) -------------
  if (live && l < P.M) {
    if (P.col.agent_collide) P.col.agent_collide[(size_t)b * P.M + l] = (uint8_t)((P.collision_check && !latched && !aborted) ? my_flag : 0);
    if (P.col.conflict_index) P.col.conflict_index[(size_t)b * P.M + l] = (P.collision_check && !latched && !aborted && my_flag) ? my_cidx : -1;
    if (P.col.conflict_point) {
      const bool hit = P.collision_check && !latched && !aborted && my_flag;
      P.col.conflict_point[((size_t)b * P.M + l) * 2] = hit ? (float)my_qx : nanf("");
      P.col.conflict_point[((size_t)b * P.M + l) * 2 + 1] = hit ? (float)my_qy : nanf("");
    }
  }
  if (l < P.M) {
    s_oobs[l * 4 + 0][g] = has_veh ? (float)ox : 0.f;
    s_oobs[l * 4 + 1][g] = has_veh ? (float)oy : 0.f;
    s_oobs[l * 4 + 2][g] = has_veh ? (float)incx : 0.f;
    s_oobs[l * 4 + 3][g] = has_veh ? (float)incy : 0.f;
  }
  if (LPP < MPC_MAX_OBSTACLES && l == 0) {
    for (int m = LPP; m < P.M; ++m)                     // more vehicles than lanes: not reachable with LPP >= M
      for (int c = 0; c < 4; ++c) s_oobs[m * 4 + c][g] = 0.f;
  }
  if (l == 0) {
    // ---- weights, reference-speed profile (update_reference_states, pure_mpc.py:678-724) -----------
    float w_s = P.w_speed, w_c = P.w_control, w_d = P.w_diff;
    if (P.weights) { w_s = P.weights[(size_t)bb * 3]; w_c = P.weights[(size_t)bb * 3 + 1]; w_d = P.weights[(size_t)bb * 3 + 2]; }
    if (is_col) w_s = 100.f;                              // pure_mpc.py:143-147
    float vr_a = 0.f, vr_slope = 0.f, vr_b = (float)s_ref[0][2];
    int vr_n = 0;
    bool override_v = false;
    if (P.ref_speed) {
      const float rs = P.ref_speed[bb];
      if (rs == rs) { override_v = true; vr_b = fminf(fmaxf(rs, 0.f), 30.f); }   // np.clip(., 0, 30), takes precedence
    }
    if (!override_v && is_col && cmin >= 0) {
      int stop = cmin - kSafetyBuffer;
      stop = stop > ego_index + 1 ? stop : ego_index + 1;
      stop = stop < kNRef - 1 ? stop : kNRef - 1;
      const int n = stop - ego_index;
      if (n > 0) {
        vr_n = n; vr_a = (float)ev; vr_b = 0.f;
        vr_slope = n > 1 ? (float)(-ev / (double)(n - 1)) : 0.f;   // np.linspace(v, 0, n)
        stop_index = stop;
      }
    }
    s_of[0][g] = (float)ex; s_of[1][g] = (float)ey; s_of[2][g] = (float)eth; s_of[3][g] = (float)ev;
    s_of[4][g] = w_s; s_of[5][g] = w_c; s_of[6][g] = w_d;
    s_of[7][g] = vr_a; s_of[8][g] = vr_slope; s_of[9][g] = vr_b;
    s_oi[0][g] = ego_index; s_oi[1][g] = vr_n; s_oi[2][g] = n_obs; s_oi[3][g] = mem; s_oi[4][g] = memo; s_oi[5][g] = stop_index;
    s_ou[0][g] = (uint8_t)is_col; s_ou[1][g] = (uint8_t)any_deg;
  }
  __syncthreads();
  const int nb = P.count - (int)blockIdx.x * PPB < PPB ? P.count - (int)blockIdx.x * PPB : PPB;   // live environments of this block
  const size_t b0 = (size_t)P.first + (size_t)blockIdx.x * PPB;
  const size_t SB = (size_t)P.B;
  for (int q = threadIdx.x; q < P.M * 4 * PPB; q += blockDim.x) {
    const int plane = q / PPB, e = q % PPB;
    if (e < nb) P.ws.obstacles[(size_t)plane * SB + b0 + e] = s_oobs[plane][e];
  }
  for (int q = threadIdx.x; q < kFloatRows * PPB; q += blockDim.x) {
    const int row = q / PPB, e = q % PPB;
    if (e >= nb) continue;
    const float v = s_of[row][e];
    float* dst = row < 4 ? P.ws.s0 + (size_t)row * SB : row == 4 ? P.ws.w_speed : row == 5 ? P.ws.w_control : row == 6 ? P.ws.w_diff
               : row == 7 ? P.ws.vr_a : row == 8 ? P.ws.vr_slope : P.ws.vr_b;
    dst[b0 + e] = v;
  }
  for (int q = threadIdx.x; q < kIntRows * PPB; q += blockDim.x) {
    const int row = q / PPB, e = q % PPB;
    if (e >= nb) continue;
    const int v = s_oi[row][e];
    int32_t* dst = row == 0 ? P.ws.ego_index : row == 1 ? P.ws.vr_n : row == 2 ? P.ws.n_obs
                 : row == 3 ? (P.collision_check ? P.latch.collision_memory : nullptr) : row == 4 ? (P.collision_check ? P.latch.memo_conflict : nullptr)
                 : P.col.stop_index;
    if (dst) dst[b0 + e] = v;
    if (row == 0 && P.col.ego_index) P.col.ego_index[b0 + e] = v;
  }
  for (int q = threadIdx.x; q < 2 * PPB; q += blockDim.x) {
    const int row = q / PPB, e = q % PPB;
    if (e >= nb) continue;
    const uint8_t v = s_ou[row][e];
    if (row == 0) {
      P.ws.is_collide[b0 + e] = v;
      if (P.collision_check) P.latch.is_collide[b0 + e] = v;
      if (P.col.is_collide) P.col.is_collide[b0 + e] = v;
    } else if (P.col.degenerate) {
      P.col.degenerate[b0 + e] = v;
    }
  }
}

cudaError_t launch_prepare(const PrepareParams& p, cudaStream_t stream) {
  if (p.B <= 0 || p.count <= 0) return cudaSuccess;
  if (p.M <= 8) {
    const int ppb = 256 / 8;
    k_prepare<8><<<(p.count + ppb - 1) / ppb, 256, 0, stream>>>(p);
  } else {
    const int ppb = 256 / 16;
    k_prepare<16><<<(p.count + ppb - 1) / ppb, 256, 0, stream>>>(p);
  }
  return cudaGetLastError();
}

}  // namespace mpcb
