// nexoclom_b200 -- host-side preparation of a line-of-sight call (K5): the ladder of KD-ball
// centres, the constants of the membership test and the per-line ball count.  Host code only
// (no CUDA headers), shared by nx_api.cu and the test-only host build of the membership test.
// Reference: data_simulation/compute_iteration.py:151-222.
#pragma once
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <string>
#include <vector>

#include "nx_image.cuh"

namespace nx {

struct LosConsts {
  double sin_dphi;
  double cos_margin2;     // (cos(dphi) (1 - 1e-9))^2   conservative reject, exact-order path
  double cos_loose2;      // (cos(dphi) (1 - 1e-6))^2   conservative reject, FMA path
  double cos_accept2;     // (cos(dphi) (1 + 1e-9))^2   sure accept, no acos needed
  int cover;              // 1: in-cone points between the first and last ball centre are in a ball
  double inv_log_ratio;   // 1 / log(1 + sin dphi)
  double log_t0;          // log(sin dphi)
  int kwin;
  int nladder;
};

// Most ladder entries one call may use.  The reference builds t_0 = sin(dphi),
// t_{k+1} = t_k (1 + sin dphi) up to the longest boresight distance dd, about
// ln(dd / sin dphi) / log1p(sin dphi) entries: 432 for 1 deg at 30 R_p, 2.2e6 for 2" at
// 1.5e4 R_p, 4.8e6 for 1" at 5e4 R_p.  2^25 entries are 512 MB of ladder + squared ball radii
// on the device.  A call that needs more fails; it never truncates the ladder (packets past a
// truncated ladder would silently not be members).
#define NX_LOS_LADDER_MAX (1 << 25)

// "" if dphi is a usable cone half-angle [rad]: finite, > 0 and < pi/2 (the cone tests compare
// squared cosines, the balls need sin(2 dphi) > 0).
inline std::string los_dphi_error(double dphi) {
  if (dphi > 0.0 && dphi < NX_PI / 2) return std::string();
  char buf[160];
  std::snprintf(buf, sizeof(buf), "dphi = %.17g rad: the cone half-angle must be finite, > 0 and < pi/2",
                dphi);
  return buf;
}

// Constants of a line-of-sight call and the ladder of KD-ball centres (compute_iteration.py:
// 151-170), given the longest boresight distance `ddmax` to the outer edge.  Returns "" or the
// reason the call cannot run (bad dphi, a ladder above NX_LOS_LADDER_MAX entries).
inline std::string los_constants(const LosParams& lp, double ddmax, std::vector<double>& ladder,
                                 std::vector<double>& wid2, LosConsts& lc) {
  std::string err = los_dphi_error(lp.dphi);
  if (!err.empty()) return err;
  const double s = std::sin(lp.dphi);
  const double s2 = std::sin(lp.dphi * 2);
  ladder.clear();
  ladder.push_back(s);
  while (ladder.back() < ddmax) {
    if (ladder.size() >= (size_t)NX_LOS_LADDER_MAX) {
      char buf[256];
      std::snprintf(buf, sizeof(buf),
                    "dphi = %.6g rad (%.4g arcsec) out to %.6g R_p needs about %.4g KD-ball ladder "
                    "entries, more than the %d one call may use",
                    lp.dphi, lp.dphi * (180.0 / NX_PI) * 3600.0, ddmax,
                    std::log(ddmax / s) / std::log1p(s) + 1.0, NX_LOS_LADDER_MAX);
      ladder.clear();
      return buf;
    }
    const double t = ladder.back();
    ladder.push_back(t + t * s);
  }
  wid2.resize(ladder.size());
  for (size_t k = 0; k < ladder.size(); ++k) { const double w = ladder[k] * s2; wid2[k] = w * w; }
  lc.sin_dphi = s;
  const double cd = std::cos(lp.dphi);
  lc.cos_margin2 = (cd * (1 - 1e-9)) * (cd * (1 - 1e-9));
  lc.cos_loose2 = (cd * (1 - 1e-6)) * (cd * (1 - 1e-6));
  lc.cos_accept2 = (cd * (1 + 1e-9)) * (cd * (1 + 1e-9));
  // nearest ball centre is <= t_k s/2 away along the axis, the cone is <= t_k (1+s) tan(dphi)
  // wide there, the ball radius is t_k sin(2 dphi): covered if the sum of squares fits with
  // 10 % to spare
  const double td = std::tan(lp.dphi);
  lc.cover = (0.25 * s * s + (1 + s) * (1 + s) * td * td <= 0.9 * s2 * s2) ? 1 : 0;
  lc.inv_log_ratio = 1.0 / std::log1p(s);
  lc.log_t0 = std::log(s);
  const double w1 = std::log1p(s2) * lc.inv_log_ratio;
  const double w2 = -std::log1p(-s2) * lc.inv_log_ratio;
  lc.kwin = (int)std::ceil(w1 > w2 ? w1 : w2) + 2;
  lc.nladder = (int)ladder.size();
  return std::string();
}

// Boresight distance from the observer to the outer edge, in the reference's arithmetic order
// (k_los_prepare computes the same on the device); NaN if the boresight misses the sphere.
inline double los_dd(const double* los, long long nlos, long long i, double outeredge) {
  const double x = los[i], y = los[nlos + i], z = los[2 * nlos + i];
  const double bx = los[3 * nlos + i], by = los[4 * nlos + i], bz = los[5 * nlos + i];
  const double b = 2 * ((x * bx + y * by) + z * bz);
  const double nrm = std::sqrt((x * x + y * y) + z * z);
  const double c = nrm * nrm - outeredge * outeredge;
  return (-b + std::sqrt(b * b - 4 * 1 * c)) / 2;
}

// Balls of one line: the first k with t_k >= dd is its last entry; NaN dd -> a single entry
// (k_los_finish does the same on the device).
inline int los_nball(const std::vector<double>& ladder, double dd) {
  int k = 0;
  if (dd == dd) {
    k = (int)(std::lower_bound(ladder.begin(), ladder.end(), dd) - ladder.begin());
    if (k >= (int)ladder.size()) k = (int)ladder.size() - 1;
  }
  return k + 1;
}

// Host version of the per-line preparation (nx_los_used; the accumulate calls do the same on
// the device: k_los_prepare / k_los_finish in nx_los_grid.cu).
inline std::string los_prepare(const double* los, long long nlos, const LosParams& lp,
                               std::vector<int>& nball, std::vector<double>& ladder,
                               std::vector<double>& wid2, LosConsts& lc) {
  std::vector<double> dd(nlos);
  double ddmax = 0.0;
  for (long long i = 0; i < nlos; ++i) {
    dd[i] = los_dd(los, nlos, i, lp.outeredge);
    if (dd[i] > ddmax) ddmax = dd[i];
  }
  std::string err = los_constants(lp, ddmax, ladder, wid2, lc);
  if (!err.empty()) return err;
  nball.resize(nlos);
  for (long long i = 0; i < nlos; ++i) nball[i] = los_nball(ladder, dd[i]);
  return std::string();
}

}  // namespace nx
