// TEST-ONLY: the line-of-sight membership of K5 -- the ladder and constants of a call
// (nx_los.h: los_prepare), the exact test (nx_image.cuh: los_hit) and the weight (los_weight) --
// compiled with g++ under the same flags as hostcheck.cpp (no FMA contraction), so
// tests/test_los_membership.py can check them against the oracle on machines without a GPU.
// Never loaded by nexoclom_b200.
#include <cstring>

#include "../../nexoclom_b200/csrc/nx_physics.cuh"
#include "../../nexoclom_b200/csrc/nx_tables.h"
#include "../../nexoclom_b200/csrc/nx_image.cuh"
#include "../../nexoclom_b200/csrc/nx_los.h"

using namespace nx;

// the ladder of the last successful hc_los_prepare
static std::vector<double> g_ladder, g_wid2;

// Per-line preparation of nlos lines (los: 6 x nlos, rows x, y, z, xbore, ybore, zbore): the
// ball count of every line, the call's constants (sin_dphi, cos_margin2, cos_loose2,
// cos_accept2, cover, inv_log_ratio, log_t0, kwin, nladder) and the ladder length.  Returns 0,
// or -1 with the reason in err.
extern "C" int hc_los_prepare(const double* los, long long nlos, double dphi, double outeredge,
                              int* nball, double* consts, long long* nladder, char* err,
                              int errlen) {
  LosParams lp{};
  lp.dphi = dphi;
  lp.outeredge = outeredge;
  std::vector<int> nb;
  LosConsts lc{};
  const std::string e = los_prepare(los, nlos, lp, nb, g_ladder, g_wid2, lc);
  if (!e.empty()) {
    std::snprintf(err, errlen, "%s", e.c_str());
    g_ladder.clear(); g_wid2.clear();
    return -1;
  }
  std::memcpy(nball, nb.data(), nb.size() * sizeof(int));
  const double c[9] = {lc.sin_dphi, lc.cos_margin2, lc.cos_loose2, lc.cos_accept2, (double)lc.cover,
                       lc.inv_log_ratio, lc.log_t0, (double)lc.kwin, (double)lc.nladder};
  std::memcpy(consts, c, sizeof(c));
  *nladder = (long long)g_ladder.size();
  return 0;
}

extern "C" void hc_los_ladder(double* ladder, double* wid2) {
  std::memcpy(ladder, g_ladder.data(), g_ladder.size() * sizeof(double));
  std::memcpy(wid2, g_wid2.data(), g_wid2.size() * sizeof(double));
}

// los_hit and los_weight of every (line, packet) pair over the ladder of the last
// hc_los_prepare with the same dphi.  cover < 0: the call's `cover`, else forced;
// accept_off: cos_accept2 = +inf (every in-cone candidate goes through acos).  hit and weight
// are (nlos, n) row-major; weight is 0 where there is no hit.
extern "C" int hc_los_members(const double* los, long long nlos, const double* dist_plan,
                              const int* nball, long long n, const double* x, const double* y,
                              const double* z, const double* vy, const double* frac, double dphi,
                              double vrplanet, double rp_cm, int nt, const int* sizes,
                              const double* gv, const double* gg, int cover, int accept_off,
                              unsigned char* hit, double* weight) {
  if (g_ladder.empty()) return -1;
  LosParams lp{};
  lp.dphi = dphi; lp.vrplanet = vrplanet; lp.rp_cm = rp_cm; lp.quantity = 1;
  std::vector<double> l2, w2;
  LosConsts lc{};
  if (!los_constants(lp, 0.0, l2, w2, lc).empty()) return -1;
  if (cover >= 0) lc.cover = cover;
  if (accept_off) lc.cos_accept2 = INFINITY;
  std::vector<HostInterp> store(nt);
  GTables G{};
  G.n = nt;
  size_t off = 0;
  for (int t = 0; t < nt; ++t) {
    store[t] = make_interp(gv + off, gg + off, sizes[t]);
    InterpTable& T = G.t[t];
    T.x = store[t].x.data(); T.f = store[t].f.data(); T.slope = store[t].slope.data();
    T.bucket = store[t].bucket.data(); T.n = (int)store[t].x.size(); T.nbucket = store[t].nbucket;
    T.blo = store[t].blo; T.binvw = store[t].binvw;
    off += sizes[t];
  }
  for (long long l = 0; l < nlos; ++l) {
    LosRay L;
    L.xs = los[l]; L.ys = los[nlos + l]; L.zs = los[2 * nlos + l];
    L.bx = los[3 * nlos + l]; L.by = los[4 * nlos + l]; L.bz = los[5 * nlos + l];
    L.dist_plan = dist_plan[l];
    L.nball = nball[l];
    if (L.nball > (int)g_ladder.size()) return -1;
    for (long long i = 0; i < n; ++i) {
      double losrad, d2;
      const bool h = los_hit(L, lp.dphi, lc.cos_margin2, lc.cos_accept2, lc.cover, g_ladder.data(),
                             g_wid2.data(), lc.inv_log_ratio, lc.log_t0, lc.kwin, x[i], y[i], z[i],
                             losrad, d2);
      hit[l * n + i] = h;
      weight[l * n + i] = h ? los_weight(L, lp, G, lc.sin_dphi, frac[i], vy[i], losrad, d2) : 0.0;
    }
  }
  return 0;
}
