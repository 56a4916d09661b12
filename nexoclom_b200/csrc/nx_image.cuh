// nexoclom_b200 -- per-packet image / line-of-sight math (K4, K5).
// Reference: data_simulation/ModelImage.py:229-274, ModelResult.py:140-170,
// math/histogram.py:28-39 (np.histogram2d), data_simulation/compute_iteration.py:151-222.
#pragma once
#include "nx_physics.cuh"

namespace nx {

#define NX_MAX_GTABLES 4

struct ImageParams {
  double M[9];
  double x0, x1, z0, z1;
  double apix;
  double vrplanet;
  int32_t nx, nz;
  int32_t quantity;      // 0 column, 1 radiance
  int32_t round_f32;
  int32_t skip_dead;
  int32_t reserved;
};

struct LosParams {
  double dphi, outeredge, vrplanet, rp_cm;
  int32_t quantity, round_f32, skip_dead, reserved;
};

struct GTables {
  InterpTable t[NX_MAX_GTABLES];
  FastTable f[NX_MAX_GTABLES];      // record form of the same tables (kernels)
  // the SUM of the tables on the union of their nodes (built on upload when n > 1): a sum of
  // piecewise-linear functions is piecewise linear on the union grid, so the fast path needs
  // one lookup instead of n (values agree with the sum of n np.interp to rounding)
  FastTable fsum;
  int n;
  int has_sum;
};

NX_HD double round_f32(double v) { return (double)(float)v; }

// np.histogram2d bin of v for edges = linspace(lo, hi, n+1):
// edges[k] = k*step + lo (k < n), edges[n] = hi; bin = searchsorted(edges, v,
// 'right') - 1, the right edge belongs to the last bin.  Returns -1 if outside.
NX_HD double hist_edge(int k, int n, double lo, double hi, double step) {
  return (k == n) ? hi : add_rn(mul_rn((double)k, step), lo);
}
NX_HD int hist_bin(double v, int n, double lo, double hi, double step) {
  if (!(v >= lo && v <= hi)) return -1;
  int k = (int)((v - lo) / step);
  k = k < 0 ? 0 : (k > n - 1 ? n - 1 : k);
  while (k > 0 && hist_edge(k, n, lo, hi, step) > v) --k;
  while (k < n - 1 && hist_edge(k + 1, n, lo, hi, step) <= v) ++k;
  return k;
}

// same bin from a reciprocal first guess (the two correction loops make the result
// independent of the guess; they run 0 or 1 times)
NX_HD int hist_bin_fast(double v, int n, double lo, double hi, double step, double inv_step) {
  if (!(v >= lo && v <= hi)) return -1;
  int k = (int)((v - lo) * inv_step);
  k = k < 0 ? 0 : (k > n - 1 ? n - 1 : k);
  while (k > 0 && hist_edge(k, n, lo, hi, step) > v) --k;
  while (k < n - 1 && hist_edge(k + 1, n, lo, hi, step) <= v) ++k;
  return k;
}

// Surface longitude / latitude of a deposition event at (x, y, z): the bounce's convention
// (nx_surface.cuh::bounce), lon = fmod(atan2(x, -y) + 2 pi, 2 pi), lat = atan2(z, |(x, y)|).
NX_HD void deposit_lonlat(double x, double y, double z, double& lon, double& lat) {
  lon = fmod(add_rn(atan2(x, -y), NX_TWO_PI), NX_TWO_PI);
  lat = atan2(z, sqrt(add_rn(mul_rn(x, x), mul_rn(y, y))));
}

// Deposition map cell (lon-major: ilon * nlat + ilat) on np.histogram2d's axes
// linspace(0, 2 pi, nlon + 1) x linspace(-pi/2, pi/2, nlat + 1), the axes of make_source_map;
// -1 outside.
NX_HD int deposit_cell(double lon, double lat, int nlon, int nlat) {
  const double half_pi = NX_PI / 2.0;
  const int i = hist_bin(lon, nlon, 0.0, NX_TWO_PI, NX_TWO_PI / nlon);
  const int j = hist_bin(lat, nlat, -half_pi, half_pi, (half_pi - -half_pi) / nlat);
  return (i < 0 || j < 0) ? -1 : i * nlat + j;
}

// Ion-production grid cell of (x, y, z), row-major (ix * ny + iy) * nz + iz, by
// np.histogramdd's rule per axis (hist_bin_fast); -1 outside the box or NaN.
NX_HD long long ion_cell(const IonOut& g, double x, double y, double z) {
  const int i = hist_bin_fast(x, g.n[0], g.lo[0], g.hi[0], g.step[0], g.inv_step[0]);
  const int j = hist_bin_fast(y, g.n[1], g.lo[1], g.hi[1], g.step[1], g.inv_step[1]);
  const int k = hist_bin_fast(z, g.n[2], g.lo[2], g.hi[2], g.step[2], g.inv_step[2]);
  if (i < 0 || j < 0 || k < 0) return -1;
  return ((long long)i * g.n[1] + j) * g.n[2] + k;
}

// The steps and reciprocals of the grid's axes, as ImageSteps forms them.
NX_HD void ion_steps(IonOut& g) {
  for (int a = 0; a < 3; ++a) {
    g.step[a] = (g.hi[a] - g.lo[a]) / g.n[a];
    g.inv_step[a] = 1.0 / g.step[a];
  }
}

// Ion production of one accepted adaptive step (declared in nx_physics.cuh).
template <class Sink>
NX_COLD void ion_record(Sink& I, double loss, double x, double y, double z) {
  const long long c = ion_cell(I.g, x, y, z);
  if (c < 0) {
    I.out_sum += loss;
    I.out_n += 1;
    return;
  }
#if defined(__CUDA_ARCH__)
  atomicAdd(I.g.sum + c, loss);
  atomicAdd(I.g.cnt + c, 1ull);
#else
  I.g.sum[c] += loss;
  I.g.cnt[c] += 1;
#endif
}

// per-launch constants of the image kernels
struct ImageSteps {
  double step_x, step_z;          // bin widths, as np.histogram2d's linspace gives them
  double inv_step_x, inv_step_z;
  double wscale;                  // 1/apix (column) or 1/(1e6 apix) (radiance)
};
NX_HD ImageSteps image_steps(const ImageParams& ip) {
  ImageSteps t;
  t.step_x = (ip.x1 - ip.x0) / ip.nx; t.step_z = (ip.z1 - ip.z0) / ip.nz;
  t.inv_step_x = 1.0 / t.step_x; t.inv_step_z = 1.0 / t.step_z;
  t.wscale = (ip.quantity == 1) ? 1.0 / (1e6 * ip.apix) : 1.0 / ip.apix;
  return t;
}

// Sum of g-values over the emission lines at radial velocity rv [R_p/s]
// (ModelResult.py:152-157: gg = 0 + g_1 + g_2 ...).
NX_HD double gvalue_sum(const GTables& G, double rv) {
  double gg = 0.0;
#pragma unroll
  for (int i = 0; i < NX_MAX_GTABLES; ++i)
    if (i < G.n) gg = add_rn(gg, interp(G.t[i], rv));
  return gg;
}
// same sum through the record tables (value differs from np.interp by <= 1 ulp:
// fma(slope, x - lo, f) instead of slope*(x - lo) + f)
NX_HD double gvalue_sum_fast(const GTables& G, double rv) {
  if (G.has_sum) return interp_fast<false>(G.fsum, rv);
  double gg = 0.0;
#pragma unroll
  for (int i = 0; i < NX_MAX_GTABLES; ++i)
    if (i < G.n) gg += interp_fast<false>(G.f[i], rv);
  return gg;
}

// One packet's contribution to the image.  Returns the flat pixel index
// ix*nz + iz (or -1) and the weight.
template <bool FASTG = false>
NX_HD int image_packet(const ImageParams& ip, const GTables& G, double step_x, double step_z,
                       double x, double y, double z, double vy, double frac, double& weight) {
  if (ip.round_f32) { x = round_f32(x); y = round_f32(y); z = round_f32(z);
                      vy = round_f32(vy); frac = round_f32(frac); }
  // rotate to the observer frame (np.matmul -> FMA-chained dot, ModelImage.py:249)
  const double xo = fma(ip.M[2], z, fma(ip.M[1], y, ip.M[0] * x));
  const double yo = fma(ip.M[5], z, fma(ip.M[4], y, ip.M[3] * x));
  const double zo = fma(ip.M[8], z, fma(ip.M[7], y, ip.M[6] * x));
  // occultation by the planet (ModelImage.py:252-254)
  const double so = add_rn(mul_rn(xo, xo), mul_rn(zo, zo));
  const bool inview = (so > NX_ONE_PLUS_ULP) || (yo < 0.0);
  double f = mul_rn(frac, inview ? 1.0 : 0.0);
  if (ip.quantity == 1) {
    const bool lit = out_of_shadow(x, y, z);                    // ModelImage.py:257-258
    const double rv = add_rn(vy, ip.vrplanet);                  // ModelImage.py:242
    const double gg = FASTG ? gvalue_sum_fast(G, rv) : gvalue_sum(G, rv);
    f = div_rn(mul_rn(mul_rn(f, lit ? 1.0 : 0.0), gg), 1e6);    // ModelResult.py:161
  }
  weight = div_rn(f, ip.apix);                                  // ModelImage.py:262
  const int ix = hist_bin(xo, ip.nx, ip.x0, ip.x1, step_x);
  const int iz = hist_bin(zo, ip.nz, ip.z0, ip.z1, step_z);
  if (ix < 0 || iz < 0) return -1;
  return ix * ip.nz + iz;
}

// Kernel form: identical pixel (bit-exact), weight through one reciprocal scale
// instead of the two divisions (<= 2 ulp from the form above; the gate is 1e-6).
NX_HD int image_packet_fast(const ImageParams& ip, const GTables& G, const ImageSteps& t,
                            double x, double y, double z, double vy, double frac,
                            double& weight, int* ix_out = nullptr, int* iz_out = nullptr) {
  if (ip.round_f32) { x = round_f32(x); y = round_f32(y); z = round_f32(z);
                      vy = round_f32(vy); frac = round_f32(frac); }
  const double xo = fma(ip.M[2], z, fma(ip.M[1], y, ip.M[0] * x));
  const double yo = fma(ip.M[5], z, fma(ip.M[4], y, ip.M[3] * x));
  const double zo = fma(ip.M[8], z, fma(ip.M[7], y, ip.M[6] * x));
  const double so = add_rn(mul_rn(xo, xo), mul_rn(zo, zo));
  const bool inview = (so > NX_ONE_PLUS_ULP) || (yo < 0.0);
  double f = inview ? frac : 0.0;
  if (ip.quantity == 1) {
    const bool lit = out_of_shadow(x, y, z);
    f = lit ? f * gvalue_sum_fast(G, add_rn(vy, ip.vrplanet)) : 0.0;
  }
  weight = f * t.wscale;
  const int ix = hist_bin_fast(xo, ip.nx, ip.x0, ip.x1, t.step_x, t.inv_step_x);
  const int iz = hist_bin_fast(zo, ip.nz, ip.z0, ip.z1, t.step_z, t.inv_step_z);
  if (ix < 0 || iz < 0) return -1;
  if (ix_out) { *ix_out = ix; *iz_out = iz; }
  return ix * ip.nz + iz;
}

// The trajectory sink of one launch (k_trace_adaptive, a __grid_constant__ kernel parameter
// the lanes read through TraceSink::o): the image (img_sum == nullptr: none) with K4's
// parameters and g-value tables (their records stay in global memory), and the grid
// (grid.sum == nullptr: none), whose OUTSIDE slot is index n[0] * n[1] * n[2].
struct TraceOut {
  double* img_sum;
  unsigned long long* img_cnt;
  ImageParams ip;
  ImageSteps is;
  GTables G;
  IonOut grid;
  double endtime;           // T
};

// One accepted step of the trajectory sink (declared in nx_physics.cuh).  The dwell of the
// step, weighted by the inverse probability that a packet of its age is still in flight,
//   a = (h * T) / (age0 + (t - 0.5 * h)),   age0 = T - t0,
// every operation an f64 op rounded to nearest (both terms of the sum are >= 0, the second
// > 0).  The image adds w * a at the midpoint's pixel, w being K4's weight of the midpoint
// (image_packet_fast, which carries the frac), and one count; the grid adds frac * a at the
// midpoint's cell (ion_cell) and one count, or to the lane's OUTSIDE share.
template <class Sink>
NX_COLD void trace_record(Sink& Tr, double x, double y, double z, double vy, double frac,
                          double h, double t) {
  const TraceOut& o = *Tr.o;
  const double a = div_rn(mul_rn(h, o.endtime), add_rn(Tr.age0, sub_rn(t, mul_rn(0.5, h))));
  if (o.img_sum) {
    double w;
    const int pix = image_packet_fast(o.ip, o.G, o.is, x, y, z, vy, frac, w);
    if (pix >= 0) {
      const double v = mul_rn(w, a);
#if defined(__CUDA_ARCH__)
      if (v != 0.0) atomicAdd(o.img_sum + pix, v);
      atomicAdd(o.img_cnt + pix, 1ull);
#else
      o.img_sum[pix] += v;
      o.img_cnt[pix] += 1;
#endif
    }
  }
  if (o.grid.sum) {
    const double d = mul_rn(frac, a);
    const long long c = ion_cell(o.grid, x, y, z);
    if (c < 0) {
      Tr.out_sum += d;
      Tr.out_n += 1;
      return;
    }
#if defined(__CUDA_ARCH__)
    atomicAdd(o.grid.sum + c, d);
    atomicAdd(o.grid.cnt + c, 1ull);
#else
    o.grid.sum[c] += d;
    o.grid.cnt[c] += 1;
#endif
  }
}

// ---------------------------------------------------------------------------
// Lines of sight
// ---------------------------------------------------------------------------
struct LosRay {            // per-LOS constants prepared by nx_los_prepare
  double xs, ys, zs;       // spacecraft position
  double bx, by, bz;       // boresight (unit)
  double dist_plan;        // planet-truncation distance or 1e30
  int nball;               // number of KD-ball centres on the ladder
};

// Exact membership test, same arithmetic as compute_iteration.py:175-185 plus
// the KD-tree candidate filter (:164-173): the packet must lie in at least one
// ball |p - (x_sc + bore t_k)| <= t_k sin(2 dphi).  `ladder` = t_k, `wid2` =
// (t_k sin 2dphi)^2, `kwin` = half-width of the ball-index window to search.
// Two shortcuts keep the common hit cheap without changing any decision:
//  * a packet whose cos^2 exceeds cos_accept2 = (cos(dphi)(1+1e-9))^2 is inside the
//    cone by a margin far above the rounding of acos(): no sqrt / div / acos;
//  * if `cover` is set (host: the balls overlap enough, true for dphi up to ~20 deg),
//    every in-cone point with t_0 <= losrad <= t_last lies in the ball whose centre is
//    nearest, with a factor ~3 to spare: no log / window search.
// Outputs losrad and the squared distance d2 (the weight takes its sqrt).
NX_HD bool los_hit(const LosRay& L, double dphi, double cos_margin2, double cos_accept2,
                   int cover, const double* ladder, const double* wid2, double inv_log_ratio,
                   double log_t0, int kwin,
                   double px, double py, double pz, double& losrad, double& d2) {
  const double rx = sub_rn(px, L.xs), ry = sub_rn(py, L.ys), rz = sub_rn(pz, L.zs);
  losrad = add_rn(add_rn(mul_rn(rx, L.bx), mul_rn(ry, L.by)), mul_rn(rz, L.bz));
  d2 = add_rn(add_rn(mul_rn(rx, rx), mul_rn(ry, ry)), mul_rn(rz, rz));
  // cheap conservative reject: cos(ang) < cos(dphi) - margin
  const double l2 = mul_rn(losrad, losrad);
  if (!(losrad > 0.0) || l2 < mul_rn(d2, cos_margin2)) return false;
  if (!(losrad < L.dist_plan)) return false;
  if (!(l2 > mul_rn(d2, cos_accept2))) {
    double cosang = div_rn(losrad, sqrt(d2));
    if (cosang > 1.0) cosang = 1.0;
    if (!(acos(cosang) <= dphi)) return false;
  }
  // KD-ball candidate filter
  if (cover && losrad >= ladder[0] && losrad <= ladder[L.nball - 1]) return true;
  int k0 = (int)((log(losrad) - log_t0) * inv_log_ratio);
  int lo = k0 - kwin, hi = k0 + kwin;
  if (lo < 0) lo = 0;
  if (hi > L.nball - 1) hi = L.nball - 1;
  for (int k = lo; k <= hi; ++k) {
    const double t = ladder[k];
    const double cx = add_rn(L.xs, mul_rn(L.bx, t));
    const double cy = add_rn(L.ys, mul_rn(L.by, t));
    const double cz = add_rn(L.zs, mul_rn(L.bz, t));
    const double ex = sub_rn(px, cx), ey = sub_rn(py, cy), ez = sub_rn(pz, cz);
    const double e2 = add_rn(add_rn(mul_rn(ex, ex), mul_rn(ey, ey)), mul_rn(ez, ez));
    if (e2 <= wid2[k]) return true;
  }
  return false;
}

// Radiance weight of a hit packet (compute_iteration.py:193-206).
NX_HD double los_weight(const LosRay& L, const LosParams& lp, const GTables& G,
                        double sin_dphi, double frac, double vy, double losrad, double d2) {
  if (!(frac != 0.0)) return frac;            // 0 * finite g-value / area = 0 (keeps NaN)
  const double dist = sqrt(d2);
  const double rv = add_rn(vy, lp.vrplanet);
  const double gg = gvalue_sum(G, rv);
  const double w = div_rn(mul_rn(mul_rn(frac, 1.0), gg), 1e6);          // sunlit flag = 1 here (Q16)
  const double ds = mul_rn(dist, sin_dphi);
  const double apix = mul_rn(mul_rn(NX_PI, mul_rn(ds, ds)), mul_rn(lp.rp_cm, lp.rp_cm));
  double wt = div_rn(w, apix);
  // shadow test at the LOS foot-point (compute_iteration.py:202-206)
  const double hx = add_rn(L.xs, mul_rn(L.bx, losrad));
  const double hy = add_rn(L.ys, mul_rn(L.by, losrad));
  const double hz = add_rn(L.zs, mul_rn(L.bz, losrad));
  const double sh = add_rn(mul_rn(hx, hx), mul_rn(hz, hz));
  const bool lit = (sh > NX_ONE_PLUS_ULP) || (hy < 0.0);
  return mul_rn(wt, lit ? 1.0 : 0.0);
}

// ---------------------------------------------------------------------------
// Doppler spectra (LOSSpectrum): the velocity of a hit row along the boresight, in km/s,
// positive away from the observer, v = ((vx*bx + vy*by) + vz*bz) * vscale, every operation an
// IEEE float64 op rounded to nearest (vscale = R_p in km).
// ---------------------------------------------------------------------------
NX_HD double los_doppler(double vx, double vy, double vz, double bx, double by, double bz,
                         double vscale) {
  return mul_rn(add_rn(add_rn(mul_rn(vx, bx), mul_rn(vy, by)), mul_rn(vz, bz)), vscale);
}
// Spectrum column of v for edges = np.linspace(vmin, vmax, nbins + 1), step = (vmax - vmin) /
// nbins: 0 below vmin, 1 + the np.histogram bin inside [vmin, vmax] (vmax in the last bin),
// nbins + 1 above vmax (NaN included).
NX_HD int spectrum_column(double v, int nbins, double vmin, double vmax, double step) {
  if (v < vmin) return 0;
  if (!(v <= vmax)) return nbins + 1;
  return hist_bin(v, nbins, vmin, vmax, step) + 1;
}

// ---------------------------------------------------------------------------
// Number density (K7): is the saved row (x, y, z), float32 values widened to double, inside
// the ball of radius r around p?  d2 = (dx*dx + dy*dy) + dz*dz <= r*r, every operation an
// IEEE float64 op rounded to nearest, no contraction: NumPy's order for
// ((X - p)**2).sum(axis=1) <= r**2 on a float64 copy of the float32 columns.
// ---------------------------------------------------------------------------
NX_HD bool density_member(double x, double y, double z, double px, double py, double pz,
                          double r) {
  const double dx = sub_rn(x, px), dy = sub_rn(y, py), dz = sub_rn(z, pz);
  const double d2 = add_rn(add_rn(mul_rn(dx, dx), mul_rn(dy, dy)), mul_rn(dz, dz));
  return d2 <= mul_rn(r, r);
}

}  // namespace nx
