// nexoclom_b200 -- surface interaction (bounce / stick / thermal accommodation),
// the counter-based RNG and the constant-step driver step.
// NX_HD like nx_physics.cuh: inlined into kernels, and compiled by g++ for
// tests/_hostcheck.
#pragma once
#include "nx_fast.cuh"
#include "nx_image.cuh"
#include "nx_physics.cuh"

namespace nx {


// ---------------------------------------------------------------------------
// Philox4x32-10 (Salmon et al. 2011).  counter = (id_lo, id_hi, draw, stream),
// key = (seed_lo, seed_hi).  Results depend only on (seed, global packet id,
// stream, draw) -> independent of launch geometry and GPU count.
// ---------------------------------------------------------------------------
enum RngStream { STREAM_INIT = 0, STREAM_BOUNCE = 1 };

NX_HD void philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3,
                         uint32_t k0, uint32_t k1, uint32_t* out) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint64_t p0 = (uint64_t)0xD2511F53u * c0;
    const uint64_t p1 = (uint64_t)0xCD9E8D57u * c2;
    const uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0;
    const uint32_t n1 = (uint32_t)p1;
    const uint32_t n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1;
    const uint32_t n3 = (uint32_t)p0;
    c0 = n0; c1 = n1; c2 = n2; c3 = n3;
    k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
  }
  out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

// 53-bit uniform in [0,1) from two 32-bit words (same construction as NumPy's
// Generator.random: (a>>5)*2^26 + (b>>6), scaled by 2^-53).
NX_HD double u53(uint32_t a, uint32_t b) {
  return (double)(((uint64_t)(a >> 5) << 26) | (uint64_t)(b >> 6)) * (1.0 / 9007199254740992.0);
}

NX_HD void uniform_pair(uint64_t seed, uint64_t id, uint32_t stream, uint32_t draw,
                        double& u0, double& u1) {
  uint32_t w[4];
  philox4x32_10((uint32_t)id, (uint32_t)(id >> 32), draw, stream,
                (uint32_t)seed, (uint32_t)(seed >> 32), w);
  u0 = u53(w[0], w[1]);
  u1 = u53(w[2], w[3]);
}

// ---------------------------------------------------------------------------
// Mercury surface temperature -- reference surface_temperature.py:4-19
// ---------------------------------------------------------------------------
NX_HD double surface_temperature(double t1, double lon, double lat) {
  const double t0 = 100.0;
  if ((lon <= NX_PI / 2) || (lon >= 3 * NX_PI / 2)) {
    const double cc = fabs(mul_rn(cos(lon), cos(lat)));
    return add_rn(t0, mul_rn(t1, sqrt(sqrt(cc))));      // |.|**0.25
  }
  return t0;
}

// ---------------------------------------------------------------------------
// Bicubic tensor B-spline, FITPACK bispev/fpbspl evaluation order
// (what scipy RectBivariateSpline.ev runs; reference SurfaceInteraction.py:56-58)
// ---------------------------------------------------------------------------
NX_HD int spl_interval(const double* t, int nt, double& arg) {
  // FITPACK fpbisp: l = k1; while (arg >= t(l+1) && l != nk1) l++  (1-based).
  // The interior knots of an interpolating spline on a linspace grid are uniform,
  // so l is first guessed by division and then corrected with the same
  // comparisons -- identical result, no 200-iteration scan.
  const int k1 = 4, nk1 = nt - k1;          // 1-based: tb=t(k1), te=t(nk1+1)
  const double tb = t[k1 - 1], te = t[nk1];
  if (arg < tb) arg = tb;
  if (arg > te) arg = te;
  int l = k1;
  if (nk1 > k1) {
    const double dtk = (te - tb) / (double)(nk1 - k1 + 1);   // mean knot spacing
    int g = k1 + (int)((arg - tb) / dtk);
    l = g < k1 ? k1 : (g > nk1 ? nk1 : g);
    while (l > k1 && arg < t[l - 1]) --l;        // need t(l) <= arg
    while (l != nk1 && !(arg < t[l])) ++l;       // and arg < t(l+1) unless l == nk1
  }
  return l;
}

NX_HD void spl_basis(const double* t, double x, int l, double* h) {
  double hh[3];
  h[0] = 1.0;
#pragma unroll
  for (int j = 1; j <= 3; ++j) {
#pragma unroll
    for (int i = 0; i < j; ++i) hh[i] = h[i];
    h[0] = 0.0;
#pragma unroll
    for (int i = 0; i < j; ++i) {
      const int li = l + i + 1, lj = li - j;            // 1-based
      const double tli = t[li - 1], tlj = t[lj - 1];
      const double f = div_rn(hh[i], sub_rn(tli, tlj));
      h[i] = add_rn(h[i], mul_rn(f, sub_rn(tli, x)));
      h[i + 1] = mul_rn(f, sub_rn(x, tlj));
    }
  }
}

NX_HD double spline2d_ev(const Spline2D& S, double x, double y) {
  double wx[4], wy[4];
  const int lx = spl_interval(S.tx, S.ntx, x);
  spl_basis(S.tx, x, lx, wx);
  const int ly = spl_interval(S.ty, S.nty, y);
  spl_basis(S.ty, y, ly, wy);
  const int nky1 = S.nty - 4;
  int l1 = (lx - 4) * nky1 + (ly - 4);
  double sp = 0.0;
#pragma unroll
  for (int i1 = 0; i1 < 4; ++i1) {
#pragma unroll
    for (int j1 = 0; j1 < 4; ++j1)
      sp = add_rn(sp, mul_rn(mul_rn(S.c[l1 + j1], wx[i1]), wy[j1]));
    l1 += nky1;
  }
  return sp;
}

// ---------------------------------------------------------------------------
// Unit emission direction in the local frame at `pos` -- reference
// bouncepackets.py:5-36 and source_distribution.py:229-252 (v_tan0 multiplies
// NORTH, v_tan1 multiplies EAST: quirk Q18).
// ---------------------------------------------------------------------------
NX_HD void local_direction(double x, double y, double z, double alt, double az, double* d) {
  const double v_rad = sin(alt);
  const double ca = cos(alt);
  const double v_tan0 = mul_rn(ca, cos(az));
  const double v_tan1 = mul_rn(ca, sin(az));
  const double rn = sqrt(add_rn(add_rn(mul_rn(x, x), mul_rn(y, y)), mul_rn(z, z)));
  const double ex = y, ey = -x;
  const double en = sqrt(add_rn(add_rn(mul_rn(ex, ex), mul_rn(ey, ey)), 0.0));
  const double nx_ = mul_rn(-z, x), ny_ = mul_rn(-z, y), nz_ = add_rn(mul_rn(x, x), mul_rn(y, y));
  const double nn = sqrt(add_rn(add_rn(mul_rn(nx_, nx_), mul_rn(ny_, ny_)), mul_rn(nz_, nz_)));
  const double r[3] = {div_rn(x, rn), div_rn(y, rn), div_rn(z, rn)};
  const double e[3] = {div_rn(ex, en), div_rn(ey, en), div_rn(0.0, en)};
  const double n[3] = {div_rn(nx_, nn), div_rn(ny_, nn), div_rn(nz_, nn)};
#pragma unroll
  for (int k = 0; k < 3; ++k)
    d[k] = add_rn(add_rn(mul_rn(v_tan0, n[k]), mul_rn(v_tan1, e[k])), mul_rn(v_rad, r[k]));
}

// ---------------------------------------------------------------------------
// Surface impact -- reference bouncepackets.py:39-100.  `s` is the post-step
// state (inside the planet), r_hit its radius.  Position is moved back to the
// surface, speed from energy conservation (+ accommodation), direction cosine
// law, frac reduced by the sticking coefficient.  Remaining time untouched (Q17).
// ---------------------------------------------------------------------------
NX_HD void bounce(const RunParams& p, const Spline2D& S, double* s, double r_hit,
                  double u_alt, double u_az, double u_prob) {
  double x = s[1], y = s[2], z = s[3];
  const double vx = s[4], vy = s[5], vz = s[6];
  const double a = add_rn(add_rn(mul_rn(vx, vx), mul_rn(vy, vy)), mul_rn(vz, vz));
  const double b = mul_rn(2.0, add_rn(add_rn(mul_rn(x, vx), mul_rn(y, vy)), mul_rn(z, vz)));
  const double c = sub_rn(add_rn(add_rn(mul_rn(x, x), mul_rn(y, y)), mul_rn(z, z)), 1.0);
  const double disc = sqrt(sub_rn(mul_rn(b, b), mul_rn(mul_rn(4.0, a), c)));
  const double two_a = mul_rn(2.0, a);
  const double t0 = div_rn(sub_rn(-b, disc), two_a);
  const double t1 = div_rn(add_rn(-b, disc), two_a);
  const double t = fmin(t0, t1);
  x = add_rn(x, mul_rn(vx, t)); y = add_rn(y, mul_rn(vy, t)); z = add_rn(z, mul_rn(vz, t));

  const double pe = mul_rn(mul_rn(2.0, p.GM), sub_rn(div_rn(1.0, r_hit), 1.0));
  double v_old2 = add_rn(a, pe);
  if (v_old2 < 0.0) v_old2 = 0.0;

  double dir[3];
  local_direction(x, y, z, asin(u_alt), mul_rn(NX_TWO_PI, u_az), dir);

  const bool need_lonlat = (p.accomfactor != 0.0) || (p.sticktype == STICK_TEMPERATURE);
  double tsurf = 0.0;
  if (need_lonlat) {
    const double lon = fmod(add_rn(atan2(x, -y), NX_TWO_PI), NX_TWO_PI);
    const double lat = asin(z);
    tsurf = surface_temperature(p.surf_t1, lon, lat);
  }
  double v_new;
  if (p.accomfactor == 0.0) {
    v_new = sqrt(v_old2);
  } else {
    const double v_emit = div_rn(spline2d_ev(S, tsurf, u_prob), p.planet_radius_km);
    const double af = p.accomfactor;
    v_new = sqrt(add_rn(mul_rn(mul_rn(v_emit, v_emit), af), mul_rn(v_old2, sub_rn(1.0, af))));
  }
  s[1] = x; s[2] = y; s[3] = z;
  s[4] = mul_rn(dir[0], v_new); s[5] = mul_rn(dir[1], v_new); s[6] = mul_rn(dir[2], v_new);

  if (p.sticktype == STICK_TEMPERATURE) {
    double coef = add_rn(mul_rn(p.stick_A[0], exp(mul_rn(p.stick_A[1], tsurf))), p.stick_A[2]);
    if (coef > 1.0) coef = 1.0;
    if (coef < 0.0) coef = 0.0;
    s[7] = mul_rn(s[7], sub_rn(1.0, coef));
  } else if (p.stickcoef > 0.0) {
    s[7] = mul_rn(s[7], sub_rn(1.0, p.stickcoef));
  }
}

// ---------------------------------------------------------------------------
// One step of the constant-step driver -- reference Output.py:384-431.
// Returns true while the packet is still alive (frac > 0).  A packet that dies
// keeps its final position with frac = 0, time = 0 for THIS step; all later
// rows of the reference's dense tensor are zero.
// ---------------------------------------------------------------------------
// Fast-arithmetic bounce: same physics as bounce(), with the trigonometry of the
// reference folded analytically for a point on the unit sphere:
//   sin(asin(u)) = u, cos(asin(u)) = sqrt(1-u^2);
//   cos(lon) cos(lat) = -y  (x = sin lon cos lat, y = -cos lon cos lat, z = sin lat),
//   dayside (lon <= pi/2 or lon >= 3pi/2)  <=>  y <= 0,
// so no asin / atan2 / fmod is needed for the surface temperature.
NX_HD void bounce_fast(const RunParams& p, const Spline2D& S, double* s, double r_hit,
                       double u_alt, double u_az, double u_prob) {
  double x = s[1], y = s[2], z = s[3];
  const double vx = s[4], vy = s[5], vz = s[6];
  const double a = fma(vz, vz, fma(vy, vy, vx * vx));
  const double b = 2.0 * fma(z, vz, fma(y, vy, x * vx));
  const double c = fma(z, z, fma(y, y, x * x)) - 1.0;
  const double disc = sqrt(fma(b, b, -4.0 * a * c));
  const double inv2a = 1.0 / (2.0 * a);
  const double t = fmin((-b - disc) * inv2a, (-b + disc) * inv2a);
  x = fma(vx, t, x); y = fma(vy, t, y); z = fma(vz, t, z);

  double v_old2 = a + (2.0 * p.GM) * (1.0 / r_hit - 1.0);
  if (v_old2 < 0.0) v_old2 = 0.0;

  // cosine-law direction in the local frame (rad, east, north)
  const double v_rad = u_alt, ca = sqrt(fmax(1.0 - u_alt * u_alt, 0.0));
  double sa, cz;
#if defined(__CUDA_ARCH__)
  sincospi(2.0 * u_az, &sa, &cz);
#else
  sa = sin(NX_TWO_PI * u_az); cz = cos(NX_TWO_PI * u_az);
#endif
  const double v_tan0 = ca * cz, v_tan1 = ca * sa;
  const double rxy2 = fma(y, y, x * x);
  const double rinv = rsqrt_h(rxy2 + z * z), einv = rsqrt_h(rxy2);
  const double nn = rsqrt_h(fma(rxy2, rxy2, (z * z) * rxy2));
  const double nx_ = -z * x * nn, ny_ = -z * y * nn, nz_ = rxy2 * nn;
  const double ex = y * einv, ey = -x * einv;
  const double dx = fma(v_rad, x * rinv, fma(v_tan1, ex, v_tan0 * nx_));
  const double dy = fma(v_rad, y * rinv, fma(v_tan1, ey, v_tan0 * ny_));
  const double dz = fma(v_rad, z * rinv, v_tan0 * nz_);

  const bool need_t = (p.accomfactor != 0.0) || (p.sticktype == STICK_TEMPERATURE);
  double tsurf = 100.0;
  if (need_t && y <= 0.0) tsurf = fma(p.surf_t1, sqrt(sqrt(fabs(y))), 100.0);
  double v_new;
  if (p.accomfactor == 0.0) {
    v_new = sqrt(v_old2);
  } else {
    const double v_emit = spline2d_ev(S, tsurf, u_prob) / p.planet_radius_km;
    const double af = p.accomfactor;
    v_new = sqrt(fma(v_emit * v_emit, af, v_old2 * (1.0 - af)));
  }
  s[1] = x; s[2] = y; s[3] = z;
  s[4] = dx * v_new; s[5] = dy * v_new; s[6] = dz * v_new;
  if (p.sticktype == STICK_TEMPERATURE) {
    double coef = fma(p.stick_A[0], exp(p.stick_A[1] * tsurf), p.stick_A[2]);
    coef = fmin(fmax(coef, 0.0), 1.0);
    s[7] *= (1.0 - coef);
  } else if (p.stickcoef > 0.0) {
    s[7] *= (1.0 - p.stickcoef);
  }
}

// Surface interaction of the adaptive driver's BOUNCE builds (declared in nx_physics.cuh).
template <bool FAST>
NX_COLD void adaptive_surface(const RunParams& p, const Spline2D& S, double* s, double r2,
                              uint64_t seed, uint64_t id, uint32_t k) {
  double u_alt, u_az, u_prob, unused;
  uniform_pair(seed, id, STREAM_BOUNCE, 2u * k, u_alt, u_az);
  uniform_pair(seed, id, STREAM_BOUNCE, 2u * k + 1u, u_prob, unused);
  if (FAST) bounce_fast(p, S, s, sqrt(r2), u_alt, u_az, u_prob);
  else bounce(p, S, s, sqrt(r2), u_alt, u_az, u_prob);
}

// Deposition events of one accepted adaptive step (declared in nx_physics.cuh).
template <class Sink>
NX_COLD void deposit_record(Sink& D, bool surf, double x, double y, double z, double dep,
                            int fate, double ff) {
  if (surf) {
    D.sum[DEP_SURFACE] += dep;
    D.n[DEP_SURFACE] += 1;
    double lon, lat;
    deposit_lonlat(x, y, z, lon, lat);
    const int c = deposit_cell(lon, lat, D.nlon, D.nlat);
    if (c >= 0) {
#if defined(__CUDA_ARCH__)
      atomicAdd(D.map + c, dep);
      atomicAdd(D.cnt + c, 1ull);
#else
      D.map[c] += dep;
      D.cnt[c] += 1;
#endif
    }
  }
  if (fate >= 0) {
    D.sum[fate] += ff;
    D.n[fate] += 1;
  }
}

// post-step handling shared by the strict and the fast constant step
template <bool FAST>
NX_HD bool constant_step_finish(const RunParams& p, const Spline2D& S, double* nx, double* s,
                                uint64_t seed, uint64_t id, uint32_t stepidx) {
  const double r = sqrt(add_rn(add_rn(mul_rn(nx[1], nx[1]), mul_rn(nx[2], nx[2])), mul_rn(nx[3], nx[3])));
  if (sub_rn(r, 1.0) < 0.0) {
    if (p.sticktype == STICK_CONSTANT && p.stickcoef == 1.0) {
      nx[7] = 0.0;
    } else {
      double u_alt, u_az, u_prob, unused;
      uniform_pair(seed, id, STREAM_BOUNCE, 2u * stepidx, u_alt, u_az);
      uniform_pair(seed, id, STREAM_BOUNCE, 2u * stepidx + 1u, u_prob, unused);
      if (FAST) bounce_fast(p, S, nx, r, u_alt, u_az, u_prob);
      else bounce(p, S, nx, r, u_alt, u_az, u_prob);
    }
  }
  for (int m = 0; m < p.nmoons; ++m) {     // extension: packets that hit a moon stick to it
    double mx, my;
    moon_position(p, m, nx[0], mx, my);
    const double dx = nx[1] - mx, dy = nx[2] - my;
    if (dx * dx + dy * dy + nx[3] * nx[3] < p.moon_r2[m]) nx[7] = 0.0;
  }
  if (r > p.outeredge) nx[7] = 0.0;
  if (nx[7] < 1e-10) nx[7] = 0.0;
  if (nx[7] == 0.0) nx[0] = 0.0;
#pragma unroll
  for (int k = 0; k < 8; ++k) s[k] = nx[k];
  return nx[7] > 0.0;
}

template <bool STRICT>
NX_HD bool constant_step(const RunParams& p, const InterpTable& T, const Spline2D& S,
                         double* s, uint64_t seed, uint64_t id, uint32_t stepidx) {
  double nx[8];
  dp_step<STRICT, false>(p, T, s, p.step_size, nx, nullptr);
  return constant_step_finish<false>(p, S, nx, s, seed, id, stepidx);
}

// fast arithmetic (Nystrom stages of nx_fast.cuh), same decisions
template <int GR, int RP, int LOSS>
NX_HD bool constant_step_fast(const RunParams& p, const FastTable& T, const Spline2D& S,
                              double* s, uint64_t seed, uint64_t id, uint32_t stepidx) {
  double q[6], d[6], fn, df;
  fast_stages<GR, RP, LOSS, false>(p, T, s, p.step_size, q, fn, d, df);
  double nx[8] = {s[0] - p.step_size, q[0], q[1], q[2], q[3], q[4], q[5], fn};
  return constant_step_finish<true>(p, S, nx, s, seed, id, stepidx);
}

// --- split form of the fast constant step, for kernels that batch the bounces ---
// stage part: s <- post-step state (before any surface interaction); returns r.
template <int GR, int RP, int LOSS>
NX_HD double constant_stages_fast(const RunParams& p, const FastTable& T, double* s,
                                  const double* hc = nullptr) {
  double q[6], d[6], fn, df;
  fast_stages<GR, RP, LOSS, false>(p, T, s, p.step_size, q, fn, d, df, nullptr, hc);
  s[0] -= p.step_size;
#pragma unroll
  for (int k = 0; k < 6; ++k) s[1 + k] = q[k];
  s[7] = fn;
  return sqrt(add_rn(add_rn(mul_rn(q[0], q[0]), mul_rn(q[1], q[1])), mul_rn(q[2], q[2])));
}
// surface interaction of a packet whose post-step radius r is below the surface
NX_HD void constant_bounce_fast(const RunParams& p, const Spline2D& S, double* s, double r,
                                uint64_t seed, uint64_t id, uint32_t stepidx) {
  double u_alt, u_az, u_prob, unused;
  uniform_pair(seed, id, STREAM_BOUNCE, 2u * stepidx, u_alt, u_az);
  uniform_pair(seed, id, STREAM_BOUNCE, 2u * stepidx + 1u, u_prob, unused);
  bounce_fast(p, S, s, r, u_alt, u_az, u_prob);
}
// escape / vanish / done tests (Output.py:409-416); r is the pre-bounce radius
NX_HD bool constant_post(const RunParams& p, double* s, double r) {
  if (r > p.outeredge) s[7] = 0.0;
  if (s[7] < 1e-10) s[7] = 0.0;
  if (s[7] == 0.0) s[0] = 0.0;
  return s[7] > 0.0;
}

NX_HD bool constant_step_fast_rt(const RunParams& p, const FastTable& T, const Spline2D& S,
                                 double* s, uint64_t seed, uint64_t id, uint32_t stepidx) {
  const int key = (p.gravity ? 4 : 0) | (p.radpres ? 2 : 0);
#define NX_CASE(G, R)                                                                          \
  if (key == ((G) * 4 + (R) * 2)) {                                                            \
    if (p.loss_mode == LOSS_PHOTO) return constant_step_fast<G, R, LOSS_PHOTO>(p, T, S, s, seed, id, stepidx);       \
    if (p.loss_mode == LOSS_LIFETIME) return constant_step_fast<G, R, LOSS_LIFETIME>(p, T, S, s, seed, id, stepidx); \
    return constant_step_fast<G, R, LOSS_NONE>(p, T, S, s, seed, id, stepidx);                 \
  }
  NX_CASE(1, 1) NX_CASE(1, 0) NX_CASE(0, 1) NX_CASE(0, 0)
#undef NX_CASE
  return false;
}

}  // namespace nx
