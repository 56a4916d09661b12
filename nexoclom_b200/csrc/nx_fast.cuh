// nexoclom_b200 -- throughput-oriented adaptive step (STRICT = false product path).
//
// Same algorithm and the same accept / reject DECISIONS as adaptive_attempt<true>
// (reference Output.py:249-353 + rk5.py + state.py), re-associated for the FP64
// pipe of sm_100a:
//   * stage sums are FMA chains started from the base state, written on the scaled
//     accelerations K_j = h a_j only (Nystrom form: stage velocities are never
//     stored -> 30 fewer registers -> one more resident block per SM); tableau
//     constants come from the constant bank;
//   * gravity uses one MUFU.RSQ64H seed + one third-order correction;
//   * frac is advanced as f*exp(dlogf) (== exp(log f + dlogf) in exact arithmetic),
//     so no log/exp pair per step and no per-stage log-frac bookkeeping;
//   * the radiation-pressure table is looked up through a bucket index + 32-byte
//     interval records (one LDS.U16 + two LDS.128, no search loop in the common case);
//   * accept test is "every delta_j < scale_j" (exactly equivalent to
//     max_j fl(delta_j/scale_j) < 1 for correctly rounded division); the
//     quotient itself is only formed on the reject path, with Newton reciprocals;
//   * forces / loss mode are template parameters (no per-stage uniform branches).
// Differences from the NumPy operation order are a few ulp per step; parity
// against the oracle stays ~1e-14 (gate 1e-8), see tests/test_hostcheck.py.
#pragma once
#include <string.h>

#include "nx_physics.cuh"

namespace nx {

// Dormand-Prince coefficients (reference rk5.py:5-18) and the derived "Nystrom"
// constants that let the position stages be written on the accelerations alone
// (so the six stage velocities never have to be stored):
//   v_m = v0 + sum_{j<m} a_mj K_j,                 K_j = h a_j
//   p_m = p0 + c_m (h v0) + sum_{j<m-1} (h A2_mj) K_j,  A2_mj = sum_{i=j+1}^{m-1} a_mi a_ij
//   h sum_{i<6} bd_i kv_i = BDS (h v0) + sum_{j<5} (h BD2_j) K_j
constexpr double dpc_a(int n, int i) {
  switch (n * 8 + i) {
    case 1 * 8 + 0: return 0.2;
    case 2 * 8 + 0: return 3. / 40.;  case 2 * 8 + 1: return 9. / 40.;
    case 3 * 8 + 0: return 44. / 45.; case 3 * 8 + 1: return -56. / 15.; case 3 * 8 + 2: return 32. / 9.;
    case 4 * 8 + 0: return 19372. / 6561.; case 4 * 8 + 1: return -25360. / 2187.;
    case 4 * 8 + 2: return 64448. / 6561.; case 4 * 8 + 3: return -212. / 729.;
    case 5 * 8 + 0: return 9017. / 3168.; case 5 * 8 + 1: return -355. / 33.;
    case 5 * 8 + 2: return 46732. / 5247.; case 5 * 8 + 3: return 49. / 176.;
    case 5 * 8 + 4: return -5103. / 18656.;
    case 6 * 8 + 0: return 35. / 384.; case 6 * 8 + 1: return 0.;
    case 6 * 8 + 2: return 500. / 1113.; case 6 * 8 + 3: return 125. / 192.;
    case 6 * 8 + 4: return -2187. / 6784.; case 6 * 8 + 5: return 11. / 84.;
    default: return 0.;
  }
}
constexpr double dpc_bd(int i) {
  switch (i) {
    case 0: return 35. / 384. - 5179. / 57600.;
    case 2: return 500. / 1113. - 7571. / 16695.;
    case 3: return 125. / 192. - 393. / 640.;
    case 4: return -2187. / 6784. - -92097. / 339200.;
    case 5: return 11. / 84. - 187. / 2100.;
    default: return 0.;
  }
}
constexpr double dpc_c(int m) { double s = 0; for (int i = 0; i < m; ++i) s += dpc_a(m, i); return s; }
constexpr double dpc_a2(int m, int j) {
  double s = 0;
  for (int i = j + 1; i < m; ++i) s += dpc_a(m, i) * dpc_a(i, j);
  return s;
}
constexpr double dpc_bds() { double s = 0; for (int i = 0; i < 6; ++i) s += dpc_bd(i); return s; }
constexpr double dpc_bd2(int j) {
  double s = 0;
  for (int i = j + 1; i < 6; ++i) s += dpc_bd(i) * dpc_a(i, j);
  return s;
}
constexpr double dpc_bsum() { double s = 0; for (int i = 0; i < 6; ++i) s += dpc_a(6, i); return s; }
// evaluated once at compile time (usable from device code without relaxed constexpr)
constexpr double kDpcBsum = dpc_bsum();
constexpr double kDpcBds = dpc_bds();

#define NX_ROW(f, m) f(m, 0), f(m, 1), f(m, 2), f(m, 3), f(m, 4), f(m, 5), 0., 0.
#define NX_TAB(f) {NX_ROW(f, 0), NX_ROW(f, 1), NX_ROW(f, 2), NX_ROW(f, 3), NX_ROW(f, 4), \
                   NX_ROW(f, 5), NX_ROW(f, 6)}
#define NX_VEC6(f) {f(0), f(1), f(2), f(3), f(4), f(5), 0., 0.}
#define NX_VEC7(f) {f(0), f(1), f(2), f(3), f(4), f(5), f(6), 0.}

#if defined(__CUDACC__)
__constant__ double c_dp_a[56] = NX_TAB(dpc_a);
__constant__ double c_dp_a2[56] = NX_TAB(dpc_a2);
__constant__ double c_dp_c[8] = NX_VEC7(dpc_c);
__constant__ double c_dp_bd[8] = NX_VEC6(dpc_bd);
__constant__ double c_dp_bd2[8] = NX_VEC6(dpc_bd2);
#endif
static const double h_dp_a[56] = NX_TAB(dpc_a);
static const double h_dp_a2[56] = NX_TAB(dpc_a2);
static const double h_dp_c[8] = NX_VEC7(dpc_c);
static const double h_dp_bd[8] = NX_VEC6(dpc_bd);
static const double h_dp_bd2[8] = NX_VEC6(dpc_bd2);

#if defined(__CUDA_ARCH__)
#define NX_CONST(name, k) c_##name[k]
#else
#define NX_CONST(name, k) h_##name[k]
#endif
NX_HD double dp_a(int m, int j) { return NX_CONST(dp_a, m * 8 + j); }
NX_HD double dp_a2(int m, int j) { return NX_CONST(dp_a2, m * 8 + j); }
NX_HD double dp_c(int m) { return NX_CONST(dp_c, m); }
NX_HD double dp_bd(int i) { return NX_CONST(dp_bd, i); }
NX_HD double dp_bd2(int j) { return NX_CONST(dp_bd2, j); }

// Comparisons of NON-NEGATIVE doubles through their bit patterns: integer compares
// run on the ALU pipe and leave the (half-rate) FP64 pipe to the arithmetic.
NX_HD long long dbits(double a) {
#if defined(__CUDA_ARCH__)
  return __double_as_longlong(a);
#else
  long long r; memcpy(&r, &a, 8); return r;
#endif
}
NX_HD bool lt_nonneg(double a, double b) { return dbits(a) < dbits(b); }   // a, b >= 0 (NaN > all)
NX_HD bool is_negative(double a) { return dbits(a) < 0 && a != 0.0; }
NX_HD double max_nonneg(double a, double b) { return lt_nonneg(a, b) ? b : a; }

// 1/sqrt(a): hardware seed + one third-order (Halley) step  -> ~0.2 ulp
NX_HD double rsqrt_h(double a) {
#if defined(__CUDA_ARCH__)
  double y;
  asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(a));
  const double t = a * y;
  const double e = fma(-t, y, 1.0);
  const double q = fma(0.375, e, 0.5) * e;
  return fma(y, q, y);
#else
  return 1.0 / sqrt(a);
#endif
}

// 1/a to ~2^-40: hardware seed + one Newton step (only feeds the step-size
// update on the reject path, never a decision)
NX_HD double rcp_n(double a) {
#if defined(__CUDA_ARCH__)
  double r;
  asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(a));
  const double e = fma(-a, r, 1.0);
  return fma(r, e, r);
#else
  return 1.0 / a;
#endif
}

// exp(d) for the small log-frac increments of one step
NX_HD double exp_step(double d) {
  if (fabs(d) < 0.03125) {
    double p = 1.0 / 5040.0;
    p = fma(p, d, 1.0 / 720.0);
    p = fma(p, d, 1.0 / 120.0);
    p = fma(p, d, 1.0 / 24.0);
    p = fma(p, d, 1.0 / 6.0);
    p = fma(p, d, 0.5);
    p = fma(p, d, 1.0);
    return fma(p, d, 1.0);
  }
  return exp(d);
}

// sin / cos of a small angle (|d| < ~0.2 rad: moon phase advanced over one step)
NX_HD void sincos_small(double d, double& sn, double& cs) {
  const double d2 = d * d;
  double ps = -1.0 / 39916800.0;                       // -1/11!
  ps = fma(ps, d2, 1.0 / 362880.0);
  ps = fma(ps, d2, -1.0 / 5040.0);
  ps = fma(ps, d2, 1.0 / 120.0);
  ps = fma(ps, d2, -1.0 / 6.0);
  sn = fma(ps * d2, d, d);
  double pc = 1.0 / 479001600.0;                       // 1/12!
  pc = fma(pc, d2, -1.0 / 3628800.0);
  pc = fma(pc, d2, 1.0 / 40320.0);
  pc = fma(pc, d2, -1.0 / 720.0);
  pc = fma(pc, d2, 1.0 / 24.0);
  pc = fma(pc, d2, -0.5);
  cs = fma(pc, d2, 1.0);
}

// The six Dormand-Prince stages in Nystrom form.  Inputs s[0..7], step h.
// Outputs: nx[6] = new position / velocity, fn = new frac; if ERR also the error
// vector d[6] = |h sum_{i<6} bd_i k_i| (stage 7 not included: quirk Q1) and
// delta_f for the log-frac component.
// MO = 1: one moon (the extension of RunParams) acts on the packets: its phase at the stage
// time tau - c_n h is phi_0 + omega c_n h, evaluated by angle addition from one sincos per
// step; `moon_end` receives the moon's position at the end of the step (impact test).
// `hc` (constant-step driver: h is the same for every packet and step): the products
// h * A2_mj (index m * 8 + j) and h * GM (index 56) formed once on the host -- the same
// correctly rounded products, 16 fewer FP64 multiplies per step.
#define NX_STEPCOEF_COUNT 57
template <int GR, int RP, int LOSS, bool ERR, int MO = 0>
NX_HD void fast_stages(const RunParams& p, const FastTable& T, const double* s, double h,
                       double* nx, double& fn, double* d, double& delta_f,
                       double* moon_end = nullptr, const double* hc = nullptr) {
  double K[6][3];                      // K_j = h * accel_j  (the only per-stage storage)
  const double hv0 = h * s[4], hv1 = h * s[5], hv2 = h * s[6];
  const double hGM = hc ? hc[56] : h * p.GM;
  double ms0 = 0.0, mc0 = 1.0, hGMm = 0.0, hGMi = 0.0, mx = 0.0, my = 0.0;
  if (MO) {
    const double phi0 = p.moon_phi[0] - p.moon_omega[0] * s[0];
#if defined(__CUDA_ARCH__)
    sincos(phi0, &ms0, &mc0);
#else
    ms0 = sin(phi0); mc0 = cos(phi0);
#endif
    hGMm = h * p.moon_GM[0];
    const double ai = 1.0 / p.moon_a[0];
    hGMi = hGMm * (ai * ai) * ai;
  }
  unsigned litmask = 0;
  int rec_hint = 0;                    // table record of the previous stage's lookup
  (void)rec_hint;
  double px = s[1], py = s[2], pz = s[3], vx = s[4], vy = s[5], vz = s[6];
#pragma unroll
  for (int n = 0; n < 6; ++n) {
    const double s2 = fma(pz, pz, px * px);
    // K_n = h * accel: h is folded into GM, the radiation term is scaled once
    double kx = 0.0, ky = 0.0, kz = 0.0;
    if (GR) {
      const double r2 = fma(py, py, s2);
      const double ri = rsqrt_h(r2);
      const double g = (hGM * ri) * (ri * ri);
      kx = g * px; ky = g * py; kz = g * pz;
      if (MO) {
        double sd, cd;
        sincos_small(p.moon_omega[0] * (dp_c(n) * h), sd, cd);
        const double sn = fma(ms0, cd, mc0 * sd), cs = fma(mc0, cd, -(ms0 * sd));
        mx = -p.moon_a[0] * sn; my = p.moon_a[0] * cs;
        const double dx = px - mx, dy = py - my;
        const double di = rsqrt_h(fma(pz, pz, fma(dy, dy, dx * dx)));
        const double gm = (hGMm * di) * (di * di);
        kx = fma(gm, dx, fma(hGMi, mx, kx));
        ky = fma(gm, dy, fma(hGMi, my, ky));
        kz = fma(gm, pz, kz);
      }
    }
    bool lit = true;
    if (RP || LOSS == LOSS_PHOTO)
      lit = (dbits(s2) > dbits(NX_ONE_PLUS_ULP)) || (dbits(py) < 0);   // s2 >= 0
    if (RP) {
      // adaptive kernels: stages 1-5 first try the record stage 0 ended in (K2 21.10 -> 21.00 ms,
      // the streaming kernel 24.6 -> 24.0 ms); the constant-step kernel, short of registers,
      // is faster with the plain lookup (2.49e10 against 2.47e10 packet-steps/s)
      const double ar = !ERR ? interp_fast(T, vy + p.vrplanet)
                        : n == 0 ? interp_fast_hint<false>(T, vy + p.vrplanet, rec_hint)
                                 : interp_fast_hint<true>(T, vy + p.vrplanet, rec_hint);
      ky = fma(lit ? h : 0.0, ar, ky);
    }
    if (LOSS == LOSS_PHOTO) litmask |= (lit ? 1u : 0u) << n;
    K[n][0] = kx; K[n][1] = ky; K[n][2] = kz;

    const int m = n + 1;
    const double cm = dp_c(m);
    double ap0 = fma(cm, hv0, s[1]), ap1 = fma(cm, hv1, s[2]), ap2 = fma(cm, hv2, s[3]);
    double av0 = s[4], av1 = s[5], av2 = s[6];
#pragma unroll
    for (int j = 0; j <= n; ++j) {
      if (!(m == 6 && j == 1)) {                       // b[1] = 0
        const double a = dp_a(m, j);
        av0 = fma(a, K[j][0], av0); av1 = fma(a, K[j][1], av1); av2 = fma(a, K[j][2], av2);
      }
      if (j < n) {
        const double ha2 = hc ? hc[m * 8 + j] : h * dp_a2(m, j);
        ap0 = fma(ha2, K[j][0], ap0); ap1 = fma(ha2, K[j][1], ap1); ap2 = fma(ha2, K[j][2], ap2);
      }
    }
    px = ap0; py = ap1; pz = ap2; vx = av0; vy = av1; vz = av2;
  }
  nx[0] = px; nx[1] = py; nx[2] = pz; nx[3] = vx; nx[4] = vy; nx[5] = vz;
  if (MO && moon_end) { moon_end[0] = mx; moon_end[1] = my; }     // stage 5 sits at tau - h

  // fractional content: dlogf = -h sum b_i rate_i ; error term h sum bd_i rate_i
  double sb = 0.0, sbd = 0.0;
  if (LOSS == LOSS_LIFETIME) {
    sb = p.loss_rate * kDpcBsum;
    sbd = p.loss_rate * kDpcBds;
  } else if (LOSS == LOSS_PHOTO) {
#pragma unroll
    for (int i = 0; i < 6; ++i) {
      if (i == 1) continue;
      const double r = (litmask >> i) & 1u ? p.loss_rate : 0.0;
      sb = fma(dp_a(6, i), r, sb);
      if (ERR) sbd = fma(dp_bd(i), r, sbd);
    }
  }
  fn = (LOSS == LOSS_NONE) ? s[7] : s[7] * exp_step(-(h * sb));
  if (ERR) {
    delta_f = fabs(h * sbd);
    const double bds = kDpcBds;
    double ep0 = bds * hv0, ep1 = bds * hv1, ep2 = bds * hv2;
    double ev0 = dp_bd(0) * K[0][0], ev1 = dp_bd(0) * K[0][1], ev2 = dp_bd(0) * K[0][2];
#pragma unroll
    for (int j = 0; j < 5; ++j) {
      const double hb = h * dp_bd2(j);
      ep0 = fma(hb, K[j][0], ep0); ep1 = fma(hb, K[j][1], ep1); ep2 = fma(hb, K[j][2], ep2);
    }
#pragma unroll
    for (int i = 2; i < 6; ++i) {
      const double b = dp_bd(i);
      ev0 = fma(b, K[i][0], ev0); ev1 = fma(b, K[i][1], ev1); ev2 = fma(b, K[i][2], ev2);
    }
    d[0] = fabs(ep0); d[1] = fabs(ep1); d[2] = fabs(ep2);
    d[3] = fabs(ev0); d[4] = fabs(ev1); d[5] = fabs(ev2);
  }
}

// One attempted adaptive step, fast arithmetic.  Same contract as
// adaptive_attempt<>(): s[0..7] = time,x,y,z,vx,vy,vz,frac; returns AttemptFlags.
// BOUNCE, S, seed, id, k, SINK, D, ION, I, TRACE, Tr: as in adaptive_attempt<>().
template <int GR, int RP, int LOSS, int MO = 0, bool BOUNCE = false, bool SINK = false,
          bool ION = false, bool TRACE = false>
NX_HD int adaptive_attempt_fast(const RunParams& p, const FastTable& T, double* s,
                                double& step, const Spline2D* S = nullptr, uint64_t seed = 0,
                                uint64_t id = 0, uint32_t k = 0, DepositSink* D = nullptr,
                                IonSink* I = nullptr, TraceSink* Tr = nullptr) {
  const double res = p.resolution;
  const double resv = 0.1 * res;
  const double h = fmin(s[0], step);
  double nx[6], d[6], fn, delta_f, moon_end[2] = {0.0, 0.0};
  fast_stages<GR, RP, LOSS, true, MO>(p, T, s, h, nx, fn, d, delta_f, moon_end);
  double px = nx[0], py = nx[1], pz = nx[2], vx = nx[3], vy = nx[4], vz = nx[5];
  // accept  <=>  every delta_j < scale_j  (== max_j fl(delta_j/scale_j) < 1).  The
  // quotient itself (Newton reciprocal, ~2^-40) only sizes the next step after a
  // reject and screens the "no error" case (Q4); it is formed for every lane so
  // that the warp does not split into an accept and a reject instruction stream.
  const double sf = fma(fabs(fn), res, res);
  bool ok = lt_nonneg(delta_f, sf);
  double errmax = delta_f * rcp_n(sf);
  double dsum = delta_f;
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    const double sp = fma(fabs(nx[k]), res, res);
    const double sv = fma(fabs(nx[3 + k]), resv, resv);
    ok = ok && lt_nonneg(d[k], sp) && lt_nonneg(d[3 + k], sv);
    errmax = max_nonneg(errmax, max_nonneg(d[k] * rcp_n(sp), d[3 + k] * rcp_n(sv)));
    dsum += d[k] + d[3 + k];
  }
  const bool tiny = errmax < 1e-7;                                   // quirk Q4
  const bool accept = ok && !tiny;

  // step-size update of a rejected attempt (reference Output.py:333-342)
  const double htried = tiny ? h * 10.0 : h;
  double e = errmax;
  if ((fn - s[7] > sf) && (errmax > 1.0)) e = 1.1;                  // quirk Q9
  if (tiny) e = 1.0;
  const double grow = rsqrt_h(e * rsqrt_h(e));                       // e^-0.25
  const double cand = (0.95 * htried) * grow;

  int flags = 0;
  if (!(dsum <= 1.7976931348623157e308)) flags |= ATT_BAD_ERRMAX;    // NaN / inf deltas
  if (accept) {
    if (ION) {                             // before a bounce moves the packet
      const double loss = s[7] - fn;
      if (loss != 0.0) ion_record(*I, loss, (s[1] + px) * 0.5, (s[2] + py) * 0.5, (s[3] + pz) * 0.5);
    }
    if (TRACE)
      trace_record(*Tr, (s[1] + px) * 0.5, (s[2] + py) * 0.5, (s[3] + pz) * 0.5, (s[5] + vy) * 0.5,
                   (s[7] + fn) * 0.5, h, s[0]);
    const double r2 = fma(pz, pz, fma(py, py, px * px));
    double f = fn;
    double dep = 0.0, ff = 0.0;            // SINK: deposited frac, frac of the fate event
    int fate = -1;
    if (fn < 0.0) flags |= ATT_NEG_FRAC;
    if (r2 < 1.0) {
      if (BOUNCE && !perfect_sticking(p)) {  // bounce, then K3's tests on the new state
        double b[8] = {0.0, px, py, pz, vx, vy, vz, fn};
        adaptive_surface<true>(p, *S, b, r2, seed, id, k);
        px = b[1]; py = b[2]; pz = b[3]; vx = b[4]; vy = b[5]; vz = b[6]; f = b[7];
        if (SINK) dep = fn - f;
        flags |= ATT_BOUNCED;
      } else {
        if (SINK) dep = fn;
        f = 0.0;                           // impact, stickcoef == 1 (Q6)
      }
    }
    if (MO) {                              // impact on the moon
      const double dx = px - moon_end[0], dy = py - moon_end[1];
      if (fma(pz, pz, fma(dy, dy, dx * dx)) < p.moon_r2[0]) {
        if (SINK && f != 0.0) { fate = DEP_MOON; ff = f; }
        f = 0.0;
      }
    }
    if (r2 > p.outeredge) {                // escape: r^2 vs outeredge (Q7)
      if (SINK && f != 0.0) { fate = DEP_ESCAPED; ff = f; }
      f = 0.0;
    }
    if (f < 1e-10) {                       // vanish (Q8)
      if (SINK && f != 0.0) { fate = DEP_VANISHED; ff = f; }
      f = 0.0;
    }
    if (SINK && (r2 < 1.0 || fate >= 0)) deposit_record(*D, r2 < 1.0, px, py, pz, dep, fate, ff);
    s[0] = (f == 0.0) ? 0.0 : s[0] - h;
    s[1] = px; s[2] = py; s[3] = pz; s[4] = vx; s[5] = vy; s[6] = vz;
    s[7] = f;
    flags |= ATT_ACCEPTED;
  } else {
    if (!(fabs(cand) <= 1.7976931348623157e308)) flags |= ATT_BAD_STEP;
    step = fmax(cand, 0.1 * htried);
  }
  if (s[0] > res && s[7] > 0.0) flags |= ATT_LIVE;
  return flags;
}

// runtime dispatch over the compile-time force / loss combinations
template <bool BOUNCE = false, bool SINK = false, bool ION = false, bool TRACE = false>
NX_HD int adaptive_attempt_fast_rt(const RunParams& p, const FastTable& T, double* s,
                                   double& step, const Spline2D* S = nullptr, uint64_t seed = 0,
                                   uint64_t id = 0, uint32_t k = 0,
                                   DepositSink* D = nullptr, IonSink* I = nullptr,
                                   TraceSink* Tr = nullptr) {
#define NX_ARGS p, T, s, step, S, seed, id, k, D, I, Tr
  if (p.nmoons == 1 && p.gravity) {
    if (p.radpres) {
      if (p.loss_mode == LOSS_PHOTO) return adaptive_attempt_fast<1, 1, LOSS_PHOTO, 1, BOUNCE, SINK, ION, TRACE>(NX_ARGS);
      if (p.loss_mode == LOSS_LIFETIME) return adaptive_attempt_fast<1, 1, LOSS_LIFETIME, 1, BOUNCE, SINK, ION, TRACE>(NX_ARGS);
      return adaptive_attempt_fast<1, 1, LOSS_NONE, 1, BOUNCE, SINK, ION, TRACE>(NX_ARGS);
    }
    if (p.loss_mode == LOSS_PHOTO) return adaptive_attempt_fast<1, 0, LOSS_PHOTO, 1, BOUNCE, SINK, ION, TRACE>(NX_ARGS);
    if (p.loss_mode == LOSS_LIFETIME) return adaptive_attempt_fast<1, 0, LOSS_LIFETIME, 1, BOUNCE, SINK, ION, TRACE>(NX_ARGS);
    return adaptive_attempt_fast<1, 0, LOSS_NONE, 1, BOUNCE, SINK, ION, TRACE>(NX_ARGS);
  }
  const int key = (p.gravity ? 4 : 0) | (p.radpres ? 2 : 0);
#define NX_CASE(G, R)                                                                    \
  if (key == ((G) * 4 + (R) * 2)) {                                                      \
    if (p.loss_mode == LOSS_PHOTO) return adaptive_attempt_fast<G, R, LOSS_PHOTO, 0, BOUNCE, SINK, ION, TRACE>(NX_ARGS);       \
    if (p.loss_mode == LOSS_LIFETIME) return adaptive_attempt_fast<G, R, LOSS_LIFETIME, 0, BOUNCE, SINK, ION, TRACE>(NX_ARGS); \
    return adaptive_attempt_fast<G, R, LOSS_NONE, 0, BOUNCE, SINK, ION, TRACE>(NX_ARGS);                     \
  }
  NX_CASE(1, 1) NX_CASE(1, 0) NX_CASE(0, 1) NX_CASE(0, 0)
#undef NX_CASE
#undef NX_ARGS
  return 0;
}

}  // namespace nx
