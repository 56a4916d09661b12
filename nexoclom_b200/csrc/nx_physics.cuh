// nexoclom_b200 -- per-packet physics shared by every kernel.
//
// Everything here is a pure function of its arguments (NX_HD = __host__ __device__)
// so the SAME source is (a) inlined into the sm_100a kernels and (b) compiled by
// g++ into tests/_hostcheck (a test-only library used to debug logic on machines
// without a GPU; never loaded by the product).
//
// Arithmetic policy (template parameter STRICT):
//   STRICT = true : IEEE ops in the reference's NumPy operation order, no FMA
//                   contraction (reference rk5.py:31-36, state.py:19-36).
//   STRICT = false: FMA-contracted stage assembly, rsqrt-based gravity; differs
//                   from the reference by a few ulp per step (well inside the 1e-8
//                   gate, see DESIGN.md section 4).
#pragma once
#include <math.h>
#include <stdint.h>

#if defined(__CUDACC__)
#define NX_HD __host__ __device__ __forceinline__
#else
#define NX_HD inline
#endif

namespace nx {

// ---------------------------------------------------------------------------
// POD parameter blocks (mirrored by ctypes structures in nexoclom_b200/_lib.py)
// ---------------------------------------------------------------------------
enum LossMode { LOSS_NONE = 0, LOSS_LIFETIME = 1, LOSS_PHOTO = 2 };
enum StickType { STICK_CONSTANT = 0, STICK_TEMPERATURE = 1 };

#define NX_MAX_MOONS 4
struct RunParams {
  double GM;              // R_p^3 / s^2, NEGATIVE (reference SSObject.py:53)
  double vrplanet;        // R_p / s
  double loss_rate;       // LOSS_LIFETIME: 1/lifetime ; LOSS_PHOTO: photo rate [1/s]
  double outeredge;       // R_p (adaptive driver compares r^2 with it: quirk Q7)
  double resolution;      // adaptive tolerance (reference Options.resolution)
  double step_size;       // constant step [s]; 0 = adaptive
  double endtime;         // s
  double stickcoef;       // constant sticking coefficient
  double accomfactor;     // thermal accommodation factor (0 = none)
  double stick_A[3];      // T-dependent sticking  A0*exp(A1*T)+A2
  double surf_t1;         // 600 + 125 (cos(taa) - 1)/2  (surface_temperature.py:9)
  double planet_radius_km;
  double radpres_amax;    // max |a_rad| [R_p/s^2]; only orders the K2 work queue
  int32_t gravity;
  int32_t radpres;
  int32_t loss_mode;      // LossMode
  int32_t sticktype;      // StickType
  int32_t strict_math;    // 1 = STRICT kernels
  int32_t nmoons;         // moons whose gravity acts on the packets (0: the reference's case)
  // Moons on circular, prograde, equatorial orbits (extension: the reference asserts when the
  // planet has moons, Output.py:153-155; conventions of docs/nexoclom/inputfiles.rst:72-77).
  // Position at time-remaining tau: a (-sin phi, cos phi, 0), phi = moon_phi - moon_omega tau
  // (phi = 0: superior conjunction, pi/2: over the dawn terminator).
  double moon_GM[NX_MAX_MOONS];      // R_p^3/s^2, negative
  double moon_a[NX_MAX_MOONS];       // R_p
  double moon_omega[NX_MAX_MOONS];   // rad/s
  double moon_phi[NX_MAX_MOONS];     // rad, at the time of the observation (tau = 0)
  double moon_r2[NX_MAX_MOONS];      // (moon radius / R_p)^2: impact test
};

// np.interp table + slopes + a uniform bucket index that accelerates the search
// (the interval found is exactly the one numpy's binary search finds).
struct InterpTable {
  const double* x;
  const double* f;
  const double* slope;          // (f[j+1]-f[j])/(x[j+1]-x[j])
  const unsigned short* bucket; // largest j with x[j] <= blo + b/binvw
  int n;
  int nbucket;
  double blo;
  double binvw;
};

// bicubic tensor-product B-spline (scipy RectBivariateSpline tck)
struct Spline2D {
  const double* tx; const double* ty; const double* c;
  int ntx; int nty;            // number of knots; coefficient grid is (ntx-4) x (nty-4)
};

// ---------------------------------------------------------------------------
// rounding-controlled primitives
// ---------------------------------------------------------------------------
#if defined(__CUDA_ARCH__)
NX_HD double mul_rn(double a, double b) { return __dmul_rn(a, b); }
NX_HD double add_rn(double a, double b) { return __dadd_rn(a, b); }
NX_HD double sub_rn(double a, double b) { return __dsub_rn(a, b); }
NX_HD double div_rn(double a, double b) { return __ddiv_rn(a, b); }
NX_HD double rsqrt_fast(double a) { return rsqrt(a); }
#else
// host build is compiled with -ffp-contract=off
NX_HD double mul_rn(double a, double b) { return a * b; }
NX_HD double add_rn(double a, double b) { return a + b; }
NX_HD double sub_rn(double a, double b) { return a - b; }
NX_HD double div_rn(double a, double b) { return a / b; }
NX_HD double rsqrt_fast(double a) { return 1.0 / sqrt(a); }
#endif

template <bool STRICT> NX_HD double madd(double a, double b, double c) {
  if (STRICT) return add_rn(mul_rn(a, b), c);
  return fma(a, b, c);
}
template <bool STRICT> NX_HD double msub(double c, double a, double b) {  // c - a*b
  if (STRICT) return sub_rn(c, mul_rn(a, b));
  return fma(-a, b, c);
}

// r^3 correctly rounded (error-free products + one compensated sum).  NumPy's
// ``r**3`` goes through its SIMD pow, which equals the correctly rounded cube in
// ~95% of cases (and is off by 1 ulp otherwise) -- this is the closest
// deterministic stand-in (see DESIGN.md section 4).
NX_HD double cube_cr(double r) {
  double p = mul_rn(r, r);
  double e = fma(r, r, -p);
  double q = mul_rn(p, r);
  double e2 = fma(p, r, -q);
  return add_rn(q, add_rn(e2, mul_rn(e, r)));
}

// sqrt(x^2+z^2) > 1  <=>  x^2+z^2 > 1+2^-52 for correctly rounded sqrt.
#define NX_ONE_PLUS_ULP 1.0000000000000002
#define NX_PI 3.141592653589793
#define NX_TWO_PI 6.283185307179586

// ---------------------------------------------------------------------------
// np.interp (numpy/core/src/multiarray/compiled_base.c: arr_interp) semantics:
// clamped ends, exact-node shortcut, slope*(x-xj)+fj without FMA.
// ---------------------------------------------------------------------------
// index j with x[j] <= v < x[j+1] for x[0] <= v <= x[n-1] (j = n-1 iff v == x[n-1]):
// the bucket index bounds the search to [bucket[b], bucket[b+1]], a short
// bisection finishes it (what numpy's binary_search_with_guess returns).
NX_HD int interp_locate(const InterpTable& T, double v) {
  const int n = T.n;
  int b = (int)((v - T.blo) * T.binvw);
  b = b < 0 ? 0 : (b >= T.nbucket ? T.nbucket - 1 : b);
  int lo = T.bucket[b];
  int hi = (b + 1 < T.nbucket) ? (int)T.bucket[b + 1] + 1 : n - 1;
  if (lo > 0) --lo;                       // slack for the rounding of b
  if (hi > n - 1) hi = n - 1;
  while (lo > 0 && T.x[lo] > v) --lo;
  while (hi < n - 1 && T.x[hi] <= v) ++hi;
  // invariant: x[lo] <= v, and (v < x[hi] or hi == n-1)
  while (hi - lo > 1) {
    const int mid = (lo + hi) >> 1;
    if (T.x[mid] <= v) lo = mid; else hi = mid;
  }
  if (hi == n - 1 && T.x[hi] <= v) lo = hi;
  return lo;
}

NX_HD double interp(const InterpTable& T, double x) {
  const int n = T.n;
  if (x != x) return x;
  if (x > T.x[n - 1]) return T.f[n - 1];
  if (x < T.x[0]) return T.f[0];
  const int j = interp_locate(T, x);
  if (j == n - 1) return T.f[j];
  const double xj = T.x[j];
  if (xj == x) return T.f[j];
  return add_rn(mul_rn(T.slope[j], sub_rn(x, xj)), T.f[j]);
}

// Record-form table of the fast path (see nx_tables.h: make_fast_table).
struct InterpRec { double lo, hi, f, slope; };
struct FastTable {
  const InterpRec* rec;
  const unsigned short* bucket;
  int nrec, nbucket;
  double blo, binvw, boff;
};

// np.interp through the record table: bucket -> record, then at most two steps to the
// following records (guaranteed by the table builder, nx_tables.h); clamp records make
// the ends branch-free and pad records keep +inf in bounds.
// GLOBAL_BUCKET: the bucket index is known to live in global memory (read through the
// read-only path); false when it may have been staged in shared memory (K4's g tables).
template <bool GLOBAL_BUCKET = true>
NX_HD double interp_fast(const FastTable& T, double v) {
#if defined(__CUDA_ARCH__)
  int b = __double2int_rz(fma(v, T.binvw, T.boff));    // boff = -blo*binvw; NaN -> 0
  b = max(0, min(b, T.nbucket - 1));
  int idx = GLOBAL_BUCKET ? (int)__ldg(T.bucket + b)   // 64 KB index, L1-resident
                          : (int)T.bucket[b];
#else
  int b = (v == v) ? (int)fmax(fmin((v - T.blo) * T.binvw, 2e9), -2e9) : 0;
  b = b < 0 ? 0 : (b >= T.nbucket ? T.nbucket - 1 : b);
  int idx = T.bucket[b];
#endif
  InterpRec r = T.rec[idx];
  if (v >= r.hi) {                             // the bucket holds a node and v is past it
    r = T.rec[idx + 1];
    if (v >= r.hi) r = T.rec[idx + 2];         // ... a pair of near-coincident nodes
  }
  return fma(r.slope, v - r.lo, r.f);
}

// The same lookup with a hint: `idx` is the record the previous lookup of this packet ended in.
// The six stages of one step evaluate the table at nearly the same velocity, so the hinted
// record almost always still holds v: two compares replace the bucket arithmetic and the
// dependent index load.  The records partition the axis, so a hinted hit IS the record the
// full lookup would return (bit-identical results).  TRY_HINT = false: plain lookup that
// leaves its record in idx.
template <bool TRY_HINT>
NX_HD double interp_fast_hint(const FastTable& T, double v, int& idx) {
  InterpRec r;
  bool hit = false;
  if (TRY_HINT) {
    r = T.rec[idx];
    hit = (v >= r.lo) && (v < r.hi);
  }
  if (!hit) {
#if defined(__CUDA_ARCH__)
    int b = __double2int_rz(fma(v, T.binvw, T.boff));
    b = max(0, min(b, T.nbucket - 1));
    idx = (int)__ldg(T.bucket + b);
#else
    int b = (v == v) ? (int)fmax(fmin((v - T.blo) * T.binvw, 2e9), -2e9) : 0;
    b = b < 0 ? 0 : (b >= T.nbucket ? T.nbucket - 1 : b);
    idx = T.bucket[b];
#endif
    r = T.rec[idx];
    if (v >= r.hi) {
      r = T.rec[++idx];
      if (v >= r.hi) r = T.rec[++idx];
    }
  }
  return fma(r.slope, v - r.lo, r.f);
}

// ---------------------------------------------------------------------------
// RHS -- reference particle_tracking/state.py:17-74
// ---------------------------------------------------------------------------
NX_HD bool out_of_shadow(double x, double y, double z) {
  const double s = add_rn(mul_rn(x, x), mul_rn(z, z));
  return (s > NX_ONE_PLUS_ULP) || (y < 0.0);
}

// moon position / phase at time-remaining tau
NX_HD void moon_position(const RunParams& p, int m, double tau, double& mx, double& my) {
  const double phi = p.moon_phi[m] - p.moon_omega[m] * tau;
  mx = -p.moon_a[m] * sin(phi);
  my = p.moon_a[m] * cos(phi);
}

template <bool STRICT>
NX_HD void rhs(const RunParams& p, const InterpTable& T,
               double x, double y, double z, double vy,
               double& ax, double& ay, double& az, double& rate, double tau = 0.0) {
  if (p.gravity) {
    if (STRICT) {
      const double r2 = add_rn(add_rn(mul_rn(x, x), mul_rn(y, y)), mul_rn(z, z));
      const double r3 = cube_cr(sqrt(r2));
      ax = div_rn(mul_rn(p.GM, x), r3);
      ay = div_rn(mul_rn(p.GM, y), r3);
      az = div_rn(mul_rn(p.GM, z), r3);
    } else {
      const double r2 = fma(z, z, fma(y, y, x * x));
      const double ri = rsqrt_fast(r2);
      const double g = p.GM * (ri * ri) * ri;
      ax = g * x; ay = g * y; az = g * z;
    }
    // moons (state.py:5-10 docstring: sum over objects of GM (x - x_obj) / r_obj^3), in the
    // planet-centred frame: direct term + the planet's own acceleration towards the moon
    for (int m = 0; m < p.nmoons; ++m) {
      double mx, my;
      moon_position(p, m, tau, mx, my);
      const double dx = x - mx, dy = y - my;
      const double d2 = dx * dx + dy * dy + z * z;
      const double di = 1.0 / sqrt(d2);
      const double gd = p.moon_GM[m] * di * di * di;
      const double ai = 1.0 / p.moon_a[m];
      const double gi = p.moon_GM[m] * ai * ai * ai;
      ax += gd * dx + gi * mx;
      ay += gd * dy + gi * my;
      az += gd * z;
    }
  } else {
    ax = 0.0; ay = 0.0; az = 0.0;
  }
  bool lit = true;
  if (p.radpres || p.loss_mode == LOSS_PHOTO) lit = out_of_shadow(x, y, z);
  if (p.radpres) {
    const double vv = add_rn(vy, p.vrplanet);
    const double ar = mul_rn(interp(T, vv), lit ? 1.0 : 0.0);
    ay = add_rn(ay, ar);
  }
  if (p.loss_mode == LOSS_LIFETIME) rate = p.loss_rate;
  else if (p.loss_mode == LOSS_PHOTO) rate = lit ? p.loss_rate : 0.0;
  else rate = 0.0;
}

// ---------------------------------------------------------------------------
// Dormand-Prince 5(4) -- reference particle_tracking/rk5.py:5-54
// ---------------------------------------------------------------------------
struct DP {
  static NX_HD double c(int n) {
    switch (n) { case 1: return 0.2; case 2: return 0.3; case 3: return 0.8;
                 case 4: return 8. / 9.; case 5: return 1.; case 6: return 1.; default: return 0.; }
  }
  static NX_HD double a(int n, int i) {
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
  // bd = b - bs, evaluated in double exactly as NumPy does (rk5.py:10)
  static NX_HD double bd(int i) {
    switch (i) {
      case 0: return 35. / 384. - 5179. / 57600.;
      case 2: return 500. / 1113. - 7571. / 16695.;
      case 3: return 125. / 192. - 393. / 640.;
      case 4: return -2187. / 6784. - -92097. / 339200.;
      case 5: return 11. / 84. - 187. / 2100.;
      default: return 0.;
    }
  }
};

// Packet state: s[0]=time remaining, s[1..3]=pos, s[4..6]=vel, s[7]=frac.
// One DP step of size h.  out[] = new state (out[7] is frac, not log frac),
// delta[j] (j=0..6 for x,y,z,vx,vy,vz,log-frac) = |h * sum_{i<6} bd_i k_i| -- the
// 7th stage is NOT part of the estimate (quirk Q1).
template <bool STRICT, bool WANT_ERR>
NX_HD void dp_step(const RunParams& p, const InterpTable& T, const double* s, double h,
                   double* out, double* delta) {
  double kv[6][3], ka[6][3], kr[6];
  const double lf0 = log(s[7]);
  double px = s[1], py = s[2], pz = s[3], vx = s[4], vy = s[5], vz = s[6], lf = lf0;
#pragma unroll
  for (int n = 0; n < 6; ++n) {
    kv[n][0] = vx; kv[n][1] = vy; kv[n][2] = vz;
    rhs<STRICT>(p, T, px, py, pz, vy, ka[n][0], ka[n][1], ka[n][2], kr[n],
                p.nmoons ? s[0] - DP::c(n) * h : 0.0);
    double ap[3], av[3], af;
    {
      const double ha = mul_rn(h, DP::a(n + 1, 0));
#pragma unroll
      for (int k = 0; k < 3; ++k) { ap[k] = mul_rn(ha, kv[0][k]); av[k] = mul_rn(ha, ka[0][k]); }
      af = -mul_rn(ha, kr[0]);
    }
#pragma unroll
    for (int i = 1; i <= n; ++i) {
      if (DP::a(n + 1, i) == 0.) continue;          // b[1] = 0: adds exactly 0
      const double ha = mul_rn(h, DP::a(n + 1, i));
#pragma unroll
      for (int k = 0; k < 3; ++k) {
        ap[k] = madd<STRICT>(ha, kv[i][k], ap[k]);
        av[k] = madd<STRICT>(ha, ka[i][k], av[k]);
      }
      af = msub<STRICT>(af, ha, kr[i]);
    }
    px = add_rn(ap[0], s[1]); py = add_rn(ap[1], s[2]); pz = add_rn(ap[2], s[3]);
    vx = add_rn(av[0], s[4]); vy = add_rn(av[1], s[5]); vz = add_rn(av[2], s[6]);
    lf = add_rn(af, lf0);
  }
  out[0] = sub_rn(s[0], h);
  out[1] = px; out[2] = py; out[3] = pz; out[4] = vx; out[5] = vy; out[6] = vz;
  out[7] = exp(lf);
  if (WANT_ERR) {
    double dp[3], dv[3], df;
#pragma unroll
    for (int k = 0; k < 3; ++k) { dp[k] = mul_rn(DP::bd(0), kv[0][k]); dv[k] = mul_rn(DP::bd(0), ka[0][k]); }
    df = mul_rn(DP::bd(0), kr[0]);
#pragma unroll
    for (int i = 2; i < 6; ++i) {
#pragma unroll
      for (int k = 0; k < 3; ++k) {
        dp[k] = madd<STRICT>(DP::bd(i), kv[i][k], dp[k]);
        dv[k] = madd<STRICT>(DP::bd(i), ka[i][k], dv[k]);
      }
      df = madd<STRICT>(DP::bd(i), kr[i], df);
    }
#pragma unroll
    for (int k = 0; k < 3; ++k) { delta[k] = fabs(mul_rn(h, dp[k])); delta[3 + k] = fabs(mul_rn(h, dv[k])); }
    delta[6] = fabs(mul_rn(h, df));
  }
}

// ---------------------------------------------------------------------------
// One attempted step of the adaptive driver -- reference Output.py:249-353.
// Returns a bit mask.
// ---------------------------------------------------------------------------
enum AttemptFlags {
  ATT_ACCEPTED = 1,       // step accepted and state advanced
  ATT_LIVE = 2,           // packet still needs steps: (time > res) & (frac > 0)
  ATT_BAD_ERRMAX = 4,     // non-finite errmax            (reference assert :284)
  ATT_NEG_FRAC = 8,       // accepted negative frac        (reference assert :287)
  ATT_BAD_STEP = 16,      // non-finite / unchanged step   (reference asserts :337-339)
  ATT_BOUNCED = 256       // accepted step ended in a surface interaction (BOUNCE builds only;
                          // above the kernels' status bits, never reported as one)
};

// Surface interaction of an accepted adaptive step that ended inside the planet (r2 < 1),
// for BOUNCE builds of the attempt functions: K3's bounce (FAST: bounce_fast) with r =
// sqrt(r2) and the deviates uniform_pair(seed, id, STREAM_BOUNCE, 2k) and (.., 2k + 1), k = the
// packet's accepted steps counting this one.  s[1..7] is updated in place.  Defined in
// nx_surface.cuh; on the device it is an out-of-line call, so the rarely taken bounce (spline,
// trigonometry, Philox) adds neither registers nor instruction-cache footprint to the step loop.
#if defined(__CUDACC__)
#define NX_COLD __host__ __device__ __noinline__
#else
#define NX_COLD inline
#endif
template <bool FAST>
NX_COLD void adaptive_surface(const RunParams& p, const Spline2D& S, double* s, double r2,
                              uint64_t seed, uint64_t id, uint32_t k);

// Bounce inputs of the adaptive driver: everything but constant sticking of exactly 1.
NX_HD bool perfect_sticking(const RunParams& p) {
  return p.sticktype == STICK_CONSTANT && p.stickcoef == 1.0;
}

// Where the frac of the packets goes (SINK builds of the adaptive driver, ModelDeposition);
// the order of nx_deposit_bucket in nexoclom_b200.h.
enum DepositBucket {
  DEP_SURFACE = 0,        // deposited on the planet's surface (mapped)
  DEP_MOON = 1,           // hit a moon
  DEP_ESCAPED = 2,        // r^2 > outeredge (Q7)
  DEP_VANISHED = 3,       // frac < 1e-10 (Q8)
  DEP_REMAINING = 4,      // still in flight when the packet retires
  DEP_SOURCE = 5,         // initial frac > 0 of the packets handed to the kernel
  DEP_NBUCKET = 6
};

// One lane's deposition sink: the device map (nlon x nlat cells, longitude major) and this
// lane's bucket sums and counts, reduced when the kernel ends.
struct DepositSink {
  double* map;
  unsigned long long* cnt;
  int nlon, nlat;
  double sum[DEP_NBUCKET];
  unsigned long long n[DEP_NBUCKET];
};

// Records the events of one accepted step (SINK builds): surf = the step ended inside the
// planet, `dep` of frac deposited at the surface point (x, y, z) into the map and SURFACE;
// fate >= 0: the bucket that took the remaining frac ff (MOON, ESCAPED, VANISHED).  Defined in
// nx_surface.cuh, an out-of-line call like adaptive_surface().
template <class Sink>
NX_COLD void deposit_record(Sink& D, bool surf, double x, double y, double z, double dep,
                            int fate, double ff);

// The ion-production grid (ION builds of the adaptive driver, ModelIonization): n[0] x n[1] x
// n[2] cells, row-major, of f64 frac sums and u64 step counts, then one OUTSIDE slot (index
// n[0] * n[1] * n[2]) in each; per axis np.histogramdd's edges linspace(lo, hi, n + 1), with
// the bin widths and their reciprocals formed once per launch as ImageSteps does.
struct IonOut {
  double* sum;
  unsigned long long* cnt;
  double lo[3], hi[3], step[3], inv_step[3];
  int n[3];
};

// One lane's ion sink: the grid, and this lane's OUTSIDE sum and count, reduced when the
// kernel ends.
struct IonSink {
  IonOut g;
  double out_sum;
  unsigned long long out_n;
};

// Records the frac `loss` one accepted step lost in flight at its chord midpoint (x, y, z):
// one f64 and one u64 atomic add to its cell, or the lane's OUTSIDE slot (outside the box, or
// NaN).  Defined in nx_image.cuh, an out-of-line call like deposit_record().
template <class Sink>
NX_COLD void ion_record(Sink& I, double loss, double x, double y, double z);

// The trajectory sink (TRACE builds of the adaptive driver, ModelTrajectoryImage /
// ModelTrajectoryDensity): an image and / or a grid that every accepted step adds to, weighted
// by the time the packet spends on it.  TraceOut (nx_image.cuh) is the launch's image, grid and
// g-value tables; the lane keeps age0 = T - t0 of the packet it holds (T = endtime, t0 = its
// initial time remaining) and its OUTSIDE share of the grid, reduced when the kernel ends.
struct TraceOut;
struct TraceSink {
  const TraceOut* o;
  double age0;
  double out_sum;
  unsigned long long out_n;
};

// Records one accepted step of length h from time remaining t, at the midpoint (x, y, z, vy,
// frac) of the state before it and the Runge-Kutta state.  Defined in nx_image.cuh, an
// out-of-line call like ion_record().
template <class Sink>
NX_COLD void trace_record(Sink& Tr, double x, double y, double z, double vy, double frac,
                          double h, double t);

// BOUNCE = false: the reference's driver (a packet that hits the surface sticks, Q6).
// BOUNCE = true: accepted steps that end inside the planet go through adaptive_surface()
// unless the sticking is perfect; S / seed / id / k feed it (unused otherwise).
// SINK = true: every surface, moon, escape and vanish event goes to deposit_record(*D); the
// state the attempt computes is the same as without the sink.
// ION = true: every accepted step that changes the frac goes to ion_record(*I) with
// frac before - frac of the Runge-Kutta step, at the midpoint of the step's chord (before a
// bounce moves the packet); the state is again the same as without it.
// TRACE = true: every accepted step goes to trace_record(*Tr) with its length, the time
// remaining before it and the midpoint of the state before it and the Runge-Kutta state (each
// component (s + s_rk) * 0.5, before any surface, moon, escape or vanish handling).
template <bool STRICT, bool BOUNCE = false, bool SINK = false, bool ION = false,
          bool TRACE = false>
NX_HD int adaptive_attempt(const RunParams& p, const InterpTable& T, double* s, double& step,
                           const Spline2D* S = nullptr, uint64_t seed = 0, uint64_t id = 0,
                           uint32_t k = 0, DepositSink* D = nullptr, IonSink* I = nullptr,
                           TraceSink* Tr = nullptr) {
  const double res = p.resolution;
  const double resv = mul_rn(0.1, res);
  const double h = fmin(s[0], step);
  double nx[8], delta[7];
  dp_step<STRICT, true>(p, T, s, h, nx, delta);

  double errmax = 0.0;
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    const double sx = madd<true>(fabs(nx[1 + k]), res, res);
    const double sv = madd<true>(fabs(nx[4 + k]), resv, resv);
    errmax = fmax(errmax, div_rn(delta[k], sx));
    errmax = fmax(errmax, div_rn(delta[3 + k], sv));
  }
  const double sf = madd<true>(fabs(nx[7]), res, res);
  errmax = fmax(errmax, div_rn(delta[6], sf));

  int flags = 0;
  if (!(fabs(errmax) <= 1.7976931348623157e308)) flags |= ATT_BAD_ERRMAX;
  if (nx[7] < 0.0 && errmax < 1.0) flags |= ATT_NEG_FRAC;
  if ((sub_rn(nx[7], s[7]) > sf) && (errmax > 1.0)) errmax = 1.1;      // quirk Q9
  double htried = h;
  if (errmax < 1e-7) { errmax = 1.0; htried = mul_rn(h, 10.0); }       // quirk Q4
  if (errmax < 1.0) {
    if (ION) {
      const double loss = sub_rn(s[7], nx[7]);
      if (loss != 0.0)
        ion_record(*I, loss, mul_rn(add_rn(s[1], nx[1]), 0.5), mul_rn(add_rn(s[2], nx[2]), 0.5),
                   mul_rn(add_rn(s[3], nx[3]), 0.5));
    }
    if (TRACE)
      trace_record(*Tr, mul_rn(add_rn(s[1], nx[1]), 0.5), mul_rn(add_rn(s[2], nx[2]), 0.5),
                   mul_rn(add_rn(s[3], nx[3]), 0.5), mul_rn(add_rn(s[5], nx[5]), 0.5),
                   mul_rn(add_rn(s[7], nx[7]), 0.5), h, s[0]);
    const double r2 = add_rn(add_rn(mul_rn(nx[1], nx[1]), mul_rn(nx[2], nx[2])), mul_rn(nx[3], nx[3]));
    double f = nx[7];
    double dep = 0.0, ff = 0.0;            // SINK: deposited frac, frac of the fate event
    int fate = -1;
    if (r2 < 1.0) {
      if (BOUNCE && !perfect_sticking(p)) {  // bounce, then K3's tests on the new state
        adaptive_surface<false>(p, *S, nx, r2, seed, id, k);
        if (SINK) dep = f - nx[7];
        f = nx[7];
        flags |= ATT_BOUNCED;
      } else {
        if (SINK) dep = f;
        f = 0.0;                           // impact, stickcoef == 1 (Q6)
      }
    }
    for (int m = 0; m < p.nmoons; ++m) {   // impact on a moon (same rule, moon surface)
      double mx, my;
      moon_position(p, m, nx[0], mx, my);
      const double dx = nx[1] - mx, dy = nx[2] - my;
      if (dx * dx + dy * dy + nx[3] * nx[3] < p.moon_r2[m]) {
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
    if (SINK && (r2 < 1.0 || fate >= 0)) deposit_record(*D, r2 < 1.0, nx[1], nx[2], nx[3], dep, fate, ff);
    s[0] = (f == 0.0) ? 0.0 : nx[0];
#pragma unroll
    for (int k = 1; k < 7; ++k) s[k] = nx[k];
    s[7] = f;
    flags |= ATT_ACCEPTED;
  } else {
    const double old = htried;
    const double grow = STRICT ? pow(errmax, -0.25) : rsqrt_fast(sqrt(errmax));
    const double cand = mul_rn(mul_rn(0.95, old), grow);
    if (!(fabs(cand) <= 1.7976931348623157e308)) flags |= ATT_BAD_STEP;
    step = fmax(cand, mul_rn(0.1, old));
  }
  if (s[0] > res && s[7] > 0.0) flags |= ATT_LIVE;
  return flags;
}

}  // namespace nx
