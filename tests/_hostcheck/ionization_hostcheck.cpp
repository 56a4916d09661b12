// TEST-ONLY: the adaptive driver's ion-production sink (adaptive_attempt<.., ION = true> and
// adaptive_attempt_fast<.., ION = true>, the attempt functions k_ionize_adaptive<MODE, BOUNCE>
// runs) and the grid's bin helper, compiled with g++ under the flags of hostcheck.cpp (no FMA
// contraction), so tests/test_ionization.py can check them against the oracle on machines
// without a GPU.  Never loaded by nexoclom_b200.
#include "../../nexoclom_b200/csrc/nx_physics.cuh"
#include "../../nexoclom_b200/csrc/nx_fast.cuh"
#include "../../nexoclom_b200/csrc/nx_tables.h"
#include "../../nexoclom_b200/csrc/nx_surface.cuh"
#include "../../nexoclom_b200/csrc/nx_image.cuh"

using namespace nx;

static IonOut ion_grid(const double* lo, const double* hi, const int* n) {
  IonOut g{};
  for (int a = 0; a < 3; ++a) { g.lo[a] = lo[a]; g.hi[a] = hi[a]; g.n[a] = n[a]; }
  ion_steps(g);
  return g;
}

// Cell of (x, y, z) on the grid lo..hi in n[0] x n[1] x n[2] cells (ion_cell), -1 outside.
extern "C" long long hc_ion_cell(double x, double y, double z, const double* lo,
                                 const double* hi, const int* n) {
  return ion_cell(ion_grid(lo, hi, n), x, y, z);
}

// X: n x 8 row-major, integrated in place from a 1000 s first step, packets in order (sums in
// packet order).  bounce = 1: the bounce build (deviates keyed by seed, first_id + i), as
// nx_integrate_adaptive_ionize selects it for sticking != 1.  sum / cnt: the grid's
// n[0] * n[1] * n[2] cells then OUTSIDE, added to.  strict = 1: NumPy operation order, 0: the
// fast path.  Returns the status bits of the attempts.
extern "C" int hc_integrate_adaptive_ionize(long n, double* X, unsigned* att, unsigned* acc,
                                            const RunParams* p, const double* rpv,
                                            const double* rpa, int nrp, const double* tx, int ntx,
                                            const double* ty, int nty, const double* c,
                                            unsigned long long seed, unsigned long long first_id,
                                            int strict, int bounce, const double* lo,
                                            const double* hi, const int* ncell, double* sum,
                                            unsigned long long* cnt) {
  HostInterp hi_; InterpTable T{};
  HostFastTable hf; FastTable F{};
  if (nrp > 0) {
    hi_ = make_interp(rpv, rpa, nrp); T = {hi_.x.data(), hi_.f.data(), hi_.slope.data(), hi_.bucket.data(),
                                           (int)hi_.x.size(), hi_.nbucket, hi_.blo, hi_.binvw};
    hf = make_fast_table(rpv, rpa, nrp, 32768);
    F.rec = reinterpret_cast<const InterpRec*>(hf.rec.data()); F.bucket = hf.bucket.data();
    F.nrec = hf.nrec; F.nbucket = hf.nbucket; F.blo = hf.blo; F.binvw = hf.binvw; F.boff = -hf.blo * hf.binvw;
  }
  const Spline2D S{tx, ty, c, ntx, nty};
  IonSink I;
  I.g = ion_grid(lo, hi, ncell);
  I.g.sum = sum; I.g.cnt = cnt;
  const long long out = (long long)ncell[0] * ncell[1] * ncell[2];
  I.out_sum = sum[out]; I.out_n = cnt[out];
  int status = 0;
  for (long i = 0; i < n; ++i) {
    double* s = X + 8 * i;
    double step = 1000.0;
    att[i] = acc[i] = 0;
    bool live = (s[0] > p->resolution) && (s[7] > 0.0);
    while (live) {
      const uint64_t id = first_id + i;
      int fl;
      if (bounce)
        fl = strict ? adaptive_attempt<true, true, false, true>(*p, T, s, step, &S, seed, id, acc[i] + 1, nullptr, &I)
                    : adaptive_attempt_fast_rt<true, false, true>(*p, F, s, step, &S, seed, id, acc[i] + 1, nullptr, &I);
      else
        fl = strict ? adaptive_attempt<true, false, false, true>(*p, T, s, step, nullptr, 0, 0, 0, nullptr, &I)
                    : adaptive_attempt_fast_rt<false, false, true>(*p, F, s, step, nullptr, 0, 0, 0, nullptr, &I);
      att[i]++;
      if (fl & ATT_ACCEPTED) acc[i]++;
      status |= fl & ~(ATT_ACCEPTED | ATT_LIVE | ATT_BOUNCED);
      live = fl & ATT_LIVE;
    }
  }
  sum[out] = I.out_sum; cnt[out] = I.out_n;
  return status;
}
