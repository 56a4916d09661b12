// TEST-ONLY: the adaptive driver with surface bounce (adaptive_attempt<.., true> and
// adaptive_attempt_fast<.., true>, the attempt functions k_integrate_adaptive<MODE, true> runs)
// compiled with g++ under the flags of hostcheck.cpp (no FMA contraction), so
// tests/test_adaptive_bounce.py can check it against the oracle on machines without a GPU.
// Never loaded by nexoclom_b200.
#include "../../nexoclom_b200/csrc/nx_physics.cuh"
#include "../../nexoclom_b200/csrc/nx_fast.cuh"
#include "../../nexoclom_b200/csrc/nx_tables.h"
#include "../../nexoclom_b200/csrc/nx_surface.cuh"

using namespace nx;

// X: n x 8 row-major, integrated in place from a 1000 s first step; att / acc / bnc: per
// packet attempted and accepted steps and bounces.  strict = 1: NumPy operation order, 0: the
// product's fast path.  Returns the status bits of the attempts.
extern "C" int hc_integrate_adaptive_bounce(long n, double* X, unsigned* att, unsigned* acc,
                                            unsigned* bnc, const RunParams* p, const double* rpv,
                                            const double* rpa, int nrp, const double* tx, int ntx,
                                            const double* ty, int nty, const double* c,
                                            unsigned long long seed, unsigned long long first_id,
                                            int strict) {
  HostInterp hi; InterpTable T{};
  HostFastTable hf; FastTable F{};
  if (nrp > 0) {
    hi = make_interp(rpv, rpa, nrp); T = {hi.x.data(), hi.f.data(), hi.slope.data(), hi.bucket.data(),
                                          (int)hi.x.size(), hi.nbucket, hi.blo, hi.binvw};
    hf = make_fast_table(rpv, rpa, nrp, 32768);
    F.rec = reinterpret_cast<const InterpRec*>(hf.rec.data()); F.bucket = hf.bucket.data();
    F.nrec = hf.nrec; F.nbucket = hf.nbucket; F.blo = hf.blo; F.binvw = hf.binvw; F.boff = -hf.blo * hf.binvw;
  }
  const Spline2D S{tx, ty, c, ntx, nty};
  int status = 0;
  for (long i = 0; i < n; ++i) {
    double* s = X + 8 * i;
    double step = 1000.0;
    att[i] = acc[i] = bnc[i] = 0;
    bool live = (s[0] > p->resolution) && (s[7] > 0.0);
    while (live) {
      const int fl = strict ? adaptive_attempt<true, true>(*p, T, s, step, &S, seed, first_id + i, acc[i] + 1)
                            : adaptive_attempt_fast_rt<true>(*p, F, s, step, &S, seed, first_id + i, acc[i] + 1);
      att[i]++;
      if (fl & ATT_ACCEPTED) acc[i]++;
      if (fl & ATT_BOUNCED) bnc[i]++;
      status |= fl & ~(ATT_ACCEPTED | ATT_LIVE | ATT_BOUNCED);
      live = fl & ATT_LIVE;
    }
  }
  return status;
}
