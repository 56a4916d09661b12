// TEST-ONLY: the adaptive driver's deposition sink (adaptive_attempt<.., SINK = true> and
// adaptive_attempt_fast<.., SINK = true>, the attempt functions k_integrate_adaptive<MODE,
// BOUNCE, true> runs, with the kernel's SOURCE / REMAINING bookkeeping) and the map's bin
// helper, compiled with g++ under the flags of hostcheck.cpp (no FMA contraction), so
// tests/test_deposition.py can check them against the oracle on machines without a GPU.
// Never loaded by nexoclom_b200.
#include "../../nexoclom_b200/csrc/nx_physics.cuh"
#include "../../nexoclom_b200/csrc/nx_fast.cuh"
#include "../../nexoclom_b200/csrc/nx_tables.h"
#include "../../nexoclom_b200/csrc/nx_surface.cuh"
#include "../../nexoclom_b200/csrc/nx_image.cuh"

using namespace nx;

// Cell of (lon, lat) on the deposition map (deposit_cell), -1 outside.
extern "C" int hc_deposit_cell(double lon, double lat, int nlon, int nlat) {
  return deposit_cell(lon, lat, nlon, nlat);
}

// X: n x 8 row-major, integrated in place from a 1000 s first step, packets in order (sums in
// packet order).  bounce = 1: the bounce build (deviates keyed by seed, first_id + i), as
// nx_integrate_adaptive_deposit selects it for sticking != 1.  map / cnt: nlon x nlat, buckets /
// bucket_n: DEP_NBUCKET, all added to.  strict = 1: NumPy operation order, 0: the fast path.
// Returns the status bits of the attempts.
extern "C" int hc_integrate_adaptive_deposit(long n, double* X, unsigned* att, unsigned* acc,
                                             const RunParams* p, const double* rpv,
                                             const double* rpa, int nrp, const double* tx, int ntx,
                                             const double* ty, int nty, const double* c,
                                             unsigned long long seed, unsigned long long first_id,
                                             int strict, int bounce, int nlon, int nlat,
                                             double* map, unsigned long long* cnt, double* buckets,
                                             unsigned long long* bucket_n) {
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
  DepositSink D;
  D.map = map; D.cnt = cnt; D.nlon = nlon; D.nlat = nlat;
  for (int b = 0; b < DEP_NBUCKET; ++b) { D.sum[b] = buckets[b]; D.n[b] = bucket_n[b]; }
  int status = 0;
  for (long i = 0; i < n; ++i) {
    double* s = X + 8 * i;
    double step = 1000.0;
    att[i] = acc[i] = 0;
    bool live = (s[0] > p->resolution) && (s[7] > 0.0);
    if (s[7] > 0.0) { D.sum[DEP_SOURCE] += s[7]; ++D.n[DEP_SOURCE]; }
    while (live) {
      const uint64_t id = first_id + i;
      int fl;
      if (bounce)
        fl = strict ? adaptive_attempt<true, true, true>(*p, T, s, step, &S, seed, id, acc[i] + 1, &D)
                    : adaptive_attempt_fast_rt<true, true>(*p, F, s, step, &S, seed, id, acc[i] + 1, &D);
      else
        fl = strict ? adaptive_attempt<true, false, true>(*p, T, s, step, nullptr, 0, 0, 0, &D)
                    : adaptive_attempt_fast_rt<false, true>(*p, F, s, step, nullptr, 0, 0, 0, &D);
      att[i]++;
      if (fl & ATT_ACCEPTED) acc[i]++;
      status |= fl & ~(ATT_ACCEPTED | ATT_LIVE | ATT_BOUNCED);
      live = fl & ATT_LIVE;
    }
    if (s[7] > 0.0) { D.sum[DEP_REMAINING] += s[7]; ++D.n[DEP_REMAINING]; }
  }
  for (int b = 0; b < DEP_NBUCKET; ++b) { buckets[b] = D.sum[b]; bucket_n[b] = D.n[b]; }
  return status;
}
