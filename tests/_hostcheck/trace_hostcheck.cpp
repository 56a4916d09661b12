// TEST-ONLY: the adaptive driver's trajectory sink (adaptive_attempt<.., TRACE = true> and
// adaptive_attempt_fast<.., TRACE = true>, the attempt functions k_trace_adaptive<MODE, BOUNCE>
// runs, and trace_record), compiled with g++ under the flags of hostcheck.cpp (no FMA
// contraction), so tests/test_trace.py can check them against the oracle on machines without a
// GPU.  Never loaded by nexoclom_b200.
#include <vector>

#include "../../nexoclom_b200/csrc/nx_physics.cuh"
#include "../../nexoclom_b200/csrc/nx_fast.cuh"
#include "../../nexoclom_b200/csrc/nx_tables.h"
#include "../../nexoclom_b200/csrc/nx_surface.cuh"
#include "../../nexoclom_b200/csrc/nx_image.cuh"

using namespace nx;

// X: n x 8 row-major, integrated in place from a 1000 s first step, packets in order (sums in
// packet order); the packets' initial times X[8 * i] are their t0.  bounce = 1: the bounce
// build (deviates keyed by seed, first_id + i).  strict = 1: NumPy operation order, 0: the
// fast path.  ip == NULL: no image, else image / image_cnt (ip->nx * ip->nz) are added to,
// radiance through the nt g-value tables (sizes, v, g concatenated), as the kernel reads them
// (record tables, no sum table).  ncell == NULL: no grid, else sum / cnt (the cells, then
// OUTSIDE) are added to.  Returns the status bits of the attempts.
extern "C" int hc_integrate_adaptive_trace(long n, double* X, unsigned* att, unsigned* acc,
                                           const RunParams* p, const double* rpv,
                                           const double* rpa, int nrp, const double* tx, int ntx,
                                           const double* ty, int nty, const double* c,
                                           unsigned long long seed, unsigned long long first_id,
                                           int strict, int bounce, const ImageParams* ip,
                                           int nt, const int* sizes, const double* gv,
                                           const double* gg, double* image,
                                           unsigned long long* image_cnt, const double* lo,
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
  TraceOut o{};
  o.endtime = p->endtime;
  std::vector<HostFastTable> gstore(nt > 0 ? nt : 0);
  if (ip) {
    o.img_sum = image; o.img_cnt = image_cnt;
    o.ip = *ip;
    o.is = image_steps(o.ip);
    o.G.n = nt;
    size_t off = 0;
    for (int t = 0; t < nt; ++t) {
      gstore[t] = make_fast_table(gv + off, gg + off, sizes[t], 256);
      FastTable& f = o.G.f[t];
      f.rec = reinterpret_cast<const InterpRec*>(gstore[t].rec.data()); f.bucket = gstore[t].bucket.data();
      f.nrec = gstore[t].nrec; f.nbucket = gstore[t].nbucket; f.blo = gstore[t].blo;
      f.binvw = gstore[t].binvw; f.boff = -gstore[t].blo * gstore[t].binvw;
      off += sizes[t];
    }
  }
  long long out = 0;
  if (ncell) {
    for (int a = 0; a < 3; ++a) { o.grid.lo[a] = lo[a]; o.grid.hi[a] = hi[a]; o.grid.n[a] = ncell[a]; }
    ion_steps(o.grid);
    o.grid.sum = sum; o.grid.cnt = cnt;
    out = (long long)ncell[0] * ncell[1] * ncell[2];
  }
  TraceSink Tr;
  Tr.o = &o;
  Tr.out_sum = ncell ? sum[out] : 0.0;
  Tr.out_n = ncell ? cnt[out] : 0;
  int status = 0;
  for (long i = 0; i < n; ++i) {
    double* s = X + 8 * i;
    double step = 1000.0;
    att[i] = acc[i] = 0;
    bool live = (s[0] > p->resolution) && (s[7] > 0.0);
    if (live) Tr.age0 = sub_rn(o.endtime, s[0]);
    while (live) {
      const uint64_t id = first_id + i;
      int fl;
      if (bounce)
        fl = strict ? adaptive_attempt<true, true, false, false, true>(*p, T, s, step, &S, seed, id, acc[i] + 1, nullptr, nullptr, &Tr)
                    : adaptive_attempt_fast_rt<true, false, false, true>(*p, F, s, step, &S, seed, id, acc[i] + 1, nullptr, nullptr, &Tr);
      else
        fl = strict ? adaptive_attempt<true, false, false, false, true>(*p, T, s, step, nullptr, 0, 0, 0, nullptr, nullptr, &Tr)
                    : adaptive_attempt_fast_rt<false, false, false, true>(*p, F, s, step, nullptr, 0, 0, 0, nullptr, nullptr, &Tr);
      att[i]++;
      if (fl & ATT_ACCEPTED) acc[i]++;
      status |= fl & ~(ATT_ACCEPTED | ATT_LIVE | ATT_BOUNCED);
      live = fl & ATT_LIVE;
    }
  }
  if (ncell) { sum[out] = Tr.out_sum; cnt[out] = Tr.out_n; }
  return status;
}
