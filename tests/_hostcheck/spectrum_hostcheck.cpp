// TEST-ONLY: the Doppler velocity and spectrum column of LOSSpectrum (nx_image.cuh: los_doppler,
// spectrum_column) compiled with g++ under the same flags as hostcheck.cpp (no FMA
// contraction), so tests/test_spectrum.py can check them against NumPy bit for bit on machines
// without a GPU.  Never loaded by nexoclom_b200.
#include "../../nexoclom_b200/csrc/nx_physics.cuh"
#include "../../nexoclom_b200/csrc/nx_image.cuh"

using namespace nx;

// velocity of n rows (float32 vx, vy, vz) along one boresight
extern "C" void hc_los_doppler(long n, const float* vx, const float* vy, const float* vz, double bx,
                               double by, double bz, double vscale, double* v) {
  for (long i = 0; i < n; ++i) v[i] = los_doppler(vx[i], vy[i], vz[i], bx, by, bz, vscale);
}

// spectrum column of n velocities, step as nx_los_spectrum computes it
extern "C" void hc_spectrum_column(long n, const double* v, double vmin, double vmax, int nbins,
                                   int32_t* col) {
  const double step = (vmax - vmin) / nbins;
  for (long i = 0; i < n; ++i) col[i] = spectrum_column(v[i], nbins, vmin, vmax, step);
}
