// TEST-ONLY: the K7 membership predicate (nx_image.cuh: density_member) compiled with g++
// under the same flags as hostcheck.cpp (no FMA contraction), so tests/test_density.py can
// check it against NumPy bit for bit on machines without a GPU.  Never loaded by
// nexoclom_b200.
#include "../../nexoclom_b200/csrc/nx_physics.cuh"
#include "../../nexoclom_b200/csrc/nx_image.cuh"

using namespace nx;

// membership of n rows (float32 x, y, z) in one ball
extern "C" void hc_density_member(long n, const float* x, const float* y, const float* z,
                                  double px, double py, double pz, double r, uint8_t* member) {
  for (long i = 0; i < n; ++i) member[i] = density_member(x[i], y[i], z[i], px, py, pz, r) ? 1 : 0;
}
