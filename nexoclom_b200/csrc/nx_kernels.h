// Internal interface between the kernels (nx_kernels.cu) and the C ABI (nx_api.cu).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "nx_image.cuh"
#include "nx_init.cuh"
#include "nx_los.h"
#include "nx_physics.cuh"
#include "nx_surface.cuh"

// One 512-thread block per SM for the persistent integrators: the lookup tables are staged
// once per SM instead of four times (26.5 KB each), which leaves the L1 large enough for the
// 64 KB bucket index (measured K2, 1e7 packets: 4 x 128 threads 22.2 ms, 2 x 256 21.7, 1 x 512 21.3)
#ifndef NX_INT_THREADS
#define NX_INT_THREADS 512
#endif
#ifdef NX_INT_MINBLOCKS_OVERRIDE
#define NX_INT_MINBLOCKS NX_INT_MINBLOCKS_OVERRIDE
#else
#define NX_INT_MINBLOCKS 1
#endif
#define NX_LOS_THREADS 128

namespace nx {

struct StateCols { double* c[9]; };    // time,x,y,z,vx,vy,vz,frac,step_size
struct X0Cols { double* c[14]; };
// Device table K3 appends the rows of a constant-step run to (cursor == nullptr: no sink;
// cap == 0: count the rows only)
struct RowSink {
  double* cols;                  // 8 columns time..frac, stride `stride`
  unsigned* index;               // packet index of the row (within the launch)
  unsigned short* step;          // step number of the row
  unsigned long long* cursor;    // rows appended so far (may run past cap: overflow)
  unsigned long long cap;
  size_t stride;
  int skip_dead, to_f32;
};

// ---- K5 spatial culling (nx_los_grid.cu) ----
// Cell grid of K5.  Exospheric packets pile up near the planet (most of them end on its
// surface), so the grid is uniform in u = asinh(v / scale) per axis instead of in v:
// cell index = floor(G/2 + k * asinh(v / scale)); cells are scale/k wide at the origin and
// grow ~ |v| / k far out, where the cone of a line of sight is wide anyway.
struct LosGrid { int G; double half, scale, inv_scale, k; };
#define NX_LOS_GRID_MAX 160       // cells per axis the work arrays are allocated for
// packets in cell order: one 32-byte record (x, y, z, vy) per packet -- a candidate costs
// exactly one DRAM sector -- plus frac and the original index for the (rare) hits
struct LosSorted { double4* pos; double* frac; unsigned* idx; };
struct LosGridWork {
  int G = 128;                 // cells per axis of the current grid
  int G_fixed = 0;             // option "los_grid": > 0 pins G, 0 = sized from the packet count
  double scale = 1.0;          // R_p: where the asinh grid turns from uniform to logarithmic
  LosGrid grid{};
  LosSorted sorted{};
  unsigned *cell_id = nullptr, *count = nullptr, *start = nullptr, *block_sum = nullptr,
           *total = nullptr;
  unsigned long long* extent_bits = nullptr;
  long long cap = 0;
  // candidate (line of sight, sorted packet) pairs between k_los_candidates and k_los_resolve
  uint2* pairs = nullptr;
  unsigned long long pairs_cap = 0;
  unsigned long long* pair_cursor = nullptr;
  long long batch_hint = 0;    // lines of sight per batch that half-filled `pairs` last time
  unsigned long long pairs_cap_fixed = 0;   // option "los_pair_cap" (tests: force several batches)
};
// Doppler spectrum of the hits instead of the per-line sums (nx_los_spectrum): the exact test
// and the weight stay K5's; every hit adds its weight and 1 to column spectrum_column(v) of its
// line (row-major (nlos, nbins + 2)).  vx / vz are columns 4 and 6 of the packet table, read
// at the hit's row (vy is in the sorted record).
struct LosSpectrum {
  const double* vx;
  const double* vz;
  double vmin, vmax, step, vscale;
  int nbins;
  double* sum;
  unsigned long long* count;
};
cudaError_t launch_los_grid_build(cudaStream_t st, int device, StateCols P, long long n,
                                  const LosParams& lp, LosGridWork& w);
cudaError_t launch_los_grid(cudaStream_t st, LosGridWork& w, long long nlos,
                            const double* los, const double* dist_plan, const int* nball,
                            const double* ladder, const double* wid2, const LosParams& lp,
                            const LosConsts& lc, const GTables& G, double* radiance,
                            unsigned long long* npack, unsigned char* included,
                            unsigned long long* nused = nullptr, const long long* used_off = nullptr,
                            unsigned long long* used_cursor = nullptr, unsigned* used_idx = nullptr,
                            const unsigned* order = nullptr, unsigned long long* kept_pairs = nullptr,
                            const LosSpectrum* spec = nullptr);
cudaError_t launch_los_resolve(cudaStream_t st, LosGridWork& w, unsigned long long np, long long nlos,
                               const double* los, const double* dist_plan, const int* nball,
                               const double* ladder, const double* wid2, const LosParams& lp,
                               const LosConsts& lc, const GTables& G, double* radiance,
                               unsigned long long* npack, unsigned char* included,
                               unsigned long long* nused, const long long* used_off,
                               unsigned long long* used_cursor, unsigned* used_idx);

// K7 number density over the grid launch_los_grid_build made with round_f32 = 1 (F32
// records): pts SoA with stride npts, order = the points' processing order; box[6 * B],
// nitem[B], item_off[B + 1] scratch for B = min(npts, 2^20) points, cursor one u32.
// s1 / s2 / count are added to.
cudaError_t launch_density(cudaStream_t st, int device, const LosGridWork& w, long long npts,
                           const double* pts, const double* rad, const unsigned* order,
                           int* box, unsigned* nitem, unsigned* item_off, unsigned* cursor,
                           double* s1, double* s2, unsigned long long* count, int* nlaunch);
#define NX_DENSITY_BATCH (1 << 20)  // points per plan / scan / query round (item ids fit u32)

// per-call preparation of the lines of sight on the device (nx_los_grid.cu)
#define NX_LOS_KEY_BINS 32768
cudaError_t launch_los_prepare(cudaStream_t st, const double* los, long long nlos, double outeredge,
                               double* dd, unsigned* key, unsigned* hist,
                               unsigned long long* ddmax_bits);
cudaError_t launch_los_finish(cudaStream_t st, const double* dd, const double* ladder, int nladder,
                              long long nlos, int* nball, const unsigned* key, unsigned* hist,
                              unsigned* order);

size_t table_smem_bytes(const InterpTable& g);

cudaError_t launch_init_state(cudaStream_t st, X0Cols X, long long n,
                              const SourceParams& sp, const SourceMap& map,
                              const InterpTable& speed, const InterpTable& lon1d, uint64_t seed,
                              uint64_t first_id, bool fast);
// deviate columns: u_time, u_sinlat, u_lon, lon_in, lat_in (both null: uniform band), u_speed,
// z_normal, u_alt, u_az
cudaError_t launch_init_from_deviates(cudaStream_t st, X0Cols X, long long n,
                                      const SourceParams& sp, const InterpTable& speed,
                                      const InterpTable& lon1d, const double* const* dev);
cudaError_t launch_fill(cudaStream_t st, double* p, long long n, double v);
cudaError_t launch_image_finish(cudaStream_t st, const double* img, const unsigned long long* cnt,
                                double scale, double* img_out, double* cnt_out, long long npix);
cudaError_t launch_cost_order(cudaStream_t st, int device, StateCols P, long long n,
                              const RunParams& p, int model, unsigned char* bucket,
                              unsigned* hist_cursor, unsigned* perm, bool to_surface = true);
// Deposition sink of K2 (nx_integrate_adaptive_deposit): the nlon x nlat map (f64 sums and
// u64 counts, longitude major) and the DEP_NBUCKET bucket sums and counts, all device memory
// the kernel adds to.
struct DepositOut {
  double* map;
  unsigned long long* cnt;
  double* bucket;
  unsigned long long* bucket_n;
  int nlon, nlat;
};
// In: columns the initial state is read from (X0 slab right after K1, else == P).
// S != nullptr: packets bounce (totals[2] counts the bounces), deviates keyed by
// (seed, first_id + packet index); nullptr: the reference's driver (Q6).
// dep != nullptr: the same run through the kernel's SINK build, which adds its events to *dep.
// ion != nullptr (dep == nullptr, a run with a loss term): the same run through
// k_ionize_adaptive, which adds the frac lost in flight to the grid *ion.
// trace != nullptr (the others nullptr, a run without moons): the same run through
// k_trace_adaptive, which adds every accepted step to the image and / or grid of *trace.
cudaError_t launch_integrate_adaptive(cudaStream_t st, int device, StateCols In, StateCols P,
                                      long long n, const RunParams& p, const InterpTable& T,
                                      const FastTable& F, const unsigned* perm,
                                      unsigned long long* queue, unsigned long long* totals,
                                      unsigned* att, unsigned* acc, int* status,
                                      const Spline2D* S = nullptr, uint64_t seed = 0,
                                      uint64_t first_id = 0, const DepositOut* dep = nullptr,
                                      const IonOut* ion = nullptr,
                                      const TraceOut* trace = nullptr);
#define NX_STREAM_GROUP 128          // == NX_GROUP: segment sizes are multiples of this
#define NX_STREAM_MAX_SEG 32
#define NX_STREAM_CURSORS 256        // >= NX_NCLASS x 32 u64 cursors
cudaError_t debug_begin(cudaStream_t st);                       // no-ops unless NX_STREAM_DEBUG
cudaError_t debug_read(unsigned long long* out, int count);
// in0/in_stride: the 8 immutable input columns (time..frac); P: where the final state goes;
// cls: nullptr, or one byte per packet (padded to 32) preset to 0xFF -- the cost class is
// computed by the first pass that meets a packet and read back by the later ones
cudaError_t launch_integrate_adaptive_stream(cudaStream_t st, int device, const double* in0,
                                             size_t in_stride, double step0, StateCols P,
                                             long long n, const RunParams& p,
                                             const InterpTable& T, const FastTable& F,
                                             long long seg, int nseg, int model,
                                             unsigned long long* cursor, const unsigned* arrived,
                                             unsigned char* cls, unsigned long long* totals,
                                             unsigned* att, unsigned* acc, int* status);
cudaError_t launch_integrate_constant(cudaStream_t st, int device, StateCols In, StateCols P,
                                      long long n, const RunParams& p, const InterpTable& T,
                                      const FastTable& F,
                                      const Spline2D& S, uint64_t seed, uint64_t first_id,
                                      int nsteps, const ImageParams& ip, const GTables& G,
                                      double* image, unsigned long long* counts, double* traj,
                                      const RowSink& rows,
                                      unsigned long long* queue, unsigned long long* totals,
                                      int* status);
cudaError_t launch_image_accumulate(cudaStream_t st, int device, StateCols P, long long n,
                                    const ImageParams& ip, const GTables& G, double* image,
                                    unsigned long long* counts, int mode = 0);
// Velocity axis of an image cube (ModelImageCube): edges = linspace(vmin, vmax, nbins + 1),
// step = (vmax - vmin) / nbins, vscale = R_p in km; cell = pixel * (nbins + 2) + column
struct CubeAxis {
  double vmin, vmax, step, vscale;
  int nbins;
};
cudaError_t launch_image_cube(cudaStream_t st, int device, StateCols P, long long n,
                              const ImageParams& ip, const GTables& G, const CubeAxis& ax,
                              double* cube, unsigned long long* counts);
cudaError_t launch_los_accumulate(cudaStream_t st, int device, StateCols P, long long n,
                                  long long nlos, const double* los, const double* dist_plan,
                                  const int* nball, const double* ladder, const double* wid2,
                                  const LosParams& lp, const LosConsts& lc, const GTables& G,
                                  double* radiance, unsigned long long* npack,
                                  unsigned char* included);
// ---- K6 source maps (nx_source_map.cu) ----
struct SourceMapParams {
  double smear;            // smear_radius [rad]
  double vmax;             // ceil(max speed) [km/s]
  int32_t nlon, nlat, nvel, nalt, naz;
  int32_t weight_is_frac;  // todo == 'source': weight = X0.frac; 'available': weight = 1
};
struct SourceMapOut {
  double *abundance_hist;                 // [nlon][nlat]   np.histogram2d of the included packets
  double *speed_dist, *altitude_dist, *azimuth_dist;     // whole-planet histograms
  unsigned long long *n_included, *n_total;              // [nlon*nlat]
  double *abundance;                      // [nlon*nlat]    smeared: sum of weights in the ball
  double *speed_map, *altitude_map, *azimuth_map;        // [nlon*nlat][nbins]
};
cudaError_t launch_source_map(cudaStream_t st, long long n, const SourceMapParams& sp,
                              const double* lon, const double* lat, const double* v,
                              const double* alt, const double* az, const double* frac,
                              const double* plon, const double* plat, const double* pcos,
                              const double* pthr, const SourceMapOut& out);

cudaError_t launch_fp64_peak(cudaStream_t st, int device, double* out, int iters, int* blocks,
                             int* threads);
cudaError_t launch_copy(cudaStream_t st, int device, const double* src, double* dst,
                        long long n);

}  // namespace nx

namespace nx {
// ---- device-side Output.save: stable compaction + f32 rounding (nx_compact.cu) ----
long long compact_tiles(long long n);
cudaError_t launch_compact_count(cudaStream_t st, const double* frac, long long n, int skip_dead,
                                 unsigned* tile_count, unsigned long long* total);
cudaError_t launch_compact_scatter(cudaStream_t st, StateCols P, long long n, int skip_dead,
                                   int to_f32, int have_step, const unsigned* tile_offset,
                                   double* out, size_t out_stride, unsigned* index);
cudaError_t launch_to_f32(cudaStream_t st, const double* src, size_t src_stride, long long n,
                          int ncols, float* dst);
}  // namespace nx
