/* nexoclom_b200 -- C ABI of the B200-native nexoclom hot path.
 *
 * The reference (mburger-stsci/nexoclom v3.7.4) is pure Python and has no FFI
 * layer; each entry point below replaces the body of a Python function that
 * takes plain ndarrays, and is bound from Python with ctypes
 * (nexoclom_b200/_lib.py; the stub a reference maintainer would add is shown
 * in INTEGRATION.md).  Citations are relative to the reference tree.
 *
 * Conventions
 *   - every function returns 0 on success; < 0 = CUDA error (message via
 *     nx_last_error); > 0 = violated numerical invariant (bit mask, see
 *     NX_INV_*), mirroring the reference's bare `assert`s.
 *   - host buffers are caller-owned, contiguous, little-endian f64 / i64 / u8;
 *     packet tables are structure-of-arrays: one pointer per column.
 *   - `*_dev` variants take DEVICE pointers (e.g. torch tensors' data_ptr())
 *     for results that stay on the GPU for a following NCCL all-reduce.
 *   - one nx_ctx per (process, GPU); calls on a ctx are serialised by the
 *     caller; the library keeps no global mutable state.
 *   - units: length = planet radii, time = s, GM < 0, Sun at -y.
 */
#ifndef NEXOCLOM_B200_H
#define NEXOCLOM_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct nx_ctx nx_ctx;
typedef struct nx_packets nx_packets;   /* a compacted packet table resident on the GPU   */
typedef struct nx_comm nx_comm;         /* the ranks of one sharded run (NCCL communicator) */

/* invariant bits (positive return values / nx_status) */
#define NX_INV_BAD_ERRMAX 4   /* non-finite errmax        (Output.py:284)      */
#define NX_INV_NEG_FRAC   8   /* accepted negative frac   (Output.py:287-288)  */
#define NX_INV_BAD_STEP   16  /* non-finite step size     (Output.py:337-339)  */
#define NX_INV_BAD_STATE  32  /* non-finite packet state  (Output.py:388-389)  */
#define NX_INV_STARVED    64  /* host-buffer path: a segment never arrived (20 s watchdog) */
#define NX_INV_NO_PROGRESS 128 /* adaptive driver: a packet used 2^22 attempted steps; the
                                 reference's loop (Output.py:248-353) would never end   */

/* packet-state columns (Output.py:247, :370) */
enum { NX_COL_TIME = 0, NX_COL_X, NX_COL_Y, NX_COL_Z, NX_COL_VX, NX_COL_VY, NX_COL_VZ,
       NX_COL_FRAC, NX_NCOL_STATE };
/* X0 columns (Output.py:180-182) */
enum { NX_X0_TIME = 0, NX_X0_X, NX_X0_Y, NX_X0_Z, NX_X0_VX, NX_X0_VY, NX_X0_VZ, NX_X0_FRAC,
       NX_X0_V, NX_X0_LONGITUDE, NX_X0_LATITUDE, NX_X0_LOCAL_TIME, NX_X0_ALTITUDE,
       NX_X0_AZIMUTH, NX_NCOL_X0 };

/* Per-run scalars (what Output.__init__ builds, Output.py:102-133). */
typedef struct nx_run_params {
  double GM;               /* R_p^3/s^2, negative (SSObject.py:53)                 */
  double vrplanet;         /* R_p/s (planet_dist.py:67)                            */
  double loss_rate;        /* loss_mode 1: 1/lifetime; 2: photo rate (LossInfo.py) */
  double outeredge;        /* Options.outeredge                                    */
  double resolution;       /* Options.resolution (adaptive)                        */
  double step_size;        /* Options.step_size; 0 = adaptive                      */
  double endtime;          /* Options.endtime [s]                                  */
  double stickcoef;        /* SurfaceInteraction.stickcoef                         */
  double accomfactor;      /* SurfaceInteraction.accomfactor                       */
  double stick_A[3];       /* SurfaceInteraction.A (temperature dependent)         */
  double surf_t1;          /* 600+125(cos taa-1)/2 (surface_temperature.py:9)      */
  double planet_radius_km;
  double radpres_amax;     /* max |radiation accel| of the table (scheduling heuristic only) */
  int32_t gravity, radpres;
  int32_t loss_mode;       /* 0 none, 1 constant lifetime, 2 photo x sunlit        */
  int32_t sticktype;       /* 0 constant, 1 temperature dependent                  */
  int32_t strict_math;     /* 1: NumPy operation order without FMA contraction     */
  int32_t nmoons;          /* 0 = the reference's case (it asserts for planets with moons,
                              Output.py:153-155); > 0: extension, see DESIGN.md           */
  /* moons on circular prograde equatorial orbits; position at time-remaining tau:
     a (-sin phi, cos phi, 0), phi = moon_phi - moon_omega tau (inputfiles.rst:72-77)      */
  double moon_GM[4];       /* R_p^3/s^2, negative                                       */
  double moon_a[4];        /* R_p                                                        */
  double moon_omega[4];    /* rad/s                                                      */
  double moon_phi[4];      /* rad at the time of the observation                         */
  double moon_r2[4];       /* (moon radius / R_p)^2                                      */
} nx_run_params;

/* Initial-state distributions (source_distribution.py:37-283). */
enum { NX_SPATIAL_UNIFORM = 0, NX_SPATIAL_MAP = 1, NX_SPATIAL_LON1D = 2 };
enum { NX_SPEED_FLAT = 0, NX_SPEED_GAUSSIAN = 1, NX_SPEED_TABLE = 2 };
enum { NX_ANGULAR_RADIAL = 0, NX_ANGULAR_ISOTROPIC = 1, NX_ANGULAR_2D = 2 };
typedef struct nx_source_params {
  int32_t spatial_type, speed_type, angular_type, is_planet;
  double exobase;
  double sinlat0, sinlat1;   /* uniform: sin(latitude) range                        */
  double lon0, lon1;         /* uniform: longitude range (lon1 > lon0, may be > 2pi) */
  double vprob, vsigma, delv;/* km/s                                                */
  double v_scale;            /* km/s -> R_p/s  (1/R_km)                             */
  double sinalt0, sinalt1;   /* isotropic: sin(altitude) range; 2d: cos(altitude)   */
  double az0, az1;           /* isotropic: azimuth range                            */
  double endtime;
  int32_t random_time;       /* 1: time = U*endtime (adaptive); 0: time = endtime   */
  int32_t map_nx, map_ny;    /* source map grid (surface map / surface spot)        */
  int32_t map_lat_is_sin;    /* 1: y-axis is sin(lat) (surface map); 0: lat (spot)  */
  double map_fmax;
  int32_t start_is_moon;     /* extension: StartPoint is a moon (see nx_run_params)      */
  int32_t reserved;
  double moon_a, moon_omega, moon_phi, moon_radius;   /* R_p, rad/s, rad, R_p            */
} nx_source_params;

/* Image accumulation (ModelImage.py:229-274). */
typedef struct nx_image_params {
  double M[9];               /* row-major rotation Sun frame -> observer frame      */
  double x0, x1, z0, z1;     /* image range [R_p]                                   */
  double apix;               /* pixel area [cm^2]; weights are divided by it        */
  double vrplanet;           /* R_p/s                                               */
  int32_t nx, nz;
  int32_t quantity;          /* 0 column, 1 radiance                                */
  int32_t round_f32;         /* 1: round x,y,z,vy,frac to f32 first (Output.save)   */
  int32_t skip_dead;         /* 1: ignore frac == 0 packets (compress=True)         */
  int32_t reserved;
} nx_image_params;

/* Line-of-sight accumulation (compute_iteration.py:90-240). */
typedef struct nx_los_params {
  double dphi;               /* cone half-angle [rad], finite, > 0 and < pi/2       */
  double outeredge;          /* R_p                                                 */
  double vrplanet;           /* R_p/s                                               */
  double rp_cm;              /* planet radius [cm]                                  */
  int32_t quantity;          /* 1 radiance (only one the reference supports)        */
  int32_t round_f32;
  int32_t skip_dead;
  int32_t reserved;
} nx_los_params;

/* ---- context ---------------------------------------------------------------- */
int nx_ctx_create(int device, nx_ctx** out);
int nx_ctx_destroy(nx_ctx* ctx);
/* adopt a caller-owned cudaStream_t (e.g. torch.cuda.current_stream().cuda_stream) */
int nx_ctx_set_stream(nx_ctx* ctx, void* cuda_stream);
/* the cudaStream_t the context enqueues on (its own, or the adopted one) */
int nx_ctx_stream(nx_ctx* ctx, void** cuda_stream);
int nx_ctx_sync(nx_ctx* ctx);
/* tuning switches: "order_packets" (cost model of the K2 work queue: 0 natural order,
 * 1 ballistic flight time (default), 2 + radiation-pressure perturbation);
 * "schedule" (host-buffer path: 1 one streaming class-ordered kernel (default), 0 one
 * sort + kernel per chunk; 2 = developer mode, streaming kernel over the resident X0);
 * "class_cache" (streaming kernel: 1 keep each packet's cost class between passes (default));
 * "los_mode" (0 auto, 1 brute force, 2 cell grid); "los_grid" (cells per axis)         */
int nx_ctx_set_option(nx_ctx* ctx, const char* name, int value);
const char* nx_last_error(nx_ctx* ctx);
int nx_status(nx_ctx* ctx, int* invariant_bits);

/* ---- tables (replaces the table objects Output.__init__ attaches:
 *      self.radpres, self.loss_info, self.surfaceint; Output.py:113-133) ------- */
int nx_tables_upload(nx_ctx* ctx, const nx_run_params* p,
                     const double* radpres_v, const double* radpres_a, int n_radpres,
                     const double* spl_tx, int ntx, const double* spl_ty, int nty,
                     const double* spl_c);
/* g-value tables for radiance weighting (ModelResult.py:152-161): `ntables`
 * tables concatenated in v[] / g[] with lengths sizes[]; v in R_p/s.            */
int nx_gtables_upload(nx_ctx* ctx, int ntables, const int* sizes,
                      const double* v, const double* g);

/* ---- packets ------------------------------------------------------------------ */
int nx_packets_resize(nx_ctx* ctx, long long n);
/* import mode: reference-generated initial state, cols[8] = time,x,y,z,vx,vy,vz,frac */
int nx_import_state(nx_ctx* ctx, long long n, const double* const* cols);
int nx_export_state(nx_ctx* ctx, long long n, double* const* cols);
int nx_export_x0(nx_ctx* ctx, long long n, double* const* cols /* NX_NCOL_X0 */);
int nx_export_stats(nx_ctx* ctx, long long n, uint32_t* attempted, uint32_t* accepted);
int nx_export_step(nx_ctx* ctx, long long n, double* step_size);
int nx_state_device_ptr(nx_ctx* ctx, int column, void** dev_ptr);

/* ---- K1: initial state (source_distribution.py:37-283, Output.py:136-147) ---- */
int nx_sourcemap_upload(nx_ctx* ctx, const double* fmap, int nx, int ny,
                        const double* xaxis, const double* yaxis);
int nx_speedtable_upload(nx_ctx* ctx, const double* cdf, const double* v, int n);
/* inverse CDF of a longitude-only source map (source_distribution.py:72-76 ->
 * random_deviates_1d, randomdeviates.py:29-33): spatial_type NX_SPATIAL_LON1D           */
int nx_lontable_upload(nx_ctx* ctx, const double* cdf, const double* lon, int n);
/* Draws n packets with global ids [first_id, first_id + n) into the context's X0 columns
 * (112 B per packet).  The packets' current state IS X0[0:8] until an integrator has run;
 * nx_export_state / nx_state_device_ptr / K4 / K5 materialise a copy on demand.          */
int nx_init_state(nx_ctx* ctx, const nx_source_params* sp, uint64_t seed,
                  uint64_t first_id, long long n);
/* Import mode for reference-generated DEVIATES: the same deviate -> state transform as
 * nx_init_state (source_distribution.py:47-62, 137-283) on caller-supplied host columns of
 * length n.  lon_in / lat_in: surface points sampled elsewhere (map rejection sampling), or
 * both NULL for the uniform band drawn from u_sinlat / u_lon; unused deviates may be NULL. */
int nx_init_state_deviates(nx_ctx* ctx, const nx_source_params* sp, long long n,
                           const double* u_time, const double* u_sinlat, const double* u_lon,
                           const double* lon_in, const double* lat_in, const double* u_speed,
                           const double* z_normal, const double* u_alt, const double* u_az);
/* Make the resident initial state (X0[0:8], from nx_init_state or the host-buffer path) the
 * packets' current state again, without copying: the next integrator call re-runs it.      */
int nx_rewind_state(nx_ctx* ctx);

/* ---- K2: adaptive driver (Output.py:221-366 + rk5.py + state.py) ------------- */
int nx_integrate_adaptive(nx_ctx* ctx, long long n,
                          unsigned long long* attempted_steps,
                          unsigned long long* accepted_steps);

/* End-to-end variant: imports `cols` (8 host columns time..frac, ideally pinned) and
 * integrates them while they are still arriving: the copy engine delivers the packets
 * in `nchunks` (<= 32) segments behind ONE persistent kernel that consumes every
 * segment as soon as it is resident, longest packets first.  The imported initial
 * state stays in the context's X0 columns (nx_export_x0, columns 0-7), the final state
 * goes to the state columns.  Same results as nx_import_state + nx_integrate_adaptive
 * (bit-identical; reference Output.py:180-182 + 221-366 on imported X0).              */
int nx_integrate_adaptive_host(nx_ctx* ctx, long long n, const double* const* cols, int nchunks,
                               unsigned long long* attempted_steps,
                               unsigned long long* accepted_steps);

/* K2 with surface bounce (an extension: the reference's adaptive driver asserts 'Not set up'
 * unless stickcoef == 1, Output.py:309-315).  An accepted step that ends inside the planet
 * goes through K3's surface interaction (bouncepackets.py: back-trace to r = 1, rebound speed,
 * cosine-law direction, accommodation, constant or temperature-dependent sticking) with the
 * deviates uniform_pair(seed, first_id + i, STREAM_BOUNCE, 2k) and (.., 2k + 1), k = the
 * packet's accepted steps counting this one; then moon impact, escape (r^2 > outeredge),
 * vanish and time = 0 for a dead packet as in K3.  Results do not depend on the launch
 * geometry, the packet order or the number of GPUs.  Perfect sticking gives exactly
 * nx_integrate_adaptive's results.  Preconditions of nx_integrate_constant: tables uploaded,
 * the accommodation spline when accomfactor > 0.  `bounces` receives the number of surface
 * interactions of the run.                                                                  */
int nx_integrate_adaptive_bounce(nx_ctx* ctx, long long n, uint64_t seed, uint64_t first_id,
                                 unsigned long long* attempted_steps,
                                 unsigned long long* accepted_steps,
                                 unsigned long long* bounces);

/* ---- context-owned accumulators (image, cube, deposition, ion production, trajectory) -----
 * Each product below sums on the device into its own accumulator of `nsum` f64 sums and
 * `ncount` i64 counts (the product states the shape), so one product's calls leave the others
 * alone.  Its begin validates the shape and zeroes the accumulator (the device block is reused
 * when large enough); its add sums into it, any number of times.  nx_product_fetch copies sums
 * and counts to the host (either may be NULL; page-locked destinations from nx_host_alloc get
 * the DMA directly, the driver stages pageable ones) and waits.  nx_product_device_ptrs returns
 * the device buffers (fused K3 image, NCCL).  nx_product_allreduce sums them over the ranks of
 * `comm` in place on the context's stream, the one collective of a sharded product; a non-NULL
 * *total (e.g. ModelImage's totalsource) rides along: this rank's share on entry, the sum on
 * return (the call then waits).  nx_product_end waits for the stream and frees the block.
 * Before begin, or after end, each returns -1 with "<product> begin not called".  None of them
 * drops the candidate pairs nx_los_used_fill reads.                                          */
typedef enum {
  NX_PRODUCT_IMAGE = 0,
  NX_PRODUCT_CUBE = 1,
  NX_PRODUCT_DEPOSIT = 2,
  NX_PRODUCT_IONIZE = 3,
  NX_PRODUCT_TRACE = 4
} nx_product;
int nx_product_fetch(nx_ctx* ctx, nx_product which, double* sums, long long* counts);
int nx_product_device_ptrs(nx_ctx* ctx, nx_product which, void** sums, void** counts);
int nx_product_allreduce(nx_ctx* ctx, nx_product which, nx_comm* comm, double* total);
int nx_product_end(nx_ctx* ctx, nx_product which);

/* ---- K2d: surface deposition maps and the source's loss budget (ModelDeposition) ----------
 * An extension (the reference records neither).  nx_integrate_adaptive_deposit runs the
 * adaptive driver on the resident packets exactly as nx_integrate_adaptive (perfect sticking)
 * or nx_integrate_adaptive_bounce (any other sticking, deviates keyed by seed / first_id)
 * would, same preconditions, same final state and step totals, and adds to the sink of
 * nx_deposit_begin where the frac of the packets went:
 *   SURFACE    per accepted step that ends inside the planet: the frac that stays there
 *              (all of it for perfect sticking, frac before - frac after a bounce), mapped at
 *              the post-step point (perfect sticking) or the bounce point, lon =
 *              fmod(atan2(x, -y) + 2 pi, 2 pi), lat = atan2(z, sqrt(x*x + y*y)), on
 *              np.histogram2d's axes linspace(0, 2 pi, nlon + 1) x linspace(-pi/2, pi/2,
 *              nlat + 1), longitude major; one event per such step, whatever its amount
 *   MOON / ESCAPED (r^2 > outeredge) / VANISHED (frac < 1e-10): the frac the first of these
 *              tests (in the driver's order) sets to zero
 *   REMAINING  the frac of packets that retire alive (time <= resolution or the attempt cap)
 *              or are passed through without integration
 *   SOURCE     the initial frac > 0 of the packets handed to the kernel
 * The frac lost in flight (photo-ionisation, lifetime) is SOURCE minus the other buckets.
 * The sink is the NX_PRODUCT_DEPOSIT accumulator, nsum = ncount = nlon * nlat + NX_DEP_NBUCKET:
 * the map cells, then the buckets in nx_deposit_bucket order, each an f64 sum and an event
 * count.  begin validates nlon, nlat >= 1 (nlon * nlat < 2^31).                              */
typedef enum {
  NX_DEP_SURFACE = 0,
  NX_DEP_MOON = 1,
  NX_DEP_ESCAPED = 2,
  NX_DEP_VANISHED = 3,
  NX_DEP_REMAINING = 4,
  NX_DEP_SOURCE = 5,
  NX_DEP_NBUCKET = 6
} nx_deposit_bucket;
int nx_deposit_begin(nx_ctx* ctx, int nlon, int nlat);
int nx_integrate_adaptive_deposit(nx_ctx* ctx, long long n, uint64_t seed, uint64_t first_id,
                                  unsigned long long* attempted_steps,
                                  unsigned long long* accepted_steps,
                                  unsigned long long* bounces);

/* ---- K2i: 3-D ion production maps (ModelIonization) ----------------------------------------
 * An extension (the reference has no such product).  nx_integrate_adaptive_ionize runs the
 * adaptive driver on the resident packets exactly as nx_integrate_adaptive_deposit would (the
 * same preconditions, the same kernel choice: perfect sticking or bounce, deviates keyed by
 * seed / first_id, the same final state and step totals), and adds to the grid of
 * nx_ionize_begin where the frac was lost in flight.  For every accepted step, before any
 * surface, moon, escape or vanish handling:
 *   loss       frac before the step - frac of the Runge-Kutta step (one f64 subtraction); a
 *              step with loss == 0 is not recorded, a negative loss (a step across the shadow
 *              edge) is recorded as it is
 *   where      the midpoint of the step's chord, (x + x_rk) * 0.5 per axis, x_rk taken before
 *              a bounce moves the packet; planet frame (R_p, Sun toward -y)
 *   binning    np.histogramdd's rule on linspace(lo[k], hi[k], n[k] + 1) per axis, the last
 *              right edge in the last cell; a midpoint outside the box, or NaN, goes to OUTSIDE
 * Summed over the grid and OUTSIDE, the loss is ModelDeposition's LOST (SOURCE minus the other
 * buckets), up to rounding.  The run needs a loss process (loss_mode 1 or 2): -1 otherwise.
 * The sink is the NX_PRODUCT_IONIZE accumulator, nsum = ncount = nx * ny * nz + 1: the cells,
 * row-major (nx, ny, nz), then OUTSIDE, each an f64 loss sum and a count of recorded steps.
 * begin validates n[k] >= 1, lo[k] < hi[k] (finite) and nx * ny * nz + 1 < 2^31.  Every
 * recorded step is one f64 and one u64 atomic add; a 100^3 grid (16 MB) stays in the B200's
 * 126 MB L2, a 200^3 grid (128 MB) does not.                                                 */
typedef struct nx_ion_grid {
  double lo[3], hi[3];        /* box edges per axis (x, y, z), R_p                           */
  int32_t n[3];               /* cells per axis                                              */
  int32_t reserved;
} nx_ion_grid;
int nx_ionize_begin(nx_ctx* ctx, const nx_ion_grid* grid);
int nx_integrate_adaptive_ionize(nx_ctx* ctx, long long n, uint64_t seed, uint64_t first_id,
                                 unsigned long long* attempted_steps,
                                 unsigned long long* accepted_steps,
                                 unsigned long long* bounces);

/* ---- K2t: images and density grids from every accepted step (ModelTrajectoryImage,
 * ModelTrajectoryDensity) -------------------------------------------------------------------
 * An extension (the reference has no such product).  nx_integrate_adaptive_trace runs the
 * adaptive driver on the resident packets exactly as nx_integrate_adaptive_ionize would (the
 * same preconditions, the same kernel choice: perfect sticking or bounce, deviates keyed by
 * seed / first_id, the same final state and step totals), and adds every accepted step to the
 * image and / or grid of nx_trace_begin.  With T = endtime, t0 the packet's time remaining when
 * the kernel loads it (its release time in an imported or K1 X0), t the time remaining before
 * the step, h the step, and every operation an f64 op rounded to nearest:
 *   midpoint   m = (s + s_rk) * 0.5 per component, s the state before the step, s_rk the
 *              Runge-Kutta state before any surface, moon, escape or vanish handling
 *   dwell      a = (h * T) / ((T - t0) + (t - 0.5 * h)): the step's length over the chance
 *              (T - age) / T that a packet released uniformly in (0, T] is still in flight at
 *              the midpoint's age, so the sums estimate the steady state the snapshot does
 *   image      K4's pixel and weight w of m (nx_image_accumulate with round_f32 = 0; w carries
 *              m's frac, and the sunlit mask and g-values for radiance): w * a and one count
 *   grid       m's position binned as in nx_ionize_begin: frac(m) * a and one count, OUTSIDE
 *              for a midpoint outside the box or NaN
 * ModelImage's image is sums * atoms_per_packet; this image is sums * atoms_per_packet / T
 * with the same expectation.  A step is represented by its midpoint (not split over the pixels
 * or cells its chord crosses); a step that ends inside the planet counts its full h.
 * The sink is the NX_PRODUCT_TRACE accumulator, nsum = ncount = (image ? nx * nz : 0) + (grid ?
 * gx * gy * gz + 1 : 0): the pixels (ix * nz + iz), then the grid's cells (row-major) and
 * OUTSIDE, each an f64 sum and a count of recorded steps.  begin takes either or both (NULL:
 * none; both NULL is -1), validates the image (nx, nz >= 1, x0 < x1 and z0 < z1 finite, apix >
 * 0, quantity 0 or 1) and the grid as nx_ionize_begin does, and keeps copies of both.
 * nx_integrate_adaptive_trace returns -1 for a run with moons (the forces then depend on the
 * time, so a step's sample is not the snapshot's state) and for a radiance image without
 * g-value tables.  Every recorded step is one f64 and one u64 atomic add per product.       */
int nx_trace_begin(nx_ctx* ctx, const nx_image_params* image, const nx_ion_grid* grid);
int nx_integrate_adaptive_trace(nx_ctx* ctx, long long n, uint64_t seed, uint64_t first_id,
                                unsigned long long* attempted_steps,
                                unsigned long long* accepted_steps,
                                unsigned long long* bounces);

/* ---- K3: constant-step driver with bounce (Output.py:368-455, bouncepackets.py)
 * Optional fused per-step image accumulation (image_dev / counts_dev device
 * pointers, may be NULL) and optional dense trajectory sink traj_host
 * [n][8][nsteps] (small n only; NULL otherwise).                                 */
int nx_integrate_constant(nx_ctx* ctx, long long n, uint64_t seed, uint64_t first_id,
                          const nx_image_params* img, void* image_dev, void* counts_dev,
                          double* traj_host, unsigned long long* packet_steps);

/* Row-table variant: every row of the reference's results[N, 8, nsteps] tensor (Output.py:
 * 376-449) that Output.save would keep (frac > 0 when skip_dead; float32-rounded when
 * round_f32) is appended to a NEW resident packet table (index = packet number within the
 * launch, step = step number; row order is unspecified).  ModelImage / LOSResult then run K4
 * / K5 over the bound table -- any Output of a constant-step run, at any size, without the
 * dense tensor ever existing (compute_iteration.py:118-222 works on these rows).           */
int nx_integrate_constant_rows(nx_ctx* ctx, long long n, uint64_t seed, uint64_t first_id,
                               int skip_dead, int round_f32, nx_packets** out, long long* nrows,
                               unsigned long long* packet_steps);

/* ---- K4: image (ModelImage.create_image + packet_weighting + Histogram2d) ---- */
int nx_image_accumulate(nx_ctx* ctx, long long n, const nx_image_params* ip,
                        double* image /* nx*nz */, long long* counts /* nx*nz */);
int nx_image_accumulate_dev(nx_ctx* ctx, long long n, const nx_image_params* ip,
                            void* image_dev, void* counts_dev);
/* The same into the NX_PRODUCT_IMAGE accumulator, nsum = ncount = nx * nz (row-major (nx, nz)):
 * every add bins the bound packet table (or the slab) into it -- ModelImage sums its output
 * files this way (ModelImage.py:92-99).  ModelImage never ends it, so its block only grows. */
int nx_image_begin(nx_ctx* ctx, int nx, int nz);
int nx_image_add(nx_ctx* ctx, long long n, const nx_image_params* ip);
/* What ModelImage keeps (ModelImage.py:92-105): image * scale (scale = atoms_per_packet) and the
 * packet image as float64, converted on the device, one copy.  Destinations obtained from
 * nx_host_alloc (page-locked) receive the DMA directly, pageable ones are staged.            */
int nx_image_fetch_scaled(nx_ctx* ctx, double scale, double* image, double* counts);
/* Page-locked host memory for result arrays (no reference counterpart: the reference's results
 * are NumPy arrays; these let the device write them without a staging copy).                  */
int nx_host_alloc(long long bytes, void** out);
int nx_host_free(void* p);

/* ---- K5: lines of sight (compute_iteration.py:151-222) ------------------------
 * los[6*nlos] SoA: x,y,z,xbore,ybore,zbore; dist_from_plan[nlos] as computed at
 * compute_iteration.py:105-115.                                                  */
int nx_los_accumulate(nx_ctx* ctx, long long n, long long nlos, const double* los,
                      const double* dist_from_plan, const nx_los_params* lp,
                      double* radiance, long long* npackets, uint8_t* included);
int nx_los_accumulate_dev(nx_ctx* ctx, long long n, long long nlos, void* los_dev,
                          void* dist_dev, const nx_los_params* lp,
                          void* radiance_dev, void* npackets_dev, void* included_dev);

/* `used` packet sets (compute_iteration.py:143-144, 210-211; consumed by
 * LOSResultFitted): packets with weight > 0 per line of sight, as CSR.  Call once
 * with used_indices == NULL to get used_count[nlos]; build used_offsets[nlos+1]
 * (exclusive prefix sum) and call again to fill used_indices[used_offsets[nlos]]
 * (original packet indices, unordered within a line of sight).                   */
int nx_los_used(nx_ctx* ctx, long long n, long long nlos, const double* los,
                const double* dist_from_plan, const nx_los_params* lp,
                const long long* used_offsets, long long* used_count, uint32_t* used_indices);
/* The `used` / `used0` packet sets of compute_iteration.py:143-144, 210-211 without a second
 * search: nx_los_accumulate that also returns used_count[nlos] from the same pass and keeps its
 * candidate pairs on the device; nx_los_used_fill then writes the CSR indices
 * (used_offsets = prefix sums of used_count) by repeating only the exact test over those pairs
 * when nothing happened in between, else by searching again.                                 */
int nx_los_accumulate_counted(nx_ctx* ctx, long long n, long long nlos, const double* los,
                              const double* dist_from_plan, const nx_los_params* lp,
                              double* radiance, long long* npackets, uint8_t* included,
                              long long* used_count);
int nx_los_used_fill(nx_ctx* ctx, long long n, long long nlos, const double* los,
                     const double* dist_from_plan, const nx_los_params* lp,
                     const long long* used_offsets, uint32_t* used_indices);

/* ---- Doppler line profiles along lines of sight (LOSSpectrum) ------------------
 * The hits of nx_los_accumulate (same test, same rows, same weight w) binned by the velocity
 * of the row along the boresight, v = ((vx*bx + vy*by) + vz*bz) * vscale [km/s, planet rest
 * frame, positive = receding], every operation float64 rounded to nearest; vx, vy, vz are
 * float32-rounded when lp->round_f32.  Bins follow np.histogram on edges = linspace(vmin,
 * vmax, nbins + 1) (vmax belongs to the last bin).  Always runs the cell-grid search; more
 * than 2^32 packets per GPU are rejected.                                                  */
typedef struct nx_spectrum_params {
  double vmin, vmax;      /* km/s; edges = linspace(vmin, vmax, nbins + 1)          */
  double vscale;          /* km/s per R_p/s (the planet radius in km)               */
  int32_t nbins;          /* >= 1                                                   */
  int32_t reserved;
} nx_spectrum_params;
/* spectrum / counts: row-major (nlos, nbins + 2); column 0 = v < vmin, 1..nbins = bins,
 * nbins + 1 = v > vmax.  Overwritten (like nx_los_accumulate).  Resets the candidate pairs
 * nx_los_accumulate_counted keeps for nx_los_used_fill.                                 */
int nx_los_spectrum(nx_ctx* ctx, long long n, long long nlos, const double* los,
                    const double* dist_from_plan, const nx_los_params* lp,
                    const nx_spectrum_params* sp, double* spectrum, long long* counts);

/* ---- Doppler-resolved image cubes (ModelImageCube) -----------------------------
 * K4's rows, pixel and weight (nx_image_add: same rows, occulted / shadowed rows counted with
 * w = 0) with a velocity axis: v = ((vx*M[3] + vy*M[4]) + vz*M[5]) * sp->vscale [km/s], every
 * operation float64 rounded to nearest, M the observer rotation of ip (row 1: the observer sits
 * at -y_obs, so v > 0 recedes; planet rest frame); vx, vy, vz float32-rounded when
 * ip->round_f32.  Columns as nx_los_spectrum: 0 = v < vmin, 1..nbins = np.histogram on
 * linspace(vmin, vmax, nbins + 1), nbins + 1 = v > vmax (NaN included).  Layout row-major
 * (nx, nz, nbins + 2), so the sum over the last axis is K4's image and counts.
 * The cube is the NX_PRODUCT_CUBE accumulator, nsum = ncount = nx * nz * (nbins + 2) < 2^31
 * (16 B per cell; nx_product_end releases it).  add bins the bound packet table (or the slab)
 * into it (any number of tables; checks dims, the velocity axis, g-tables for radiance and n
 * before any launch).                                                                      */
int nx_cube_begin(nx_ctx* ctx, int nx, int nz, int nbins);
int nx_cube_add(nx_ctx* ctx, long long n, const nx_image_params* ip,
                const nx_spectrum_params* sp);

/* ---- K7: number density at sample points (ModelDensity) ------------------------
 * Over the rows of the bound packet table (or the slab), float32-rounded, frac == 0 rows
 * dropped: a row is a member of ball i when d2 <= radius[i]^2, with dx = x - pts[i] etc. and
 * d2 = (dx*dx + dy*dy) + dz*dz, every operation an IEEE float64 op rounded to nearest.
 * pts[3*npts] SoA: x[npts], y[npts], z[npts] in R_p (the frame of Output.X);
 * radius[npts] > 0 in R_p.  ADDS to the caller's buffers (several tables can be summed):
 * s1[i] += sum frac, s2[i] += sum frac^2, count[i] += member rows.  Counts are exact; the
 * sums are atomics, so their last bits depend on the order of the additions.
 * Resets the candidate pairs nx_los_accumulate_counted keeps for nx_los_used_fill.        */
int nx_density_accumulate(nx_ctx* ctx, long long n, long long npts, const double* pts,
                          const double* radius, double* s1, double* s2,
                          unsigned long long* count);

/* ---- K6: source maps (data_simulation/make_source_map.py:11-175) ----------------
 * Whole-planet and per-grid-point (haversine ball of radius smear_radius*cos(lat_point),
 * sklearn BallTree.query_radius) histograms of the initial states.  All arrays are host
 * buffers: six packet columns of length n (longitude, latitude [rad], speed [km/s],
 * altitude, azimuth [rad], frac); point_lon[nlon] / point_lat[nlat] = bin centres of the
 * abundance histogram, point_radius[nlat] = smear_radius*cos(point_lat) as the caller's
 * NumPy computed them.  Outputs (caller-allocated, overwritten): abundance_hist
 * [nlon*nlat], speed_dist[nvel], altitude_dist[nalt], azimuth_dist[naz], n_included /
 * n_total [nlon*nlat], abundance[nlon*nlat], speed_map[nlon*nlat*nvel], altitude_map
 * [..*nalt], azimuth_map[..*naz]; point index = ilon*nlat + ilat.                      */
typedef struct nx_source_map_params {
  double smear_radius;
  double vmax;
  int32_t nlon, nlat, nvel, nalt, naz;
  int32_t weight_is_frac;   /* 1: todo = 'source' (weight = frac), 0: 'available' (weight = 1) */
} nx_source_map_params;
int nx_source_map(nx_ctx* ctx, long long n, const nx_source_map_params* p,
                  const double* longitude, const double* latitude, const double* speed_kms,
                  const double* altitude, const double* azimuth, const double* frac,
                  const double* point_lon, const double* point_lat, const double* point_radius,
                  double* abundance_hist, double* speed_dist, double* altitude_dist,
                  double* azimuth_dist, long long* n_included, long long* n_total,
                  double* abundance, double* speed_map, double* altitude_map,
                  double* azimuth_map);

/* ---- resident packet tables: Output.save on the device (Output.py:522-543) ------
 * nx_compact_state copies the current state of the first n packets into a new table:
 * rows with frac == 0 dropped when skip_dead (compress=True, :526-527; the f64 value is
 * tested, as the reference does before its down-cast), every column rounded to float32 when
 * round_f32 (:528-543; kept as f64 bit patterns so K4 / K5 read what Output.restore would
 * hand them), original packet index kept; row order is the packet order.  The table stays
 * on the GPU until nx_packets_free; nx_packets_bind makes K4 / K5 / nx_export_state read it
 * instead of the context's slab (NULL: back to the slab; integrators unbind).
 * nx_packets_export writes the columns time,x,y,z,vx,vy,vz,frac,step_size as float32 (cols
 * has 9 entries, any may be NULL; step_size exists for tables made by nx_compact_state) and
 * the indices as int32 -- the only packet bytes that cross PCIe
 * when a run is saved.  nx_packets_upload is the inverse (a restored Output file).          */
int nx_compact_state(nx_ctx* ctx, long long n, int skip_dead, int round_f32, nx_packets** out,
                     long long* count);
int nx_packets_upload(nx_ctx* ctx, long long n, const double* const* cols /* 8 */,
                      const uint32_t* index, nx_packets** out);
int nx_packets_bind(nx_ctx* ctx, nx_packets* table);
int nx_packets_count(nx_ctx* ctx, nx_packets* table, long long* count);
int nx_packets_export(nx_ctx* ctx, nx_packets* table, float* const* cols /* 9 */, int32_t* index,
                      uint16_t* step /* constant-step row tables; may be NULL */);
int nx_packets_free(nx_ctx* ctx, nx_packets* table);

/* ---- multi-GPU: one all-reduce (sum) per product (SURVEY 8e; the reference has no
 * collective: Input.py:243-249 loops chunks serially).  Packets are sharded by global id
 * (first_id of nx_init_state / nx_integrate_constant), per-rank images and LOS columns are
 * summed in place.  Rank 0 calls nx_comm_unique_id and hands the 128 bytes to the other ranks
 * (file, socket, MPI, torch.distributed store ...); every rank then calls nx_comm_create.
 * NCCL (libnccl.so.2) is loaded on first use.                                                */
#define NX_COMM_ID_BYTES 128
#define NX_DTYPE_F64 0
#define NX_DTYPE_I64 1
int nx_comm_unique_id(void* out128);
int nx_comm_create(int device, const void* unique_id128, int rank, int world, nx_comm** out);
int nx_allreduce(nx_comm* comm, void* dev_buffer, long long count, int dtype, void* cuda_stream);
int nx_allreduce_host(nx_comm* comm, void* host_buffer, long long count, int dtype);
int nx_comm_rank(nx_comm* comm, int* rank, int* world);
int nx_comm_destroy(nx_comm* comm);
const char* nx_comm_last_error(void);

/* ---- measurement --------------------------------------------------------------- */
int nx_last_kernel_ms(nx_ctx* ctx, float* ms);          /* CUDA-event time of last K* */
int nx_kernel_launches(nx_ctx* ctx, unsigned long long* count);
int nx_measure_fp64_peak(nx_ctx* ctx, double* tflops);  /* DFMA-chain microbenchmark  */
int nx_measure_copy_bw(nx_ctx* ctx, long long bytes, double* gbs);

#ifdef __cplusplus
}
#endif
#endif /* NEXOCLOM_B200_H */
