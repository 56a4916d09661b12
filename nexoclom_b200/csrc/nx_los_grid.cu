// nexoclom_b200 -- K5 with spatial culling.
//
// The reference evaluates every spectrum against the union of ~425 KD-tree balls
// along the boresight and then applies a cone test (compute_iteration.py:151-222).
// The membership rule depends only on (line of sight, packet), so any candidate
// generator that does not miss a member gives identical results.  Here:
//
//   1. live packets are binned into a uniform G^3 cell grid over their bounding
//      cube and copied into cell order (counting sort: count / scan / scatter);
//      the cell id is (ix*G + iy)*G + iz, so the packets of a run of cells along z
//      are one contiguous range;
//   2. one WARP per line of sight marches along the boresight in segments of one
//      cell size; the axis-aligned box around a segment, inflated by the cone
//      radius at its far end, yields a rectangle of (ix, iy) columns and a z-range;
//      the warp streams the contiguous packet range of every column (coalesced);
//   3. a packet is tested in exactly one segment -- the one that contains its
//      axial coordinate losrad -- so overlapping boxes never double count;
//   4. survivors of that ownership test go through the same exact membership /
//      weighting code as the brute-force kernel (nx_image.cuh: los_hit, los_weight).
#include <cuda_runtime.h>
#include <stdint.h>
#include <string.h>

#include "nx_image.cuh"
#include "nx_kernels.h"

namespace nx {

#define FULL_MASK 0xffffffffu
#ifndef NX_LOS_SEG_CELLS
#define NX_LOS_SEG_CELLS 12.0     // march segment length in finest local cells (with the pieces below: 6: 17.7 ms, 8: 17.0, 12: 16.0, 16: 16.2)
#endif

// ---- 1. bounding cube: max |coordinate| over live packets ----------------------
__global__ void __launch_bounds__(256)
k_los_extent(StateCols P, long long n, int skip_dead, int round32, unsigned long long* out) {
  // out[0] = bits of max |coordinate|, out[1] = number of packets that enter the grid
  double m = 0.0;
  unsigned long long live = 0;
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    if (skip_dead && !(P.c[7][i] > 0.0)) continue;
    double x = P.c[1][i], y = P.c[2][i], z = P.c[3][i];
    if (round32) { x = round_f32(x); y = round_f32(y); z = round_f32(z); }
    m = fmax(m, fmax(fabs(x), fmax(fabs(y), fabs(z))));
    ++live;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    m = fmax(m, __shfl_xor_sync(FULL_MASK, m, o));
    live += __shfl_xor_sync(FULL_MASK, live, o);
  }
  if ((threadIdx.x & 31) == 0) {
    atomicMax(out, (unsigned long long)__double_as_longlong(m));
    if (live) atomicAdd(out + 1, live);
  }
}

__device__ __forceinline__ int cell_of(double v, const LosGrid& g) {
  int c = __double2int_rd(fma(g.k, asinh(v * g.inv_scale), 0.5 * g.G));
  return max(0, min(c, g.G - 1));
}
// width of the cell that holds coordinate v
__device__ __forceinline__ double cell_width(double v, const LosGrid& g) {
  return sqrt(fma(v, v, g.scale * g.scale)) / g.k;
}

// ---- 2. counting sort into cell order -------------------------------------------
__global__ void __launch_bounds__(256)
k_los_cell_count(StateCols P, long long n, LosGrid g, int skip_dead, int round32,
                 unsigned* __restrict__ cell_id, unsigned* __restrict__ count) {
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    unsigned id = 0xffffffffu;
    if (!(skip_dead && !(P.c[7][i] > 0.0))) {
      double x = P.c[1][i], y = P.c[2][i], z = P.c[3][i];
      if (round32) { x = round_f32(x); y = round_f32(y); z = round_f32(z); }
      const int ix = cell_of(x, g), iy = cell_of(y, g), iz = cell_of(z, g);
      id = (unsigned)((ix * g.G + iy) * g.G + iz);
      atomicAdd(&count[id], 1u);
    }
    cell_id[i] = id;
  }
}

// exclusive scan of `count` (ncell entries) into start[0..ncell]; three passes
#define NX_SCAN_ELEMS 4096
__global__ void __launch_bounds__(1024)
k_scan_partial(const unsigned* __restrict__ in, unsigned* __restrict__ out,
               unsigned* __restrict__ block_sum, int n) {
  __shared__ unsigned warp_tot[32];
  const int base = blockIdx.x * NX_SCAN_ELEMS + threadIdx.x * 4;
  unsigned v[4], s = 0;
#pragma unroll
  for (int k = 0; k < 4; ++k) { v[k] = (base + k < n) ? in[base + k] : 0u; s += v[k]; }
  unsigned incl = s;
  const unsigned lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const unsigned t = __shfl_up_sync(FULL_MASK, incl, o);
    if (lane >= (unsigned)o) incl += t;
  }
  if (lane == 31) warp_tot[warp] = incl;
  __syncthreads();
  if (warp == 0) {
    unsigned w = warp_tot[lane], wi = w;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const unsigned t = __shfl_up_sync(FULL_MASK, wi, o);
      if (lane >= (unsigned)o) wi += t;
    }
    warp_tot[lane] = wi - w;                  // exclusive warp offsets
    if (lane == 31) block_sum[blockIdx.x] = wi;
  }
  __syncthreads();
  unsigned run = warp_tot[warp] + incl - s;   // exclusive prefix of this thread
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    if (base + k < n) out[base + k] = run;
    run += v[k];
  }
}

__global__ void __launch_bounds__(1024)
k_scan_top(unsigned* __restrict__ block_sum, int nblocks, unsigned* __restrict__ total) {
  // single block: sequential over chunks of 1024 (nblocks <= a few thousand)
  __shared__ unsigned warp_tot[32];
  __shared__ unsigned carry;
  if (threadIdx.x == 0) carry = 0;
  __syncthreads();
  for (int b0 = 0; b0 < nblocks; b0 += 1024) {
    const int i = b0 + threadIdx.x;
    const unsigned v = (i < nblocks) ? block_sum[i] : 0u;
    unsigned incl = v;
    const unsigned lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const unsigned t = __shfl_up_sync(FULL_MASK, incl, o);
      if (lane >= (unsigned)o) incl += t;
    }
    if (lane == 31) warp_tot[warp] = incl;
    __syncthreads();
    if (warp == 0) {
      unsigned w = warp_tot[lane], wi = w;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const unsigned t = __shfl_up_sync(FULL_MASK, wi, o);
        if (lane >= (unsigned)o) wi += t;
      }
      warp_tot[lane] = wi - w;
    }
    __syncthreads();
    const unsigned excl = carry + warp_tot[warp] + incl - v;
    if (i < nblocks) block_sum[i] = excl;
    __syncthreads();
    if (threadIdx.x == 1023) carry = excl + v;
    __syncthreads();
  }
  if (threadIdx.x == 0) *total = carry;
}

__global__ void __launch_bounds__(1024)
k_scan_add(unsigned* __restrict__ out, const unsigned* __restrict__ block_sum, int n,
           const unsigned* __restrict__ total) {
  const int base = blockIdx.x * NX_SCAN_ELEMS + threadIdx.x * 4;
  const unsigned add = block_sum[blockIdx.x];
#pragma unroll
  for (int k = 0; k < 4; ++k)
    if (base + k < n) out[base + k] += add;
  if (blockIdx.x == 0 && threadIdx.x == 0) out[n] = *total;
}

// F32: the packets are float32-rounded (what a saved Output holds, quirk Q14), so x, y, z, vy
// and frac are stored as floats -- a candidate costs 16 bytes instead of 32
template <bool F32>
__global__ void __launch_bounds__(256)
k_los_cell_scatter(StateCols P, long long n, int round32, const unsigned* __restrict__ cell_id,
                   const unsigned* __restrict__ start, unsigned* __restrict__ cursor,
                   LosSorted S) {
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    const unsigned id = cell_id[i];
    if (id == 0xffffffffu) continue;
    const unsigned pos = start[id] + atomicAdd(&cursor[id], 1u);
    double x = P.c[1][i], y = P.c[2][i], z = P.c[3][i], vy = P.c[5][i], fr = P.c[7][i];
    if (round32) { x = round_f32(x); y = round_f32(y); z = round_f32(z); vy = round_f32(vy); fr = round_f32(fr); }
    if (F32) {
      reinterpret_cast<float4*>(S.pos)[pos] = make_float4((float)x, (float)y, (float)z, (float)vy);
      reinterpret_cast<float*>(S.frac)[pos] = (float)fr;
    } else {
      S.pos[pos] = make_double4(x, y, z, vy); S.frac[pos] = fr;
    }
    S.idx[pos] = (unsigned)i;
  }
}

// ---- 3. candidates: one warp per line of sight, lean ------------------------------------
// The march only decides which (line of sight, packet) pairs deserve the exact test: segment
// ownership, the cone with a safety margin and the planet cut -- the first rejects of los_hit,
// in the same arithmetic.  Survivors go to a global pair list (through a per-warp
// shared-memory buffer: one atomic per ~100 pairs) and are resolved by k_los_resolve, one
// THREAD per pair.  Keeping acos / log / the ball search / the g-value lookups out of this
// kernel matters because it is bound by DRAM latency (round 1 ncu: long_scoreboard 9.3 cycles
// per issue, 72 registers -> 17 resident warps per SM): at ~40 registers three times as many
// warps are in flight, and the exact test runs on full warps instead of on the ~15 % of the
// lanes that hit.
__device__ __forceinline__ float4 load_rec(const float4* p) { return __ldg(p); }
__device__ __forceinline__ double4 load_rec(const double4* p) { return *p; }
template <bool F32> struct LosRec { typedef double4 type; };
template <> struct LosRec<true> { typedef float4 type; };
#define NX_LOS_WARPS 8              // warps per block of the candidate kernel
#define NX_LOS_BUF 128              // pairs buffered per warp
#ifndef NX_LOS_SUB
#define NX_LOS_SUB 12               // pieces a march segment is cut into for the cell ranges (<= 31)
#endif
#ifndef NX_LOS_MINBLOCKS
#define NX_LOS_MINBLOCKS 4          // 64 registers: 32 resident warps per SM
#endif

template <bool F32>
__global__ void __launch_bounds__(32 * NX_LOS_WARPS, NX_LOS_MINBLOCKS)
k_los_candidates(LosSorted S, LosGrid g, const unsigned* __restrict__ start, long long nlos,
                 long long first, long long count, const double* __restrict__ los,
                 const double* __restrict__ dist_plan, const int* __restrict__ nball,
                 const double* __restrict__ ladder, double dphi, double cos_margin2,
                 const unsigned* __restrict__ order, uint2* __restrict__ pairs,
                 unsigned long long* __restrict__ cursor, unsigned long long cap) {
  typedef typename LosRec<F32>::type RecT;
  __shared__ unsigned buf_all[NX_LOS_WARPS][NX_LOS_BUF];
  __shared__ __align__(16) int sub_all[NX_LOS_WARPS][NX_LOS_SUB * 8];
  const unsigned lane = threadIdx.x & 31u;
  unsigned* buf = buf_all[threadIdx.x >> 5];
  const RecT* __restrict__ recs = reinterpret_cast<const RecT*>(S.pos);
  const double s2 = sin(2.0 * dphi);
  const double tan_phi = tan(dphi) * (1.0 + 1e-9);
  // persistent warps: a line of sight costs anything between a few and thousands of
  // iterations, so every warp takes the next one from a ticket counter when it is done
  for (;;) {
  long long w_ = 0;
  if (lane == 0) w_ = (long long)atomicAdd(cursor + 1, 1ull);
  w_ = __shfl_sync(FULL_MASK, w_, 0);
  if (w_ >= count) return;
  // lines of sight are processed in a spatially coherent order (host: Morton order of the
  // points of closest approach) so that neighbouring warps stream the same cells out of L2
  const long long l = order ? (long long)order[first + w_] : first + w_;
  const double xs = los[l], ys = los[nlos + l], zs = los[2 * nlos + l];
  const double bx = los[3 * nlos + l], by = los[4 * nlos + l], bz = los[5 * nlos + l];
  const double dplan = dist_plan[l];

  // farthest axial distance at which a packet can still be a member: planet
  // truncation, last KD ball, and the far side of the packet cube
  double t_end = ladder[nball[l] - 1] * (1.0 + s2);
  if (dplan < t_end) t_end = dplan;
  const double reach = sqrt(xs * xs + ys * ys + zs * zs) + 1.7320508075688772 * g.half;
  if (reach < t_end) t_end = reach;

  int nbuf = 0;                                       // warp-uniform
  auto flush = [&]() {
    unsigned long long base = 0;
    if (lane == 0) base = atomicAdd(cursor, (unsigned long long)nbuf);
    base = __shfl_sync(FULL_MASK, base, 0);
    for (int i = (int)lane; i < nbuf; i += 32)
      if (base + i < cap) pairs[base + i] = make_uint2((unsigned)l, buf[i]);
    nbuf = 0;
    __syncwarp();
  };
  double t0 = 0.0, t1 = 0.0;
  auto keep = [&](double px, double py, double pz) {
    // same arithmetic as los_hit, so that every packet has exactly one owner segment and no
    // member is lost
    const double rx = sub_rn(px, xs), ry = sub_rn(py, ys), rz = sub_rn(pz, zs);
    const double lr = add_rn(add_rn(mul_rn(rx, bx), mul_rn(ry, by)), mul_rn(rz, bz));
    const double d2 = add_rn(add_rn(mul_rn(rx, rx), mul_rn(ry, ry)), mul_rn(rz, rz));
    return (lr >= t0 && lr < t1) && (lr > 0.0) && !(mul_rn(lr, lr) < mul_rn(d2, cos_margin2)) &&
           (lr < dplan);
  };
  while (t1 < t_end) {
    // segment [t0, t1): about one cell of the finest axis long, never shorter than the
    // cone is wide there; t1 of one segment IS t0 of the next (same double)
    t0 = t1;
    const double cx = xs + bx * t0, cy = ys + by * t0, cz = zs + bz * t0;
    const double dt = fmax(NX_LOS_SEG_CELLS *
                               fmin(cell_width(cx, g), fmin(cell_width(cy, g), cell_width(cz, g))),
                           2.0 * t0 * tan_phi);
    t1 = t0 + dt;
    const double rho = t1 * tan_phi + 1e-9 * (1.0 + t1);
    const double ex = xs + bx * t1, ey = ys + by * t1, ez = zs + bz * t1;
    const double xlo = fmin(cx, ex) - rho, xhi = fmax(cx, ex) + rho;
    const double ylo = fmin(cy, ey) - rho, yhi = fmax(cy, ey) + rho;
    const double zlo = fmin(cz, ez) - rho, zhi = fmax(cz, ez) + rho;
    // boxes entirely outside the packet cube hold nothing
    if (xlo > g.half || xhi < -g.half || ylo > g.half || yhi < -g.half || zlo > g.half ||
        zhi < -g.half)
      continue;
    // The axis-aligned box of a diagonal segment holds several times the cells its cone
    // touches.  The segment is therefore cut into NX_LOS_SUB pieces: lane j takes the axis
    // point at t0 + j dt / NX_LOS_SUB (the last one at t1), the cells of that point +- rho per
    // axis; piece j is the hull of points j and j + 1 (cell_of is monotone, so the hull of the
    // cell indices is the cell range of the hull).  A packet the segment owns sits within rho
    // of the axis point at its own axial coordinate, i.e. inside one of the pieces.
    int plo[3], phi[3];
    {
      const int j = min((int)lane, NX_LOS_SUB);
      const double tj = j == NX_LOS_SUB ? t1 : t0 + dt * ((double)j * (1.0 / NX_LOS_SUB));
      const double ax = xs + bx * tj, ay = ys + by * tj, az = zs + bz * tj;
      plo[0] = cell_of(ax - rho, g); phi[0] = cell_of(ax + rho, g);
      plo[1] = cell_of(ay - rho, g); phi[1] = cell_of(ay + rho, g);
      plo[2] = cell_of(az - rho, g); phi[2] = cell_of(az + rho, g);
    }
    int* sb = sub_all[threadIdx.x >> 5];
    __syncwarp();                                     // the previous segment's readers are done
#pragma unroll
    for (int a = 0; a < 3; ++a) {
      const int nlo = __shfl_down_sync(FULL_MASK, plo[a], 1), nhi = __shfl_down_sync(FULL_MASK, phi[a], 1);
      if (lane < NX_LOS_SUB) {
        sb[lane * 8 + 2 * a] = min(plo[a], nlo);
        sb[lane * 8 + 2 * a + 1] = max(phi[a], nhi);
      }
    }
    __syncwarp();
    const bool pt = lane <= NX_LOS_SUB;
    const int ix0 = __reduce_min_sync(FULL_MASK, pt ? plo[0] : 0x7fffffff);
    const int ix1 = __reduce_max_sync(FULL_MASK, pt ? phi[0] : -1);
    const int iy0 = __reduce_min_sync(FULL_MASK, pt ? plo[1] : 0x7fffffff);
    const int iy1 = __reduce_max_sync(FULL_MASK, pt ? phi[1] : -1);
    // the (ix, iy) columns of the box: every lane finds the z cells the pieces reach in ITS
    // column and fetches that packet range (the dependent index loads of up to 32 columns are
    // in flight together), then the warp streams the ranges one after the other, two records
    // per lane in flight; columns no piece touches stay empty
    const int nyr = iy1 - iy0 + 1, ncol = (ix1 - ix0 + 1) * nyr;
    for (int c0 = 0; c0 < ncol; c0 += 32) {
      const int c = c0 + (int)lane;
      unsigned p0v = 0u, p1v = 0u;
      if (c < ncol) {
        const int ix = ix0 + c / nyr, iy = iy0 + c % nyr;
        int iz0 = 0x7fffffff, iz1 = -1;
#pragma unroll
        for (int j = 0; j < NX_LOS_SUB; ++j) {
          const int4 q = *reinterpret_cast<const int4*>(sb + j * 8);        // x lo, x hi, y lo, y hi
          const int2 qz = *reinterpret_cast<const int2*>(sb + j * 8 + 4);   // z lo, z hi
          if (ix >= q.x && ix <= q.y && iy >= q.z && iy <= q.w) { iz0 = min(iz0, qz.x); iz1 = max(iz1, qz.y); }
        }
        if (iz1 >= iz0) {
          const unsigned row = (unsigned)((ix * g.G + iy) * g.G);
          p0v = __ldg(start + row + iz0); p1v = __ldg(start + row + iz1 + 1);
        }
      }
      const int nc = min(32, ncol - c0);
      for (int k = 0; k < nc; ++k) {
        const unsigned p0 = __shfl_sync(FULL_MASK, p0v, k), p1 = __shfl_sync(FULL_MASK, p1v, k);
        for (unsigned qb = p0; qb < p1; qb += 64) {
          const unsigned q0 = qb + lane, q1 = q0 + 32u;
          const bool in0 = q0 < p1, in1 = q1 < p1;
          RecT a, b;
          if (in0) a = load_rec(recs + q0);
          if (in1) b = load_rec(recs + q1);
          const bool k0 = in0 && keep(a.x, a.y, a.z);
          const bool k1 = in1 && keep(b.x, b.y, b.z);
          const unsigned m0 = __ballot_sync(FULL_MASK, k0), m1 = __ballot_sync(FULL_MASK, k1);
          if (m0 | m1) {
            if (k0) buf[nbuf + __popc(m0 & ((1u << lane) - 1u))] = q0;
            nbuf += __popc(m0);
            if (k1) buf[nbuf + __popc(m1 & ((1u << lane) - 1u))] = q1;
            nbuf += __popc(m1);
            __syncwarp();
            if (nbuf > NX_LOS_BUF - 64) flush();
          }
        }
      }
    }
  }
  if (nbuf) flush();
  }
}

// ---- 4. exact membership + weight, one thread per candidate pair -----------------------
// SPEC: the Doppler spectrum variant (nx_los_spectrum) -- the same test and weight, added to
// the hit's (line, velocity column) cell of sp instead of the per-line sums.
template <bool F32, bool SPEC>
__global__ void __launch_bounds__(256)
k_los_resolve(LosSorted S, const uint2* __restrict__ pairs, unsigned long long npairs,
              long long nlos, const double* __restrict__ los,
              const double* __restrict__ dist_plan, const int* __restrict__ nball,
              const double* __restrict__ ladder, const double* __restrict__ wid2, LosParams lp,
              LosConsts lc, GTables G, double* __restrict__ radiance,
              unsigned long long* __restrict__ npack, unsigned char* __restrict__ included,
              unsigned long long* __restrict__ nused, const long long* __restrict__ used_off,
              unsigned long long* __restrict__ used_cursor, unsigned* __restrict__ used_idx,
              LosSpectrum sp) {
  typedef typename LosRec<F32>::type RecT;
  const unsigned lane = threadIdx.x & 31u;
  const unsigned long long stride = (unsigned long long)gridDim.x * blockDim.x;
  // whole warps iterate together (the tail is padded with inactive lanes) so that the
  // per-warp aggregation below can use full-mask collectives
  const unsigned long long rounded = (npairs + 31ull) & ~31ull;
  for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
       i < rounded; i += stride) {
    const bool valid = i < npairs;
    unsigned l = 0xffffffffu;
    double w = 0.0;
    bool hit = false;
    unsigned cell = 0xffffffffu;       // SPEC: l * (nbins + 2) + velocity column of a hit
    if (valid) {
      const uint2 pr = pairs[i];
      l = pr.x;
      const unsigned q = pr.y;
      LosRay L;
      L.xs = los[l]; L.ys = los[nlos + l]; L.zs = los[2 * nlos + l];
      L.bx = los[3 * nlos + l]; L.by = los[4 * nlos + l]; L.bz = los[5 * nlos + l];
      L.dist_plan = dist_plan[l];
      L.nball = nball[l];
      const RecT r = load_rec(reinterpret_cast<const RecT*>(S.pos) + q);
      double losrad, dist;
      if (los_hit(L, lp.dphi, lc.cos_margin2, lc.cos_accept2, lc.cover, ladder, wid2,
                  lc.inv_log_ratio, lc.log_t0, lc.kwin, r.x, r.y, r.z, losrad, dist)) {
        hit = true;
        const double fr = F32 ? (double)reinterpret_cast<const float*>(S.frac)[q] : S.frac[q];
        w = los_weight(L, lp, G, lc.sin_dphi, fr, r.w, losrad, dist);
        const unsigned pidx = S.idx[q];
        if (SPEC) {
          // vx, vz gathered from the table at the hit's row (the records carry x, y, z, vy only)
          double vx = sp.vx[pidx], vz = sp.vz[pidx];
          if (lp.round_f32) { vx = round_f32(vx); vz = round_f32(vz); }
          const double v = los_doppler(vx, r.w, vz, L.bx, L.by, L.bz, sp.vscale);
          cell = l * (unsigned)(sp.nbins + 2) +
                 (unsigned)spectrum_column(v, sp.nbins, sp.vmin, sp.vmax, sp.step);
        } else {
          if (included) included[pidx] = 1;
          if (w > 0.0 && used_idx)               // `used` packets (compute_iteration.py:210-211)
            used_idx[used_off[l] + atomicAdd(&used_cursor[l], 1ull)] = pidx;
        }
      }
    }
    if (SPEC) {
      // Pairs of one line are adjacent but their velocity columns are not: the lanes with equal
      // cells combine (the lowest lane adds the group's weights in lane order) before the
      // global f64 / u64 atomics.
      const unsigned hitm = __ballot_sync(FULL_MASK, hit);
      if (hitm) {
        const unsigned grp = __match_any_sync(FULL_MASK, cell);
        double acc = 0.0;
        for (int k = 0; k < 32; ++k) {
          const double wk = __shfl_sync(FULL_MASK, w, k);
          if ((grp >> k) & 1u) acc += wk;
        }
        if (hit && lane == (unsigned)(__ffs(grp) - 1)) {
          atomicAdd(&sp.count[cell], (unsigned long long)__popc(grp));
          if (acc != 0.0) atomicAdd(&sp.sum[cell], acc);
        }
      }
      continue;
    }
    // pairs of one line of sight sit next to each other in the list: one atomic per run of
    // equal l within the warp (segmented reduction over the lanes, in lane order)
    const unsigned prev = __shfl_up_sync(FULL_MASK, l, 1);
    const bool head = lane == 0 || prev != l;
    const unsigned heads = __ballot_sync(FULL_MASK, head);
    const unsigned hitm = __ballot_sync(FULL_MASK, hit);
    const unsigned usedm = __ballot_sync(FULL_MASK, hit && w > 0.0);
    // end of my run = next head after my lane
    const unsigned after = heads & ~((2u << lane) - 1u);
    const int run_end = after ? __ffs(after) - 1 : 32;
    // the head of a run adds up its weights in lane order (every lane takes part in the shuffles)
    double acc = 0.0;
    if (heads == 1u) {
      // the usual case (a line of sight has thousands of pairs): the whole warp is one run
      acc = w;
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(FULL_MASK, acc, o);
    } else {
      for (int k = 0; k < 32; ++k) {
        const double wk = __shfl_sync(FULL_MASK, w, k);
        if (head && k >= (int)lane && k < run_end) acc += wk;
      }
    }
    if (head && valid) {
      const unsigned runmask = (run_end >= 32 ? 0xffffffffu : ((1u << run_end) - 1u)) & ~((1u << lane) - 1u);
      const unsigned nh = __popc(hitm & runmask), nu = __popc(usedm & runmask);
      if (nh) {
        if (npack) atomicAdd(&npack[l], (unsigned long long)nh);
        if (radiance && acc != 0.0) atomicAdd(&radiance[l], acc);
        if (nused && nu) atomicAdd(&nused[l], (unsigned long long)nu);
      }
    }
  }
}

// ---- host-side launch sequence ------------------------------------------------------
// k_los_resolve over np pairs in w.pairs: records F32 or not, spectrum (spec) or per-line sums
static void launch_resolve_pairs(cudaStream_t st, LosGridWork& w, unsigned long long np, long long nlos,
                                 const double* los, const double* dist_plan, const int* nball,
                                 const double* ladder, const double* wid2, const LosParams& lp,
                                 const LosConsts& lc, const GTables& G, double* radiance,
                                 unsigned long long* npack, unsigned char* included,
                                 unsigned long long* nused, const long long* used_off,
                                 unsigned long long* used_cursor, unsigned* used_idx,
                                 const LosSpectrum* spec) {
  int sms = 148, dev = 0;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  long long rb = (long long)((np + 255) / 256);
  if (rb > (long long)sms * 16) rb = (long long)sms * 16;
  const LosSpectrum sp = spec ? *spec : LosSpectrum{};
#define NX_RESOLVE(F32, SPEC)                                                                  \
  k_los_resolve<F32, SPEC><<<(unsigned)rb, 256, 0, st>>>(                                      \
      w.sorted, w.pairs, np, nlos, los, dist_plan, nball, ladder, wid2, lp, lc, G, radiance,   \
      npack, included, nused, used_off, used_cursor, used_idx, sp)
  if (spec) {
    if (lp.round_f32) NX_RESOLVE(true, true); else NX_RESOLVE(false, true);
  } else {
    if (lp.round_f32) NX_RESOLVE(true, false); else NX_RESOLVE(false, false);
  }
#undef NX_RESOLVE
}

cudaError_t launch_los_grid_build(cudaStream_t st, int device, StateCols P, long long n,
                                  const LosParams& lp, LosGridWork& w) {
  int sms = 148;
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device);
  const int blocks = sms * 8;
  cudaError_t e;
  if ((e = cudaMemsetAsync(w.extent_bits, 0, 2 * sizeof(unsigned long long), st)) != cudaSuccess) return e;
  k_los_extent<<<blocks, 256, 0, st>>>(P, n, lp.skip_dead, lp.round_f32, w.extent_bits);
  unsigned long long bits[2] = {0, 0};
  if ((e = cudaMemcpyAsync(bits, w.extent_bits, sizeof(bits), cudaMemcpyDeviceToHost, st)) != cudaSuccess) return e;
  if ((e = cudaStreamSynchronize(st)) != cudaSuccess) return e;
  double ext;
  memcpy(&ext, &bits[0], sizeof(ext));
  if (!(ext > 0.0)) ext = 1.0;
  // cells per axis: fixed by the option "los_grid", else ~0.55 n^(1/3) in steps of 32
  // (measured on 1e5 lines of sight: 1.9e6 packets -> 64 best, 1e7 -> 96..128)
  int G = w.G_fixed;
  if (G <= 0) {
    G = (int)(0.55 * cbrt((double)(bits[1] ? bits[1] : 1)) / 32.0 + 0.5) * 32;
    G = G < 32 ? 32 : (G > NX_LOS_GRID_MAX ? NX_LOS_GRID_MAX : G);
  }
  w.G = G;
  w.grid.G = w.G;
  w.grid.half = ext * (1.0 + 1e-9) + 1e-9;
  // scale: one planet radius (cells ~0.06 R_p at the planet for G = 128, half = 25);
  // a cloud smaller than that gets a nearly uniform grid
  w.grid.scale = w.grid.half < w.scale ? w.grid.half : w.scale;
  w.grid.inv_scale = 1.0 / w.grid.scale;
  w.grid.k = 0.5 * w.G / asinh(w.grid.half * w.grid.inv_scale);
  const int ncell = w.G * w.G * w.G;
  if ((e = cudaMemsetAsync(w.count, 0, (size_t)ncell * sizeof(unsigned), st)) != cudaSuccess) return e;
  k_los_cell_count<<<blocks, 256, 0, st>>>(P, n, w.grid, lp.skip_dead, lp.round_f32, w.cell_id, w.count);
  const int nb = (ncell + NX_SCAN_ELEMS - 1) / NX_SCAN_ELEMS;
  k_scan_partial<<<nb, 1024, 0, st>>>(w.count, w.start, w.block_sum, ncell);
  k_scan_top<<<1, 1024, 0, st>>>(w.block_sum, nb, w.total);
  k_scan_add<<<nb, 1024, 0, st>>>(w.start, w.block_sum, ncell, w.total);
  if ((e = cudaMemsetAsync(w.count, 0, (size_t)ncell * sizeof(unsigned), st)) != cudaSuccess) return e;
  if (lp.round_f32)
    k_los_cell_scatter<true><<<blocks, 256, 0, st>>>(P, n, lp.round_f32, w.cell_id, w.start, w.count, w.sorted);
  else
    k_los_cell_scatter<false><<<blocks, 256, 0, st>>>(P, n, lp.round_f32, w.cell_id, w.start, w.count, w.sorted);
  return cudaGetLastError();
}

cudaError_t launch_los_grid(cudaStream_t st, LosGridWork& w, long long nlos,
                            const double* los, const double* dist_plan, const int* nball,
                            const double* ladder, const double* wid2, const LosParams& lp,
                            const LosConsts& lc, const GTables& G, double* radiance,
                            unsigned long long* npack, unsigned char* included,
                            unsigned long long* nused, const long long* used_off,
                            unsigned long long* used_cursor, unsigned* used_idx,
                            const unsigned* order, unsigned long long* kept_pairs,
                            const LosSpectrum* spec) {
  // Lines of sight go through in batches sized so that the candidate pairs of a batch fit the
  // pair buffer (about half full: the size of the next batch follows the pairs per line of
  // sight seen so far); a batch that overflows is repeated with half as many lines.
  int sms = 148, dev = 0;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  const unsigned long long cap = w.pairs_cap;
  long long batch = w.batch_hint > 0 ? w.batch_hint : nlos;
  long long first = 0;
  cudaError_t e;
  while (first < nlos) {
    long long cnt = batch < nlos - first ? batch : nlos - first;
    if ((e = cudaMemsetAsync(w.pair_cursor, 0, 2 * sizeof(unsigned long long), st)) != cudaSuccess) return e;
    long long blocks = (cnt + NX_LOS_WARPS - 1) / NX_LOS_WARPS;
    if (blocks > (long long)sms * NX_LOS_MINBLOCKS) blocks = (long long)sms * NX_LOS_MINBLOCKS;
    if (lp.round_f32)
      k_los_candidates<true><<<(unsigned)blocks, 32 * NX_LOS_WARPS, 0, st>>>(
          w.sorted, w.grid, w.start, nlos, first, cnt, los, dist_plan, nball, ladder, lp.dphi,
          lc.cos_margin2, order, w.pairs, w.pair_cursor, cap);
    else
      k_los_candidates<false><<<(unsigned)blocks, 32 * NX_LOS_WARPS, 0, st>>>(
          w.sorted, w.grid, w.start, nlos, first, cnt, los, dist_plan, nball, ladder, lp.dphi,
          lc.cos_margin2, order, w.pairs, w.pair_cursor, cap);
    unsigned long long np = 0;
    if ((e = cudaMemcpyAsync(&np, w.pair_cursor, sizeof(np), cudaMemcpyDeviceToHost, st)) != cudaSuccess) return e;
    if ((e = cudaStreamSynchronize(st)) != cudaSuccess) return e;
    if (np > cap) {
      // the cursor counted every pair the batch wanted to write: size the repeat from it
      if (cnt == 1) return cudaErrorMemoryAllocation;     // cannot happen: cap >= packets + slack
      long long fit = (long long)(0.8 * (double)cap / ((double)np / (double)cnt));
      if (fit > cnt / 2) fit = cnt / 2;
      batch = fit > 1 ? fit : 1;
      continue;
    }
    if (np)
      launch_resolve_pairs(st, w, np, nlos, los, dist_plan, nball, ladder, wid2, lp, lc, G, radiance,
                           npack, included, nused, used_off, used_cursor, used_idx, spec);
    // one batch covered every line of sight: its pairs stay valid in w.pairs
    if (kept_pairs) *kept_pairs = (first == 0 && cnt == nlos) ? np : 0ull;
    const bool whole = first == 0 && cnt == nlos;      // the whole sweep fitted one batch
    first += cnt;
    const double per = (double)np / (double)cnt;
    // (lines of sight run in Morton order: their pair counts drift from batch to batch, and an
    // overflowing batch is thrown away -- at 0.9 four of eleven candidate passes were, at 1e8 packets)
    long long next = per > 0.0 ? (long long)(0.65 * (double)cap / per) : nlos;
    if (next < 256) next = 256;
    if (whole) next = nlos;              // try the same again (an overflow is sized from its count)
    batch = next;
    w.batch_hint = batch;
  }
  return cudaGetLastError();
}

// ---------------------------------------------------------------------------
// Per-call preparation of the lines of sight, on the device (round 1 did this on the host:
// 4 ms per 1e5 lines).  compute_iteration.py:151-170 builds, per spectrum, a ladder of KD-ball
// centres t_0 = sin(dphi), t_{k+1} = t_k + t_k sin(dphi) up to the distance `dd` at which the
// boresight leaves the outer edge; the ladder is common to all lines (the host builds its
// ~430 entries once the longest `dd` is known), a line needs its own entry count only.
//   k_los_prepare : dd per line (the reference's arithmetic order), the running maximum, and
//                   the 15-bit Morton key of the point of closest approach to the planet
//                   (0.4 R_p cells over +-6.4 R_p) + its histogram: lines of sight run in
//                   Morton order, so that warps that run together stream the same
//                   near-planet cells
//   k_los_key_scan: exclusive scan of the 32768-bin histogram (one block)
//   k_los_finish  : nball = lower_bound(ladder, dd) + 1 and the counting-sort scatter
// ---------------------------------------------------------------------------
#define NX_LOS_KEYS 32768
__device__ __forceinline__ unsigned morton_spread5(unsigned v) {
  unsigned r = 0;
#pragma unroll
  for (int b = 0; b < 5; ++b) r |= ((v >> b) & 1u) << (3 * b);
  return r;
}
__global__ void __launch_bounds__(256)
k_los_prepare(const double* __restrict__ los, long long nlos, double outeredge,
              double* __restrict__ dd_out, unsigned* __restrict__ key_out,
              unsigned* __restrict__ hist, unsigned long long* __restrict__ ddmax_bits) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  double dd = 0.0;
  if (i < nlos) {
    const double x = los[i], y = los[nlos + i], z = los[2 * nlos + i];
    const double bx = los[3 * nlos + i], by = los[4 * nlos + i], bz = los[5 * nlos + i];
    const double b = 2 * ((x * bx + y * by) + z * bz);
    const double nrm = sqrt((x * x + y * y) + z * z);
    const double c = nrm * nrm - outeredge * outeredge;
    dd = (-b + sqrt(b * b - 4 * 1 * c)) / 2;
    dd_out[i] = dd;
    if (key_out) {
      double t = -(x * bx + y * by + z * bz);
      if (!(t > 0.0)) t = 0.0;
      const double cpa[3] = {x + bx * t, y + by * t, z + bz * t};
      unsigned q[3];
#pragma unroll
      for (int a = 0; a < 3; ++a) {
        double v = (cpa[a] + 6.4) / 0.4;
        v = v < 0.0 ? 0.0 : (v > 31.0 ? 31.0 : v);
        q[a] = (v == v) ? (unsigned)v : 0u;
      }
      const unsigned key = morton_spread5(q[0]) | (morton_spread5(q[1]) << 1) | (morton_spread5(q[2]) << 2);
      key_out[i] = key;
      atomicAdd(&hist[key], 1u);
    }
  }
  // block maximum of the positive, non-NaN dd (bit patterns of positive doubles are ordered)
  unsigned long long bits = (dd > 0.0) ? (unsigned long long)__double_as_longlong(dd) : 0ull;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const unsigned long long other = __shfl_xor_sync(0xffffffffu, bits, o);
    bits = other > bits ? other : bits;
  }
  if ((threadIdx.x & 31) == 0 && bits) atomicMax(ddmax_bits, bits);
}
__global__ void __launch_bounds__(1024) k_los_key_scan(unsigned* __restrict__ hist) {
  __shared__ unsigned part[1024];
  const int per = NX_LOS_KEYS / 1024;
  unsigned local[NX_LOS_KEYS / 1024];
  unsigned run = 0;
#pragma unroll
  for (int k = 0; k < per; ++k) { local[k] = run; run += hist[threadIdx.x * per + k]; }
  part[threadIdx.x] = run;
  __syncthreads();
  for (int o = 1; o < 1024; o <<= 1) {
    const unsigned v = threadIdx.x >= (unsigned)o ? part[threadIdx.x - o] : 0u;
    __syncthreads();
    part[threadIdx.x] += v;
    __syncthreads();
  }
  const unsigned base = part[threadIdx.x] - run;
#pragma unroll
  for (int k = 0; k < per; ++k) hist[threadIdx.x * per + k] = base + local[k];
}
__global__ void __launch_bounds__(256)
k_los_finish(const double* __restrict__ dd, const double* __restrict__ ladder, int nladder,
             long long nlos, int* __restrict__ nball, const unsigned* __restrict__ key,
             unsigned* __restrict__ cursor, unsigned* __restrict__ order) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= nlos) return;
  const double d = dd[i];
  int k = 0;
  if (d == d) {                           // first k with t_k >= dd; NaN dd -> single entry
    int lo = 0, hi = nladder;
    while (lo < hi) {
      const int mid = (lo + hi) >> 1;
      if (ladder[mid] < d) lo = mid + 1; else hi = mid;
    }
    k = lo >= nladder ? nladder - 1 : lo;
  }
  nball[i] = k + 1;
  if (order) order[atomicAdd(&cursor[key[i]], 1u)] = (unsigned)i;
}

cudaError_t launch_los_prepare(cudaStream_t st, const double* los, long long nlos, double outeredge,
                               double* dd, unsigned* key, unsigned* hist,
                               unsigned long long* ddmax_bits) {
  cudaError_t e;
  if ((e = cudaMemsetAsync(ddmax_bits, 0, sizeof(unsigned long long), st)) != cudaSuccess) return e;
  if (key && (e = cudaMemsetAsync(hist, 0, NX_LOS_KEYS * sizeof(unsigned), st)) != cudaSuccess) return e;
  k_los_prepare<<<(unsigned)((nlos + 255) / 256), 256, 0, st>>>(los, nlos, outeredge, dd, key, hist,
                                                                  ddmax_bits);
  return cudaGetLastError();
}
cudaError_t launch_los_finish(cudaStream_t st, const double* dd, const double* ladder, int nladder,
                              long long nlos, int* nball, const unsigned* key, unsigned* hist,
                              unsigned* order) {
  if (order) k_los_key_scan<<<1, 1024, 0, st>>>(hist);
  k_los_finish<<<(unsigned)((nlos + 255) / 256), 256, 0, st>>>(dd, ladder, nladder, nlos, nball, key,
                                                                 hist, order);
  return cudaGetLastError();
}

// The exact test + weights over a pair list that is already on the device (the pairs a
// single-batch launch_los_grid left in w.pairs).
cudaError_t launch_los_resolve(cudaStream_t st, LosGridWork& w, unsigned long long np, long long nlos,
                               const double* los, const double* dist_plan, const int* nball,
                               const double* ladder, const double* wid2, const LosParams& lp,
                               const LosConsts& lc, const GTables& G, double* radiance,
                               unsigned long long* npack, unsigned char* included,
                               unsigned long long* nused, const long long* used_off,
                               unsigned long long* used_cursor, unsigned* used_idx) {
  if (!np) return cudaSuccess;
  launch_resolve_pairs(st, w, np, nlos, los, dist_plan, nball, ladder, wid2, lp, lc, G, radiance,
                       npack, included, nused, used_off, used_cursor, used_idx, nullptr);
  return cudaGetLastError();
}

// ---------------------------------------------------------------------------
// K7: number density, sums over the saved rows inside a ball around every sample point
// (ModelDensity).  The rows are the ones K5 reads (float32-rounded, frac == 0 dropped), in
// the same cell order, so the grid is launch_los_grid_build's.
//   k_density_plan: per point (in the host's Morton order) the cell box of [p - r, p + r]
//                   per axis (cell_of is monotone: an index range per axis) and the number
//                   of work items, one per 32 (ix, iy) columns of the box;
//   scan          : the three K5 scan kernels turn the item counts into item offsets;
//   k_density     : persistent warps take items from a ticket counter; lane c of the warp
//                   finds the packet range of column c of the item (the z cells of the box),
//                   then the warp streams the ranges, coalesced, through the exact membership
//                   test (nx_image.cuh: density_member) and adds S1 = sum frac,
//                   S2 = sum frac^2 and the member count of the item to the point's totals
//                   with f64 / u64 atomics.  A ball near the planet spans hundreds of columns
//                   and most of the packets: its items spread over many warps instead of
//                   keeping one warp busy after the others are done.
// ---------------------------------------------------------------------------
#define NX_DENSITY_WARPS 8
#define NX_DENSITY_MINBLOCKS 4      // <= 64 registers: 32 resident warps per SM
#define NX_DENSITY_COLS 32          // (ix, iy) columns per work item (one per lane)

__global__ void __launch_bounds__(256)
k_density_plan(long long npts, long long stride, const double* __restrict__ pts,
               const double* __restrict__ rad, const unsigned* __restrict__ order, LosGrid g,
               int* __restrict__ box, unsigned* __restrict__ nitem) {
  const long long j = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= npts) return;
  const long long i = order[j];
  const double p[3] = {pts[i], pts[stride + i], pts[2 * stride + i]};
  // a member's |x - p| can exceed r by the rounding of d2: pad the box by far more
  const double rr = rad[i] * (1.0 + 1e-9) + 1e-12;
  int lo[3], hi[3];
  bool empty = !(rr > 0.0);
#pragma unroll
  for (int a = 0; a < 3; ++a) {
    if (p[a] - rr > g.half || p[a] + rr < -g.half) empty = true;       // outside the packet cube
    lo[a] = cell_of(p[a] - rr, g);
    hi[a] = cell_of(p[a] + rr, g);
  }
#pragma unroll
  for (int a = 0; a < 3; ++a) { box[6 * j + 2 * a] = lo[a]; box[6 * j + 2 * a + 1] = hi[a]; }
  const unsigned ncol = (unsigned)((hi[0] - lo[0] + 1) * (hi[1] - lo[1] + 1));
  nitem[j] = empty ? 0u : (ncol + NX_DENSITY_COLS - 1) / NX_DENSITY_COLS;
}

__global__ void __launch_bounds__(32 * NX_DENSITY_WARPS, NX_DENSITY_MINBLOCKS)
k_density(LosSorted S, LosGrid g, const unsigned* __restrict__ start, long long npts,
          const int* __restrict__ box, const unsigned* __restrict__ item_off,
          const unsigned* __restrict__ nitems, const unsigned* __restrict__ order, long long stride,
          const double* __restrict__ pts, const double* __restrict__ rad, double* __restrict__ s1,
          double* __restrict__ s2, unsigned long long* __restrict__ count,
          unsigned* __restrict__ cursor) {
  const unsigned lane = threadIdx.x & 31u;
  const float4* __restrict__ recs = reinterpret_cast<const float4*>(S.pos);
  const float* __restrict__ fracs = reinterpret_cast<const float*>(S.frac);
  const unsigned total = *nitems;
  for (;;) {
    unsigned t = 0;
    if (lane == 0) t = atomicAdd(cursor, 1u);
    t = __shfl_sync(FULL_MASK, t, 0);
    if (t >= total) return;
    // the point of item t: the last slot j with item_off[j] <= t (item_off[npts] = total > t)
    long long lo = 0, hi = npts;
    while (hi - lo > 1) {
      const long long mid = (lo + hi) >> 1;
      if (__ldg(item_off + mid) <= t) lo = mid; else hi = mid;
    }
    const long long j = lo;
    const long long i = order[j];
    const double px = pts[i], py = pts[stride + i], pz = pts[2 * stride + i], r = rad[i];
    const int ix0 = box[6 * j], ix1 = box[6 * j + 1], iy0 = box[6 * j + 2], iy1 = box[6 * j + 3];
    const int iz0 = box[6 * j + 4], iz1 = box[6 * j + 5];
    const int ny = iy1 - iy0 + 1, ncol = (ix1 - ix0 + 1) * ny;
    const int c0 = (int)(t - item_off[j]) * NX_DENSITY_COLS;
    const int c = c0 + (int)lane;
    unsigned p0v = 0u, p1v = 0u;
    if (c < ncol) {
      const unsigned row = (unsigned)(((ix0 + c / ny) * g.G + iy0 + c % ny) * g.G);
      p0v = __ldg(start + row + iz0);
      p1v = __ldg(start + row + iz1 + 1);
    }
    const int nc = min(NX_DENSITY_COLS, ncol - c0);
    double a1 = 0.0, a2 = 0.0;
    unsigned m = 0;
    for (int k = 0; k < nc; ++k) {
      const unsigned p0 = __shfl_sync(FULL_MASK, p0v, k), p1 = __shfl_sync(FULL_MASK, p1v, k);
      for (unsigned qb = p0; qb < p1; qb += 64) {
        const unsigned q0 = qb + lane, q1 = q0 + 32u;
        float4 ra, rb;
        if (q0 < p1) ra = __ldg(recs + q0);
        if (q1 < p1) rb = __ldg(recs + q1);
        if (q0 < p1 && density_member(ra.x, ra.y, ra.z, px, py, pz, r)) {
          const double f = (double)__ldg(fracs + q0);
          a1 += f; a2 += f * f; ++m;           // f * f: exact (24-bit mantissas)
        }
        if (q1 < p1 && density_member(rb.x, rb.y, rb.z, px, py, pz, r)) {
          const double f = (double)__ldg(fracs + q1);
          a1 += f; a2 += f * f; ++m;
        }
      }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      a1 += __shfl_xor_sync(FULL_MASK, a1, o);
      a2 += __shfl_xor_sync(FULL_MASK, a2, o);
      m += __shfl_xor_sync(FULL_MASK, m, o);
    }
    if (lane == 0 && m) {
      atomicAdd(s1 + i, a1);
      atomicAdd(s2 + i, a2);
      atomicAdd(count + i, (unsigned long long)m);
    }
  }
}

cudaError_t launch_density(cudaStream_t st, int device, const LosGridWork& w, long long npts,
                           const double* pts, const double* rad, const unsigned* order,
                           int* box, unsigned* nitem, unsigned* item_off, unsigned* cursor, double* s1,
                           double* s2, unsigned long long* count, int* nlaunch) {
  int sms = 148;
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device);
  cudaError_t e;
  for (long long first = 0; first < npts; first += NX_DENSITY_BATCH) {
    const long long nb = npts - first < NX_DENSITY_BATCH ? npts - first : NX_DENSITY_BATCH;
    k_density_plan<<<(unsigned)((nb + 255) / 256), 256, 0, st>>>(nb, npts, pts, rad, order + first,
                                                                  w.grid, box, nitem);
    // item counts -> offsets; item_off[nb] = the item total
    const int nsb = (int)((nb + NX_SCAN_ELEMS - 1) / NX_SCAN_ELEMS);
    k_scan_partial<<<nsb, 1024, 0, st>>>(nitem, item_off, w.block_sum, (int)nb);
    k_scan_top<<<1, 1024, 0, st>>>(w.block_sum, nsb, w.total);
    k_scan_add<<<nsb, 1024, 0, st>>>(item_off, w.block_sum, (int)nb, w.total);
    if ((e = cudaMemsetAsync(cursor, 0, sizeof(unsigned), st)) != cudaSuccess) return e;
    // the item total stays on the device: the warps read it, the host does not wait for it
    k_density<<<(unsigned)sms * NX_DENSITY_MINBLOCKS, 32 * NX_DENSITY_WARPS, 0, st>>>(
        w.sorted, w.grid, w.start, nb, box, item_off, w.total, order + first, npts, pts, rad, s1,
        s2, count, cursor);
    if (nlaunch) *nlaunch += 5;
  }
  return cudaGetLastError();
}

}  // namespace nx
