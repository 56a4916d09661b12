// nexoclom_b200 -- sm_100a kernels K1..K5.
//
//  K1 k_init_state            HBM-write bound   (14 + 9 f64 columns per packet)
//  K2 k_integrate_adaptive    FP64-pipe bound   persistent lanes, per-lane refill
//  K3 k_integrate_constant    FP64-pipe bound   + fused per-step image atomics
//  K4 k_image_accumulate      HBM-read bound    40 B/packet + L2 atomics
//  K5 k_los_accumulate        FP64-pipe bound   LOS-per-thread x packet tiles in smem
//
// Packet state lives in HBM as structure-of-arrays (one f64 column per field, all
// columns of one slab, column stride = capacity rounded to 32) so that a warp's
// loads/stores of one field are one or two fully-used 128-byte lines.
#include <cuda_runtime.h>
#include <stdint.h>

#include <cmath>

#include "nx_fast.cuh"
#include "nx_image.cuh"
#include "nx_init.cuh"
#include "nx_kernels.h"
#include "nx_physics.cuh"
#include "nx_surface.cuh"

namespace nx {

#define FULL_MASK 0xffffffffu

#ifdef NX_STREAM_DEBUG
// developer instrumentation of K2 (never compiled into the product library):
// [0] start ns, [1..8] first time class c ran out, [16] last warp exit ns, [17] warp
// iterations, [18] feeder scans, [32..] live lane-steps per 0.25 ms of run time
__device__ unsigned long long g_dbg[512];
__device__ __forceinline__ unsigned long long dbg_now() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
  return t;
}
#define NX_DBG_ITER(havemask)                                                        \
  do {                                                                               \
    ++dbg_iters;                                                                     \
    const unsigned hm_ = (havemask);   /* evaluated by ALL lanes (it is a ballot) */   \
    if ((threadIdx.x & 31u) == 0) {                                                  \
      unsigned long long b_ = (dbg_now() - g_dbg[0]) / 250000ull;                    \
      if (b_ > 400) b_ = 400;                                                        \
      atomicAdd(&g_dbg[32 + b_], (unsigned long long)__popc(hm_));                   \
    }                                                                                \
  } while (0)
#else
#define NX_DBG_ITER(havemask) do { } while (0)
#endif

// ---------------------------------------------------------------------------
// shared-memory staging of an np.interp table (x, f, slope, bucket index)
// ---------------------------------------------------------------------------
__device__ __forceinline__ size_t stage_table(const InterpTable& g, InterpTable& s,
                                              unsigned char* base) {
  // pointers are ALWAYS derived from the shared-memory base so that the compiler
  // can prove the address space (LDS instead of generic LD)
  double* sx = reinterpret_cast<double*>(base);
  double* sf = sx + g.n;
  double* ss = sf + g.n;
  unsigned short* sb = reinterpret_cast<unsigned short*>(ss + g.n);
  for (int i = threadIdx.x; i < g.n; i += blockDim.x) {
    sx[i] = g.x[i]; sf[i] = g.f[i]; ss[i] = g.slope[i];
  }
  const int nb = g.n ? g.nbucket : 0;
  for (int i = threadIdx.x; i < nb; i += blockDim.x) sb[i] = g.bucket[i];
  s.x = sx; s.f = sf; s.slope = ss; s.bucket = sb;
  s.n = g.n; s.nbucket = g.nbucket; s.blo = g.blo; s.binvw = g.binvw;
  size_t bytes = (size_t)g.n * 24 + (size_t)nb * 2;
  return (bytes + 15) & ~(size_t)15;
}

// fast path: interval records in shared memory, the (large) bucket index stays in
// global memory and is served by L1
// with_bucket: small bucket indices (the g-value tables of K4: a few hundred buckets) are
// staged too, so a lookup never leaves shared memory -- with a ~200 KB shared-memory
// carve-out the L1 that would serve a global bucket index is down to a few KB.
#define NX_SMEM_BUCKET_MAX 8192
__device__ __forceinline__ void stage_fast_table(const FastTable& g, FastTable& s,
                                                 unsigned char* base, bool with_bucket = false) {
  double4* sr = reinterpret_cast<double4*>(base);
  const double4* gr = reinterpret_cast<const double4*>(g.rec);
  for (int i = threadIdx.x; i < g.nrec; i += blockDim.x) sr[i] = gr[i];   // 32 B per record
  s.rec = reinterpret_cast<const InterpRec*>(sr);
  s.bucket = g.bucket;
  if (with_bucket && g.nbucket <= NX_SMEM_BUCKET_MAX) {
    unsigned short* sb = reinterpret_cast<unsigned short*>(sr + g.nrec);
    for (int i = threadIdx.x; i < g.nbucket; i += blockDim.x) sb[i] = g.bucket[i];
    s.bucket = sb;
  }
  s.nrec = g.nrec; s.nbucket = g.nbucket; s.blo = g.blo; s.binvw = g.binvw; s.boff = g.boff;
}

__device__ __forceinline__ size_t fast_table_smem_bytes_dev(const FastTable& g) {
  size_t b = (size_t)g.nrec * 32;
  if (g.nbucket <= NX_SMEM_BUCKET_MAX) b += ((size_t)g.nbucket * 2 + 15) & ~(size_t)15;
  return b;
}
size_t fast_table_smem_bytes(const FastTable& g, bool with_bucket = false) {
  size_t b = (size_t)g.nrec * 32;
  if (with_bucket && g.nbucket <= NX_SMEM_BUCKET_MAX) b += ((size_t)g.nbucket * 2 + 15) & ~(size_t)15;
  return b;
}

// g-value tables of K4 in shared memory: the sum table alone when there is one
__device__ __forceinline__ size_t stage_gtables(const GTables& Gg, GTables& G, unsigned char* base) {
  G.n = Gg.n; G.has_sum = Gg.has_sum;
  size_t off = 0;
  if (Gg.has_sum) {
    stage_fast_table(Gg.fsum, G.fsum, base, true);
    return fast_table_smem_bytes_dev(Gg.fsum);
  }
#pragma unroll
  for (int t = 0; t < NX_MAX_GTABLES; ++t)
    if (t < Gg.n) { stage_fast_table(Gg.f[t], G.f[t], base + off, true); off += fast_table_smem_bytes_dev(Gg.f[t]); }
  return off;
}
static size_t gtables_smem_bytes(const GTables& G) {
  if (G.has_sum) return fast_table_smem_bytes(G.fsum, true);
  size_t b = 0;
  for (int t = 0; t < G.n; ++t) b += fast_table_smem_bytes(G.f[t], true);
  return b;
}

size_t table_smem_bytes(const InterpTable& g) {
  if (g.n == 0) return 0;
  size_t bytes = (size_t)g.n * 24 + (size_t)g.nbucket * 2;
  return (bytes + 15) & ~(size_t)15;
}

// ---------------------------------------------------------------------------
// K1: initial state
// ---------------------------------------------------------------------------
// Only the 14 X0 columns are written (112 B per packet, the algorithmic minimum): the
// integrators read their input straight from the first eight of them and write the final
// state to the state slab, so the initial state is never stored twice.  A lane computes one
// packet; lanes 2j / 2j+1 then swap halves with one shuffle per column pair so that every
// store is a 16-byte STG of two consecutive packets (even lanes: columns 0,2,..,12, odd
// lanes: columns 1,3,..,13; 16 lanes x 16 B = one full 256-byte row segment per column).
template <bool FAST>
__global__ void __launch_bounds__(256)
k_init_state(X0Cols X, long long n, SourceParams sp, SourceMap map, InterpTable speed,
             InterpTable lon1d, uint64_t seed, uint64_t first_id) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long ic = i < n ? i : n - 1;            // whole warps run the shuffles
  const unsigned lane = threadIdx.x & 31u;
  double x0[14];
  init_packet<FAST>(sp, map, speed, seed, first_id + (uint64_t)ic, x0, lon1d);
  const bool odd = lane & 1u;
  const long long pair0 = i & ~1LL;                  // first packet of this lane pair
  const bool full = pair0 + 1 < n;                   // both packets of the pair exist
#pragma unroll
  for (int k = 0; k < 14; k += 2) {
    const double mine = odd ? x0[k] : x0[k + 1];
    const double other = __shfl_xor_sync(FULL_MASK, mine, 1);
    if (full) {
      if (!odd) __stcs(reinterpret_cast<double2*>(X.c[k] + pair0), make_double2(x0[k], other));
      else __stcs(reinterpret_cast<double2*>(X.c[k + 1] + pair0), make_double2(other, x0[k + 1]));
    } else if (i < n) {                              // last packet of an odd n
      X.c[k][i] = x0[k]; X.c[k + 1][i] = x0[k + 1];
    }
  }
}

// The pure deviate -> state transform of K1 on caller-supplied deviates (import mode for
// reference-generated draws; the parity tests replay the reference's recorded deviates
// through this entry on the device).  lon_in / lat_in: surface points sampled elsewhere
// (rejection sampling on a map), or null for the uniform band.
__global__ void __launch_bounds__(256)
k_init_from_deviates(X0Cols X, long long n, SourceParams sp, InterpTable speed,
                     InterpTable lon1d, const double* __restrict__ u_time, const double* __restrict__ u_sinlat,
                     const double* __restrict__ u_lon, const double* __restrict__ lon_in,
                     const double* __restrict__ lat_in, const double* __restrict__ u_speed,
                     const double* __restrict__ z_normal, const double* __restrict__ u_alt,
                     const double* __restrict__ u_az) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  double lon, lat;
  if (lon_in) { lon = lon_in[i]; lat = lat_in[i]; }
  else if (sp.spatial_type == SPATIAL_LON1D) { lon = interp(lon1d, u_lon[i]); lat = 0.0; }
  else uniform_lonlat(sp, u_sinlat[i], u_lon[i], lon, lat);
  double x0[14];
  init_packet_finish(sp, speed, u_time[i], lon, lat, u_speed[i], z_normal[i], u_alt[i], u_az[i],
                     x0);
#pragma unroll
  for (int k = 0; k < 14; ++k) X.c[k][i] = x0[k];
}

__global__ void k_fill(double* p, long long n, double v) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) p[i] = v;
}

// ---------------------------------------------------------------------------
// K2: adaptive driver.  Persistent lanes: every lane owns one packet at a time
// and runs whole attempted steps; a lane whose packet finished stores it and
// claims the next unprocessed packet from a global counter (warp-aggregated
// atomicAdd), so warps stay full although step counts per packet differ by
// orders of magnitude (p50 ~ 40, max ~ 4000).
// ---------------------------------------------------------------------------
// ---------------------------------------------------------------------------
// Per-warp packet feeder: the work queue is consumed in batches of 32 packets
// that are copied global -> shared memory with cp.async (LDGSTS) one batch AHEAD
// of their use, so a lane that finishes its packet picks the next one out of
// shared memory instead of stalling the whole warp on a chain of dependent
// global loads (queue index -> permutation -> 9 state columns).
// Layout per warp: 2 buffers x (8 columns x 32 doubles + 32 indices).
// ---------------------------------------------------------------------------
#define NX_FEED_COLS 8     // time,x,y,z,vx,vy,vz,frac; the step size starts at 1000 s (Output.py:246)
#define NX_FEED_BYTES_PER_WARP (2 * (NX_FEED_COLS * 32 * 8 + 32 * 4))
#define NX_INVALID 0xffffffffu
// The reference's adaptive loop never ends for a packet that makes no progress (errmax == 0
// on every attempt: no forces, no loss, v = 0 -- Output.py:294-300 rejects the step and grows
// it forever).  On the GPU that would be a kernel that cannot be interrupted, so a packet is
// retired as it is after this many attempted steps and status bit NX_INV_NO_PROGRESS is set
// (the longest packet of the 1e7-packet Na run needs 5 434).
#define NX_ATTEMPT_CAP (1u << 22)
#define NX_ST_NO_PROGRESS 128
#define NX_INITIAL_STEP 1000.0        // every packet starts with a 1000 s step (Output.py:246)

__device__ __forceinline__ void cp_async8(void* smem, const void* gmem) {
  const unsigned s = (unsigned)__cvta_generic_to_shared(smem);
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(s), "l"(gmem) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_group 0;" ::: "memory"); }

struct PacketFeeder {
  double* vals;              // this warp's staging area: [2][9][32]
  unsigned* ids;             // [2][32]
  const StateCols* P;
  const unsigned* perm;
  unsigned long long* queue;
  long long n;
  unsigned lane;
  unsigned pnext;            // queue entry this lane will prefetch next (NX_INVALID: none)
  int buf, pos, cnt;         // buffer being consumed, read position, packets in it
  int cnt_pending;           // packets of the batch in flight into buffer buf^1
  bool queue_done;

  __device__ __forceinline__ void claim_indices() {
    // claim the next 32 queue entries; the permutation load is NOT waited for here
    unsigned long long base = 0;
    if (!queue_done) {
      if (lane == 0) base = atomicAdd(queue, 32ull);
      base = __shfl_sync(FULL_MASK, base, 0);
      if ((long long)base + 32 >= n) queue_done = true;
      const long long q = (long long)base + lane;
      pnext = (q < n) ? (perm ? __ldg(perm + q) : (unsigned)q) : NX_INVALID;
    } else {
      pnext = NX_INVALID;
    }
  }
  __device__ __forceinline__ void issue_prefetch() {
    const unsigned my = pnext;
    const unsigned valid = __ballot_sync(FULL_MASK, my != NX_INVALID);
    cnt_pending = __popc(valid);
    if (cnt_pending) {
      const int b = buf ^ 1;
      if (my != NX_INVALID) {
        double* dst = vals + (size_t)b * NX_FEED_COLS * 32 + lane;
#pragma unroll
        for (int k = 0; k < NX_FEED_COLS; ++k) cp_async8(dst + k * 32, P->c[k] + my);
        ids[b * 32 + lane] = my;
      }
      cp_async_commit();
    }
    claim_indices();
  }
  __device__ __forceinline__ void init(unsigned char* smem, const StateCols* P_,
                                       const unsigned* perm_, unsigned long long* queue_,
                                       long long n_) {
    const unsigned warp = threadIdx.x >> 5;
    lane = threadIdx.x & 31u;
    vals = reinterpret_cast<double*>(smem + (size_t)warp * NX_FEED_BYTES_PER_WARP);
    ids = reinterpret_cast<unsigned*>(vals + 2 * NX_FEED_COLS * 32);
    P = P_; perm = perm_; queue = queue_; n = n_;
    buf = 0; pos = 0; cnt = 0; cnt_pending = 0; queue_done = false; pnext = NX_INVALID;
    claim_indices();
    issue_prefetch();
  }
  // make the pending batch current; returns false when nothing is left
  __device__ __forceinline__ bool advance() {
    if (cnt_pending == 0) return false;
    cp_async_wait_all();
    __syncwarp();
    buf ^= 1; pos = 0; cnt = cnt_pending;
    issue_prefetch();
    return true;
  }
};

// MODE: -1 = strict (NumPy operation order, runtime force flags);
//       otherwise fast arithmetic with compile-time forces:
//       MODE = GR*8 + RP*4 + LOSS.
// BOUNCE: packets that hit the surface bounce (adaptive_attempt<.., true>), the deviates of
// packet idx are keyed by (seed, first_id + idx); totals[2] receives the number of bounces.
// S / seed / first_id are unused otherwise.
// SINK: the deposition sink (ModelDeposition): the attempts record every surface, moon, escape
// and vanish event (deposit_record), the kernel the initial frac (SOURCE) and the frac of the
// packets that retire alive (REMAINING); Dep is unused otherwise.  The final state and the
// step totals are the same as without the sink.
// ION: the ion-production sink (ModelIonization, k_ionize_adaptive): the attempts record the
// frac every accepted step loses in flight (ion_record), each lane its OUTSIDE share, reduced
// here; Ion is unused otherwise.  The final state and the step totals are again unchanged.
// TRACE: the trajectory sink (ModelTrajectoryImage / ModelTrajectoryDensity,
// k_trace_adaptive): the lane keeps T - t0 of its packet from the moment it loads it, the
// attempts record every accepted step (trace_record) into *Tro, each lane its OUTSIDE share of
// the grid, reduced here; Tro is unused otherwise.  The final state and the step totals are
// again unchanged.
// The persistent lane loop of the kernels (feeder, refill, step totals), inlined into each.
template <int MODE, bool BOUNCE, bool SINK, bool ION, bool TRACE = false>
__device__ __forceinline__ void
adaptive_lanes(const StateCols& In, const StateCols& P, long long n, const RunParams& p,
               const InterpTable& Tg, const FastTable& Fg, const unsigned* __restrict__ perm,
               unsigned long long* __restrict__ queue, unsigned long long* __restrict__ totals,
               unsigned* __restrict__ att_out, unsigned* __restrict__ acc_out,
               int* __restrict__ status, unsigned table_bytes, const Spline2D& S, uint64_t seed,
               uint64_t first_id, const DepositOut& Dep, const IonOut& Ion,
               const TraceOut* Tro = nullptr) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  InterpTable T;
  FastTable F;
  if (MODE < 0) stage_table(Tg, T, smem_raw);
  else stage_fast_table(Fg, F, smem_raw);
  PacketFeeder feed;
  feed.init(smem_raw + table_bytes, &In, perm, queue, n);
  __syncthreads();

  // In: where the initial state is read (the X0 slab right after K1, else the state slab
  // itself); P: where the final state goes.  Packets that need no integration are passed
  // through when the two differ.
  const bool pass_through = In.c[0] != P.c[0];
  const unsigned lane = threadIdx.x & 31u;
  bool have = false, drained = false;
  unsigned idx = 0;
  double s[8], step = 0.0;
  unsigned att = 0, acc = 0;
  unsigned long long tot_att = 0, tot_acc = 0, tot_bnc = 0;
  int st = 0;
  DepositSink D;                 // SINK: lives in local memory, touched on events only
  if (SINK) {
    D.map = Dep.map; D.cnt = Dep.cnt; D.nlon = Dep.nlon; D.nlat = Dep.nlat;
#pragma unroll
    for (int b = 0; b < DEP_NBUCKET; ++b) { D.sum[b] = 0.0; D.n[b] = 0; }
  }
  IonSink I;                     // ION: lives in local memory, the grid read by ion_record
  if (ION) { I.g = Ion; I.out_sum = 0.0; I.out_n = 0; }
  TraceSink Tr;                  // TRACE: lives in local memory, the launch's sink read through o
  if (TRACE) { Tr.o = Tro; Tr.age0 = 0.0; Tr.out_sum = 0.0; Tr.out_n = 0; }
#ifdef NX_STREAM_DEBUG
  unsigned long long dbg_iters = 0;
#endif

  for (;;) {
    unsigned need = __ballot_sync(FULL_MASK, !have);
    while (need && !drained) {
      if (feed.pos == feed.cnt && !feed.advance()) { drained = true; break; }
      const int take = min(__popc(need), feed.cnt - feed.pos);
      const int rank = __popc(need & ((1u << lane) - 1u));
      if (!have && rank < take) {
        const int slot = feed.pos + rank;
        const double* v = feed.vals + (size_t)feed.buf * NX_FEED_COLS * 32 + slot;
#pragma unroll
        for (int k = 0; k < 8; ++k) s[k] = v[k * 32];
        step = NX_INITIAL_STEP;
        idx = feed.ids[feed.buf * 32 + slot];
        att = 0; acc = 0;
        have = (s[0] > p.resolution) && (s[7] > 0.0);
        if (TRACE && have) Tr.age0 = sub_rn(Tro->endtime, s[0]);
        if (SINK && s[7] > 0.0) {
          D.sum[DEP_SOURCE] += s[7]; ++D.n[DEP_SOURCE];
          if (!have) { D.sum[DEP_REMAINING] += s[7]; ++D.n[DEP_REMAINING]; }
        }
        if (!have) {
          att_out[idx] = 0; acc_out[idx] = 0;
          if (pass_through) {
#pragma unroll
            for (int k = 0; k < 8; ++k) __stcs(P.c[k] + idx, s[k]);
            __stcs(P.c[8] + idx, step);
          }
        }
      }
      feed.pos += take;
      need = __ballot_sync(FULL_MASK, !have);
    }
    if (!__any_sync(FULL_MASK, have)) {
      if (drained) break;
      continue;
    }
    NX_DBG_ITER(__ballot_sync(FULL_MASK, have));
    if (have) {
      int fl;
      if (MODE < 0)
        fl = adaptive_attempt<true, BOUNCE, SINK, ION, TRACE>(p, T, s, step, &S, seed,
                                                              first_id + idx, acc + 1,
                                                              SINK ? &D : nullptr,
                                                              ION ? &I : nullptr,
                                                              TRACE ? &Tr : nullptr);
      else
        fl = adaptive_attempt_fast<(MODE >> 3) & 1, (MODE >> 2) & 1, MODE & 3, (MODE >> 4) & 1, BOUNCE,
                                   SINK, ION, TRACE>(p, F, s, step, &S, seed, first_id + idx,
                                                     acc + 1, SINK ? &D : nullptr,
                                                     ION ? &I : nullptr, TRACE ? &Tr : nullptr);
      ++att;
      if (fl & ATT_ACCEPTED) ++acc;
      if (BOUNCE && (fl & ATT_BOUNCED)) ++tot_bnc;
      st |= fl & ~(ATT_ACCEPTED | ATT_LIVE | (BOUNCE ? ATT_BOUNCED : 0));
      if (att >= NX_ATTEMPT_CAP) { st |= NX_ST_NO_PROGRESS; fl &= ~ATT_LIVE; }
      if (!(fl & ATT_LIVE)) {
#pragma unroll
        for (int k = 0; k < 8; ++k) __stcs(P.c[k] + idx, s[k]);
        __stcs(P.c[8] + idx, step);
        att_out[idx] = att; acc_out[idx] = acc;
        tot_att += att; tot_acc += acc;
        if (SINK && s[7] > 0.0) { D.sum[DEP_REMAINING] += s[7]; ++D.n[DEP_REMAINING]; }
        have = false;
      }
    }
  }
  // block-level totals
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    tot_att += __shfl_xor_sync(FULL_MASK, tot_att, o);
    tot_acc += __shfl_xor_sync(FULL_MASK, tot_acc, o);
    if (BOUNCE) tot_bnc += __shfl_xor_sync(FULL_MASK, tot_bnc, o);
    st |= __shfl_xor_sync(FULL_MASK, st, o);
  }
  if (lane == 0) {
    if (tot_att) atomicAdd(&totals[0], tot_att);
    if (tot_acc) atomicAdd(&totals[1], tot_acc);
    if (BOUNCE && tot_bnc) atomicAdd(&totals[2], tot_bnc);
    if (st) atomicOr(status, st);
#ifdef NX_STREAM_DEBUG
    atomicMax(&g_dbg[16], dbg_now());
    atomicAdd(&g_dbg[17], dbg_iters);
#endif
  }
  if (SINK) {
#pragma unroll
    for (int b = 0; b < DEP_NBUCKET; ++b) {
      double v = D.sum[b];
      unsigned long long c = D.n[b];
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        v += __shfl_xor_sync(FULL_MASK, v, o);
        c += __shfl_xor_sync(FULL_MASK, c, o);
      }
      if (lane == 0 && c) {
        atomicAdd(Dep.bucket + b, v);
        atomicAdd(Dep.bucket_n + b, c);
      }
    }
  }
  if (ION) {
    double v = I.out_sum;
    unsigned long long c = I.out_n;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      v += __shfl_xor_sync(FULL_MASK, v, o);
      c += __shfl_xor_sync(FULL_MASK, c, o);
    }
    if (lane == 0 && c) {
      const long long out = (long long)Ion.n[0] * Ion.n[1] * Ion.n[2];
      atomicAdd(Ion.sum + out, v);
      atomicAdd(Ion.cnt + out, c);
    }
  }
  if (TRACE && Tro->grid.sum) {
    double v = Tr.out_sum;
    unsigned long long c = Tr.out_n;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      v += __shfl_xor_sync(FULL_MASK, v, o);
      c += __shfl_xor_sync(FULL_MASK, c, o);
    }
    if (lane == 0 && c) {
      const IonOut& g = Tro->grid;
      const long long out = (long long)g.n[0] * g.n[1] * g.n[2];
      atomicAdd(g.sum + out, v);
      atomicAdd(g.cnt + out, c);
    }
  }
}

template <int MODE, bool BOUNCE = false, bool SINK = false>
__global__ void __launch_bounds__(NX_INT_THREADS, NX_INT_MINBLOCKS)
k_integrate_adaptive(StateCols In, StateCols P, long long n, RunParams p, InterpTable Tg,
                     FastTable Fg, const unsigned* __restrict__ perm,
                     unsigned long long* __restrict__ queue,
                     unsigned long long* __restrict__ totals,
                     unsigned* __restrict__ att_out, unsigned* __restrict__ acc_out,
                     int* __restrict__ status, unsigned table_bytes, Spline2D S, uint64_t seed,
                     uint64_t first_id, DepositOut Dep) {
  adaptive_lanes<MODE, BOUNCE, SINK, false>(In, P, n, p, Tg, Fg, perm, queue, totals, att_out,
                                            acc_out, status, table_bytes, S, seed, first_id, Dep,
                                            IonOut{});
}

// K2i: the adaptive driver with the ion-production sink (ModelIonization).  Built only where
// the run has a loss term: the strict kernel and MODE & 3 = LOSS_LIFETIME or LOSS_PHOTO.
template <int MODE, bool BOUNCE>
__global__ void __launch_bounds__(NX_INT_THREADS, NX_INT_MINBLOCKS)
k_ionize_adaptive(StateCols In, StateCols P, long long n, RunParams p, InterpTable Tg,
                  FastTable Fg, const unsigned* __restrict__ perm,
                  unsigned long long* __restrict__ queue,
                  unsigned long long* __restrict__ totals,
                  unsigned* __restrict__ att_out, unsigned* __restrict__ acc_out,
                  int* __restrict__ status, unsigned table_bytes, Spline2D S, uint64_t seed,
                  uint64_t first_id, IonOut Ion) {
  adaptive_lanes<MODE, BOUNCE, false, true>(In, P, n, p, Tg, Fg, perm, queue, totals, att_out,
                                            acc_out, status, table_bytes, S, seed, first_id,
                                            DepositOut{}, Ion);
}

// K2t: the adaptive driver with the trajectory sink (ModelTrajectoryImage /
// ModelTrajectoryDensity).  Built for every kernel the dispatch selects for a run without
// moons: the fast MODEs without bit 16, with and without bounce, and the strict kernel.
template <int MODE, bool BOUNCE>
__global__ void __launch_bounds__(NX_INT_THREADS, NX_INT_MINBLOCKS)
k_trace_adaptive(StateCols In, StateCols P, long long n, RunParams p, InterpTable Tg,
                 FastTable Fg, const unsigned* __restrict__ perm,
                 unsigned long long* __restrict__ queue,
                 unsigned long long* __restrict__ totals,
                 unsigned* __restrict__ att_out, unsigned* __restrict__ acc_out,
                 int* __restrict__ status, unsigned table_bytes, Spline2D S, uint64_t seed,
                 uint64_t first_id, const __grid_constant__ TraceOut Tro) {
  adaptive_lanes<MODE, BOUNCE, false, false, true>(In, P, n, p, Tg, Fg, perm, queue, totals,
                                                   att_out, acc_out, status, table_bytes, S, seed,
                                                   first_id, DepositOut{}, IonOut{}, &Tro);
}

// ---------------------------------------------------------------------------
// Longest-first scheduling.  Attempted steps per packet span 1 .. ~10^4, and one
// packet's steps are strictly sequential, so a long packet claimed late leaves
// the whole GPU waiting for one lane.  k_cost_* predict the step count from the
// Kepler flight time and the position-error step bound h ~ 40 res (1+r)/v, bin
// it in half-octaves and counting-sort packet indices, longest first.  The
// prediction only orders the queue; it never touches the physics.
// ---------------------------------------------------------------------------
#define NX_NBUCKET 32

// Predicted attempted steps of a packet, in float (it only orders the queue): Kepler flight
// time to the surface for bound orbits that dip below it, else the time the packet has left,
// over the position-error step bound.  to_surface = false (bounce runs: a packet that reaches
// the surface goes on hopping) always budgets the time left.
__device__ __forceinline__ float cost_estimate_f(const RunParams& p, int model, float res, float mu,
                                                float amax, double td, double xd, double yd,
                                                double zd, double vxd, double vyd, double vzd,
                                                bool to_surface = true) {
  const float t = (float)td, x = (float)xd, y = (float)yd, z = (float)zd;
  const float vx = (float)vxd, vy = (float)vyd, vz = (float)vzd;
  const float r2 = x * x + y * y + z * z, r = sqrtf(r2);
  const float v2 = vx * vx + vy * vy + vz * vz, v = sqrtf(v2);
  const float rv = x * vx + y * vy + z * vz;
  float tfl = t;
  const float en = 0.5f * v2 - mu / r;
  if (to_surface && p.gravity && en < 0.0f && mu > 0.0f) {
    const float a = -mu / (2.0f * en);
    const float l2 = fmaxf(r2 * v2 - rv * rv, 0.0f);
    const float e = sqrtf(fmaxf(1.0f + 2.0f * en * l2 / (mu * mu), 0.0f));
    if (a * (1.0f - e) < 1.0f && e > 1e-6f) {
      const float c1 = fminf(fmaxf((1.0f - 1.0f / a) / e, -1.0f), 1.0f);
      const float c0 = fminf(fmaxf((1.0f - r / a) / e, -1.0f), 1.0f);
      const float E1 = acosf(c1);
      float E0 = acosf(c0);
      if (rv < 0.0f) E0 = 6.2831853f - E0;
      const float Ei = 6.2831853f - E1;
      const float dM = (Ei - e * sinf(Ei)) - (E0 - e * sinf(E0));
      const float tk = dM * sqrtf(a * a * a / mu);
      bool perturbed = (model == 2) && p.radpres && (amax * tk > 0.15f * v);
      // model 3 (default): radiation pressure of the order of the local gravity lifts a hop
      // off the surface for good once the launch speed passes a sharp threshold (Na at
      // Mercury, amax = 0.98 g: v > 0.43 v_esc; those packets are 1 % of the run, 22 % of its
      // steps and held EVERY packet above 3000 steps, yet the ballistic hop predicted ~100).
      // With u = v / v_esc(r): flagged when 4.5 (amax / g) u^2 > (1 - u^2)^2  (u > 0.40 there)
      if (model == 3 && p.radpres) {
        const float u2 = 0.5f * v2 * r / mu, w = 1.0f - u2;
        perturbed = 4.5f * amax * r2 * u2 > mu * w * w;
      }
      if (tk > 0.0f && tk < tfl && !perturbed) tfl = tk;
    }
  }
  return tfl * v / (40.0f * res * (1.0f + r)) + 4.0f;
}
__device__ __forceinline__ int cost_bucket(const RunParams& p, int model, double t, double x, double y,
                                           double z, double vx, double vy, double vz, double f,
                                           bool to_surface) {
  if (!(t > p.resolution) || !(f > 0.0)) return 0;
  const float est = cost_estimate_f(p, model, (float)p.resolution, (float)fabs(p.GM),
                                    (float)p.radpres_amax, t, x, y, z, vx, vy, vz, to_surface);
  const int b = (int)(2.0f * log2f(est));
  return b < 0 ? 0 : (b > NX_NBUCKET - 1 ? NX_NBUCKET - 1 : b);
}

__global__ void __launch_bounds__(256)
k_cost_histogram(StateCols P, long long n, RunParams p, int model, bool to_surface,
                 unsigned char* __restrict__ bucket, unsigned* __restrict__ hist) {
  __shared__ unsigned sh[8][NX_NBUCKET];            // one histogram per warp (most packets
  sh[threadIdx.x >> 5][threadIdx.x & 31] = 0;       // share three or four buckets)
  __syncthreads();
  unsigned* mine = sh[threadIdx.x >> 5];
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    const int b = cost_bucket(p, model, P.c[0][i], P.c[1][i], P.c[2][i], P.c[3][i], P.c[4][i],
                              P.c[5][i], P.c[6][i], P.c[7][i], to_surface);
    bucket[i] = (unsigned char)b;
    atomicAdd(&mine[b], 1u);
  }
  __syncthreads();
  if (threadIdx.x < NX_NBUCKET) {
    unsigned c = 0;
#pragma unroll
    for (int w = 0; w < 8; ++w) c += sh[w][threadIdx.x];
    if (c) atomicAdd(&hist[threadIdx.x], c);
  }
}

// cursor[b] = number of packets in buckets > b  (descending order of cost)
__global__ void k_cost_offsets(const unsigned* __restrict__ hist, unsigned* __restrict__ cursor) {
  if (threadIdx.x == 0) {
    unsigned run = 0;
    for (int b = NX_NBUCKET - 1; b >= 0; --b) { cursor[b] = run; run += hist[b]; }
  }
}

#define NX_SCATTER_ITEMS 8
__global__ void __launch_bounds__(256)
k_cost_scatter(long long n, const unsigned char* __restrict__ bucket,
               unsigned* __restrict__ cursor, unsigned* __restrict__ perm) {
  __shared__ unsigned cnt[NX_NBUCKET], base[NX_NBUCKET];
  if (threadIdx.x < NX_NBUCKET) cnt[threadIdx.x] = 0;
  __syncthreads();
  const long long first = (long long)blockIdx.x * (256 * NX_SCATTER_ITEMS);
  int b[NX_SCATTER_ITEMS];
  unsigned r[NX_SCATTER_ITEMS];
#pragma unroll
  for (int k = 0; k < NX_SCATTER_ITEMS; ++k) {
    const long long i = first + (long long)k * 256 + threadIdx.x;
    b[k] = (i < n) ? bucket[i] : -1;
    r[k] = (b[k] >= 0) ? atomicAdd(&cnt[b[k]], 1u) : 0u;
  }
  __syncthreads();
  if (threadIdx.x < NX_NBUCKET)
    base[threadIdx.x] = cnt[threadIdx.x] ? atomicAdd(&cursor[threadIdx.x], cnt[threadIdx.x]) : 0u;
  __syncthreads();
#pragma unroll
  for (int k = 0; k < NX_SCATTER_ITEMS; ++k) {
    const long long i = first + (long long)k * 256 + threadIdx.x;
    if (b[k] >= 0) perm[base[b[k]] + r[k]] = (unsigned)i;
  }
}

// ---------------------------------------------------------------------------
// K2, class-ordered streaming queue (the default schedule).
//
// The sort above costs three extra kernels, turns every column access of K2 into a
// scattered 8-byte access, and cannot start before ALL packets are on the device.
// Here the queue stays in natural (coalesced) order and is walked NX_NCLASS times:
// pass c only hands out packets whose predicted cost class is c (longest class
// first), so long packets still start first, but a batch is 32 CONSECUTIVE packets
// (nine 256-byte rows, 16-byte cp.async.cg).  The packet range is cut into up to 32
// segments; segment s may be used once *arrived > s, which lets ONE persistent
// kernel integrate while the copy engine is still delivering later segments
// (nx_integrate_adaptive_host): lanes prefer the longest class of any segment that
// has arrived, so there is a single tail at the very end of the run instead of
// one per chunk.  The class is recomputed from the packet's INITIAL state in every
// pass (float arithmetic, deterministic): the kernel reads the initial state from
// one slab (the context's X0 columns, where the host-buffer path lands its copies)
// and writes the final state to the state slab, so the input is immutable while
// the kernel runs and every packet is handed out exactly once, in the pass of its
// class.
// ---------------------------------------------------------------------------
// measured on B200, 1e7 Na packets through the host path, 16 segments: 6 classes at
// 1024 / 2.83^c: 26.9 ms; 8 classes at 2048 / 2^c: 27.6 ms; 4 classes at 512 / 4^c: 27.7 ms
#ifndef NX_NCLASS
#define NX_NCLASS 6
#endif
#ifndef NX_CLASS_TOP
#define NX_CLASS_TOP 1024.0f         // class 0: predicted steps >= TOP; class c: >= TOP / RATIO^c
#endif
#ifndef NX_CLASS_RATIO
#define NX_CLASS_RATIO 2.83f
#endif
#define NX_GROUP 128                 // packets claimed per atomic
#define NX_SFEED_COLS 8              // time,x,y,z,vx,vy,vz,frac (the step size starts as a constant)
#define NX_SFEED_BYTES_PER_WARP (2 * NX_SFEED_COLS * 32 * 8 + 32)
#ifndef NX_SCAN_MAX
#define NX_SCAN_MAX 3                // batches scanned per step while some lane is live
#endif
#define NX_STREAM_TIMEOUT_NS 20000000000ull   // watchdog of a lane starved of segments

__device__ __forceinline__ void cp_async16_cg(void* smem, const void* gmem) {
  const unsigned s = (unsigned)__cvta_generic_to_shared(smem);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(s), "l"(gmem) : "memory");
}
__device__ __forceinline__ unsigned ld_volatile_u32(const unsigned* p) {
  unsigned v;
  asm volatile("ld.volatile.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ unsigned long long global_timer_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
  return t;
}

#define NX_FEED_INLINE __forceinline__
// cost_estimate_f() folded into NX_NCLASS classes (0 = longest)
__device__ NX_FEED_INLINE int cost_class(const RunParams& p, int model, float res, float mu,
                                          float amax, double td, double xd, double yd, double zd,
                                          double vxd, double vyd, double vzd, double fd) {
  if (!(td > p.resolution) || !(fd > 0.0)) return NX_NCLASS - 1;
  const float est = cost_estimate_f(p, model, res, mu, amax, td, xd, yd, zd, vxd, vyd, vzd);
  int cls = 0;
  float thr = NX_CLASS_TOP;
#pragma unroll
  for (int c = 0; c < NX_NCLASS - 1; ++c) {
    if (est < thr) cls = c + 1;
    thr *= (1.0f / NX_CLASS_RATIO);
  }
  return cls;
}

struct StreamQueue {
  long long seg;                     // packets per segment (multiple of NX_GROUP)
  int nseg;                          // <= 32
  int model;                         // cost model (ctx option order_packets)
  unsigned long long* cursor;        // [NX_NCLASS][32], zeroed before the launch
  const unsigned* arrived;           // segments [0, *arrived) are on the device; nullptr: all
  unsigned char* cls;                // class of every packet once known (0xFF: not yet), or nullptr
};

// Feeder state of one warp.  It lives in SHARED memory and is advanced by ONE
// non-inlined function: the whole queue logic (claims, class test with its acosf /
// sinf slow paths, prefetch) stays out of the integration loop, whose code then fits
// the 32 KB instruction cache like the sorted kernel's does (ncu: the inlined
// version spent 1.7 cycles per issue waiting for instructions).
struct StreamShared {
  unsigned char clsb[2][32];         // cached classes of the batch in staging buffer 0 / 1
  unsigned base_cur, base_pend;      // packet index of slot 0 of the current / pending batch
  int cnt_pend;                      // packets in the pending batch (0: none in flight)
  int cls_pend;
  int buf;                           // staging buffer holding the current batch
  unsigned grp_next, grp_end;        // claimed group still to be walked
  int grp_cls;
  unsigned exh[NX_NCLASS];           // bit s: cursor (class, segment s) is exhausted
  unsigned char order[32];           // slots of the current batch that belong to its class
};
#define NX_SFEED_STATE_BYTES 160     // >= sizeof(StreamShared), multiple of 16
#undef NX_SFEED_BYTES_PER_WARP
#define NX_SFEED_BYTES_PER_WARP (2 * NX_SFEED_COLS * 32 * 8 + NX_SFEED_STATE_BYTES)

struct StreamArgs {                  // everything the feeder needs, passed by value
  const double* col0;
  size_t stride;
  long long n, seg;
  unsigned long long* cursor;
  const unsigned* arrived;
  unsigned char* cls;
  double resolution;
  float res, mu, amax;
  int nseg, model, gravity, radpres;
};

// Make the next batch current.  Returns the number of packets of the batch that are
// handed out in this pass (their slots are in S->order), -1 when the queue is
// finished, -2 when nothing is available right now (segments still on the wire).
__device__ __noinline__ int stream_advance(StreamShared* S, double* vals, StreamArgs A) {
  const unsigned lane = threadIdx.x & 31u;
  const unsigned all_mask = A.nseg >= 32 ? 0xffffffffu : ((1u << A.nseg) - 1u);
  unsigned base_pend = S->base_pend, grp_next = S->grp_next, grp_end = S->grp_end;
  int cnt_pend = S->cnt_pend, cls_pend = S->cls_pend, buf = S->buf, grp_cls = S->grp_cls;
  unsigned exh[NX_NCLASS];
#pragma unroll
  for (int c = 0; c < NX_NCLASS; ++c) exh[c] = S->exh[c];
  __syncwarp();
  int result = -3;
  unsigned base_cur = 0;
  // two rounds at most: (0) nothing in flight -> start a copy, (1) consume it and start the next
  for (int round = 0; round < 2; ++round) {
    if (cnt_pend != 0) {
      cp_async_wait_all();
      __syncwarp();
      buf ^= 1;
      base_cur = base_pend;
      const double* v = vals + (size_t)buf * NX_SFEED_COLS * 32 + lane;
      int cls = -1;
      if ((int)lane < cnt_pend) {
        // the class found by an earlier pass came in with the rows (a stale 0xFF only
        // means the deterministic model is evaluated again)
        const int cached = A.cls ? (int)S->clsb[buf][lane] : 0xFF;
        if (NX_NCLASS == 1) cls = 0;
        else if (cached < NX_NCLASS) cls = cached;
        else {
          RunParams pp;               // only the fields cost_class reads
          pp.resolution = A.resolution; pp.gravity = A.gravity; pp.radpres = A.radpres;
          cls = cost_class(pp, A.model, A.res, A.mu, A.amax, v[0], v[32], v[64], v[96], v[128],
                           v[160], v[192], v[224]);
          if (A.cls) A.cls[base_cur + lane] = (unsigned char)cls;
        }
      }
      const unsigned match = __ballot_sync(FULL_MASK, cls == cls_pend);
      if (cls == cls_pend) S->order[__popc(match & ((1u << lane) - 1u))] = (unsigned char)lane;
      result = __popc(match);
      cnt_pend = 0;
    }
    // start the copy of the next batch into the idle buffer
    if (grp_next >= grp_end) {
      unsigned done = all_mask;
#pragma unroll
      for (int c = 0; c < NX_NCLASS; ++c) done &= exh[c];
      bool claimed = false;
      if (done != all_mask) {
        unsigned nready = (unsigned)A.nseg;
        if (A.arrived) nready = ld_volatile_u32(A.arrived);
        const unsigned ready = nready >= 32u ? 0xffffffffu : ((1u << nready) - 1u);
#pragma unroll
        for (int c = 0; c < NX_NCLASS; ++c) {
          unsigned avail = claimed ? 0u : (ready & ~exh[c]);
          while (avail) {
            const int sgm = __ffs(avail) - 1;
            unsigned long long g = 0;
            if (lane == 0) g = atomicAdd(A.cursor + c * 32 + sgm, (unsigned long long)NX_GROUP);
            g = __shfl_sync(FULL_MASK, g, 0);
            const long long first = (long long)sgm * A.seg;
            const long long count = min(A.seg, A.n - first);
            if ((long long)g + NX_GROUP >= count) {
              exh[c] |= 1u << sgm;
#ifdef NX_STREAM_DEBUG
              if (lane == 0 && sgm == A.nseg - 1) atomicCAS(&g_dbg[1 + c], 0ull, global_timer_ns());
#endif
            }
            if ((long long)g < count) {
              grp_next = (unsigned)(first + (long long)g);
              grp_end = (unsigned)min(first + count, first + (long long)g + NX_GROUP);
              grp_cls = c;
              claimed = true;
              break;
            }
            avail &= ~(1u << sgm);
          }
        }
      }
      if (!claimed && result == -3) {
        unsigned done2 = all_mask;
#pragma unroll
        for (int c = 0; c < NX_NCLASS; ++c) done2 &= exh[c];
        result = (done2 == all_mask) ? -1 : -2;
      }
    }
    if (grp_next < grp_end) {
      base_pend = grp_next;
      cnt_pend = (int)min(32u, grp_end - grp_next);
      cls_pend = grp_cls;
      grp_next += 32u;
      double* dst = vals + (size_t)(buf ^ 1) * NX_SFEED_COLS * 32;
      // 8 rows of 256 bytes = 128 chunks of 16 bytes (rows are padded to 32 packets)
#pragma unroll
      for (int i = 0; i < NX_SFEED_COLS / 2; ++i) {
        const unsigned j = lane + 32u * i;
        const unsigned col = j >> 4, part = (j & 15u) * 2u;
        cp_async16_cg(dst + col * 32u + part, A.col0 + (size_t)col * A.stride + base_pend + part);
      }
      if (A.cls && lane < 2u)
        cp_async16_cg(&S->clsb[buf ^ 1][lane * 16u], A.cls + base_pend + lane * 16u);
      cp_async_commit();
    }
    if (result != -3) break;          // a batch became current, or nothing can be had
  }
  if (lane == 0) {
    S->base_pend = base_pend; S->grp_next = grp_next; S->grp_end = grp_end;
    S->cnt_pend = cnt_pend; S->cls_pend = cls_pend; S->buf = buf; S->grp_cls = grp_cls;
    if (result >= 0) S->base_cur = base_cur;
#pragma unroll
    for (int c = 0; c < NX_NCLASS; ++c) S->exh[c] = exh[c];
  }
  __syncwarp();
  return result;
}

template <int MODE>
__global__ void __launch_bounds__(NX_INT_THREADS, NX_INT_MINBLOCKS)
k_integrate_adaptive_stream(const double* __restrict__ col0, size_t stride, double step0,
                            StateCols P, long long n, RunParams p, InterpTable Tg, FastTable Fg,
                            StreamQueue Q, unsigned long long* __restrict__ totals,
                            unsigned* __restrict__ att_out, unsigned* __restrict__ acc_out,
                            int* __restrict__ status, unsigned table_bytes) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  InterpTable T;
  FastTable F;
  if (MODE < 0) stage_table(Tg, T, smem_raw);
  else stage_fast_table(Fg, F, smem_raw);
  const unsigned lane = threadIdx.x & 31u;
  double* const vals = reinterpret_cast<double*>(smem_raw + table_bytes +
                                                 (size_t)(threadIdx.x >> 5) * NX_SFEED_BYTES_PER_WARP);
  StreamShared* const S = reinterpret_cast<StreamShared*>(vals + 2 * NX_SFEED_COLS * 32);
  for (unsigned i = lane; i < NX_SFEED_STATE_BYTES / 4; i += 32u)
    reinterpret_cast<unsigned*>(S)[i] = 0u;
  StreamArgs A;
  A.col0 = col0; A.stride = stride; A.n = n; A.seg = Q.seg; A.cursor = Q.cursor;
  A.arrived = Q.arrived; A.cls = Q.cls; A.resolution = p.resolution; A.res = (float)p.resolution;
  A.mu = (float)fabs(p.GM); A.amax = (float)p.radpres_amax; A.nseg = Q.nseg; A.model = Q.model;
  A.gravity = p.gravity; A.radpres = p.radpres;
  __syncthreads();

  bool have = false, drained = false;
  unsigned idx = 0;
  double s[8], step = 0.0;
  unsigned att = 0, acc = 0;
  unsigned long long tot_att = 0, tot_acc = 0;
  unsigned long long wait_since = 0;
  int st = 0;
  int fpos = 0, fcnt = 0;            // hand-out position / size of the current batch
#ifdef NX_STREAM_DEBUG
  unsigned long long dbg_iters = 0, dbg_scans = 0;
#endif

  for (;;) {
    unsigned need = __ballot_sync(FULL_MASK, !have);
    bool starved = false;
    int scans = 0;
    while (need && !drained) {
      if (fpos == fcnt) {
        if (scans >= NX_SCAN_MAX && need != FULL_MASK) break;   // let the live lanes step
        const int r = stream_advance(S, vals, A);
        ++scans;
#ifdef NX_STREAM_DEBUG
        ++dbg_scans;
#endif
        if (r == -1) { drained = true; break; }
        if (r == -2) { starved = true; break; }
        fpos = 0; fcnt = r;
        continue;
      }
      const int take = min(__popc(need), fcnt - fpos);
      const int rank = __popc(need & ((1u << lane) - 1u));
      if (!have && rank < take) {
        const int slot = S->order[fpos + rank];
        const double* v = vals + (size_t)S->buf * NX_SFEED_COLS * 32 + slot;
#pragma unroll
        for (int k = 0; k < 8; ++k) s[k] = v[k * 32];
        step = step0;
        idx = S->base_cur + (unsigned)slot;
        att = 0; acc = 0;
        have = (s[0] > p.resolution) && (s[7] > 0.0);
        if (!have) {                      // nothing to integrate: pass it through (att/acc pre-zeroed)
#pragma unroll
          for (int k = 0; k < 8; ++k) __stcs(P.c[k] + idx, s[k]);
          __stcs(P.c[8] + idx, step);
        }
      }
      fpos += take;
      need = __ballot_sync(FULL_MASK, !have);
    }
    if (!__any_sync(FULL_MASK, have)) {
      if (drained) break;
      if (starved) {
        // every resident segment is used up and later ones are still on the wire
        const unsigned long long now = global_timer_ns();
        if (wait_since == 0) wait_since = now;
        if (now - wait_since > NX_STREAM_TIMEOUT_NS) { st |= 64; break; }
        __nanosleep(400);
      }
      continue;
    }
    wait_since = 0;
    NX_DBG_ITER(__ballot_sync(FULL_MASK, have));
    if (have) {
      int fl;
      if (MODE < 0) fl = adaptive_attempt<true>(p, T, s, step);
      else fl = adaptive_attempt_fast<(MODE >> 3) & 1, (MODE >> 2) & 1, MODE & 3, (MODE >> 4) & 1>(p, F, s, step);
      ++att;
      if (fl & ATT_ACCEPTED) ++acc;
      st |= fl & ~(ATT_ACCEPTED | ATT_LIVE);
      if (att >= NX_ATTEMPT_CAP) { st |= NX_ST_NO_PROGRESS; fl &= ~ATT_LIVE; }
      if (!(fl & ATT_LIVE)) {
#pragma unroll
        for (int k = 0; k < 8; ++k) __stcs(P.c[k] + idx, s[k]);
        __stcs(P.c[8] + idx, step);
        att_out[idx] = att; acc_out[idx] = acc;
        tot_att += att; tot_acc += acc;
        have = false;
      }
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    tot_att += __shfl_xor_sync(FULL_MASK, tot_att, o);
    tot_acc += __shfl_xor_sync(FULL_MASK, tot_acc, o);
    st |= __shfl_xor_sync(FULL_MASK, st, o);
  }
  if (lane == 0) {
    if (tot_att) atomicAdd(&totals[0], tot_att);
    if (tot_acc) atomicAdd(&totals[1], tot_acc);
    if (st) atomicOr(status, st);
#ifdef NX_STREAM_DEBUG
    atomicMax(&g_dbg[16], global_timer_ns());
    atomicAdd(&g_dbg[17], dbg_iters);
    atomicAdd(&g_dbg[18], dbg_scans);
#endif
  }
}

// ---------------------------------------------------------------------------
// K3: constant-step driver (+ bounce) with optional fused image accumulation
// and optional dense trajectory sink.
// ---------------------------------------------------------------------------
__device__ __forceinline__ void image_add(const ImageParams& ip, const GTables& G,
                                          const ImageSteps& t, const double* s,
                                          double* image, unsigned long long* counts) {
  if (ip.skip_dead && !(s[7] > 0.0)) return;
  double w;
  const int pix = image_packet_fast(ip, G, t, s[1], s[2], s[3], s[5], s[7], w);
  if (pix >= 0) {
    if (w != 0.0) atomicAdd(&image[pix], w);
    atomicAdd(&counts[pix], 1ull);
  }
}

// K3 keeps the packets of a warp in a shared-memory POOL of NX_POOL_SLOTS slots (twice the
// warp width) and runs warp-uniform PHASES over it; a lane holds no packet between phases:
//   NEW    packets that just arrived from HBM (cp.async straight into their slot): row 0
//   STEP   32 runnable packets take one Dormand-Prince step; those that end below the
//          surface are PARKED (state + radius written back), the rest emit their row
//   BOUNCE 32 parked packets go through the surface interaction together and emit
// The surface interaction costs about two steps and ~10 % of the packets need it after any
// given step: run per lane where it occurs it leaves 20 of 32 lanes busy (round 1, ncu
// smsp__thread_inst_executed_per_inst_executed 19.9); with the pool both the step and the
// bounce code run on full warps, whatever the mix.  Results do not depend on the schedule:
// the bounce deviates are Philox draws keyed by (seed, packet id, step).
#define NX_POOL_WORDS 3
#define NX_POOL_SLOTS (32 * NX_POOL_WORDS)
#define NX_POOL_FIELDS 10      // time,x,y,z,vx,vy,vz,frac, time left in the run, radius at impact
#define NX_POOL_BYTES_PER_WARP (NX_POOL_FIELDS * NX_POOL_SLOTS * 8 + NX_POOL_SLOTS * 8 + NX_POOL_SLOTS + 32)
#define NX_POOL_BYTES_PER_WARP_ALIGNED ((NX_POOL_BYTES_PER_WARP + 15) / 16 * 16)
// measured (8e6 packets of configs[2], plain / fused image, 1e10 packet-steps/s):
// 512 threads (120 registers) 2.38 / 1.69; 640 threads (96 registers, 68 B of spills) 2.47 / 1.71
#ifndef NX_K3_THREADS
#define NX_K3_THREADS 640
#endif
struct StepCoef { double v[NX_STEPCOEF_COUNT]; };    // h-scaled tableau products (nx_fast.cuh)
enum { SLOT_FREE = 0, SLOT_LOADING = 1, SLOT_NEW = 2, SLOT_RUN = 3, SLOT_PARKED = 4 };

// census of one class of slots: lane L looks at slots L, L + 32, ...; m[w] = ballot of word w
struct SlotMask {
  unsigned m[NX_POOL_WORDS];
  __device__ __forceinline__ int count() const {
    int c = 0;
#pragma unroll
    for (int w = 0; w < NX_POOL_WORDS; ++w) c += __popc(m[w]);
    return c;
  }
};
__device__ __forceinline__ SlotMask census(const unsigned* k, unsigned what) {
  SlotMask r;
#pragma unroll
  for (int w = 0; w < NX_POOL_WORDS; ++w) r.m[w] = __ballot_sync(FULL_MASK, k[w] == what);
  return r;
}

// MODE as in k_integrate_adaptive: -1 strict, else fast with MODE = GR*8 + RP*4 + LOSS.
// ROWS: compile the row sink in (a separate instantiation keeps the plain kernel's hot loop
// as small as it was: the loop is instruction-cache bound).
template <int MODE, bool ROWS>
__global__ void __launch_bounds__(NX_K3_THREADS, 1)
k_integrate_constant(StateCols In, StateCols P, long long n, RunParams p, InterpTable Tg,
                     FastTable Fg, Spline2D S, uint64_t seed, uint64_t first_id, int nsteps,
                     ImageParams ip, GTables G, double* image, unsigned long long* counts,
                     double* traj, RowSink rows,
                     unsigned long long* __restrict__ queue,
                     unsigned long long* __restrict__ totals, int* __restrict__ status,
                     unsigned table_bytes, StepCoef hc) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  InterpTable T;
  FastTable F;
  if (MODE < 0) stage_table(Tg, T, smem_raw);
  else stage_fast_table(Fg, F, smem_raw);
  const unsigned lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
  unsigned char* pool = smem_raw + table_bytes + (size_t)warp * NX_POOL_BYTES_PER_WARP_ALIGNED;
  double* fld = reinterpret_cast<double*>(pool);                       // [FIELDS][SLOTS]
  unsigned* sidx = reinterpret_cast<unsigned*>(fld + NX_POOL_FIELDS * NX_POOL_SLOTS);
  unsigned* sct = sidx + NX_POOL_SLOTS;
  unsigned char* kind = reinterpret_cast<unsigned char*>(sct + NX_POOL_SLOTS);
  unsigned char* sel = kind + NX_POOL_SLOTS;                           // slot of lane r this phase
#pragma unroll
  for (int w = 0; w < NX_POOL_WORDS; ++w) kind[lane + 32 * w] = SLOT_FREE;
  __syncthreads();
  const bool pass_through = In.c[0] != P.c[0];     // see k_integrate_adaptive
  const ImageSteps isteps = image_steps(ip);

  bool loading = false, queue_done = false;
  unsigned long long tot = 0;
  int st = 0;

  for (;;) {
    if (loading) {                                   // the batch requested one phase ago
      cp_async_wait_all();
#pragma unroll
      for (int w = 0; w < NX_POOL_WORDS; ++w)
        if (kind[lane + 32 * w] == SLOT_LOADING) kind[lane + 32 * w] = SLOT_NEW;
      loading = false;
      __syncwarp();
    }
    unsigned kk[NX_POOL_WORDS];
#pragma unroll
    for (int w = 0; w < NX_POOL_WORDS; ++w) kk[w] = kind[lane + 32 * w];
    const SlotMask m_free = census(kk, SLOT_FREE), m_new = census(kk, SLOT_NEW),
                   m_run = census(kk, SLOT_RUN), m_park = census(kk, SLOT_PARKED);
    const int nfree = m_free.count(), nnew = m_new.count(), nrun = m_run.count(),
              npark = m_park.count();
    if (nfree == NX_POOL_SLOTS && queue_done) break;

    // refill: 32 or more free slots are filled from the global packet queue (so that the
    // NEW phases are full too); the copies land while the phase below runs
    if (!queue_done && nfree >= 32) {
      unsigned long long base = 0;
      if (lane == 0) base = atomicAdd(queue, (unsigned long long)nfree);
      base = __shfl_sync(FULL_MASK, base, 0);
      if ((long long)base + nfree >= n) queue_done = true;
      int before = 0;
#pragma unroll
      for (int w = 0; w < NX_POOL_WORDS; ++w) {
        const int j = (int)lane + 32 * w;
        if ((m_free.m[w] >> lane) & 1u) {
          const long long q = (long long)base + before + __popc(m_free.m[w] & ((1u << lane) - 1u));
          if (q < n) {
#pragma unroll
            for (int k = 0; k < 8; ++k) cp_async8(fld + k * NX_POOL_SLOTS + j, In.c[k] + q);
            fld[8 * NX_POOL_SLOTS + j] = p.endtime;      // row 0 (Output.py:379-386)
            sidx[j] = (unsigned)q;
            sct[j] = 0u;
            kind[j] = SLOT_LOADING;
          }
        }
        before += __popc(m_free.m[w]);
      }
      cp_async_commit();
      loading = true;
    }

    // phase: a full warp of parked packets first (they hold slots), else new arrivals, else
    // a step; a class that cannot fill the warp only runs when nothing else can
    int phase;
    if (npark >= 32) phase = SLOT_PARKED;
    else if (nnew >= 32) phase = SLOT_NEW;
    else if (nrun >= 32) phase = SLOT_RUN;
    else if (nrun >= npark && nrun >= nnew && nrun > 0) phase = SLOT_RUN;
    else if (npark >= nnew && npark > 0) phase = SLOT_PARKED;
    else if (nnew > 0) phase = SLOT_NEW;
    else continue;                                    // only copies in flight
    SlotMask M;
#pragma unroll
    for (int w = 0; w < NX_POOL_WORDS; ++w)
      M.m[w] = phase == SLOT_PARKED ? m_park.m[w] : (phase == SLOT_NEW ? m_new.m[w] : m_run.m[w]);
    // the r-th slot of the class goes to lane r: every slot's owner lane scatters its rank
    {
      int before = 0;
#pragma unroll
      for (int w = 0; w < NX_POOL_WORDS; ++w) {
        if ((M.m[w] >> lane) & 1u) {
          const int r = before + __popc(M.m[w] & ((1u << lane) - 1u));
          if (r < 32) sel[r] = (unsigned char)(lane + 32 * w);
        }
        before += __popc(M.m[w]);
      }
      __syncwarp();
    }
    const int navail = M.count();
    const bool act = (int)lane < navail;
    const int j = act ? (int)sel[lane] : 0;

    double s[8], curtime = 0.0, rhit = 0.0;
    unsigned idx = 0;
    int ct = 0;
    bool emit = false, live = true;
    if (act) {
#pragma unroll
      for (int k = 0; k < 8; ++k) s[k] = fld[k * NX_POOL_SLOTS + j];
      curtime = fld[8 * NX_POOL_SLOTS + j];
      idx = sidx[j];
      ct = (int)sct[j];
    }
    if (phase == SLOT_NEW) {
      if (act) { emit = true; live = s[7] > 0.0; }
    } else if (phase == SLOT_RUN) {
      if (act) {
        // non-finite state (Output.py:388-389): exponent field all ones in any component
        unsigned worst = 0u;
#pragma unroll
        for (int k = 0; k < 8; ++k) worst = max(worst, (unsigned)__double2hiint(s[k]) & 0x7fffffffu);
        if (worst >= 0x7ff00000u) st |= 32;
        ++tot;
        if (MODE < 0) {
          live = constant_step<true>(p, T, S, s, seed, first_id + (uint64_t)idx, (uint32_t)ct);
          emit = true;
        } else {
          const double r = constant_stages_fast<(MODE >> 3) & 1, (MODE >> 2) & 1, MODE & 3>(p, F, s, hc.v);
          bool hit = sub_rn(r, 1.0) < 0.0;
          if (hit && p.sticktype == STICK_CONSTANT && p.stickcoef == 1.0) { s[7] = 0.0; hit = false; }
          if (hit) {                                   // park: the bounce runs on a full warp
#pragma unroll
            for (int k = 0; k < 8; ++k) fld[k * NX_POOL_SLOTS + j] = s[k];
            fld[9 * NX_POOL_SLOTS + j] = r;
            kind[j] = SLOT_PARKED;
          } else {
            live = constant_post(p, s, r);
            emit = true;
          }
        }
      }
    } else {
      if (MODE >= 0 && act) {
        rhit = fld[9 * NX_POOL_SLOTS + j];
        constant_bounce_fast(p, S, s, rhit, seed, first_id + (uint64_t)idx, (uint32_t)ct);
        live = constant_post(p, s, rhit);
        emit = true;
      }
    }

    // One row of the reference's trajectory tensor (Output.py:376-421) is EMITTED at a
    // single place per phase -- for a packet that was just loaded (row 0), that completed
    // a step, or whose bounce was just resolved -- so the image / trajectory / retire code
    // exists once in the kernel (instruction-cache footprint).
    if (emit) {
      if (traj) {
#pragma unroll
        for (int k = 0; k < 8; ++k) traj[((size_t)idx * 8 + k) * nsteps + ct] = s[k];
      }
      if (image) image_add(ip, G, isteps, s, image, counts);
    }
    if (ROWS) {
      // Row sink: what the reference keeps of a constant-step run (Output.py:434-449 flattens
      // results[N, 8, nsteps]; Output.save drops the frac == 0 rows and rounds to float32),
      // appended to a device table with one warp-aggregated atomic per phase
      // (cap == 0: the rows are only counted).
      const bool want = emit && (!rows.skip_dead || s[7] > 0.0);
      const unsigned m = __ballot_sync(FULL_MASK, want);
      if (m) {
        const int leader = __ffs(m) - 1;
        unsigned long long base = 0;
        if ((int)lane == leader) base = atomicAdd(rows.cursor, (unsigned long long)__popc(m));
        base = __shfl_sync(FULL_MASK, base, leader);
        if (want) {
          const unsigned long long o = base + __popc(m & ((1u << lane) - 1u));
          if (o < rows.cap) {
#pragma unroll
            for (int k = 0; k < 8; ++k) {
              double v = s[k];
              if (rows.to_f32) v = (double)(float)v;
              rows.cols[(size_t)k * rows.stride + o] = v;
            }
            rows.index[o] = idx;
            rows.step[o] = (unsigned short)ct;
          }
        }
      }
    }
    if (emit) {
      const bool fresh = (ct == 0);
      ++ct;
      if (!fresh) curtime -= p.step_size;
      if (!live || !(curtime > 0.0) || ct >= nsteps) {
        if (!fresh || pass_through) {       // an unintegrated packet stays as it is
#pragma unroll
          for (int k = 0; k < 8; ++k) __stcs(P.c[k] + idx, s[k]);
        }
        kind[j] = SLOT_FREE;
      } else {
#pragma unroll
        for (int k = 0; k < 8; ++k) fld[k * NX_POOL_SLOTS + j] = s[k];
        fld[8 * NX_POOL_SLOTS + j] = curtime;
        sct[j] = (unsigned)ct;
        kind[j] = SLOT_RUN;
      }
    }
    __syncwarp();
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    tot += __shfl_xor_sync(FULL_MASK, tot, o);
    st |= __shfl_xor_sync(FULL_MASK, st, o);
  }
  if (lane == 0) {
    if (tot) atomicAdd(&totals[0], tot);
    if (st) atomicOr(status, st);
  }
}

// ---------------------------------------------------------------------------
// K4: image accumulation.  Streams x,y,z,vy,frac (40 B/packet, 16-byte vector
// loads, two packets per thread per iteration) and scatters with f64 / u64
// atomics into the L2-resident image (800x800: 5 MB + 5 MB).
// ---------------------------------------------------------------------------
__device__ __forceinline__ void image_one(const ImageParams& ip, const GTables& G,
                                          const ImageSteps& t, double x, double y, double z, double v,
                                          double f, double* image, unsigned long long* counts) {
  if (ip.skip_dead && !(f > 0.0)) return;
  double w;
  const int pix = image_packet_fast(ip, G, t, x, y, z, v, f, w);
  if (pix >= 0) {
    if (w != 0.0) atomicAdd(&image[pix], w);
    atomicAdd(&counts[pix], 1ull);
  }
}

// Two packets per thread and iteration, two iterations in flight (ten 16-byte
// loads issued before the first use); g-value tables as interval records in
// shared memory (bucket index in L1).
__global__ void __launch_bounds__(256)
k_image_accumulate(StateCols P, long long n, ImageParams ip, GTables Gg,
                   double* __restrict__ image, unsigned long long* __restrict__ counts) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  GTables G;
  stage_gtables(Gg, G, smem_raw);
  __syncthreads();
  const ImageSteps isteps = image_steps(ip);
  const long long npair = n >> 1;
  const long long stride = (long long)gridDim.x * blockDim.x;
  const double2* __restrict__ X2 = reinterpret_cast<const double2*>(P.c[1]);
  const double2* __restrict__ Y2 = reinterpret_cast<const double2*>(P.c[2]);
  const double2* __restrict__ Z2 = reinterpret_cast<const double2*>(P.c[3]);
  const double2* __restrict__ V2 = reinterpret_cast<const double2*>(P.c[5]);
  const double2* __restrict__ F2 = reinterpret_cast<const double2*>(P.c[7]);
  // software pipeline: the five loads of the NEXT pair are issued before the current
  // pair is binned (ten 16-byte loads in flight per thread); one copy of the per-packet
  // code per lane of the pair keeps the kernel inside the instruction cache
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  double2 xa, ya, za, va, fa;
  if (i < npair) {
    xa = __ldcs(X2 + i); ya = __ldcs(Y2 + i); za = __ldcs(Z2 + i);
    va = __ldcs(V2 + i); fa = __ldcs(F2 + i);
  }
  while (i < npair) {
    const long long j = i + stride;
    double2 xb = xa, yb = ya, zb = za, vb = va, fb = fa;
    if (j < npair) {
      xb = __ldcs(X2 + j); yb = __ldcs(Y2 + j); zb = __ldcs(Z2 + j);
      vb = __ldcs(V2 + j); fb = __ldcs(F2 + j);
    }
    image_one(ip, G, isteps, xa.x, ya.x, za.x, va.x, fa.x, image, counts);
    image_one(ip, G, isteps, xa.y, ya.y, za.y, va.y, fa.y, image, counts);
    xa = xb; ya = yb; za = zb; va = vb; fa = fb;
    i = j;
  }
  if ((n & 1) && blockIdx.x == 0 && threadIdx.x == 0) {
    const long long q = n - 1;
    image_one(ip, G, isteps, P.c[1][q], P.c[2][q], P.c[3][q], P.c[5][q], P.c[7][q],
              image, counts);
  }
}

// K4, privatised variant (north_star: "shared-memory-privatised histograms").  Shared-memory
// atomics are native only for 32-bit operands on sm_100a (64-bit ones, f64 and u64 alike,
// compile to ATOMS.CAST.SPIN loops), so what is privatised is the PACKET-COUNT histogram: one
// 1024-thread block per SM keeps a u32 tile of counts for the pixel rectangle around the
// projected planet -- where the packets of an exosphere run pile up -- in ~200 KB of shared
// memory (ATOMS.POPC.INC.32), and only the f64 weight of a packet goes to the L2-resident
// image as a RED.  That halves the global atomics per live packet; the tile is flushed with
// one u64 RED per non-empty pixel at the end.  Pixels outside the tile take the global path.
struct ImageTile { int ix0, iz0, w, h; };

__global__ void __launch_bounds__(1024, 1)
k_image_accumulate_tile(StateCols P, long long n, ImageParams ip, GTables Gg, ImageTile tile,
                        double* __restrict__ image, unsigned long long* __restrict__ counts) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  GTables G;
  const size_t off = stage_gtables(Gg, G, smem_raw);
  unsigned* __restrict__ tcnt = reinterpret_cast<unsigned*>(smem_raw + off);
  const int tsize = tile.w * tile.h;
  for (int i = threadIdx.x; i < tsize; i += blockDim.x) tcnt[i] = 0u;
  __syncthreads();
  const ImageSteps isteps = image_steps(ip);
  const long long npair = n >> 1;
  const long long stride = (long long)gridDim.x * blockDim.x;
  const double2* __restrict__ X2 = reinterpret_cast<const double2*>(P.c[1]);
  const double2* __restrict__ Y2 = reinterpret_cast<const double2*>(P.c[2]);
  const double2* __restrict__ Z2 = reinterpret_cast<const double2*>(P.c[3]);
  const double2* __restrict__ V2 = reinterpret_cast<const double2*>(P.c[5]);
  const double2* __restrict__ F2 = reinterpret_cast<const double2*>(P.c[7]);
  auto one = [&](double x, double y, double z, double v, double f) {
    if (ip.skip_dead && !(f > 0.0)) return;
    double w;
    int ix, iz;
    const int pix = image_packet_fast(ip, G, isteps, x, y, z, v, f, w, &ix, &iz);
    if (pix < 0) return;
    if (w != 0.0) atomicAdd(&image[pix], w);
    const unsigned tx = (unsigned)(ix - tile.ix0), tz = (unsigned)(iz - tile.iz0);
    if (tx < (unsigned)tile.w && tz < (unsigned)tile.h) atomicAdd(&tcnt[tx * tile.h + tz], 1u);
    else atomicAdd(&counts[pix], 1ull);
  };
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  double2 xa, ya, za, va, fa;
  if (i < npair) {
    xa = __ldcs(X2 + i); ya = __ldcs(Y2 + i); za = __ldcs(Z2 + i);
    va = __ldcs(V2 + i); fa = __ldcs(F2 + i);
  }
  while (i < npair) {
    const long long j = i + stride;
    double2 xb = xa, yb = ya, zb = za, vb = va, fb = fa;
    if (j < npair) {
      xb = __ldcs(X2 + j); yb = __ldcs(Y2 + j); zb = __ldcs(Z2 + j);
      vb = __ldcs(V2 + j); fb = __ldcs(F2 + j);
    }
    one(xa.x, ya.x, za.x, va.x, fa.x);
    one(xa.y, ya.y, za.y, va.y, fa.y);
    xa = xb; ya = yb; za = zb; va = vb; fa = fb;
    i = j;
  }
  if ((n & 1) && blockIdx.x == 0 && threadIdx.x == 0) {
    const long long q = n - 1;
    one(P.c[1][q], P.c[2][q], P.c[3][q], P.c[5][q], P.c[7][q]);
  }
  __syncthreads();
  for (int t = threadIdx.x; t < tsize; t += blockDim.x) {
    const unsigned c = tcnt[t];
    if (c) {
      const int tx = t / tile.h, tz = t - tx * tile.h;
      atomicAdd(&counts[(size_t)(tile.ix0 + tx) * ip.nz + (tile.iz0 + tz)], (unsigned long long)c);
    }
  }
}

// ---------------------------------------------------------------------------
// Image cube (ModelImageCube): K4's pixel and weight (image_packet_fast, unchanged) with a
// velocity axis.  v = los_doppler along row 1 of the observer rotation (the observer sits at
// -y_obs, so v > 0 recedes), column = spectrum_column (np.histogram on linspace(vmin, vmax,
// nbins + 1), 0 below, nbins + 1 above).  Streams x,y,z,vx,vy,vz,frac (56 B/row) and adds
// one f64 RED (w != 0) and one u64 RED at pixel * (nbins + 2) + column.  The host keeps
// nx * nz * (nbins + 2) below 2^31, so a cell index fits an int.
// ---------------------------------------------------------------------------
__device__ __forceinline__ void cube_one(const ImageParams& ip, const GTables& G,
                                         const ImageSteps& t, const CubeAxis& ax, double x,
                                         double y, double z, double vx, double vy, double vz,
                                         double f, double* cube, unsigned long long* counts) {
  if (ip.skip_dead && !(f > 0.0)) return;
  double w;
  const int pix = image_packet_fast(ip, G, t, x, y, z, vy, f, w);
  if (pix < 0) return;
  if (ip.round_f32) { vx = round_f32(vx); vy = round_f32(vy); vz = round_f32(vz); }
  const double v = los_doppler(vx, vy, vz, ip.M[3], ip.M[4], ip.M[5], ax.vscale);
  const int cell = pix * (ax.nbins + 2) + spectrum_column(v, ax.nbins, ax.vmin, ax.vmax, ax.step);
  if (w != 0.0) atomicAdd(&cube[cell], w);
  atomicAdd(&counts[cell], 1ull);
}

// Two rows per thread and iteration; the seven loads of the next pair are issued before the
// current pair is binned (as k_image_accumulate)
__global__ void __launch_bounds__(256)
k_image_cube(StateCols P, long long n, ImageParams ip, GTables Gg, CubeAxis ax,
             double* __restrict__ cube, unsigned long long* __restrict__ counts) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  GTables G;
  stage_gtables(Gg, G, smem_raw);
  __syncthreads();
  const ImageSteps isteps = image_steps(ip);
  const long long npair = n >> 1;
  const long long stride = (long long)gridDim.x * blockDim.x;
  const double2* __restrict__ C2[7];
#pragma unroll
  for (int k = 0; k < 7; ++k) C2[k] = reinterpret_cast<const double2*>(P.c[k + 1]);
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  double2 a[7];
  if (i < npair) {
#pragma unroll
    for (int k = 0; k < 7; ++k) a[k] = __ldcs(C2[k] + i);
  }
  while (i < npair) {
    const long long j = i + stride;
    double2 b[7];
#pragma unroll
    for (int k = 0; k < 7; ++k) b[k] = a[k];
    if (j < npair) {
#pragma unroll
      for (int k = 0; k < 7; ++k) b[k] = __ldcs(C2[k] + j);
    }
    cube_one(ip, G, isteps, ax, a[0].x, a[1].x, a[2].x, a[3].x, a[4].x, a[5].x, a[6].x, cube,
             counts);
    cube_one(ip, G, isteps, ax, a[0].y, a[1].y, a[2].y, a[3].y, a[4].y, a[5].y, a[6].y, cube,
             counts);
#pragma unroll
    for (int k = 0; k < 7; ++k) a[k] = b[k];
    i = j;
  }
  if ((n & 1) && blockIdx.x == 0 && threadIdx.x == 0) {
    const long long q = n - 1;
    cube_one(ip, G, isteps, ax, P.c[1][q], P.c[2][q], P.c[3][q], P.c[4][q], P.c[5][q], P.c[6][q],
             P.c[7][q], cube, counts);
  }
}

// ---------------------------------------------------------------------------
// K5: lines of sight.  One LOS per thread (ray constants in registers), packet
// positions staged through shared memory in tiles; every thread of the block
// reads the same packet (smem broadcast) and runs the conservative cone reject;
// the rare survivors take the exact (reference-order) path.
// ---------------------------------------------------------------------------
#define NX_LOS_TILE 1024

__global__ void __launch_bounds__(NX_LOS_THREADS)
k_los_accumulate(StateCols P, long long n, long long nlos, const double* __restrict__ los,
                 const double* __restrict__ dist_plan, const int* __restrict__ nball,
                 const double* __restrict__ ladder, const double* __restrict__ wid2,
                 LosParams lp, LosConsts lc, GTables Gg,
                 double* __restrict__ radiance, unsigned long long* __restrict__ npack,
                 unsigned char* __restrict__ included, long long chunk) {
  __shared__ double spx[NX_LOS_TILE], spy[NX_LOS_TILE], spz[NX_LOS_TILE];
  const long long l = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  LosRay L;
  const bool valid = l < nlos;
  const long long ll = valid ? l : 0;
  L.xs = los[ll]; L.ys = los[nlos + ll]; L.zs = los[2 * nlos + ll];
  L.bx = los[3 * nlos + ll]; L.by = los[4 * nlos + ll]; L.bz = los[5 * nlos + ll];
  L.dist_plan = valid ? dist_plan[ll] : -1.0;     // invalid rays reject everything
  L.nball = nball[ll];

  const long long p0 = (long long)blockIdx.y * chunk;
  const long long p1 = (p0 + chunk < n) ? p0 + chunk : n;
  double rad = 0.0;
  unsigned long long cnt = 0;
  for (long long base = p0; base < p1; base += NX_LOS_TILE) {
    const int m = (int)((p1 - base < NX_LOS_TILE) ? (p1 - base) : NX_LOS_TILE);
    __syncthreads();
    for (int j = threadIdx.x; j < m; j += blockDim.x) {
      double x = P.c[1][base + j], y = P.c[2][base + j], z = P.c[3][base + j];
      if (lp.round_f32) { x = round_f32(x); y = round_f32(y); z = round_f32(z); }
      if (lp.skip_dead && !(P.c[7][base + j] > 0.0)) x = y = z = 1e300;   // never hit
      spx[j] = x; spy[j] = y; spz[j] = z;
    }
    __syncthreads();
#pragma unroll 4
    for (int j = 0; j < m; ++j) {
      const double px = spx[j], py = spy[j], pz = spz[j];
      // conservative reject, FMA-contracted (exact path below re-evaluates)
      const double rx = px - L.xs, ry = py - L.ys, rz = pz - L.zs;
      const double lr = fma(rz, L.bz, fma(ry, L.by, rx * L.bx));
      const double d2 = fma(rz, rz, fma(ry, ry, rx * rx));
      if (lr > 0.0 && lr * lr >= d2 * lc.cos_loose2) {
        double losrad, dist;
        if (los_hit(L, lp.dphi, lc.cos_margin2, lc.cos_accept2, lc.cover, ladder, wid2,
                    lc.inv_log_ratio, lc.log_t0,
                    lc.kwin, px, py, pz, losrad, dist)) {
          ++cnt;
          double vy = P.c[5][base + j], fr = P.c[7][base + j];
          if (lp.round_f32) { vy = round_f32(vy); fr = round_f32(fr); }
          rad += los_weight(L, lp, Gg, lc.sin_dphi, fr, vy, losrad, dist);
          included[base + j] = 1;
        }
      }
    }
  }
  if (valid && cnt) {
    atomicAdd(&radiance[l], rad);
    atomicAdd(&npack[l], cnt);
  }
}

// ---------------------------------------------------------------------------
// measurement helpers
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(512, 4)
k_fp64_peak(double* out, int iters, double a, double b) {
  // 8 independent DFMA chains per thread, 2048 threads per SM, the loop unrolled 16 x (128 DFMA
  // per branch): the SASS of the loop body is DFMA only
  double x0 = threadIdx.x, x1 = x0 + 1, x2 = x0 + 2, x3 = x0 + 3, x4 = x0 + 4, x5 = x0 + 5,
         x6 = x0 + 6, x7 = x0 + 7;
#pragma unroll 16
  for (int i = 0; i < iters; ++i) {
    x0 = fma(x0, a, b); x1 = fma(x1, a, b); x2 = fma(x2, a, b); x3 = fma(x3, a, b);
    x4 = fma(x4, a, b); x5 = fma(x5, a, b); x6 = fma(x6, a, b); x7 = fma(x7, a, b);
  }
  out[(size_t)blockIdx.x * blockDim.x + threadIdx.x] = ((x0 + x1) + (x2 + x3)) + ((x4 + x5) + (x6 + x7));
}

__global__ void __launch_bounds__(256)
k_copy(const double2* __restrict__ src, double2* __restrict__ dst, long long n2) {
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n2; i += stride)
    dst[i] = src[i];
}

// ---------------------------------------------------------------------------
// launch wrappers (called from nx_api.cu)
// ---------------------------------------------------------------------------
static int sm_count(int device) {
  int v = 148;
  cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, device);
  return v;
}

cudaError_t launch_init_state(cudaStream_t st, X0Cols X, long long n,
                              const SourceParams& sp, const SourceMap& map,
                              const InterpTable& speed, const InterpTable& lon1d, uint64_t seed,
                              uint64_t first_id, bool fast) {
  const int threads = 256;
  const long long blocks = (n + threads - 1) / threads;
  if (fast) k_init_state<true><<<(unsigned)blocks, threads, 0, st>>>(X, n, sp, map, speed, lon1d, seed, first_id);
  else k_init_state<false><<<(unsigned)blocks, threads, 0, st>>>(X, n, sp, map, speed, lon1d, seed, first_id);
  return cudaGetLastError();
}

cudaError_t launch_init_from_deviates(cudaStream_t st, X0Cols X, long long n,
                                      const SourceParams& sp, const InterpTable& speed,
                                      const InterpTable& lon1d,
                                      const double* const* dev /* 9 device columns */) {
  k_init_from_deviates<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(
      X, n, sp, speed, lon1d, dev[0], dev[1], dev[2], dev[3], dev[4], dev[5], dev[6], dev[7], dev[8]);
  return cudaGetLastError();
}

// ModelImage's last two host passes (ModelImage.py:104-105: image *= atoms_per_packet; the
// packet image is a float histogram) done on the device before the image crosses PCIe
__global__ void __launch_bounds__(256)
k_image_finish(const double* __restrict__ img, const unsigned long long* __restrict__ cnt,
               double scale, double* __restrict__ img_out, double* __restrict__ cnt_out,
               long long npix) {
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < npix; i += stride) {
    img_out[i] = img[i] * scale;
    cnt_out[i] = (double)cnt[i];
  }
}
cudaError_t launch_image_finish(cudaStream_t st, const double* img, const unsigned long long* cnt,
                                double scale, double* img_out, double* cnt_out, long long npix) {
  if (npix <= 0) return cudaSuccess;
  long long blocks = (npix + 255) / 256;
  if (blocks > 148 * 8) blocks = 148 * 8;
  k_image_finish<<<(unsigned)blocks, 256, 0, st>>>(img, cnt, scale, img_out, cnt_out, npix);
  return cudaGetLastError();
}

cudaError_t launch_fill(cudaStream_t st, double* p, long long n, double v) {
  k_fill<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(p, n, v);
  return cudaGetLastError();
}

template <typename K>
static cudaError_t persistent_grid(K kernel, int device, size_t smem, int* blocks,
                                   int threads = NX_INT_THREADS) {
  cudaError_t e = cudaSuccess;
  if (smem > 48 * 1024)
    e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  int per_sm = 1;
  e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, threads, smem);
  if (e != cudaSuccess) return e;
  if (per_sm < 1) per_sm = 1;
  *blocks = per_sm * sm_count(device);
  return cudaSuccess;
}

// the ion builds: the kernels with a loss term (MODE & 3 = LOSS_LIFETIME or LOSS_PHOTO) and
// the strict kernels
constexpr bool ion_build(int mode) {
  return mode < 0 || (mode & 3) == LOSS_LIFETIME || (mode & 3) == LOSS_PHOTO;
}
// the trace builds: the kernels without a moon (MODE bit 16) and the strict kernels
constexpr bool trace_build(int mode) { return mode < 0 || !(mode & 16); }

template <typename K, typename... Args>
static cudaError_t launch_lanes(K kernel, cudaStream_t st, int device, size_t smem, long long n,
                                Args... args) {
  int blocks = 0;
  cudaError_t e = persistent_grid(kernel, device, smem, &blocks);
  if (e != cudaSuccess) return e;
  const long long need = (n + NX_INT_THREADS - 1) / NX_INT_THREADS;
  if (need < blocks) blocks = (int)(need > 0 ? need : 1);
  kernel<<<blocks, NX_INT_THREADS, smem, st>>>(args...);
  return cudaGetLastError();
}

// Ion != nullptr: the same run through k_ionize_adaptive<MODE, BOUNCE> (SINK false, MODE with
// a loss term), so the ion run selects its build by the dispatch of the plain run; Trace !=
// nullptr: through k_trace_adaptive<MODE, BOUNCE> (SINK false, MODE without a moon) alike.
template <int MODE, bool BOUNCE = false, bool SINK = false>
static cudaError_t launch_adaptive_mode(cudaStream_t st, int device, StateCols In, StateCols P,
                                        long long n,
                                        const RunParams& p, const InterpTable& T,
                                        const FastTable& F,
                                        const unsigned* perm, unsigned long long* queue,
                                        unsigned long long* totals, unsigned* att, unsigned* acc,
                                        int* status, const Spline2D& S, uint64_t seed,
                                        uint64_t first_id, const DepositOut& Dep,
                                        const IonOut* Ion, const TraceOut* Trace) {
  const size_t tbytes = (MODE < 0) ? table_smem_bytes(T) : fast_table_smem_bytes(F);
  const size_t smem = tbytes + (size_t)(NX_INT_THREADS / 32) * NX_FEED_BYTES_PER_WARP;
  if constexpr (!SINK && ion_build(MODE)) {
    if (Ion)
      return launch_lanes(k_ionize_adaptive<MODE, BOUNCE>, st, device, smem, n, In, P, n, p, T, F,
                          perm, queue, totals, att, acc, status, (unsigned)tbytes, S, seed,
                          first_id, *Ion);
  }
  if (Ion) return cudaErrorInvalidValue;         // no ion build: a run without loss
  if constexpr (!SINK && trace_build(MODE)) {
    if (Trace)
      return launch_lanes(k_trace_adaptive<MODE, BOUNCE>, st, device, smem, n, In, P, n, p, T, F,
                          perm, queue, totals, att, acc, status, (unsigned)tbytes, S, seed,
                          first_id, *Trace);
  }
  if (Trace) return cudaErrorInvalidValue;       // no trace build: a run with a moon
  return launch_lanes(k_integrate_adaptive<MODE, BOUNCE, SINK>, st, device, smem, n, In, P, n, p,
                      T, F, perm, queue, totals, att, acc, status, (unsigned)tbytes, S, seed,
                      first_id, Dep);
}

#ifdef NX_STREAM_DEBUG
__global__ void k_dbg_begin() {
  for (int i = threadIdx.x; i < 512; i += blockDim.x) g_dbg[i] = 0;
  __syncthreads();
  if (threadIdx.x == 0) g_dbg[0] = dbg_now();
}
#endif
cudaError_t debug_begin(cudaStream_t st) {
#ifdef NX_STREAM_DEBUG
  k_dbg_begin<<<1, 256, 0, st>>>();
#endif
  return cudaGetLastError();
}
cudaError_t debug_read(unsigned long long* out, int count) {
#ifdef NX_STREAM_DEBUG
  return cudaMemcpyFromSymbol(out, g_dbg, (size_t)(count > 512 ? 512 : count) * 8);
#else
  for (int i = 0; i < count; ++i) out[i] = 0;
  return cudaSuccess;
#endif
}

template <int MODE>
static cudaError_t launch_adaptive_stream_mode(cudaStream_t st, int device, const double* in0,
                                               size_t in_stride, double step0, StateCols P,
                                               long long n, const RunParams& p,
                                               const InterpTable& T, const FastTable& F,
                                               const StreamQueue& Q, unsigned long long* totals,
                                               unsigned* att, unsigned* acc, int* status) {
  const size_t tbytes = (MODE < 0) ? table_smem_bytes(T) : fast_table_smem_bytes(F);
  const size_t smem = tbytes + (size_t)(NX_INT_THREADS / 32) * NX_SFEED_BYTES_PER_WARP;
  int blocks = 0;
  cudaError_t e = persistent_grid(k_integrate_adaptive_stream<MODE>, device, smem, &blocks);
  if (e != cudaSuccess) return e;
  const long long need = (n + NX_INT_THREADS - 1) / NX_INT_THREADS;
  if (need < blocks) blocks = (int)(need > 0 ? need : 1);
  k_integrate_adaptive_stream<MODE><<<blocks, NX_INT_THREADS, smem, st>>>(
      in0, in_stride, step0, P, n, p, T, F, Q, totals, att, acc, status, (unsigned)tbytes);
  return cudaGetLastError();
}

// cursor: NX_STREAM_CURSORS zeroed u64; arrived: nullptr or a device word that the
// copy stream raises to the number of resident segments.
cudaError_t launch_integrate_adaptive_stream(cudaStream_t st, int device, const double* in0,
                                             size_t in_stride, double step0, StateCols P,
                                             long long n, const RunParams& p,
                                             const InterpTable& T, const FastTable& F,
                                             long long seg, int nseg, int model,
                                             unsigned long long* cursor, const unsigned* arrived,
                                             unsigned char* cls, unsigned long long* totals,
                                             unsigned* att, unsigned* acc, int* status) {
  StreamQueue Q;
  Q.seg = seg; Q.nseg = nseg; Q.model = model; Q.cursor = cursor; Q.arrived = arrived;
  Q.cls = cls;
#define NX_ARGS st, device, in0, in_stride, step0, P, n, p, T, F, Q, totals, att, acc, status
  // one moon + gravity: fast path with MO = 1 (MODE bit 4); more moons: generic kernel
  if (p.strict_math || p.nmoons > 1 || (p.nmoons == 1 && !p.gravity))
    return launch_adaptive_stream_mode<-1>(NX_ARGS);
  const int mode = (p.gravity ? 8 : 0) | (p.radpres ? 4 : 0) | (p.loss_mode & 3) |
                   (p.nmoons == 1 ? 16 : 0);
  switch (mode) {
    case 24: return launch_adaptive_stream_mode<24>(NX_ARGS);
    case 25: return launch_adaptive_stream_mode<25>(NX_ARGS);
    case 26: return launch_adaptive_stream_mode<26>(NX_ARGS);
    case 28: return launch_adaptive_stream_mode<28>(NX_ARGS);
    case 29: return launch_adaptive_stream_mode<29>(NX_ARGS);
    case 30: return launch_adaptive_stream_mode<30>(NX_ARGS);
    case 0: return launch_adaptive_stream_mode<0>(NX_ARGS);
    case 1: return launch_adaptive_stream_mode<1>(NX_ARGS);
    case 2: return launch_adaptive_stream_mode<2>(NX_ARGS);
    case 4: return launch_adaptive_stream_mode<4>(NX_ARGS);
    case 5: return launch_adaptive_stream_mode<5>(NX_ARGS);
    case 6: return launch_adaptive_stream_mode<6>(NX_ARGS);
    case 8: return launch_adaptive_stream_mode<8>(NX_ARGS);
    case 9: return launch_adaptive_stream_mode<9>(NX_ARGS);
    case 10: return launch_adaptive_stream_mode<10>(NX_ARGS);
    case 12: return launch_adaptive_stream_mode<12>(NX_ARGS);
    case 13: return launch_adaptive_stream_mode<13>(NX_ARGS);
    case 14: return launch_adaptive_stream_mode<14>(NX_ARGS);
    default: return cudaErrorInvalidValue;
  }
#undef NX_ARGS
}

cudaError_t launch_cost_order(cudaStream_t st, int device, StateCols P, long long n,
                              const RunParams& p, int model, unsigned char* bucket,
                              unsigned* hist_cursor, unsigned* perm, bool to_surface) {
  // hist_cursor: [0..31] histogram, [32..63] cursors
  cudaError_t e = cudaMemsetAsync(hist_cursor, 0, 2 * NX_NBUCKET * sizeof(unsigned), st);
  if (e != cudaSuccess) return e;
  long long blocks = (n + 255) / 256;
  const long long cap = (long long)sm_count(device) * 8;
  if (blocks > cap) blocks = cap;
  k_cost_histogram<<<(unsigned)blocks, 256, 0, st>>>(P, n, p, model, to_surface, bucket,
                                                      hist_cursor);
  k_cost_offsets<<<1, 32, 0, st>>>(hist_cursor, hist_cursor + NX_NBUCKET);
  const long long sb = (n + 256 * NX_SCATTER_ITEMS - 1) / (256 * NX_SCATTER_ITEMS);
  k_cost_scatter<<<(unsigned)sb, 256, 0, st>>>(n, bucket, hist_cursor + NX_NBUCKET, perm);
  return cudaGetLastError();
}

// K2 / K2b kernel selection; SINK builds exist for every kernel it can select, ion builds
// (Ion != nullptr, SINK false) for those of them with a loss term, trace builds (Trace !=
// nullptr, SINK false) for those of them without a moon.
template <bool SINK>
static cudaError_t dispatch_adaptive(cudaStream_t st, int device, StateCols In, StateCols P,
                                     long long n, const RunParams& p, const InterpTable& T,
                                     const FastTable& F, const unsigned* perm,
                                     unsigned long long* queue, unsigned long long* totals,
                                     unsigned* att, unsigned* acc, int* status,
                                     const Spline2D* S, uint64_t seed, uint64_t first_id,
                                     const DepositOut& Dep, const IonOut* Ion,
                                     const TraceOut* Trace) {
#define NX_ARGS st, device, In, P, n, p, T, F, perm, queue, totals, att, acc, status, \
                S ? *S : Spline2D{}, seed, first_id, Dep, Ion, Trace
  if (S) {
    // bounce builds: the strict kernel, and the fast kernels with gravity (one moon too);
    // runs without gravity or with more moons take the strict kernel
    if (p.strict_math || !p.gravity || p.nmoons > 1) return launch_adaptive_mode<-1, true, SINK>(NX_ARGS);
    switch ((p.radpres ? 4 : 0) | (p.loss_mode & 3) | (p.nmoons == 1 ? 16 : 0)) {
      case 16: return launch_adaptive_mode<24, true, SINK>(NX_ARGS);
      case 17: return launch_adaptive_mode<25, true, SINK>(NX_ARGS);
      case 18: return launch_adaptive_mode<26, true, SINK>(NX_ARGS);
      case 20: return launch_adaptive_mode<28, true, SINK>(NX_ARGS);
      case 21: return launch_adaptive_mode<29, true, SINK>(NX_ARGS);
      case 22: return launch_adaptive_mode<30, true, SINK>(NX_ARGS);
      case 0: return launch_adaptive_mode<8, true, SINK>(NX_ARGS);
      case 1: return launch_adaptive_mode<9, true, SINK>(NX_ARGS);
      case 2: return launch_adaptive_mode<10, true, SINK>(NX_ARGS);
      case 4: return launch_adaptive_mode<12, true, SINK>(NX_ARGS);
      case 5: return launch_adaptive_mode<13, true, SINK>(NX_ARGS);
      case 6: return launch_adaptive_mode<14, true, SINK>(NX_ARGS);
      default: return cudaErrorInvalidValue;
    }
  }
  if (p.strict_math || p.nmoons > 1 || (p.nmoons == 1 && !p.gravity))
    return launch_adaptive_mode<-1, false, SINK>(NX_ARGS);
  const int mode = (p.gravity ? 8 : 0) | (p.radpres ? 4 : 0) | (p.loss_mode & 3) |
                   (p.nmoons == 1 ? 16 : 0);
  switch (mode) {
    case 24: return launch_adaptive_mode<24, false, SINK>(NX_ARGS);
    case 25: return launch_adaptive_mode<25, false, SINK>(NX_ARGS);
    case 26: return launch_adaptive_mode<26, false, SINK>(NX_ARGS);
    case 28: return launch_adaptive_mode<28, false, SINK>(NX_ARGS);
    case 29: return launch_adaptive_mode<29, false, SINK>(NX_ARGS);
    case 30: return launch_adaptive_mode<30, false, SINK>(NX_ARGS);
    case 0: return launch_adaptive_mode<0, false, SINK>(NX_ARGS);
    case 1: return launch_adaptive_mode<1, false, SINK>(NX_ARGS);
    case 2: return launch_adaptive_mode<2, false, SINK>(NX_ARGS);
    case 4: return launch_adaptive_mode<4, false, SINK>(NX_ARGS);
    case 5: return launch_adaptive_mode<5, false, SINK>(NX_ARGS);
    case 6: return launch_adaptive_mode<6, false, SINK>(NX_ARGS);
    case 8: return launch_adaptive_mode<8, false, SINK>(NX_ARGS);
    case 9: return launch_adaptive_mode<9, false, SINK>(NX_ARGS);
    case 10: return launch_adaptive_mode<10, false, SINK>(NX_ARGS);
    case 12: return launch_adaptive_mode<12, false, SINK>(NX_ARGS);
    case 13: return launch_adaptive_mode<13, false, SINK>(NX_ARGS);
    case 14: return launch_adaptive_mode<14, false, SINK>(NX_ARGS);
    default: return cudaErrorInvalidValue;
  }
#undef NX_ARGS
}

cudaError_t launch_integrate_adaptive(cudaStream_t st, int device, StateCols In, StateCols P,
                                      long long n, const RunParams& p, const InterpTable& T,
                                      const FastTable& F, const unsigned* perm,
                                      unsigned long long* queue, unsigned long long* totals,
                                      unsigned* att, unsigned* acc, int* status,
                                      const Spline2D* S, uint64_t seed, uint64_t first_id,
                                      const DepositOut* dep, const IonOut* ion,
                                      const TraceOut* trace) {
  if ((dep != nullptr) + (ion != nullptr) + (trace != nullptr) > 1) return cudaErrorInvalidValue;
  if (dep)
    return dispatch_adaptive<true>(st, device, In, P, n, p, T, F, perm, queue, totals, att, acc,
                                   status, S, seed, first_id, *dep, nullptr, nullptr);
  return dispatch_adaptive<false>(st, device, In, P, n, p, T, F, perm, queue, totals, att, acc,
                                  status, S, seed, first_id, DepositOut{}, ion, trace);
}

template <int MODE>
static cudaError_t launch_constant_mode(cudaStream_t st, int device, StateCols In, StateCols P,
                                        long long n,
                                        const RunParams& p, const InterpTable& T,
                                        const FastTable& F, const Spline2D& S, uint64_t seed,
                                        uint64_t first_id, int nsteps, const ImageParams& ip,
                                        const GTables& G, double* image,
                                        unsigned long long* counts, double* traj,
                                        const RowSink& rows,
                                        unsigned long long* queue, unsigned long long* totals,
                                        int* status) {
  const size_t tbytes = (((MODE < 0) ? table_smem_bytes(T) : fast_table_smem_bytes(F)) + 15) & ~(size_t)15;
  const size_t smem = tbytes + (size_t)(NX_K3_THREADS / 32) * NX_POOL_BYTES_PER_WARP_ALIGNED;
  StepCoef hc;
  for (int m = 0; m < 7; ++m)
    for (int j = 0; j < 8; ++j) hc.v[m * 8 + j] = p.step_size * h_dp_a2[m * 8 + j];
  hc.v[56] = p.step_size * p.GM;
  int blocks = 0;
  const long long need = (n + 2 * NX_K3_THREADS - 1) / (2 * NX_K3_THREADS);
  cudaError_t e;
  if (rows.cursor) {
    e = persistent_grid(k_integrate_constant<MODE, true>, device, smem, &blocks, NX_K3_THREADS);
    if (e != cudaSuccess) return e;
    if (need < blocks) blocks = (int)(need > 0 ? need : 1);
    k_integrate_constant<MODE, true><<<blocks, NX_K3_THREADS, smem, st>>>(
        In, P, n, p, T, F, S, seed, first_id, nsteps, ip, G, image, counts, traj, rows, queue,
        totals, status, (unsigned)tbytes, hc);
  } else {
    e = persistent_grid(k_integrate_constant<MODE, false>, device, smem, &blocks, NX_K3_THREADS);
    if (e != cudaSuccess) return e;
    if (need < blocks) blocks = (int)(need > 0 ? need : 1);
    k_integrate_constant<MODE, false><<<blocks, NX_K3_THREADS, smem, st>>>(
        In, P, n, p, T, F, S, seed, first_id, nsteps, ip, G, image, counts, traj, rows, queue,
        totals, status, (unsigned)tbytes, hc);
  }
  return cudaGetLastError();
}

cudaError_t launch_integrate_constant(cudaStream_t st, int device, StateCols In, StateCols P,
                                      long long n, const RunParams& p, const InterpTable& T,
                                      const FastTable& F, const Spline2D& S, uint64_t seed,
                                      uint64_t first_id, int nsteps, const ImageParams& ip,
                                      const GTables& G, double* image,
                                      unsigned long long* counts, double* traj,
                                      const RowSink& rows,
                                      unsigned long long* queue, unsigned long long* totals,
                                      int* status) {
#define NX_ARGS st, device, In, P, n, p, T, F, S, seed, first_id, nsteps, ip, G, image, counts, \
                traj, rows, queue, totals, status
  if (p.strict_math || p.nmoons > 0) return launch_constant_mode<-1>(NX_ARGS);
  const int mode = (p.gravity ? 8 : 0) | (p.radpres ? 4 : 0) | (p.loss_mode & 3);
  switch (mode) {
    case 0: return launch_constant_mode<0>(NX_ARGS);
    case 1: return launch_constant_mode<1>(NX_ARGS);
    case 2: return launch_constant_mode<2>(NX_ARGS);
    case 4: return launch_constant_mode<4>(NX_ARGS);
    case 5: return launch_constant_mode<5>(NX_ARGS);
    case 6: return launch_constant_mode<6>(NX_ARGS);
    case 8: return launch_constant_mode<8>(NX_ARGS);
    case 9: return launch_constant_mode<9>(NX_ARGS);
    case 10: return launch_constant_mode<10>(NX_ARGS);
    case 12: return launch_constant_mode<12>(NX_ARGS);
    case 13: return launch_constant_mode<13>(NX_ARGS);
    case 14: return launch_constant_mode<14>(NX_ARGS);
    default: return cudaErrorInvalidValue;
  }
#undef NX_ARGS
}

cudaError_t launch_image_accumulate(cudaStream_t st, int device, StateCols P, long long n,
                                    const ImageParams& ip, const GTables& G, double* image,
                                    unsigned long long* counts, int mode) {
  size_t smem = gtables_smem_bytes(G);
  // privatised counts (mode 2): a square tile around the pixel of the projected planet centre
  const bool tiled = mode == 2;
  if (tiled) {
    const size_t budget = 227 * 1024 - 1024 - smem;
    int side = (int)std::sqrt((double)(budget / 4));
    side &= ~7;
    ImageTile tile;
    tile.w = side < ip.nx ? side : ip.nx;
    tile.h = side < ip.nz ? side : ip.nz;
    const double cx = (0.0 - ip.x0) / (ip.x1 - ip.x0) * ip.nx;
    const double cz = (0.0 - ip.z0) / (ip.z1 - ip.z0) * ip.nz;
    int ix0 = (int)cx - tile.w / 2, iz0 = (int)cz - tile.h / 2;
    if (!(cx == cx) || ix0 < 0) ix0 = 0;
    if (!(cz == cz) || iz0 < 0) iz0 = 0;
    if (ix0 > ip.nx - tile.w) ix0 = ip.nx - tile.w;
    if (iz0 > ip.nz - tile.h) iz0 = ip.nz - tile.h;
    tile.ix0 = ix0; tile.iz0 = iz0;
    const size_t total = smem + (size_t)tile.w * tile.h * 4;
    cudaError_t e = cudaFuncSetAttribute(k_image_accumulate_tile,
                                         cudaFuncAttributeMaxDynamicSharedMemorySize, (int)total);
    if (e != cudaSuccess) return e;
    long long blocks = sm_count(device);
    const long long need = ((n >> 1) + 1023) / 1024;
    if (need < blocks) blocks = need > 0 ? need : 1;
    k_image_accumulate_tile<<<(unsigned)blocks, 1024, total, st>>>(P, n, ip, G, tile, image, counts);
    return cudaGetLastError();
  }
  if (smem > 48 * 1024) {
    cudaError_t e = cudaFuncSetAttribute(k_image_accumulate,
                                         cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
  }
  int per_sm = 1;
  cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_image_accumulate, 256, smem);
  if (per_sm < 1) per_sm = 1;
  long long blocks = (long long)per_sm * sm_count(device);
  const long long need = ((n >> 1) + 255) / 256;
  if (need < blocks) blocks = need > 0 ? need : 1;
  k_image_accumulate<<<(unsigned)blocks, 256, smem, st>>>(P, n, ip, G, image, counts);
  return cudaGetLastError();
}

cudaError_t launch_image_cube(cudaStream_t st, int device, StateCols P, long long n,
                              const ImageParams& ip, const GTables& G, const CubeAxis& ax,
                              double* cube, unsigned long long* counts) {
  const size_t smem = gtables_smem_bytes(G);
  if (smem > 48 * 1024) {
    cudaError_t e = cudaFuncSetAttribute(k_image_cube, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         (int)smem);
    if (e != cudaSuccess) return e;
  }
  int per_sm = 1;
  cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_image_cube, 256, smem);
  if (per_sm < 1) per_sm = 1;
  long long blocks = (long long)per_sm * sm_count(device);
  const long long need = ((n >> 1) + 255) / 256;
  if (need < blocks) blocks = need > 0 ? need : 1;
  k_image_cube<<<(unsigned)blocks, 256, smem, st>>>(P, n, ip, G, ax, cube, counts);
  return cudaGetLastError();
}

cudaError_t launch_los_accumulate(cudaStream_t st, int device, StateCols P, long long n,
                                  long long nlos, const double* los, const double* dist_plan,
                                  const int* nball, const double* ladder, const double* wid2,
                                  const LosParams& lp, const LosConsts& lc, const GTables& G,
                                  double* radiance, unsigned long long* npack,
                                  unsigned char* included) {
  const long long bx = (nlos + NX_LOS_THREADS - 1) / NX_LOS_THREADS;
  // enough packet chunks to fill the machine a few times over
  long long target = 4LL * sm_count(device) * 4;
  long long by = (target + bx - 1) / bx;
  if (by < 1) by = 1;
  long long chunk = (n + by - 1) / by;
  chunk = ((chunk + NX_LOS_TILE - 1) / NX_LOS_TILE) * NX_LOS_TILE;
  by = (n + chunk - 1) / chunk;
  if (by > 65535) { by = 65535; chunk = (n + by - 1) / by; chunk = ((chunk + NX_LOS_TILE - 1) / NX_LOS_TILE) * NX_LOS_TILE; by = (n + chunk - 1) / chunk; }
  dim3 grid((unsigned)bx, (unsigned)by);
  k_los_accumulate<<<grid, NX_LOS_THREADS, 0, st>>>(P, n, nlos, los, dist_plan, nball, ladder,
                                                     wid2, lp, lc, G, radiance, npack, included,
                                                     chunk);
  return cudaGetLastError();
}

cudaError_t launch_fp64_peak(cudaStream_t st, int device, double* out, int iters, int* blocks,
                             int* threads) {
  *threads = 512;
  *blocks = sm_count(device) * 4;
  k_fp64_peak<<<*blocks, *threads, 0, st>>>(out, iters, 0.999999, 1e-7);
  return cudaGetLastError();
}

cudaError_t launch_copy(cudaStream_t st, int device, const double* src, double* dst,
                        long long n) {
  k_copy<<<sm_count(device) * 8, 256, 0, st>>>(reinterpret_cast<const double2*>(src),
                                               reinterpret_cast<double2*>(dst), n / 2);
  return cudaGetLastError();
}

}  // namespace nx
