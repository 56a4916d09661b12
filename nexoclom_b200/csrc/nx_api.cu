// nexoclom_b200 -- C ABI (include/nexoclom_b200.h) over the kernels.
// Host code only: context, device memory, table preparation, H2D/D2H copies,
// launches and CUDA-event timing.  No torch types, no global mutable state.
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>
#include <chrono>
#include <cstdio>
#include <cstdlib>

#include "../../include/nexoclom_b200.h"
#include "nx_kernels.h"
#include "nx_tables.h"

using namespace nx;

static_assert(sizeof(nx_run_params) == sizeof(RunParams), "RunParams layout");
static_assert(sizeof(nx_source_params) == sizeof(SourceParams), "SourceParams layout");
static_assert(sizeof(nx_image_params) == sizeof(ImageParams), "ImageParams layout");
static_assert(sizeof(nx_los_params) == sizeof(LosParams), "LosParams layout");

struct DevInterp {
  double *x = nullptr, *f = nullptr, *slope = nullptr;
  unsigned short* bucket = nullptr;
  InterpTable view{};
  double* rec = nullptr;                 // record form for the fast path
  unsigned short* fbucket = nullptr;
  FastTable fast{};
};

// A compacted packet table that stays on the GPU (device-side Output.save, nx_compact.cu)
struct nx_packets {
  long long n = 0, cap = 0;          // rows, column stride (multiple of 32)
  int ncols = 8;                     // 9: + the adaptive driver's step size
  double* cols = nullptr;            // ncols columns time..frac[, step_size]
  unsigned* index = nullptr;         // original packet index of every row
  unsigned short* step = nullptr;    // constant-step rows: step number (else nullptr)
  void* block = nullptr;             // the one stream-ordered allocation the three live in
};

// Packet tables come and go with every Output: they are carved from ONE block of the device's
// stream-ordered memory pool (cudaMallocAsync, release threshold 4 GB), so that
// creating / dropping a table costs microseconds instead of the implicit device
// synchronisation of cudaMalloc / cudaFree.  Everything else (slabs, scratch) is cudaMalloc'ed
// once and grows only; those sites trim the pool and retry when the device is full.
static cudaError_t dev_malloc(void** p, size_t bytes) {
  cudaError_t e = cudaMalloc(p, bytes);
  if (e == cudaErrorMemoryAllocation) {
    cudaGetLastError();
    int dev = 0;
    cudaMemPool_t pool;
    if (cudaGetDevice(&dev) == cudaSuccess &&
        cudaDeviceGetDefaultMemPool(&pool, dev) == cudaSuccess) {
      cudaDeviceSynchronize();
      cudaMemPoolTrimTo(pool, 0);
      e = cudaMalloc(p, bytes);
    }
  }
  return e;
}
template <class T> static cudaError_t dev_malloc(T** p, size_t bytes) {
  return dev_malloc(reinterpret_cast<void**>(p), bytes);
}
static cudaError_t table_alloc(nx_packets* h, cudaStream_t st, int ncols, bool with_step) {
  auto up = [](size_t b) { return (b + 255) / 256 * 256; };
  const size_t bc = up((size_t)ncols * h->cap * sizeof(double));
  const size_t bi = up((size_t)h->cap * sizeof(unsigned));
  const size_t bs = with_step ? up((size_t)h->cap * sizeof(unsigned short)) : 0;
  cudaError_t e = cudaMallocAsync(&h->block, bc + bi + bs, st);
  if (e != cudaSuccess) { h->block = nullptr; return e; }
  char* b = static_cast<char*>(h->block);
  h->cols = reinterpret_cast<double*>(b);
  h->index = reinterpret_cast<unsigned*>(b + bc);
  h->step = with_step ? reinterpret_cast<unsigned short*>(b + bc + bi) : nullptr;
  return cudaSuccess;
}
static void free_packets(nx_packets* h, cudaStream_t st) {
  if (!h) return;
  if (h->block) cudaFreeAsync(h->block, st);        // in stream order: after its last reader
  delete h;
}

// The context-owned accumulator of one product (nx_product): one device block of `nsum` f64
// sums, one f64 slot after them that carries a scalar through nx_product_allreduce, then, from
// the next 256-byte boundary, `ncount` u64 counts.  begin reuses a block that is large enough;
// nx_product_end frees it.  nsum == 0: begin has not been called since the last end.
struct Accum {
  void* block = nullptr;
  size_t cap = 0;                    // bytes of `block`
  long long nsum = 0, ncount = 0;
  int dims[3] = {};                  // begin's shape: image nx, nz; cube nx, nz, nbins; nlon, nlat
  static size_t count_offset(long long nsum) { return ((size_t)(nsum + 1) * 8 + 255) / 256 * 256; }
  double* sums() const { return static_cast<double*>(block); }
  unsigned long long* counts() const {
    return reinterpret_cast<unsigned long long*>(static_cast<char*>(block) + count_offset(nsum));
  }
};

struct nx_ctx {
  int device = 0;
  cudaStream_t stream = nullptr;
  bool own_stream = true;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  float last_ms = 0.f;
  unsigned long long launches = 0;
  std::string err;

  RunParams params{};
  bool have_params = false;
  DevInterp radpres;
  DevInterp speed;
  DevInterp lon1d;             // inverse CDF of a longitude-only source map
  DevInterp gtab[NX_MAX_GTABLES];
  DevInterp gsum;              // sum of the g-value tables on the union of their nodes
  GTables gtables{};
  double *spl_tx = nullptr, *spl_ty = nullptr, *spl_c = nullptr;
  Spline2D spline{};
  double* srcmap = nullptr;
  SourceMap map{};

  long long cap = 0;           // column stride (multiple of 32)
  double* state = nullptr;     // 9 columns
  double* x0 = nullptr;        // 14 columns
  // K1 writes the X0 slab only; until an integrator (or materialize()) has filled the state
  // slab, the packets' current state IS columns 0-7 of X0 (`fresh`).
  bool fresh = false;
  bool x0_valid = false;
  nx_packets* bound = nullptr; // K4 / K5 / K6 inputs come from this table instead of the slab
  // grow-only device scratch, one slot per temporary of the product calls: no cudaMalloc /
  // cudaFree (an implicit device synchronisation each) on the calls LOSResult / ModelImage
  // make once per output file, and nothing to leak on an error path
  struct Scratch { void* p = nullptr; size_t bytes = 0; } scr[32];
  Accum accum[NX_PRODUCT_IONIZE + 1];    // one per nx_product
  IonOut ion_axes{};                     // the grid of nx_ionize_begin (axes only)
  void* pinned = nullptr;      // grow-only pinned staging for small D2H results (image, LOS columns)
  size_t pinned_bytes = 0;
  unsigned* cmp_tiles = nullptr;     // compaction scratch (tile counts)
  long long cmp_tiles_cap = 0;       // X0 columns 0-7 hold an initial state (K1 or the host-buffer path)
  unsigned *att = nullptr, *acc = nullptr;
  unsigned* perm = nullptr;          // longest-first processing order
  unsigned char* cost = nullptr;     // cost bucket per packet
  unsigned* hist = nullptr;          // 32 histogram + 32 cursors
  int order_packets = 3;              // cost model: 0 none, 1 ballistic, 2 / 3 + radiation pressure (3: lift-off threshold)
  int schedule = 1;                   // K2 queue: 1 class-ordered streaming passes, 0 sort + permutation
  unsigned long long* squeue = nullptr;   // NX_STREAM_CURSORS cursors, then the `arrived` word
  unsigned* seq_host = nullptr;           // pinned 0..32: source of the `arrived` updates
  cudaStream_t copy_stream = nullptr;
  cudaEvent_t copy_ev[2] = {};
  int los_mode = 0;                  // 0 auto, 1 brute force, 2 cell grid
  int image_mode = 0;                // K4: 0 auto, 1 global atomics only, 2 privatised counts
  int class_cache = 1;               // streaming schedule: remember each packet's cost class
  int los_order = 1;                 // process lines of sight in Morton order of closest approach
  cudaStream_t pipe[16] = {};                  // H2D / compute pipeline of the host-buffer path
  cudaEvent_t pipe_ev[17] = {};
  unsigned long long* pipe_scalars = nullptr;  // 4 u64 per chunk
  unsigned* pipe_hist = nullptr;               // 64 u32 per chunk
  LosGridWork losw;
  // candidate pairs of the last nx_los_accumulate_counted call, still in losw.pairs (np > 0):
  // nx_los_used_fill resolves them again instead of repeating the whole search
  struct LosKept {
    unsigned long long np = 0;
    long long n = 0, nlos = 0;
    const void* bound = nullptr;
    LosParams lp{};
    LosConsts lc{};
    size_t nladder = 0;
  } los_kept;
  unsigned long long* scalars = nullptr;   // [0] queue, [1] total attempted, [2] total accepted
  int* status = nullptr;
  int status_host = 0;
};

#define CK(call)                                                                       \
  do {                                                                                 \
    cudaError_t e_ = (call);                                                           \
    if (e_ != cudaSuccess) {                                                           \
      ctx->err = std::string(#call) + ": " + cudaGetErrorString(e_);                   \
      return -(int)e_;                                                                 \
    }                                                                                  \
  } while (0)
// Every entry point that can change what the line-of-sight kernels read starts with ENTER: it selects
// the device and drops the candidate pairs a line-of-sight call may have left for
// nx_los_used_fill (which alone keeps them).
#define ENTER(ctx)                                                                     \
  do {                                                                                 \
    (ctx)->los_kept.np = 0;                                                            \
    CK(cudaSetDevice((ctx)->device));                                                  \
  } while (0)

static void free_interp(DevInterp& d) {
  cudaFree(d.x); cudaFree(d.f); cudaFree(d.slope); cudaFree(d.bucket);
  cudaFree(d.rec); cudaFree(d.fbucket);
  d = DevInterp{};
}

static int upload_interp(nx_ctx* ctx, DevInterp& d, const double* x, const double* f, int n,
                         bool want_fast = true, int fast_nbucket = 32768) {
  free_interp(d);
  if (n <= 0) return 0;
  HostInterp h = make_interp(x, f, n);
  CK(cudaMalloc(&d.x, n * sizeof(double)));
  CK(cudaMalloc(&d.f, n * sizeof(double)));
  CK(cudaMalloc(&d.slope, n * sizeof(double)));
  CK(cudaMalloc(&d.bucket, h.nbucket * sizeof(unsigned short)));
  CK(cudaMemcpyAsync(d.x, h.x.data(), n * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaMemcpyAsync(d.f, h.f.data(), n * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaMemcpyAsync(d.slope, h.slope.data(), n * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaMemcpyAsync(d.bucket, h.bucket.data(), h.nbucket * sizeof(unsigned short),
                     cudaMemcpyHostToDevice, ctx->stream));
  if (!want_fast) {      // inverse-CDF tables are only read through the np.interp form
    CK(cudaStreamSynchronize(ctx->stream));
    d.view.x = d.x; d.view.f = d.f; d.view.slope = d.slope; d.view.bucket = d.bucket;
    d.view.n = n; d.view.nbucket = h.nbucket; d.view.blo = h.blo; d.view.binvw = h.binvw;
    return 0;
  }
  HostFastTable hf = make_fast_table(x, f, n, fast_nbucket);
  if (hf.max_steps > NX_FAST_TABLE_MAX_STEPS) {
    ctx->err = "lookup table has more than two nodes within 1/2^22 of its range";
    return -1;
  }
  CK(cudaMalloc(&d.rec, hf.rec.size() * sizeof(double)));
  CK(cudaMalloc(&d.fbucket, hf.bucket.size() * sizeof(unsigned short)));
  CK(cudaMemcpyAsync(d.rec, hf.rec.data(), hf.rec.size() * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaMemcpyAsync(d.fbucket, hf.bucket.data(), hf.bucket.size() * sizeof(unsigned short),
                     cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  d.fast.rec = reinterpret_cast<const InterpRec*>(d.rec); d.fast.bucket = d.fbucket;
  d.fast.nrec = hf.nrec; d.fast.nbucket = hf.nbucket; d.fast.blo = hf.blo; d.fast.binvw = hf.binvw; d.fast.boff = -hf.blo * hf.binvw;
  d.view.x = d.x; d.view.f = d.f; d.view.slope = d.slope; d.view.bucket = d.bucket;
  d.view.n = n; d.view.nbucket = h.nbucket; d.view.blo = h.blo; d.view.binvw = h.binvw;
  return 0;
}

static void free_los_work(LosGridWork& w) {
  cudaFree(w.sorted.pos);
  cudaFree(w.sorted.frac); cudaFree(w.sorted.idx); cudaFree(w.cell_id); cudaFree(w.count);
  cudaFree(w.start); cudaFree(w.block_sum); cudaFree(w.total); cudaFree(w.extent_bits);
  cudaFree(w.pairs); cudaFree(w.pair_cursor);
  const int G = w.G_fixed;
  const double scale = w.scale;
  const unsigned long long pcf = w.pairs_cap_fixed;
  w = LosGridWork{};
  w.G_fixed = G;
  w.scale = scale;
  w.pairs_cap_fixed = pcf;
}

static int alloc_los_work(nx_ctx* ctx, long long n) {
  LosGridWork& w = ctx->losw;
  if (w.cap >= n && w.sorted.pos) return 0;
  free_los_work(w);
  const int gmax = w.G_fixed > NX_LOS_GRID_MAX ? w.G_fixed : NX_LOS_GRID_MAX;
  const size_t ncell = (size_t)gmax * gmax * gmax;
  const size_t nn = (size_t)n;
  CK(dev_malloc(&w.sorted.pos, nn * sizeof(double4)));
  CK(dev_malloc(&w.sorted.frac, nn * sizeof(double)));
  CK(dev_malloc(&w.sorted.idx, nn * sizeof(unsigned)));
  CK(dev_malloc(&w.cell_id, nn * sizeof(unsigned)));
  CK(cudaMalloc(&w.count, ncell * sizeof(unsigned)));
  CK(cudaMalloc(&w.start, (ncell + 1) * sizeof(unsigned)));
  CK(cudaMalloc(&w.block_sum, ((ncell + 4095) / 4096 + 1) * sizeof(unsigned)));
  CK(cudaMalloc(&w.total, sizeof(unsigned)));
  CK(cudaMalloc(&w.extent_bits, 2 * sizeof(unsigned long long)));
  // pair buffer: 32 pairs per packet, between 4 M and 512 M entries (4 GB of the 180), never
  // less than one line of sight can produce (every packet once); lines of sight are batched
  // when it cannot hold all pairs (launch_los_grid)
  unsigned long long pc = 32ull * (unsigned long long)n;
  if (pc < (1ull << 22)) pc = 1ull << 22;
  if (pc > (1ull << 29)) pc = 1ull << 29;
  if (n > 40000000LL) pc = 1ull << 30;              // 8 GB next to 40+ GB of packet slabs
  if (w.pairs_cap_fixed) pc = w.pairs_cap_fixed;    // developer option "los_pair_cap"
  if (pc < (unsigned long long)n + 1024) pc = (unsigned long long)n + 1024;
  CK(dev_malloc(&w.pairs, pc * sizeof(uint2)));
  CK(cudaMalloc(&w.pair_cursor, 2 * sizeof(unsigned long long)));   // pairs written, line-of-sight ticket
  w.pairs_cap = pc;
  w.batch_hint = 0;
  w.cap = n;
  return 0;
}

enum { SCR_LOS, SCR_DIST, SCR_RAD, SCR_NP, SCR_INC, SCR_NBALL, SCR_LADDER,
       SCR_WID2, SCR_ORDER, SCR_NUSED, SCR_CURSOR, SCR_OFF, SCR_IDX, SCR_SM_IN, SCR_SM_PTS,
       SCR_SM_OUT, SCR_SM_CNT, SCR_TMP, SCR_IMG_OUT, SCR_DD, SCR_KEY, SCR_DENS_IN, SCR_DENS_OUT,
       SCR_DENS_IDX, SCR_SPEC, SCR_NSLOTS };
static_assert(SCR_NSLOTS <= 32, "nx_ctx::scr is too small");
static int scratch_bytes(nx_ctx* ctx, int slot, size_t bytes, void** out) {
  nx_ctx::Scratch& sc = ctx->scr[slot];
  if (bytes > sc.bytes) {
    cudaFree(sc.p);
    sc.p = nullptr; sc.bytes = 0;
    const size_t want = bytes + bytes / 4 + 256;
    cudaError_t e = dev_malloc(&sc.p, want);
    if (e != cudaSuccess) { ctx->err = std::string("scratch allocation: ") + cudaGetErrorString(e); return -(int)e; }
    sc.bytes = want;
  }
  *out = sc.p;
  return 0;
}
#define SCR(slot, ptr, count)                                                              \
  do {                                                                                     \
    void* p_ = nullptr;                                                                    \
    int r_ = scratch_bytes(ctx, slot, (size_t)(count) * sizeof(*(ptr)), &p_);              \
    if (r_) return r_;                                                                     \
    (ptr) = reinterpret_cast<decltype(ptr)>(p_);                                           \
  } while (0)

static int pinned_staging(nx_ctx* ctx, size_t bytes) {
  if (bytes <= ctx->pinned_bytes) return 0;
  if (ctx->pinned) cudaFreeHost(ctx->pinned);
  ctx->pinned = nullptr; ctx->pinned_bytes = 0;
  CK(cudaHostAlloc(&ctx->pinned, bytes, cudaHostAllocDefault));
  ctx->pinned_bytes = bytes;
  return 0;
}

// ---- context-owned accumulators (image, cube, deposition, ion production) -------------------
// None of these calls ENTER: nothing here changes what the line-of-sight kernels read, so the
// candidate pairs nx_los_accumulate_counted keeps stay valid.
static const char* const accum_begin_name[] = {"nx_image_begin", "nx_cube_begin",
                                               "nx_deposit_begin", "nx_ionize_begin"};

// The accumulator of `which` when its begin has run; else NULL with the error set.
static Accum* accum_of(nx_ctx* ctx, int which) {
  if (which < NX_PRODUCT_IMAGE || which > NX_PRODUCT_IONIZE) {
    ctx->err = "unknown nx_product";
    return nullptr;
  }
  Accum& a = ctx->accum[which];
  if (!a.nsum) {
    ctx->err = std::string(accum_begin_name[which]) + " not called";
    return nullptr;
  }
  return &a;
}

// The common half of a begin, after the product has validated its shape: a zeroed block of
// nsum sums, the slot and ncount counts.
static int accum_begin(nx_ctx* ctx, nx_product which, long long nsum, long long ncount, int d0,
                       int d1, int d2) {
  Accum& a = ctx->accum[which];
  const size_t bytes = Accum::count_offset(nsum) + (size_t)ncount * 8;
  if (bytes > a.cap) {
    void* old = a.block;
    a = Accum{};
    CK(cudaFree(old));
    CK(dev_malloc(&a.block, bytes));
    a.cap = bytes;
  }
  a.nsum = nsum; a.ncount = ncount;
  a.dims[0] = d0; a.dims[1] = d1; a.dims[2] = d2;
  CK(cudaMemsetAsync(a.block, 0, bytes, ctx->stream));
  return 0;
}

int nx_product_fetch(nx_ctx* ctx, nx_product which, double* sums, long long* counts) {
  CK(cudaSetDevice(ctx->device));
  const Accum* a = accum_of(ctx, which);
  if (!a) return -1;
  // page-locked destinations (nx_host_alloc) get the DMA directly; pageable ones are staged by
  // the driver (a pinned staging buffer of the context, grow-only, would outlive a cube)
  if (sums) CK(cudaMemcpyAsync(sums, a->sums(), a->nsum * 8, cudaMemcpyDeviceToHost, ctx->stream));
  if (counts)
    CK(cudaMemcpyAsync(counts, a->counts(), a->ncount * 8, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  return 0;
}

int nx_product_device_ptrs(nx_ctx* ctx, nx_product which, void** sums, void** counts) {
  const Accum* a = accum_of(ctx, which);
  if (!a) return -1;
  if (sums) *sums = a->sums();
  if (counts) *counts = a->counts();
  return 0;
}

// The one collective of a product (SURVEY section 8e), in place on the context's stream.  With
// a total it rides in the slot after the sums and is read back (the call then waits for the
// stream); without one nothing waits.
int nx_product_allreduce(nx_ctx* ctx, nx_product which, nx_comm* comm, double* total) {
  CK(cudaSetDevice(ctx->device));
  Accum* a = accum_of(ctx, which);
  if (!a) return -1;
  double* slot = a->sums() + a->nsum;
  if (total) CK(cudaMemcpyAsync(slot, total, sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
  int r = nx_allreduce(comm, a->sums(), a->nsum + (total ? 1 : 0), NX_DTYPE_F64, ctx->stream);
  if (r == 0) r = nx_allreduce(comm, a->counts(), a->ncount, NX_DTYPE_I64, ctx->stream);
  if (r) { ctx->err = std::string("nx_product_allreduce: ") + nx_comm_last_error(); return r; }
  if (total) {
    CK(cudaMemcpyAsync(total, slot, sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
  }
  return 0;
}

int nx_product_end(nx_ctx* ctx, nx_product which) {
  CK(cudaSetDevice(ctx->device));
  Accum* a = accum_of(ctx, which);
  if (!a) return -1;
  CK(cudaStreamSynchronize(ctx->stream));
  void* block = a->block;
  *a = Accum{};
  CK(cudaFree(block));
  return 0;
}

static StateCols state_cols(nx_ctx* ctx) {
  StateCols P;
  if (ctx->bound) {
    for (int k = 0; k < 8; ++k) P.c[k] = ctx->bound->cols + (size_t)k * ctx->bound->cap;
    P.c[8] = ctx->bound->ncols > 8 ? ctx->bound->cols + (size_t)8 * ctx->bound->cap : nullptr;
    return P;
  }
  for (int k = 0; k < 9; ++k) P.c[k] = ctx->state + (size_t)k * ctx->cap;
  return P;
}
// rows the product kernels (K4 / K5) may read
static long long resident_rows(nx_ctx* ctx) { return ctx->bound ? ctx->bound->n : ctx->cap; }
static X0Cols x0_cols(nx_ctx* ctx) {
  X0Cols X;
  for (int k = 0; k < 14; ++k) X.c[k] = ctx->x0 + (size_t)k * ctx->cap;
  return X;
}

// columns the packets' CURRENT state is read from
static StateCols in_cols(nx_ctx* ctx) {
  StateCols P = state_cols(ctx);
  if (ctx->fresh && !ctx->bound)
    for (int k = 0; k < 8; ++k) P.c[k] = ctx->x0 + (size_t)k * ctx->cap;
  return P;
}
// make the state slab hold the current state (consumers that are not integrators)
static int materialize(nx_ctx* ctx) {
  if (!ctx->fresh || ctx->bound) return 0;
  StateCols P = state_cols(ctx);
  for (int k = 0; k < 8; ++k) {
    cudaError_t e = cudaMemcpyAsync(P.c[k], ctx->x0 + (size_t)k * ctx->cap,
                                    (size_t)ctx->cap * sizeof(double), cudaMemcpyDeviceToDevice,
                                    ctx->stream);
    if (e != cudaSuccess) { ctx->err = cudaGetErrorString(e); return -(int)e; }
  }
  cudaError_t e = launch_fill(ctx->stream, P.c[8], ctx->cap, 1000.0);     // Output.py:246
  if (e != cudaSuccess) { ctx->err = cudaGetErrorString(e); return -(int)e; }
  ctx->launches += 1;
  ctx->fresh = false;
  return 0;
}

static int begin_timed(nx_ctx* ctx) { CK(cudaEventRecord(ctx->ev0, ctx->stream)); return 0; }
static int end_timed(nx_ctx* ctx, int nlaunch) {
  CK(cudaEventRecord(ctx->ev1, ctx->stream));
  ctx->launches += nlaunch;
  return 0;
}

extern "C" {

int nx_ctx_create(int device, nx_ctx** out) {
  if (!out) return -1;
  *out = nullptr;
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || device < 0 || device >= ndev) {
    fprintf(stderr, "nexoclom_b200: no usable CUDA device %d (%s); there is no CPU fallback\n",
            device, e == cudaSuccess ? "index out of range" : cudaGetErrorString(e));
    return e == cudaSuccess ? -(int)cudaErrorInvalidDevice : -(int)e;
  }
  nx_ctx* ctx = new nx_ctx();
  ctx->device = device;
  if (cudaSetDevice(device) != cudaSuccess ||
      cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking) != cudaSuccess ||
      cudaEventCreate(&ctx->ev0) != cudaSuccess || cudaEventCreate(&ctx->ev1) != cudaSuccess ||
      cudaMalloc(&ctx->scalars, 8 * sizeof(unsigned long long)) != cudaSuccess ||
      cudaMalloc(&ctx->status, sizeof(int)) != cudaSuccess ||
      cudaMalloc(&ctx->squeue, (NX_STREAM_CURSORS + 1) * sizeof(unsigned long long)) != cudaSuccess ||
      cudaHostAlloc(&ctx->seq_host, 33 * sizeof(unsigned), cudaHostAllocDefault) != cudaSuccess ||
      cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking) != cudaSuccess ||
      cudaEventCreateWithFlags(&ctx->copy_ev[0], cudaEventDisableTiming) != cudaSuccess ||
      cudaEventCreateWithFlags(&ctx->copy_ev[1], cudaEventDisableTiming) != cudaSuccess ||
      cudaMemset(ctx->status, 0, sizeof(int)) != cudaSuccess) {
    fprintf(stderr, "nexoclom_b200: context setup failed: %s\n",
            cudaGetErrorString(cudaGetLastError()));
    delete ctx;
    return -2;
  }
  for (unsigned i = 0; i <= 32; ++i) ctx->seq_host[i] = i;
  {
    cudaMemPool_t pool;                       // keep freed packet tables for the next Output
    if (cudaDeviceGetDefaultMemPool(&pool, device) == cudaSuccess) {
      unsigned long long keep = 4ull << 30;   // beyond 4 GB freed blocks go back to the driver
      cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
    }
    cudaGetLastError();
  }
  *out = ctx;
  return 0;
}

int nx_ctx_destroy(nx_ctx* ctx) {
  if (!ctx) return 0;
  cudaSetDevice(ctx->device);
  cudaStreamSynchronize(ctx->stream);
  free_interp(ctx->radpres);
  free_interp(ctx->speed);
  free_interp(ctx->lon1d);
  for (auto& g : ctx->gtab) free_interp(g);
  free_interp(ctx->gsum);
  cudaFree(ctx->spl_tx); cudaFree(ctx->spl_ty); cudaFree(ctx->spl_c);
  cudaFree(ctx->srcmap);
  cudaFree(ctx->state); cudaFree(ctx->x0); cudaFree(ctx->att); cudaFree(ctx->acc);
  cudaFree(ctx->perm); cudaFree(ctx->cost); cudaFree(ctx->hist);
  free_los_work(ctx->losw);
  for (auto& s : ctx->pipe) if (s) cudaStreamDestroy(s);
  for (auto& e : ctx->pipe_ev) if (e) cudaEventDestroy(e);
  cudaFree(ctx->pipe_scalars); cudaFree(ctx->pipe_hist);
  cudaFree(ctx->scalars); cudaFree(ctx->status); cudaFree(ctx->cmp_tiles);
  for (auto& sc : ctx->scr) cudaFree(sc.p);
  for (auto& a : ctx->accum) cudaFree(a.block);
  cudaFree(ctx->squeue); cudaFreeHost(ctx->seq_host);
  if (ctx->pinned) cudaFreeHost(ctx->pinned);
  if (ctx->copy_stream) cudaStreamDestroy(ctx->copy_stream);
  for (auto& e : ctx->copy_ev) if (e) cudaEventDestroy(e);
  cudaEventDestroy(ctx->ev0); cudaEventDestroy(ctx->ev1);
  if (ctx->own_stream) cudaStreamDestroy(ctx->stream);
  delete ctx;
  return 0;
}

int nx_ctx_set_stream(nx_ctx* ctx, void* cuda_stream) {
  ENTER(ctx);
  CK(cudaStreamSynchronize(ctx->stream));
  if (ctx->own_stream) CK(cudaStreamDestroy(ctx->stream));
  ctx->stream = reinterpret_cast<cudaStream_t>(cuda_stream);
  ctx->own_stream = false;
  return 0;
}

int nx_ctx_sync(nx_ctx* ctx) {
  CK(cudaSetDevice(ctx->device));
  CK(cudaStreamSynchronize(ctx->stream));
  return 0;
}

int nx_ctx_set_option(nx_ctx* ctx, const char* name, int value) {
  ENTER(ctx);
  if (name && std::strcmp(name, "order_packets") == 0) { ctx->order_packets = value; return 0; }
  if (name && std::strcmp(name, "schedule") == 0) { ctx->schedule = value; return 0; }
  if (name && std::strcmp(name, "los_mode") == 0) { ctx->los_mode = value; return 0; }
  if (name && std::strcmp(name, "image_mode") == 0) { ctx->image_mode = value; return 0; }
  if (name && std::strcmp(name, "los_order") == 0) { ctx->los_order = value; return 0; }
  if (name && std::strcmp(name, "class_cache") == 0) { ctx->class_cache = value; return 0; }
  if (name && std::strcmp(name, "los_grid") == 0) { ctx->losw.G_fixed = value; ctx->losw.cap = 0; return 0; }
  if (name && std::strcmp(name, "los_pair_cap") == 0) {
    ctx->losw.pairs_cap_fixed = value > 0 ? (unsigned long long)value : 0ull;
    ctx->losw.cap = 0;
    return 0;
  }
  if (name && std::strcmp(name, "los_grid_scale_milli") == 0) { ctx->losw.scale = 1e-3 * value; return 0; }
  ctx->err = std::string("unknown option ") + (name ? name : "(null)");
  return -1;
}

int nx_source_map(nx_ctx* ctx, long long n, const nx_source_map_params* p_,
                  const double* longitude, const double* latitude, const double* speed_kms,
                  const double* altitude, const double* azimuth, const double* frac,
                  const double* point_lon, const double* point_lat, const double* point_radius,
                  double* abundance_hist, double* speed_dist, double* altitude_dist,
                  double* azimuth_dist, long long* n_included, long long* n_total,
                  double* abundance, double* speed_map, double* altitude_map,
                  double* azimuth_map) {
  CK(cudaSetDevice(ctx->device));
  SourceMapParams sp;
  static_assert(sizeof(SourceMapParams) == sizeof(nx_source_map_params), "ABI mirror");
  std::memcpy(&sp, p_, sizeof(sp));
  if (sp.nlon < 1 || sp.nlat < 1 || sp.nvel < 1 || sp.nalt < 1 || sp.naz < 1 || !(sp.vmax > 0.0)) {
    ctx->err = "nx_source_map: bad bin counts / vmax";
    return -1;
  }
  const size_t npts = (size_t)sp.nlon * sp.nlat;
  // per-row constants: cos(lat_p) and sklearn's reduced radius sin^2(r/2)
  std::vector<double> pcos(sp.nlat), pthr(sp.nlat);
  for (int j = 0; j < sp.nlat; ++j) {
    pcos[j] = std::cos(point_lat[j]);
    const double t = std::sin(0.5 * point_radius[j]);
    pthr[j] = t * t;
  }
  const size_t nd = (size_t)(n > 0 ? n : 1);
  const size_t out_doubles = npts + sp.nvel + sp.nalt + sp.naz + npts +
                             npts * ((size_t)sp.nvel + sp.nalt + sp.naz);
  double *d_in = nullptr, *d_pts = nullptr, *d_out = nullptr;
  unsigned long long* d_cnt = nullptr;
  SCR(SCR_SM_IN, d_in, 6 * nd);
  SCR(SCR_SM_PTS, d_pts, (size_t)sp.nlon + 3 * (size_t)sp.nlat);
  SCR(SCR_SM_OUT, d_out, out_doubles);
  SCR(SCR_SM_CNT, d_cnt, 2 * npts);
  const double* cols[6] = {longitude, latitude, speed_kms, altitude, azimuth, frac};
  for (int k = 0; k < 6; ++k)
    if (n > 0) CK(cudaMemcpyAsync(d_in + k * nd, cols[k], (size_t)n * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
  double* d_plon = d_pts; double* d_plat = d_plon + sp.nlon;
  double* d_pcos = d_plat + sp.nlat; double* d_pthr = d_pcos + sp.nlat;
  CK(cudaMemcpyAsync(d_plon, point_lon, sp.nlon * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaMemcpyAsync(d_plat, point_lat, sp.nlat * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaMemcpyAsync(d_pcos, pcos.data(), sp.nlat * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaMemcpyAsync(d_pthr, pthr.data(), sp.nlat * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaMemsetAsync(d_out, 0, out_doubles * sizeof(double), ctx->stream));
  CK(cudaMemsetAsync(d_cnt, 0, 2 * npts * sizeof(unsigned long long), ctx->stream));
  SourceMapOut o;
  double* q = d_out;
  o.abundance_hist = q; q += npts;
  o.speed_dist = q; q += sp.nvel;
  o.altitude_dist = q; q += sp.nalt;
  o.azimuth_dist = q; q += sp.naz;
  o.abundance = q; q += npts;
  o.speed_map = q; q += npts * sp.nvel;
  o.altitude_map = q; q += npts * sp.nalt;
  o.azimuth_map = q;
  o.n_included = d_cnt; o.n_total = d_cnt + npts;
  int r;
  if ((r = begin_timed(ctx))) return r;
  CK(launch_source_map(ctx->stream, n, sp, d_in, d_in + nd, d_in + 2 * nd, d_in + 3 * nd,
                       d_in + 4 * nd, d_in + 5 * nd, d_plon, d_plat, d_pcos, d_pthr, o));
  if ((r = end_timed(ctx, 1))) return r;
  auto back = [&](void* dst, const void* src, size_t bytes) {
    return cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, ctx->stream);
  };
  CK(back(abundance_hist, o.abundance_hist, npts * sizeof(double)));
  CK(back(speed_dist, o.speed_dist, sp.nvel * sizeof(double)));
  CK(back(altitude_dist, o.altitude_dist, sp.nalt * sizeof(double)));
  CK(back(azimuth_dist, o.azimuth_dist, sp.naz * sizeof(double)));
  CK(back(abundance, o.abundance, npts * sizeof(double)));
  CK(back(speed_map, o.speed_map, npts * sp.nvel * sizeof(double)));
  CK(back(altitude_map, o.altitude_map, npts * sp.nalt * sizeof(double)));
  CK(back(azimuth_map, o.azimuth_map, npts * sp.naz * sizeof(double)));
  CK(back(n_included, o.n_included, npts * sizeof(long long)));
  CK(back(n_total, o.n_total, npts * sizeof(long long)));
  CK(cudaStreamSynchronize(ctx->stream));
  return 0;
}

// developer hook: K2 instrumentation words (all zero unless built with NX_STREAM_DEBUG)
int nx_debug_queue(nx_ctx* ctx, unsigned long long* out, int count) {
  CK(cudaSetDevice(ctx->device));
  CK(cudaStreamSynchronize(ctx->stream));
  CK(debug_read(out, count));
  return 0;
}

const char* nx_last_error(nx_ctx* ctx) { return ctx ? ctx->err.c_str() : "null context"; }

int nx_status(nx_ctx* ctx, int* bits) {
  CK(cudaSetDevice(ctx->device));
  int v = 0;
  CK(cudaMemcpyAsync(&v, ctx->status, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  if (bits) *bits = v;
  return 0;
}

int nx_tables_upload(nx_ctx* ctx, const nx_run_params* p, const double* rv, const double* ra,
                     int nrp, const double* tx, int ntx, const double* ty, int nty,
                     const double* c) {
  ENTER(ctx);
  std::memcpy(&ctx->params, p, sizeof(RunParams));
  ctx->have_params = true;
  if (ctx->params.radpres && nrp < 2) {
    ctx->err = "radpres enabled but no radiation-pressure table given";
    return -1;
  }
  int r = upload_interp(ctx, ctx->radpres, rv, ra, ctx->params.radpres ? nrp : 0);
  if (r) return r;
  cudaFree(ctx->spl_tx); cudaFree(ctx->spl_ty); cudaFree(ctx->spl_c);
  ctx->spl_tx = ctx->spl_ty = ctx->spl_c = nullptr;
  ctx->spline = Spline2D{};
  if (tx && ty && c && ntx > 8 && nty > 8) {
    const size_t nc = (size_t)(ntx - 4) * (nty - 4);
    CK(cudaMalloc(&ctx->spl_tx, ntx * sizeof(double)));
    CK(cudaMalloc(&ctx->spl_ty, nty * sizeof(double)));
    CK(cudaMalloc(&ctx->spl_c, nc * sizeof(double)));
    CK(cudaMemcpyAsync(ctx->spl_tx, tx, ntx * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(ctx->spl_ty, ty, nty * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(ctx->spl_c, c, nc * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    ctx->spline = Spline2D{ctx->spl_tx, ctx->spl_ty, ctx->spl_c, ntx, nty};
  }
  return 0;
}

int nx_gtables_upload(nx_ctx* ctx, int ntables, const int* sizes, const double* v,
                      const double* g) {
  ENTER(ctx);
  if (ntables < 0 || ntables > NX_MAX_GTABLES) { ctx->err = "too many g-value tables"; return -1; }
  ctx->gtables.n = 0;
  size_t off = 0;
  for (int t = 0; t < ntables; ++t) {
    // small bucket index (doubled by the builder until <= 2 nodes per bucket): K4 stages it
    // in shared memory together with the records
    int r = upload_interp(ctx, ctx->gtab[t], v + off, g + off, sizes[t], true, 256);
    if (r) return r;
    ctx->gtables.t[t] = ctx->gtab[t].view;
    ctx->gtables.f[t] = ctx->gtab[t].fast;
    off += sizes[t];
  }
  ctx->gtables.n = ntables;
  ctx->gtables.has_sum = 0;
  if (ntables > 1) {
    // union grid and the sum of the np.interp values there (ModelResult.py:152-157 adds the
    // lines up per packet; the kernels look the sum up once)
    std::vector<double> xs(v, v + off);
    std::sort(xs.begin(), xs.end());
    xs.erase(std::unique(xs.begin(), xs.end()), xs.end());
    std::vector<double> fs(xs.size(), 0.0);
    size_t o = 0;
    for (int t = 0; t < ntables; ++t) {
      const double* x = v + o;
      const double* f = g + o;
      const int m = sizes[t];
      for (size_t k = 0; k < xs.size(); ++k) {
        const double q = xs[k];
        double val;
        if (m == 1 || q <= x[0]) val = f[0];
        else if (q >= x[m - 1]) val = f[m - 1];
        else {
          const int j = (int)(std::upper_bound(x, x + m, q) - x) - 1;
          val = (x[j] == q) ? f[j] : (f[j + 1] - f[j]) / (x[j + 1] - x[j]) * (q - x[j]) + f[j];
        }
        fs[k] = fs[k] + val;
      }
      o += m;
    }
    int r = upload_interp(ctx, ctx->gsum, xs.data(), fs.data(), (int)xs.size(), true, 256);
    if (r) return r;
    ctx->gtables.fsum = ctx->gsum.fast;
    ctx->gtables.has_sum = 1;
  }
  return 0;
}

int nx_packets_resize(nx_ctx* ctx, long long n) {
  ENTER(ctx);
  ctx->bound = nullptr;
  if (n <= ctx->cap && ctx->state) return 0;
  const long long cap = ((std::max(n, 1LL) + 31) / 32) * 32;
  cudaFree(ctx->state); cudaFree(ctx->x0); cudaFree(ctx->att); cudaFree(ctx->acc);
  cudaFree(ctx->perm); cudaFree(ctx->cost);
  ctx->state = ctx->x0 = nullptr; ctx->att = ctx->acc = nullptr; ctx->cap = 0;
  ctx->perm = nullptr; ctx->cost = nullptr;
  ctx->fresh = ctx->x0_valid = false;
  if (n >= (1LL << 32)) { ctx->err = "more than 2^32 packets per GPU"; return -1; }
  CK(dev_malloc(&ctx->state, (size_t)9 * cap * sizeof(double)));
  CK(dev_malloc(&ctx->x0, (size_t)14 * cap * sizeof(double)));
  CK(dev_malloc(&ctx->att, (size_t)cap * sizeof(unsigned)));
  CK(dev_malloc(&ctx->acc, (size_t)cap * sizeof(unsigned)));
  CK(dev_malloc(&ctx->perm, (size_t)cap * sizeof(unsigned)));
  CK(dev_malloc(&ctx->cost, (size_t)cap));
  if (!ctx->hist) CK(cudaMalloc(&ctx->hist, 64 * sizeof(unsigned)));
  CK(cudaMemsetAsync(ctx->att, 0, (size_t)cap * sizeof(unsigned), ctx->stream));
  CK(cudaMemsetAsync(ctx->acc, 0, (size_t)cap * sizeof(unsigned), ctx->stream));
  ctx->cap = cap;
  return 0;
}

int nx_import_state(nx_ctx* ctx, long long n, const double* const* cols) {
  ENTER(ctx);
  int r = nx_packets_resize(ctx, n);
  if (r) return r;
  ctx->fresh = false;
  ctx->x0_valid = false;
  StateCols P = state_cols(ctx);
  for (int k = 0; k < 8; ++k)
    CK(cudaMemcpyAsync(P.c[k], cols[k], (size_t)n * sizeof(double), cudaMemcpyHostToDevice,
                       ctx->stream));
  if (n > 0) {
    CK(launch_fill(ctx->stream, P.c[8], n, 1000.0));     // Output.py:246
    ctx->launches += 1;
  }
  return 0;
}

int nx_export_state(nx_ctx* ctx, long long n, double* const* cols) {
  CK(cudaSetDevice(ctx->device));
  if (n > resident_rows(ctx)) { ctx->err = "export: n exceeds resident packets"; return -1; }
  StateCols P = in_cols(ctx);
  for (int k = 0; k < 8; ++k)
    CK(cudaMemcpyAsync(cols[k], P.c[k], (size_t)n * sizeof(double), cudaMemcpyDeviceToHost,
                       ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  return 0;
}

int nx_export_x0(nx_ctx* ctx, long long n, double* const* cols) {
  CK(cudaSetDevice(ctx->device));
  if (n > ctx->cap) { ctx->err = "export: n exceeds resident packets"; return -1; }
  X0Cols X = x0_cols(ctx);
  for (int k = 0; k < 14; ++k)
    CK(cudaMemcpyAsync(cols[k], X.c[k], (size_t)n * sizeof(double), cudaMemcpyDeviceToHost,
                       ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  return 0;
}

int nx_export_stats(nx_ctx* ctx, long long n, uint32_t* attempted, uint32_t* accepted) {
  CK(cudaSetDevice(ctx->device));
  if (n > ctx->cap) { ctx->err = "export: n exceeds resident packets"; return -1; }
  CK(cudaMemcpyAsync(attempted, ctx->att, (size_t)n * sizeof(unsigned), cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaMemcpyAsync(accepted, ctx->acc, (size_t)n * sizeof(unsigned), cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  return 0;
}

int nx_export_step(nx_ctx* ctx, long long n, double* step) {
  CK(cudaSetDevice(ctx->device));
  if (n > ctx->cap) { ctx->err = "export: n exceeds resident packets"; return -1; }
  { int r = materialize(ctx); if (r) return r; }
  CK(cudaMemcpyAsync(step, state_cols(ctx).c[8], (size_t)n * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  return 0;
}

int nx_state_device_ptr(nx_ctx* ctx, int column, void** dev_ptr) {
  if (column < 0 || column >= 9 || !ctx->state) { ctx->err = "bad column / no packets"; return -1; }
  { int r = materialize(ctx); if (r) return r; }
  *dev_ptr = state_cols(ctx).c[column];
  return 0;
}

int nx_sourcemap_upload(nx_ctx* ctx, const double* fmap, int nx_, int ny_, const double* xaxis,
                        const double* yaxis) {
  ENTER(ctx);
  cudaFree(ctx->srcmap); ctx->srcmap = nullptr;
  CK(cudaMalloc(&ctx->srcmap, (size_t)nx_ * ny_ * sizeof(double)));
  CK(cudaMemcpyAsync(ctx->srcmap, fmap, (size_t)nx_ * ny_ * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  ctx->map.f = ctx->srcmap;
  ctx->map.x_lo = xaxis[0]; ctx->map.x_hi = xaxis[nx_ - 1];
  ctx->map.y_lo = yaxis[0]; ctx->map.y_hi = yaxis[ny_ - 1];
  return 0;
}

int nx_speedtable_upload(nx_ctx* ctx, const double* cdf, const double* v, int n) {
  ENTER(ctx);
  return upload_interp(ctx, ctx->speed, cdf, v, n, false);
}

int nx_lontable_upload(nx_ctx* ctx, const double* cdf, const double* lon, int n) {
  ENTER(ctx);
  return upload_interp(ctx, ctx->lon1d, cdf, lon, n, false);
}

int nx_init_state(nx_ctx* ctx, const nx_source_params* sp_, uint64_t seed, uint64_t first_id,
                  long long n) {
  ENTER(ctx);
  int r = nx_packets_resize(ctx, n);
  if (r) return r;
  SourceParams sp;
  std::memcpy(&sp, sp_, sizeof(sp));
  if (sp.spatial_type == SPATIAL_MAP && !ctx->srcmap) { ctx->err = "no source map uploaded"; return -1; }
  if (sp.spatial_type == SPATIAL_LON1D && ctx->lon1d.view.n == 0) { ctx->err = "no longitude table uploaded"; return -1; }
  if (sp.speed_type == SPEED_TABLE && ctx->speed.view.n == 0) { ctx->err = "no speed table uploaded"; return -1; }
  if (n == 0) return 0;
  if ((r = begin_timed(ctx))) return r;
  CK(launch_init_state(ctx->stream, x0_cols(ctx), n, sp, ctx->map, ctx->speed.view,
                       ctx->lon1d.view, seed, first_id,
                       /*fast=*/!(ctx->have_params && ctx->params.strict_math)));
  ctx->fresh = ctx->x0_valid = true;
  return end_timed(ctx, 1);
}

int nx_init_state_deviates(nx_ctx* ctx, const nx_source_params* sp_, long long n,
                           const double* u_time, const double* u_sinlat, const double* u_lon,
                           const double* lon_in, const double* lat_in, const double* u_speed,
                           const double* z_normal, const double* u_alt, const double* u_az) {
  ENTER(ctx);
  int r = nx_packets_resize(ctx, n);
  if (r) return r;
  SourceParams sp;
  std::memcpy(&sp, sp_, sizeof(sp));
  if (sp.speed_type == SPEED_TABLE && ctx->speed.view.n == 0) { ctx->err = "no speed table uploaded"; return -1; }
  if ((lon_in == nullptr) != (lat_in == nullptr)) { ctx->err = "lon_in and lat_in go together"; return -1; }
  if (sp.spatial_type == SPATIAL_LON1D && !lon_in && ctx->lon1d.view.n == 0) { ctx->err = "no longitude table uploaded"; return -1; }
  if (n == 0) return 0;
  const double* host[9] = {u_time, u_sinlat, u_lon, lon_in, lat_in, u_speed, z_normal, u_alt, u_az};
  double* slab = nullptr;
  SCR(SCR_TMP, slab, (size_t)9 * n);
  const double* dev[9];
  cudaError_t e = cudaMemsetAsync(slab, 0, (size_t)9 * n * sizeof(double), ctx->stream);
  for (int k = 0; k < 9 && e == cudaSuccess; ++k) {
    dev[k] = host[k] ? slab + (size_t)k * n : nullptr;
    if (k != 3 && k != 4) dev[k] = slab + (size_t)k * n;        // absent deviates read as 0
    if (host[k])
      e = cudaMemcpyAsync(slab + (size_t)k * n, host[k], (size_t)n * sizeof(double),
                          cudaMemcpyHostToDevice, ctx->stream);
  }
  if (e == cudaSuccess)
    e = launch_init_from_deviates(ctx->stream, x0_cols(ctx), n, sp, ctx->speed.view,
                                  ctx->lon1d.view, dev);
  if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
  if (e != cudaSuccess) { ctx->err = cudaGetErrorString(e); return -(int)e; }
  ctx->launches += 1;
  ctx->fresh = ctx->x0_valid = true;
  return 0;
}

int nx_rewind_state(nx_ctx* ctx) {
  if (!ctx->x0_valid) { ctx->err = "no initial state resident (nx_init_state first)"; return -1; }
  ctx->los_kept.np = 0;
  ctx->fresh = true;
  return 0;
}

static int check_status(nx_ctx* ctx) {
  int v = 0;
  CK(cudaMemcpyAsync(&v, ctx->status, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  ctx->status_host = v;
  if (v) {
    ctx->err = "numerical invariant violated on device (bits " + std::to_string(v) + ")";
    CK(cudaMemsetAsync(ctx->status, 0, sizeof(int), ctx->stream));
  }
  return v;
}

// K2 over the resident packets (ctx->scalars: [0] queue, [1] attempted, [2] accepted,
// [3] bounces), longest first when ordering is on, inside the caller's timed section.
// S != nullptr: packets bounce (nx_integrate_adaptive_bounce); the cost model then budgets
// every packet's remaining time, since reaching the surface no longer ends its flight.
// dep != nullptr: the SINK build of the same kernel (nx_integrate_adaptive_deposit);
// ion != nullptr: its ion build (nx_integrate_adaptive_ionize).
static int adaptive_resident(nx_ctx* ctx, long long n, const Spline2D* S, uint64_t seed,
                             uint64_t first_id, const DepositOut* dep = nullptr,
                             const IonOut* ion = nullptr) {
  const bool order = ctx->order_packets && n >= 4096;
  const bool to_surface = !S || perfect_sticking(ctx->params);
  if (order)
    CK(launch_cost_order(ctx->stream, ctx->device, in_cols(ctx), n, ctx->params,
                         ctx->order_packets, ctx->cost, ctx->hist, ctx->perm, to_surface));
  CK(launch_integrate_adaptive(ctx->stream, ctx->device, in_cols(ctx), state_cols(ctx), n,
                               ctx->params,
                               ctx->radpres.view, ctx->radpres.fast,
                               order ? ctx->perm : nullptr, ctx->scalars, ctx->scalars + 1,
                               ctx->att, ctx->acc, ctx->status, S, seed, first_id, dep, ion));
  return end_timed(ctx, order ? 4 : 1);
}

int nx_integrate_adaptive(nx_ctx* ctx, long long n, unsigned long long* attempted,
                          unsigned long long* accepted) {
  ENTER(ctx);
  if (!ctx->have_params) { ctx->err = "nx_tables_upload not called"; return -1; }
  ctx->bound = nullptr;            // integrators work on the slab
  if (n > ctx->cap) { ctx->err = "n exceeds resident packets"; return -1; }
  if (!(ctx->params.sticktype == STICK_CONSTANT && ctx->params.stickcoef == 1.0)) {
    ctx->err = "Not set up";      // reference Output.py:315 (adaptive needs stickcoef == 1)
    return -1;
  }
  CK(cudaMemsetAsync(ctx->scalars, 0, 8 * sizeof(unsigned long long), ctx->stream));
  int r;
  if (n > 0) {
    CK(debug_begin(ctx->stream));
    if ((r = begin_timed(ctx))) return r;
    if (ctx->schedule == 2 && !ctx->x0_valid) {
      ctx->err = "schedule 2 reads the X0 slab: nx_init_state first";
      return -1;
    }
    if (ctx->schedule == 2) {
      // developer option (profiling the streaming kernel with kernel replay, which cannot
      // run the concurrent copies): class-ordered passes over the X0 slab, nothing in flight
      CK(cudaMemsetAsync(ctx->squeue, 0, (NX_STREAM_CURSORS + 1) * sizeof(unsigned long long),
                         ctx->stream));
      CK(cudaMemsetAsync(ctx->att, 0, (size_t)n * sizeof(unsigned), ctx->stream));
      CK(cudaMemsetAsync(ctx->acc, 0, (size_t)n * sizeof(unsigned), ctx->stream));
      CK(cudaMemsetAsync(ctx->cost, 0xFF, (size_t)ctx->cap, ctx->stream));
      long long seg = (n + 15) / 16;
      seg = (seg + NX_STREAM_GROUP - 1) / NX_STREAM_GROUP * NX_STREAM_GROUP;
      CK(launch_integrate_adaptive_stream(ctx->stream, ctx->device, ctx->x0, (size_t)ctx->cap,
                                          1000.0, state_cols(ctx), n, ctx->params,
                                          ctx->radpres.view, ctx->radpres.fast, seg,
                                          (int)((n + seg - 1) / seg), ctx->order_packets,
                                          ctx->squeue, nullptr, ctx->class_cache ? ctx->cost : nullptr,
                                          ctx->scalars + 1, ctx->att, ctx->acc, ctx->status));
      if ((r = end_timed(ctx, 1))) return r;
    } else {
      if ((r = adaptive_resident(ctx, n, nullptr, 0, 0))) return r;
    }
    ctx->fresh = false;
  }
  unsigned long long h[3] = {0, 0, 0};
  CK(cudaMemcpyAsync(h, ctx->scalars, sizeof(h), cudaMemcpyDeviceToHost, ctx->stream));
  r = check_status(ctx);
  if (r < 0) return r;
  if (attempted) *attempted = h[1];
  if (accepted) *accepted = h[2];
  return r;
}

int nx_integrate_adaptive_bounce(nx_ctx* ctx, long long n, uint64_t seed, uint64_t first_id,
                                 unsigned long long* attempted, unsigned long long* accepted,
                                 unsigned long long* bounces) {
  ENTER(ctx);
  if (!ctx->have_params) { ctx->err = "nx_tables_upload not called"; return -1; }
  ctx->bound = nullptr;            // integrators work on the slab
  if (n > ctx->cap) { ctx->err = "n exceeds resident packets"; return -1; }
  const RunParams& p = ctx->params;
  if (!perfect_sticking(p) && p.accomfactor != 0.0 && !ctx->spl_c) {
    ctx->err = "accommodation enabled but no speed spline uploaded";
    return -1;
  }
  CK(cudaMemsetAsync(ctx->scalars, 0, 8 * sizeof(unsigned long long), ctx->stream));
  int r;
  if (n > 0) {
    if ((r = begin_timed(ctx))) return r;
    if ((r = adaptive_resident(ctx, n, &ctx->spline, seed, first_id))) return r;
    ctx->fresh = false;
  }
  unsigned long long h[4] = {0, 0, 0, 0};
  CK(cudaMemcpyAsync(h, ctx->scalars, sizeof(h), cudaMemcpyDeviceToHost, ctx->stream));
  r = check_status(ctx);
  if (r < 0) return r;
  if (attempted) *attempted = h[1];
  if (accepted) *accepted = h[2];
  if (bounces) *bounces = h[3];
  return r;
}

// ---- K2d: deposition maps and the loss budget (ModelDeposition) ----------------------------
// The sink is the NX_PRODUCT_DEPOSIT accumulator: the map cells, then the buckets, in the sums
// and in the counts.
// nx_integrate_adaptive_deposit runs the SINK build of the kernel nx_integrate_adaptive (perfect
// sticking) or nx_integrate_adaptive_bounce would run, on the resident packets: the same final
// state and step totals, plus the events added to the sink.
static_assert((int)NX_DEP_SURFACE == DEP_SURFACE && (int)NX_DEP_MOON == DEP_MOON &&
                  (int)NX_DEP_ESCAPED == DEP_ESCAPED && (int)NX_DEP_VANISHED == DEP_VANISHED &&
                  (int)NX_DEP_REMAINING == DEP_REMAINING && (int)NX_DEP_SOURCE == DEP_SOURCE &&
                  (int)NX_DEP_NBUCKET == DEP_NBUCKET,
              "nx_deposit_bucket and DepositBucket disagree");

int nx_deposit_begin(nx_ctx* ctx, int nlon, int nlat) {
  CK(cudaSetDevice(ctx->device));
  if (nlon < 1 || nlat < 1) { ctx->err = "nx_deposit_begin: nlon and nlat must be >= 1"; return -1; }
  if ((double)nlon * nlat >= 2147483648.0) {
    ctx->err = "nx_deposit_begin: nlon * nlat must be < 2^31";
    return -1;
  }
  const long long n = (long long)nlon * nlat + NX_DEP_NBUCKET;
  return accum_begin(ctx, NX_PRODUCT_DEPOSIT, n, n, nlon, nlat, 0);
}

int nx_integrate_adaptive_deposit(nx_ctx* ctx, long long n, uint64_t seed, uint64_t first_id,
                                  unsigned long long* attempted, unsigned long long* accepted,
                                  unsigned long long* bounces) {
  ENTER(ctx);
  const Accum* sink = accum_of(ctx, NX_PRODUCT_DEPOSIT);
  if (!sink) return -1;
  if (!ctx->have_params) { ctx->err = "nx_tables_upload not called"; return -1; }
  ctx->bound = nullptr;            // integrators work on the slab
  if (n < 0 || n > ctx->cap) { ctx->err = "n exceeds resident packets"; return -1; }
  const RunParams& p = ctx->params;
  const bool bounce = !perfect_sticking(p);
  if (bounce && p.accomfactor != 0.0 && !ctx->spl_c) {
    ctx->err = "accommodation enabled but no speed spline uploaded";
    return -1;
  }
  CK(cudaMemsetAsync(ctx->scalars, 0, 8 * sizeof(unsigned long long), ctx->stream));
  int r;
  if (n > 0) {
    const long long ncell = (long long)sink->dims[0] * sink->dims[1];
    DepositOut d;
    d.map = sink->sums();
    d.bucket = d.map + ncell;
    d.cnt = sink->counts();
    d.bucket_n = d.cnt + ncell;
    d.nlon = sink->dims[0]; d.nlat = sink->dims[1];
    if ((r = begin_timed(ctx))) return r;
    if ((r = adaptive_resident(ctx, n, bounce ? &ctx->spline : nullptr, seed, first_id, &d)))
      return r;
    ctx->fresh = false;
  }
  unsigned long long h[4] = {0, 0, 0, 0};
  CK(cudaMemcpyAsync(h, ctx->scalars, sizeof(h), cudaMemcpyDeviceToHost, ctx->stream));
  r = check_status(ctx);
  if (r < 0) return r;
  if (attempted) *attempted = h[1];
  if (accepted) *accepted = h[2];
  if (bounces) *bounces = h[3];
  return r;
}

// ---- K2i: ion production maps (ModelIonization) ---------------------------------------------
// The sink is the NX_PRODUCT_IONIZE accumulator: the grid's cells, row-major (nx, ny, nz), then
// OUTSIDE, in the sums and in the counts.
// nx_integrate_adaptive_ionize runs k_ionize_adaptive, the build of the kernel
// nx_integrate_adaptive (perfect sticking) or nx_integrate_adaptive_bounce would run, on the
// resident packets: the same final state and step totals, plus the loss added to the grid.
static_assert(sizeof(nx_ion_grid) == 64, "nx_ion_grid layout");

int nx_ionize_begin(nx_ctx* ctx, const nx_ion_grid* grid) {
  CK(cudaSetDevice(ctx->device));
  if (!grid) { ctx->err = "nx_ionize_begin: grid is NULL"; return -1; }
  double ncell = 1.0;
  for (int a = 0; a < 3; ++a) {
    if (grid->n[a] < 1) { ctx->err = "nx_ionize_begin: n must be >= 1 on every axis"; return -1; }
    if (!(std::isfinite(grid->lo[a]) && std::isfinite(grid->hi[a]) && grid->lo[a] < grid->hi[a])) {
      ctx->err = "nx_ionize_begin: lo < hi, both finite, on every axis";
      return -1;
    }
    ncell *= grid->n[a];
  }
  if (ncell + 1.0 >= 2147483648.0) {
    ctx->err = "nx_ionize_begin: nx * ny * nz + 1 must be < 2^31";
    return -1;
  }
  IonOut g{};
  for (int a = 0; a < 3; ++a) { g.lo[a] = grid->lo[a]; g.hi[a] = grid->hi[a]; g.n[a] = grid->n[a]; }
  ion_steps(g);
  const long long n = (long long)ncell + 1;
  int r = accum_begin(ctx, NX_PRODUCT_IONIZE, n, n, g.n[0], g.n[1], g.n[2]);
  if (r == 0) ctx->ion_axes = g;
  return r;
}

int nx_integrate_adaptive_ionize(nx_ctx* ctx, long long n, uint64_t seed, uint64_t first_id,
                                 unsigned long long* attempted, unsigned long long* accepted,
                                 unsigned long long* bounces) {
  ENTER(ctx);
  const Accum* sink = accum_of(ctx, NX_PRODUCT_IONIZE);
  if (!sink) return -1;
  if (!ctx->have_params) { ctx->err = "nx_tables_upload not called"; return -1; }
  ctx->bound = nullptr;            // integrators work on the slab
  if (n < 0 || n > ctx->cap) { ctx->err = "n exceeds resident packets"; return -1; }
  const RunParams& p = ctx->params;
  if (p.loss_mode != LOSS_LIFETIME && p.loss_mode != LOSS_PHOTO) {
    ctx->err = "nx_integrate_adaptive_ionize: the run has no loss process (loss_mode 0)";
    return -1;
  }
  const bool bounce = !perfect_sticking(p);
  if (bounce && p.accomfactor != 0.0 && !ctx->spl_c) {
    ctx->err = "accommodation enabled but no speed spline uploaded";
    return -1;
  }
  CK(cudaMemsetAsync(ctx->scalars, 0, 8 * sizeof(unsigned long long), ctx->stream));
  int r;
  if (n > 0) {
    IonOut g = ctx->ion_axes;
    g.sum = sink->sums();
    g.cnt = sink->counts();
    if ((r = begin_timed(ctx))) return r;
    if ((r = adaptive_resident(ctx, n, bounce ? &ctx->spline : nullptr, seed, first_id, nullptr,
                               &g)))
      return r;
    ctx->fresh = false;
  }
  unsigned long long h[4] = {0, 0, 0, 0};
  CK(cudaMemcpyAsync(h, ctx->scalars, sizeof(h), cudaMemcpyDeviceToHost, ctx->stream));
  r = check_status(ctx);
  if (r < 0) return r;
  if (attempted) *attempted = h[1];
  if (accepted) *accepted = h[2];
  if (bounces) *bounces = h[3];
  return r;
}

// Host-buffer variant of K2 for the end-to-end path.  schedule 1 (default): ONE
// persistent class-ordered kernel consumes the packets segment by segment while the
// copy engine is still delivering the later segments (k_integrate_adaptive_stream).
// schedule 0 (kept for A/B runs): `nchunks` ranges, each on its own stream with its
// own sort + kernel; co-resident kernels overlap one range's tail with the next.
#define NX_MAX_CHUNKS 16
int nx_integrate_adaptive_host(nx_ctx* ctx, long long n, const double* const* cols, int nchunks,
                               unsigned long long* attempted, unsigned long long* accepted) {
  ENTER(ctx);
  int r = nx_packets_resize(ctx, n);
  if (r) return r;
  if (!ctx->have_params) { ctx->err = "nx_tables_upload not called"; return -1; }
  if (!(ctx->params.sticktype == STICK_CONSTANT && ctx->params.stickcoef == 1.0)) {
    ctx->err = "Not set up";
    return -1;
  }
  if (nchunks < 1) nchunks = 1;
  if (ctx->schedule == 1) {
    // ONE persistent kernel; the copy engine delivers the packets segment by segment
    // behind it and raises `arrived` after each one (stream order on copy_stream).
    if (n == 0) { if (attempted) *attempted = 0; if (accepted) *accepted = 0; return 0; }
    if (nchunks > NX_STREAM_MAX_SEG) nchunks = NX_STREAM_MAX_SEG;
    long long seg = (n + nchunks - 1) / nchunks;
    seg = (seg + NX_STREAM_GROUP - 1) / NX_STREAM_GROUP * NX_STREAM_GROUP;
    const int nseg = (int)((n + seg - 1) / seg);
    unsigned* arrived = reinterpret_cast<unsigned*>(ctx->squeue + NX_STREAM_CURSORS);
    StateCols P = state_cols(ctx);
    CK(cudaMemsetAsync(ctx->scalars, 0, 8 * sizeof(unsigned long long), ctx->stream));
    CK(cudaMemsetAsync(ctx->squeue, 0, (NX_STREAM_CURSORS + 1) * sizeof(unsigned long long),
                       ctx->stream));
    CK(cudaMemsetAsync(ctx->att, 0, (size_t)n * sizeof(unsigned), ctx->stream));
    CK(cudaMemsetAsync(ctx->acc, 0, (size_t)n * sizeof(unsigned), ctx->stream));
    CK(cudaMemsetAsync(ctx->cost, 0xFF, (size_t)ctx->cap, ctx->stream));   // classes: unknown
    CK(debug_begin(ctx->stream));
    if ((r = begin_timed(ctx))) return r;
    CK(cudaEventRecord(ctx->copy_ev[0], ctx->stream));
    CK(cudaStreamWaitEvent(ctx->copy_stream, ctx->copy_ev[0], 0));  // `arrived` is 0 before any copy
    // the copies land in the X0 slab (the imported initial state, Output.py:180-182);
    // the kernel writes the final state and the step size (Output.py:246: 1000 s) to the state slab
    double* const in0 = ctx->x0;
    const size_t in_stride = (size_t)ctx->cap;
    CK(launch_integrate_adaptive_stream(ctx->stream, ctx->device, in0, in_stride, 1000.0, P, n,
                                        ctx->params,
                                        ctx->radpres.view, ctx->radpres.fast, seg, nseg,
                                        ctx->order_packets, ctx->squeue, arrived,
                                        ctx->class_cache ? ctx->cost : nullptr,
                                        ctx->scalars + 1, ctx->att, ctx->acc, ctx->status));
    for (int c = 0; c < nseg; ++c) {
      const long long first = (long long)c * seg, count = std::min(seg, n - first);
      for (int k = 0; k < 8; ++k)
        CK(cudaMemcpyAsync(in0 + (size_t)k * in_stride + first, cols[k] + first,
                           (size_t)count * sizeof(double), cudaMemcpyHostToDevice,
                           ctx->copy_stream));
      CK(cudaMemcpyAsync(arrived, ctx->seq_host + c + 1, sizeof(unsigned),
                         cudaMemcpyHostToDevice, ctx->copy_stream));
    }
    CK(cudaEventRecord(ctx->copy_ev[1], ctx->copy_stream));
    CK(cudaStreamWaitEvent(ctx->stream, ctx->copy_ev[1], 0));
    if ((r = end_timed(ctx, 2))) return r;
    ctx->fresh = false;
    ctx->x0_valid = true;
    unsigned long long h[3] = {0, 0, 0};
    CK(cudaMemcpyAsync(h, ctx->scalars, sizeof(h), cudaMemcpyDeviceToHost, ctx->stream));
    r = check_status(ctx);
    if (r < 0) return r;
    if (attempted) *attempted = h[1];
    if (accepted) *accepted = h[2];
    return r;
  }
  if (nchunks > NX_MAX_CHUNKS) nchunks = NX_MAX_CHUNKS;
  if (n < (long long)nchunks * 65536) nchunks = (int)std::max(1LL, n / 65536);
  if (!ctx->pipe[0]) {
    for (auto& s : ctx->pipe) CK(cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking));
    for (auto& e : ctx->pipe_ev) CK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    CK(cudaMalloc(&ctx->pipe_scalars, NX_MAX_CHUNKS * 4 * sizeof(unsigned long long)));
    CK(cudaMalloc(&ctx->pipe_hist, NX_MAX_CHUNKS * 64 * sizeof(unsigned)));
  }
  CK(cudaMemsetAsync(ctx->pipe_scalars, 0, NX_MAX_CHUNKS * 4 * sizeof(unsigned long long), ctx->stream));
  if ((r = begin_timed(ctx))) return r;
  CK(cudaEventRecord(ctx->pipe_ev[16], ctx->stream));
  for (int s = 0; s < nchunks; ++s) CK(cudaStreamWaitEvent(ctx->pipe[s], ctx->pipe_ev[16], 0));
  StateCols P = state_cols(ctx);
  ctx->fresh = ctx->x0_valid = false;
  int nlaunch = 0;
  for (int c = 0; c < nchunks; ++c) {
    const long long first = n * c / nchunks, count = n * (c + 1) / nchunks - first;
    if (count <= 0) continue;
    cudaStream_t st = ctx->pipe[c];
    StateCols Pc;
    for (int k = 0; k < 9; ++k) Pc.c[k] = P.c[k] + first;
    for (int k = 0; k < 8; ++k)
      CK(cudaMemcpyAsync(Pc.c[k], cols[k] + first, (size_t)count * sizeof(double),
                         cudaMemcpyHostToDevice, st));
    CK(launch_fill(st, Pc.c[8], count, 1000.0));
    const bool order = ctx->order_packets && count >= 4096;
    if (order)
      CK(launch_cost_order(st, ctx->device, Pc, count, ctx->params, ctx->order_packets,
                           ctx->cost + first, ctx->pipe_hist + 64 * c, ctx->perm + first));
    unsigned long long* sc = ctx->pipe_scalars + 4 * c;
    CK(launch_integrate_adaptive(st, ctx->device, Pc, Pc, count, ctx->params, ctx->radpres.view,
                                 ctx->radpres.fast, order ? ctx->perm + first : nullptr, sc, sc + 1,
                                 ctx->att + first, ctx->acc + first, ctx->status));
    nlaunch += order ? 5 : 2;
  }
  for (int s = 0; s < nchunks; ++s) {
    CK(cudaEventRecord(ctx->pipe_ev[s], ctx->pipe[s]));
    CK(cudaStreamWaitEvent(ctx->stream, ctx->pipe_ev[s], 0));
  }
  if ((r = end_timed(ctx, nlaunch))) return r;
  std::vector<unsigned long long> h((size_t)nchunks * 4, 0);
  CK(cudaMemcpyAsync(h.data(), ctx->pipe_scalars, h.size() * sizeof(unsigned long long),
                     cudaMemcpyDeviceToHost, ctx->stream));
  r = check_status(ctx);
  if (r < 0) return r;
  unsigned long long a = 0, b = 0;
  for (int c = 0; c < nchunks; ++c) { a += h[4 * c + 1]; b += h[4 * c + 2]; }
  if (attempted) *attempted = a;
  if (accepted) *accepted = b;
  return r;
}

static int integrate_constant_core(nx_ctx* ctx, long long n, uint64_t seed, uint64_t first_id,
                                   const nx_image_params* img, void* image_dev, void* counts_dev,
                                   double* traj_host, const RowSink& rows,
                                   unsigned long long* packet_steps) {
  CK(cudaSetDevice(ctx->device));
  if (!ctx->have_params) { ctx->err = "nx_tables_upload not called"; return -1; }
  ctx->bound = nullptr;            // integrators work on the slab
  if (n > ctx->cap) { ctx->err = "n exceeds resident packets"; return -1; }
  const RunParams& p = ctx->params;
  if (!(p.step_size > 0.0)) { ctx->err = "constant driver needs step_size > 0"; return -1; }
  const bool simple = (p.sticktype == STICK_CONSTANT && p.stickcoef == 1.0);
  if (!simple && p.accomfactor != 0.0 && !ctx->spl_c) {
    ctx->err = "accommodation enabled but no speed spline uploaded";
    return -1;
  }
  const int nsteps = (int)std::ceil(p.endtime / p.step_size + 1);
  ImageParams ip{};
  if (img) std::memcpy(&ip, img, sizeof(ip));
  else { ip.nx = ip.nz = 1; ip.x1 = ip.z1 = 1.0; }
  if (image_dev && ip.quantity == 1 && ctx->gtables.n == 0) {
    ctx->err = "radiance image requested but no g-value tables uploaded";
    return -1;
  }
  double* traj = nullptr;
  const size_t traj_bytes = (size_t)n * 8 * nsteps * sizeof(double);
  if (traj_host) {
    CK(dev_malloc(&traj, traj_bytes));
    cudaError_t e = cudaMemsetAsync(traj, 0, traj_bytes, ctx->stream);
    if (e != cudaSuccess) { cudaFree(traj); ctx->err = cudaGetErrorString(e); return -(int)e; }
  }
  auto fail = [&](cudaError_t e) {
    cudaFree(traj);
    ctx->err = cudaGetErrorString(e);
    return -(int)e;
  };
  cudaError_t e = cudaMemsetAsync(ctx->scalars, 0, 8 * sizeof(unsigned long long), ctx->stream);
  if (e != cudaSuccess) return fail(e);
  int r;
  if (n > 0) {
    if ((r = begin_timed(ctx))) { cudaFree(traj); return r; }
    e = launch_integrate_constant(ctx->stream, ctx->device, in_cols(ctx), state_cols(ctx), n, p,
                                  ctx->radpres.view, ctx->radpres.fast, ctx->spline, seed,
                                  first_id, nsteps, ip, ctx->gtables, (double*)image_dev,
                                  (unsigned long long*)counts_dev, traj, rows, ctx->scalars,
                                  ctx->scalars + 1, ctx->status);
    if (e != cudaSuccess) return fail(e);
    if ((r = end_timed(ctx, 1))) { cudaFree(traj); return r; }
    ctx->fresh = false;
  }
  unsigned long long h[2] = {0, 0};
  e = cudaMemcpyAsync(h, ctx->scalars, sizeof(h), cudaMemcpyDeviceToHost, ctx->stream);
  if (e == cudaSuccess && traj_host)
    e = cudaMemcpyAsync(traj_host, traj, traj_bytes, cudaMemcpyDeviceToHost, ctx->stream);
  if (e != cudaSuccess) return fail(e);
  r = check_status(ctx);
  cudaFree(traj);
  if (r < 0) return r;
  if (packet_steps) *packet_steps = h[1];
  return r;
}

int nx_integrate_constant(nx_ctx* ctx, long long n, uint64_t seed, uint64_t first_id,
                          const nx_image_params* img, void* image_dev, void* counts_dev,
                          double* traj_host, unsigned long long* packet_steps) {
  ENTER(ctx);
  return integrate_constant_core(ctx, n, seed, first_id, img, image_dev, counts_dev, traj_host,
                                 RowSink{}, packet_steps);
}

int nx_integrate_constant_rows(nx_ctx* ctx, long long n, uint64_t seed, uint64_t first_id,
                               int skip_dead, int round_f32, nx_packets** out, long long* nrows,
                               unsigned long long* packet_steps) {
  ENTER(ctx);
  if (!out) { ctx->err = "nx_integrate_constant_rows: null output"; return -1; }
  *out = nullptr;
  if (!ctx->have_params || !(ctx->params.step_size > 0.0)) {
    ctx->err = "constant driver needs nx_tables_upload with step_size > 0";
    return -1;
  }
  const int nsteps = (int)std::ceil(ctx->params.endtime / ctx->params.step_size + 1);
  if (nsteps > 65535) { ctx->err = "more than 65535 steps per packet"; return -1; }
  unsigned long long* cursor = ctx->scalars + 5;
  RowSink rows{};
  rows.cursor = cursor;
  rows.skip_dead = skip_dead; rows.to_f32 = round_f32;
  unsigned long long need = (unsigned long long)n * (unsigned long long)nsteps;
  int r;
  if (ctx->fresh && ctx->x0_valid) {
    // the initial state is immutable (X0 slab): count the rows first, allocate exactly
    r = integrate_constant_core(ctx, n, seed, first_id, nullptr, nullptr, nullptr, nullptr, rows,
                                nullptr);
    if (r < 0) return r;
    CK(cudaMemcpyAsync(&need, cursor, sizeof(need), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    ctx->fresh = true;               // rewind: second pass over the same packets
  }
  nx_packets* h = new nx_packets();
  h->cap = (((long long)std::max<unsigned long long>(need, 1ull) + 31) / 32) * 32;
  cudaError_t e = table_alloc(h, ctx->stream, 8, true);
  if (e != cudaSuccess) {
    ctx->err = std::string("row table allocation (") + std::to_string(need) + " rows): " + cudaGetErrorString(e);
    free_packets(h, ctx->stream);
    return -(int)e;
  }
  rows.cols = h->cols; rows.index = h->index; rows.step = h->step;
  rows.cap = (unsigned long long)h->cap; rows.stride = (size_t)h->cap;
  unsigned long long steps = 0;
  r = integrate_constant_core(ctx, n, seed, first_id, nullptr, nullptr, nullptr, nullptr, rows,
                              &steps);
  if (r < 0) { free_packets(h, ctx->stream); return r; }
  unsigned long long got = 0;
  e = cudaMemcpyAsync(&got, cursor, sizeof(got), cudaMemcpyDeviceToHost, ctx->stream);
  if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
  if (e != cudaSuccess || got > (unsigned long long)h->cap) {
    ctx->err = e != cudaSuccess ? cudaGetErrorString(e) : "row table overflow";
    free_packets(h, ctx->stream);
    return e != cudaSuccess ? -(int)e : -1;
  }
  h->n = (long long)got;
  *out = h;
  if (nrows) *nrows = h->n;
  if (packet_steps) *packet_steps = steps;
  return r;
}

int nx_image_accumulate_dev(nx_ctx* ctx, long long n, const nx_image_params* ip_, void* image_dev,
                            void* counts_dev) {
  CK(cudaSetDevice(ctx->device));
  if (n > resident_rows(ctx)) { ctx->err = "n exceeds resident packets"; return -1; }
  ImageParams ip;
  std::memcpy(&ip, ip_, sizeof(ip));
  if (ip.quantity == 1 && ctx->gtables.n == 0) {
    ctx->err = "radiance image requested but no g-value tables uploaded";
    return -1;
  }
  if (n == 0) return 0;
  int r;
  if ((r = materialize(ctx))) return r;
  if ((r = begin_timed(ctx))) return r;
  // auto: privatised counts pay off when most rows are live -- a compacted table, or a slab
  // binned without skip_dead; a raw slab of an adaptive run is ~99 % dead packets, where the
  // plain kernel streams faster (measured 1e7 packets: 0.075 vs 0.092 ms)
  int mode = ctx->image_mode;
  if (mode == 0) mode = (n >= (1LL << 20) && (ctx->bound || !ip.skip_dead)) ? 2 : 1;
  CK(launch_image_accumulate(ctx->stream, ctx->device, state_cols(ctx), n, ip, ctx->gtables,
                             (double*)image_dev, (unsigned long long*)counts_dev, mode));
  return end_timed(ctx, 1);
}

// The NX_PRODUCT_IMAGE accumulator: begin (allocate + zero), add (K4 into it, any number of
// packet tables).  ModelImage sums its output files on the device this way and never ends it,
// so its block only grows.
int nx_image_begin(nx_ctx* ctx, int nx_, int nz_) {
  CK(cudaSetDevice(ctx->device));
  if (nx_ < 1 || nz_ < 1) { ctx->err = "nx_image_begin: bad dims"; return -1; }
  const long long npix = (long long)nx_ * nz_;
  return accum_begin(ctx, NX_PRODUCT_IMAGE, npix, npix, nx_, nz_, 0);
}

int nx_image_add(nx_ctx* ctx, long long n, const nx_image_params* ip) {
  const Accum& a = ctx->accum[NX_PRODUCT_IMAGE];
  if (!a.nsum || ip->nx != a.dims[0] || ip->nz != a.dims[1]) {
    ctx->err = "nx_image_add: dims differ from nx_image_begin";
    return -1;
  }
  return nx_image_accumulate_dev(ctx, n, ip, a.sums(), a.counts());
}

// Page-locked host memory for results the caller wants at full PCIe rate and without a
// staging copy (ModelImage's image / packet image live in such buffers).
int nx_host_alloc(long long bytes, void** out) {
  if (!out || bytes <= 0) return -1;
  *out = nullptr;
  cudaError_t e = cudaHostAlloc(out, (size_t)bytes, cudaHostAllocDefault);
  return e == cudaSuccess ? 0 : -(int)e;
}
int nx_host_free(void* p) {
  if (!p) return 0;
  cudaError_t e = cudaFreeHost(p);
  return e == cudaSuccess ? 0 : -(int)e;
}

// image * scale and the packet counts as float64 (what ModelImage keeps: ModelImage.py:92-105),
// converted on the device and copied once.  Destinations that are page-locked (nx_host_alloc)
// receive the DMA directly; pageable ones go through the context's pinned staging buffer.
int nx_image_fetch_scaled(nx_ctx* ctx, double scale, double* image, double* counts) {
  CK(cudaSetDevice(ctx->device));
  const Accum* img = accum_of(ctx, NX_PRODUCT_IMAGE);
  if (!img) return -1;
  if (!image || !counts) { ctx->err = "nx_image_fetch_scaled: null destination"; return -1; }
  const size_t npix = (size_t)img->nsum;
  double* d_out = nullptr;
  SCR(SCR_IMG_OUT, d_out, 2 * npix);
  CK(launch_image_finish(ctx->stream, img->sums(), img->counts(), scale, d_out, d_out + npix,
                         (long long)npix));
  ctx->launches += 1;
  auto pinned = [](const void* p) {
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return false; }
    return a.type == cudaMemoryTypeHost;
  };
  if (pinned(image) && pinned(counts)) {
    CK(cudaMemcpyAsync(image, d_out, npix * 8, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(counts, d_out + npix, npix * 8, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return 0;
  }
  int r = pinned_staging(ctx, 2 * npix * 8);
  if (r) return r;
  char* st = static_cast<char*>(ctx->pinned);
  CK(cudaMemcpyAsync(st, d_out, 2 * npix * 8, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  std::memcpy(image, st, npix * 8);
  std::memcpy(counts, st + npix * 8, npix * 8);
  return 0;
}

int nx_ctx_stream(nx_ctx* ctx, void** cuda_stream) {
  if (!cuda_stream) return -1;
  *cuda_stream = ctx->stream;
  return 0;
}

int nx_image_accumulate(nx_ctx* ctx, long long n, const nx_image_params* ip, double* image,
                        long long* counts) {
  int r = nx_image_begin(ctx, ip->nx, ip->nz);
  if (r == 0) r = nx_image_add(ctx, n, ip);
  if (r == 0) r = nx_product_fetch(ctx, NX_PRODUCT_IMAGE, image, counts);
  return r;
}

// Line-of-sight parameters every K5 entry point checks before any device work.
static int check_los_params(nx_ctx* ctx, const LosParams& lp) {
  const std::string e = los_dphi_error(lp.dphi);
  if (!e.empty()) { ctx->err = e; return -1; }
  if (lp.quantity != 1) { ctx->err = "Other quantities not set up."; return -1; }   // compute_iteration.py:213
  if (ctx->gtables.n == 0) { ctx->err = "no g-value tables uploaded"; return -1; }
  return 0;
}

// The ladder, then the squared ball radii, into d_dst (2 * ladder.size() doubles) through the
// context's pinned staging, at most NX_LADDER_STAGE bytes at a time: a ladder of millions of
// entries (arcsecond cones) does not grow the staging buffer.
#define NX_LADDER_STAGE ((size_t)4 << 20)
static int stage_ladder(nx_ctx* ctx, double* d_dst, const std::vector<double>& ladder,
                        const std::vector<double>& wid2) {
  const size_t nl = ladder.size(), total = 2 * nl, per = NX_LADDER_STAGE / sizeof(double);
  { int r0 = pinned_staging(ctx, (total < per ? total : per) * sizeof(double)); if (r0) return r0; }
  double* st = static_cast<double*>(ctx->pinned);
  for (size_t a = 0; a < total; a += per) {
    const size_t b = total - a < per ? total : a + per;
    // the previous chunk has left the staging buffer (the stream is idle on the first one)
    if (a) CK(cudaStreamSynchronize(ctx->stream));
    for (size_t i = a; i < b; ++i) st[i - a] = i < nl ? ladder[i] : wid2[i - nl];
    CK(cudaMemcpyAsync(d_dst + a, st, (b - a) * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
  }
  return 0;
}

static int los_run(nx_ctx* ctx, long long n, long long nlos, const double* los_dev,
                   const double* dist_dev, const LosParams& lp, double* rad_dev,
                   unsigned long long* np_dev, unsigned char* inc_dev,
                   unsigned long long* nused_dev = nullptr, const LosSpectrum* spec = nullptr) {
  { int r0 = materialize(ctx); if (r0) return r0; }
  static const bool timing = std::getenv("NX_LOS_TIMING") != nullptr;     // developer aid
  const auto tp0 = std::chrono::steady_clock::now();
  auto lap = [&](const char* what) {
    if (timing)
      std::fprintf(stderr, "[los_run] %s at %.3f ms\n", what,
                   std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - tp0).count());
  };
  // candidate generation: brute force for small problems, cell grid otherwise
  const bool use_grid = ctx->los_mode == 2 || nused_dev || spec ||   // (`used` counts, spectra: grid path only)
                        (ctx->los_mode == 0 && (double)n * (double)nlos > 2e9 && n < (1LL << 32));
  const bool want_order = use_grid && ctx->los_order && nlos >= 1024;
  // per-line preparation on the device; the host only turns the longest boresight distance
  // (8 bytes back) into the common ladder
  int* d_nball = nullptr;
  double *d_ladder = nullptr, *d_wid2 = nullptr, *d_dd = nullptr;
  unsigned *d_order = nullptr, *d_key = nullptr;
  SCR(SCR_NBALL, d_nball, nlos);
  SCR(SCR_DD, d_dd, nlos + 1);                       // [nlos]: the running maximum (bits)
  if (want_order) {
    SCR(SCR_ORDER, d_order, nlos);
    SCR(SCR_KEY, d_key, nlos + NX_LOS_KEY_BINS);     // keys, then the key histogram / cursors
  }
  unsigned* d_hist = d_key ? d_key + nlos : nullptr;
  unsigned long long* d_ddmax = reinterpret_cast<unsigned long long*>(d_dd + nlos);
  CK(launch_los_prepare(ctx->stream, los_dev, nlos, lp.outeredge, d_dd, d_key, d_hist, d_ddmax));
  double ddmax = 0.0;
  CK(cudaMemcpyAsync(&ddmax, d_ddmax, sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  std::vector<double> ladder, wid2;
  LosConsts lc;
  { const std::string e = los_constants(lp, ddmax, ladder, wid2, lc); if (!e.empty()) { ctx->err = e; return -1; } }
  SCR(SCR_LADDER, d_ladder, 2 * ladder.size());
  d_wid2 = d_ladder + ladder.size();
  { int r0 = stage_ladder(ctx, d_ladder, ladder, wid2); if (r0) return r0; }
  CK(launch_los_finish(ctx->stream, d_dd, d_ladder, (int)ladder.size(), nlos, d_nball, d_key, d_hist,
                       d_order));
  ctx->launches += want_order ? 3 : 2;
  lap("prepared");
  int nlaunch = 1;
  int r = 0;
  if (use_grid) r = alloc_los_work(ctx, n);
  if (r == 0) r = begin_timed(ctx);
  if (r == 0) {
    cudaError_t e;
    if (use_grid) {
      e = launch_los_grid_build(ctx->stream, ctx->device, state_cols(ctx), n, lp, ctx->losw);
      unsigned long long kept = 0;
      if (e == cudaSuccess)
        e = launch_los_grid(ctx->stream, ctx->losw, nlos, los_dev, dist_dev, d_nball, d_ladder,
                            d_wid2, lp, lc, ctx->gtables, rad_dev, np_dev, inc_dev, nused_dev,
                            nullptr, nullptr, nullptr, d_order, nused_dev ? &kept : nullptr, spec);
      if (e == cudaSuccess && kept) {
        ctx->los_kept.np = kept; ctx->los_kept.n = n; ctx->los_kept.nlos = nlos;
        ctx->los_kept.bound = ctx->bound; ctx->los_kept.lc = lc;
        std::memcpy(&ctx->los_kept.lp, &lp, sizeof(lp));      // (bytes: compared with memcmp)
        ctx->los_kept.nladder = ladder.size();
      }
      nlaunch = 8;
    } else {
      e = launch_los_accumulate(ctx->stream, ctx->device, state_cols(ctx), n, nlos, los_dev,
                                dist_dev, d_nball, d_ladder, d_wid2, lp, lc, ctx->gtables,
                                rad_dev, np_dev, inc_dev);
    }
    if (e != cudaSuccess) { ctx->err = cudaGetErrorString(e); r = -(int)e; }
  }
  if (r == 0) r = end_timed(ctx, nlaunch);
  cudaError_t e = cudaStreamSynchronize(ctx->stream);
  if (r == 0 && e != cudaSuccess) { ctx->err = cudaGetErrorString(e); r = -(int)e; }
  lap("kernels");
  return r;
}

int nx_los_accumulate_dev(nx_ctx* ctx, long long n, long long nlos, void* los_dev, void* dist_dev,
                          const nx_los_params* lp_, void* radiance_dev, void* npackets_dev,
                          void* included_dev) {
  ENTER(ctx);
  if (n > resident_rows(ctx)) { ctx->err = "n exceeds resident packets"; return -1; }
  LosParams lp;
  std::memcpy(&lp, lp_, sizeof(lp));
  { int r0 = check_los_params(ctx, lp); if (r0) return r0; }
  if (n == 0 || nlos == 0) return 0;
  return los_run(ctx, n, nlos, (const double*)los_dev, (const double*)dist_dev, lp,
                 (double*)radiance_dev, (unsigned long long*)npackets_dev,
                 (unsigned char*)included_dev);
}

int nx_los_accumulate(nx_ctx* ctx, long long n, long long nlos, const double* los,
                      const double* dist_from_plan, const nx_los_params* lp_, double* radiance,
                      long long* npackets, uint8_t* included) {
  ENTER(ctx);
  if (n > resident_rows(ctx)) { ctx->err = "n exceeds resident packets"; return -1; }
  LosParams lp;
  std::memcpy(&lp, lp_, sizeof(lp));
  { int r0 = check_los_params(ctx, lp); if (r0) return r0; }
  double *d_los = nullptr, *d_dist = nullptr, *d_rad = nullptr;
  unsigned long long* d_np = nullptr;
  unsigned char* d_inc = nullptr;
  const size_t nl = (size_t)(nlos > 0 ? nlos : 1), nn = (size_t)(n > 0 ? n : 1);
  SCR(SCR_LOS, d_los, 6 * nl);
  SCR(SCR_DIST, d_dist, nl);
  SCR(SCR_RAD, d_rad, nl);
  SCR(SCR_NP, d_np, nl);
  SCR(SCR_INC, d_inc, nn);
  CK(cudaMemcpyAsync(d_los, los, 6 * (size_t)nlos * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaMemcpyAsync(d_dist, dist_from_plan, (size_t)nlos * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaMemsetAsync(d_rad, 0, nl * sizeof(double), ctx->stream));
  CK(cudaMemsetAsync(d_np, 0, nl * sizeof(unsigned long long), ctx->stream));
  CK(cudaMemsetAsync(d_inc, 0, nn, ctx->stream));
  int r = 0;
  if (n > 0 && nlos > 0) r = los_run(ctx, n, nlos, d_los, d_dist, lp, d_rad, d_np, d_inc);
  if (r == 0) {
    cudaMemcpyAsync(radiance, d_rad, (size_t)nlos * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream);
    cudaMemcpyAsync(npackets, d_np, (size_t)nlos * sizeof(long long), cudaMemcpyDeviceToHost, ctx->stream);
    if (included) cudaMemcpyAsync(included, d_inc, (size_t)n, cudaMemcpyDeviceToHost, ctx->stream);
    cudaError_t e = cudaStreamSynchronize(ctx->stream);
    if (e != cudaSuccess) { ctx->err = cudaGetErrorString(e); r = -(int)e; }
  }
  return r;
}

// nx_los_accumulate that also counts, per line of sight, the `used` packets (weight > 0,
// compute_iteration.py:210-211) in the same pass, and keeps the candidate pairs on the device
// for nx_los_used_fill.
int nx_los_accumulate_counted(nx_ctx* ctx, long long n, long long nlos, const double* los,
                              const double* dist_from_plan, const nx_los_params* lp_,
                              double* radiance, long long* npackets, uint8_t* included,
                              long long* used_count) {
  if (!used_count)
    return nx_los_accumulate(ctx, n, nlos, los, dist_from_plan, lp_, radiance, npackets, included);
  ENTER(ctx);
  if (n > resident_rows(ctx)) { ctx->err = "n exceeds resident packets"; return -1; }
  if (n >= (1LL << 32)) { ctx->err = "more than 2^32 packets per GPU"; return -1; }
  LosParams lp;
  std::memcpy(&lp, lp_, sizeof(lp));
  { int r0 = check_los_params(ctx, lp); if (r0) return r0; }
  double *d_los = nullptr, *d_dist = nullptr, *d_rad = nullptr;
  unsigned long long *d_np = nullptr, *d_nused = nullptr;
  unsigned char* d_inc = nullptr;
  const size_t nl = (size_t)(nlos > 0 ? nlos : 1), nn = (size_t)(n > 0 ? n : 1);
  SCR(SCR_LOS, d_los, 6 * nl);
  SCR(SCR_DIST, d_dist, nl);
  SCR(SCR_RAD, d_rad, nl);
  SCR(SCR_NP, d_np, nl);
  SCR(SCR_INC, d_inc, nn);
  SCR(SCR_NUSED, d_nused, nl);
  CK(cudaMemcpyAsync(d_los, los, 6 * (size_t)nlos * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaMemcpyAsync(d_dist, dist_from_plan, (size_t)nlos * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaMemsetAsync(d_rad, 0, nl * sizeof(double), ctx->stream));
  CK(cudaMemsetAsync(d_np, 0, nl * sizeof(unsigned long long), ctx->stream));
  CK(cudaMemsetAsync(d_nused, 0, nl * sizeof(unsigned long long), ctx->stream));
  CK(cudaMemsetAsync(d_inc, 0, nn, ctx->stream));
  int r = 0;
  if (n > 0 && nlos > 0) r = los_run(ctx, n, nlos, d_los, d_dist, lp, d_rad, d_np, d_inc, d_nused);
  if (r == 0) {
    cudaMemcpyAsync(radiance, d_rad, (size_t)nlos * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream);
    cudaMemcpyAsync(npackets, d_np, (size_t)nlos * sizeof(long long), cudaMemcpyDeviceToHost, ctx->stream);
    cudaMemcpyAsync(used_count, d_nused, (size_t)nlos * sizeof(long long), cudaMemcpyDeviceToHost, ctx->stream);
    if (included) cudaMemcpyAsync(included, d_inc, (size_t)n, cudaMemcpyDeviceToHost, ctx->stream);
    cudaError_t e = cudaStreamSynchronize(ctx->stream);
    if (e != cudaSuccess) { ctx->err = cudaGetErrorString(e); r = -(int)e; }
  }
  return r;
}

// The indices of the `used` packets, CSR layout given by used_offsets (the prefix sums of the
// counts nx_los_accumulate_counted returned).  When that call's candidate pairs are still on
// the device (same packets, same lines of sight, nothing in between) only the exact test is
// repeated over them; otherwise the whole search runs again (nx_los_used).
int nx_los_used_fill(nx_ctx* ctx, long long n, long long nlos, const double* los,
                     const double* dist_from_plan, const nx_los_params* lp_,
                     const long long* used_offsets, uint32_t* used_indices) {
  if (!used_offsets || !used_indices) { ctx->err = "nx_los_used_fill: null argument"; return -1; }
  LosParams lp;
  std::memcpy(&lp, lp_, sizeof(lp));
  { const std::string e = los_dphi_error(lp.dphi); if (!e.empty()) { ctx->err = e; return -1; } }
  const nx_ctx::LosKept k = ctx->los_kept;
  const bool reuse = k.np > 0 && k.n == n && k.nlos == nlos && k.bound == ctx->bound &&
                     std::memcmp(&k.lp, &lp, sizeof(lp)) == 0;
  if (!reuse) {
    std::vector<long long> count((size_t)(nlos > 0 ? nlos : 1));
    return nx_los_used(ctx, n, nlos, los, dist_from_plan, lp_, used_offsets, count.data(), used_indices);
  }
  CK(cudaSetDevice(ctx->device));
  const long long total = used_offsets[nlos];
  if (total <= 0) return 0;
  unsigned long long* d_cursor = nullptr;
  long long* d_off = nullptr;
  unsigned* d_idx = nullptr;
  SCR(SCR_CURSOR, d_cursor, (size_t)nlos);
  SCR(SCR_OFF, d_off, (size_t)(nlos + 1));
  SCR(SCR_IDX, d_idx, (size_t)total);
  CK(cudaMemsetAsync(d_cursor, 0, (size_t)nlos * sizeof(unsigned long long), ctx->stream));
  CK(cudaMemcpyAsync(d_off, used_offsets, (size_t)(nlos + 1) * sizeof(long long), cudaMemcpyHostToDevice, ctx->stream));
  const double* d_ladder = static_cast<const double*>(ctx->scr[SCR_LADDER].p);
  int r = begin_timed(ctx);
  if (r) return r;
  CK(launch_los_resolve(ctx->stream, ctx->losw, k.np, nlos,
                        static_cast<const double*>(ctx->scr[SCR_LOS].p),
                        static_cast<const double*>(ctx->scr[SCR_DIST].p),
                        static_cast<const int*>(ctx->scr[SCR_NBALL].p), d_ladder,
                        d_ladder + k.nladder, k.lp, k.lc, ctx->gtables, nullptr, nullptr, nullptr,
                        nullptr, d_off, d_cursor, d_idx));
  if ((r = end_timed(ctx, 1))) return r;
  CK(cudaMemcpyAsync(used_indices, d_idx, (size_t)total * sizeof(unsigned), cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  return 0;
}

int nx_los_used(nx_ctx* ctx, long long n, long long nlos, const double* los,
                const double* dist_from_plan, const nx_los_params* lp_, const long long* used_offsets,
                long long* used_count, uint32_t* used_indices) {
  ENTER(ctx);
  if (n > resident_rows(ctx)) { ctx->err = "n exceeds resident packets"; return -1; }
  LosParams lp;
  std::memcpy(&lp, lp_, sizeof(lp));
  { int r0 = check_los_params(ctx, lp); if (r0) return r0; }
  if (nlos <= 0) return 0;
  if (n <= 0) { for (long long i = 0; i < nlos; ++i) used_count[i] = 0; return 0; }
  if (n >= (1LL << 32)) { ctx->err = "more than 2^32 packets per GPU"; return -1; }
  { int r0 = materialize(ctx); if (r0) return r0; }
  std::vector<int> nball;
  std::vector<double> ladder, wid2;
  LosConsts lc;
  { const std::string e = los_prepare(los, nlos, lp, nball, ladder, wid2, lc); if (!e.empty()) { ctx->err = e; return -1; } }
  const long long total = used_indices ? used_offsets[nlos] : 0;
  double *d_los = nullptr, *d_dist = nullptr, *d_ladder = nullptr, *d_wid2 = nullptr;
  int* d_nball = nullptr;
  unsigned long long *d_nused = nullptr, *d_cursor = nullptr;
  long long* d_off = nullptr;
  unsigned* d_idx = nullptr;
  SCR(SCR_LOS, d_los, 6 * (size_t)nlos);
  SCR(SCR_DIST, d_dist, (size_t)nlos);
  SCR(SCR_NBALL, d_nball, (size_t)nlos);
  SCR(SCR_LADDER, d_ladder, ladder.size());
  SCR(SCR_WID2, d_wid2, wid2.size());
  SCR(SCR_NUSED, d_nused, (size_t)nlos);
  CK(cudaMemsetAsync(d_nused, 0, (size_t)nlos * sizeof(unsigned long long), ctx->stream));
  CK(cudaMemcpyAsync(d_los, los, 6 * (size_t)nlos * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaMemcpyAsync(d_dist, dist_from_plan, (size_t)nlos * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaMemcpyAsync(d_nball, nball.data(), (size_t)nlos * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaMemcpyAsync(d_ladder, ladder.data(), ladder.size() * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaMemcpyAsync(d_wid2, wid2.data(), wid2.size() * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
  if (used_indices) {
    SCR(SCR_CURSOR, d_cursor, (size_t)nlos);
    SCR(SCR_OFF, d_off, (size_t)(nlos + 1));
    SCR(SCR_IDX, d_idx, (size_t)(total > 0 ? total : 1));
    CK(cudaMemsetAsync(d_cursor, 0, (size_t)nlos * sizeof(unsigned long long), ctx->stream));
    CK(cudaMemcpyAsync(d_off, used_offsets, (size_t)(nlos + 1) * sizeof(long long), cudaMemcpyHostToDevice, ctx->stream));
  }
  int r = alloc_los_work(ctx, n);
  if (r == 0) r = begin_timed(ctx);
  if (r == 0) {
    cudaError_t e = launch_los_grid_build(ctx->stream, ctx->device, state_cols(ctx), n, lp, ctx->losw);
    if (e == cudaSuccess)
      e = launch_los_grid(ctx->stream, ctx->losw, nlos, d_los, d_dist, d_nball, d_ladder, d_wid2, lp,
                          lc, ctx->gtables, nullptr, nullptr, nullptr, d_nused, d_off, d_cursor, d_idx);
    if (e != cudaSuccess) { ctx->err = cudaGetErrorString(e); r = -(int)e; }
  }
  if (r == 0) r = end_timed(ctx, 8);
  if (r == 0) {
    static_assert(sizeof(long long) == sizeof(unsigned long long), "");
    cudaMemcpyAsync(used_count, d_nused, (size_t)nlos * sizeof(long long), cudaMemcpyDeviceToHost, ctx->stream);
    if (used_indices && total > 0)
      cudaMemcpyAsync(used_indices, d_idx, (size_t)total * sizeof(unsigned), cudaMemcpyDeviceToHost, ctx->stream);
    cudaError_t e = cudaStreamSynchronize(ctx->stream);
    if (e != cudaSuccess) { ctx->err = cudaGetErrorString(e); r = -(int)e; }
  }
  return r;
}

// ---- Doppler line profiles (LOSSpectrum): K5's hits binned by line-of-sight velocity -------
int nx_los_spectrum(nx_ctx* ctx, long long n, long long nlos, const double* los,
                    const double* dist_from_plan, const nx_los_params* lp_,
                    const nx_spectrum_params* sp_, double* spectrum, long long* counts) {
  ENTER(ctx);
  if (!lp_ || !sp_) { ctx->err = "nx_los_spectrum: null argument"; return -1; }
  if (n < 0 || nlos < 0) { ctx->err = "nx_los_spectrum: negative size"; return -1; }
  if (n > resident_rows(ctx)) { ctx->err = "n exceeds resident packets"; return -1; }
  if (n >= (1LL << 32)) { ctx->err = "more than 2^32 packets per GPU"; return -1; }
  const nx_spectrum_params sp = *sp_;
  if (sp.nbins < 1) { ctx->err = "nx_los_spectrum: nbins must be >= 1"; return -1; }
  if (!std::isfinite(sp.vmin) || !std::isfinite(sp.vmax) || !(sp.vmin < sp.vmax)) {
    ctx->err = "nx_los_spectrum: vmin < vmax, both finite, required";
    return -1;
  }
  if (!std::isfinite(sp.vscale)) { ctx->err = "nx_los_spectrum: vscale must be finite"; return -1; }
  const long long ncol = (long long)sp.nbins + 2;
  if ((double)nlos * (double)ncol >= 2147483648.0) {
    ctx->err = "nx_los_spectrum: nlos * (nbins + 2) must be < 2^31";
    return -1;
  }
  LosParams lp;
  std::memcpy(&lp, lp_, sizeof(lp));
  { int r0 = check_los_params(ctx, lp); if (r0) return r0; }
  const size_t ncell = (size_t)(nlos * ncol);
  if (nlos == 0) return 0;
  if (!los || !dist_from_plan || !spectrum || !counts) { ctx->err = "nx_los_spectrum: null argument"; return -1; }
  if (n == 0) {
    std::memset(spectrum, 0, ncell * sizeof(double));
    std::memset(counts, 0, ncell * sizeof(long long));
    return 0;
  }
  double *d_los = nullptr, *d_dist = nullptr, *d_spec = nullptr;
  SCR(SCR_LOS, d_los, 6 * (size_t)nlos);
  SCR(SCR_DIST, d_dist, (size_t)nlos);
  SCR(SCR_SPEC, d_spec, 2 * ncell);                 // sums, then the u64 counts
  LosSpectrum spec;
  const StateCols P = state_cols(ctx);
  spec.vx = P.c[4];
  spec.vz = P.c[6];
  spec.vmin = sp.vmin;
  spec.vmax = sp.vmax;
  spec.step = (sp.vmax - sp.vmin) / sp.nbins;       // np.linspace's step
  spec.vscale = sp.vscale;
  spec.nbins = sp.nbins;
  spec.sum = d_spec;
  spec.count = reinterpret_cast<unsigned long long*>(d_spec + ncell);
  CK(cudaMemcpyAsync(d_los, los, 6 * (size_t)nlos * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaMemcpyAsync(d_dist, dist_from_plan, (size_t)nlos * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaMemsetAsync(d_spec, 0, 2 * ncell * sizeof(double), ctx->stream));
  int r = los_run(ctx, n, nlos, d_los, d_dist, lp, nullptr, nullptr, nullptr, nullptr, &spec);
  if (r == 0) {
    static_assert(sizeof(long long) == sizeof(unsigned long long), "");
    CK(cudaMemcpyAsync(spectrum, d_spec, ncell * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(counts, d_spec + ncell, ncell * sizeof(long long), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
  }
  return r;
}

// ---- Doppler-resolved image cubes (ModelImageCube) -----------------------------------------
// The cube is the NX_PRODUCT_CUBE accumulator, released by nx_product_end: an 800 x 800 x 100
// cube is 0.5 GB per plane, too much to keep after the product is fetched.
int nx_cube_begin(nx_ctx* ctx, int nx_, int nz_, int nbins) {
  CK(cudaSetDevice(ctx->device));
  if (nx_ < 1 || nz_ < 1 || nbins < 1) { ctx->err = "nx_cube_begin: bad dims"; return -1; }
  if ((double)nx_ * nz_ * ((double)nbins + 2) >= 2147483648.0) {
    ctx->err = "nx_cube_begin: nx * nz * (nbins + 2) must be < 2^31";
    return -1;
  }
  const long long ncell = (long long)nx_ * nz_ * (nbins + 2);
  return accum_begin(ctx, NX_PRODUCT_CUBE, ncell, ncell, nx_, nz_, nbins);
}

int nx_cube_add(nx_ctx* ctx, long long n, const nx_image_params* ip_,
                const nx_spectrum_params* sp_) {
  CK(cudaSetDevice(ctx->device));
  const Accum* cube = accum_of(ctx, NX_PRODUCT_CUBE);
  if (!cube) return -1;
  if (!ip_ || !sp_) { ctx->err = "nx_cube_add: null argument"; return -1; }
  ImageParams ip;
  std::memcpy(&ip, ip_, sizeof(ip));
  const nx_spectrum_params sp = *sp_;
  if (ip.nx != cube->dims[0] || ip.nz != cube->dims[1] || sp.nbins != cube->dims[2]) {
    ctx->err = "nx_cube_add: dims or nbins differ from nx_cube_begin";
    return -1;
  }
  if (!std::isfinite(sp.vmin) || !std::isfinite(sp.vmax) || !(sp.vmin < sp.vmax)) {
    ctx->err = "nx_cube_add: vmin < vmax, both finite, required";
    return -1;
  }
  if (!std::isfinite(sp.vscale)) { ctx->err = "nx_cube_add: vscale must be finite"; return -1; }
  if (ip.quantity == 1 && ctx->gtables.n == 0) {
    ctx->err = "radiance cube requested but no g-value tables uploaded";
    return -1;
  }
  if (n < 0 || n > resident_rows(ctx)) { ctx->err = "n exceeds resident packets"; return -1; }
  if (n == 0) return 0;
  CubeAxis ax;
  ax.vmin = sp.vmin;
  ax.vmax = sp.vmax;
  ax.step = (sp.vmax - sp.vmin) / sp.nbins;         // np.linspace's step
  ax.vscale = sp.vscale;
  ax.nbins = sp.nbins;
  int r;
  if ((r = materialize(ctx))) return r;
  if ((r = begin_timed(ctx))) return r;
  CK(launch_image_cube(ctx->stream, ctx->device, state_cols(ctx), n, ip, ctx->gtables, ax,
                       cube->sums(), cube->counts()));
  return end_timed(ctx, 1);
}

// ---- K7: number density at sample points (ModelDensity) ------------------------------------
// The rows go through K5's cell grid (built again here, with the f32 records: this resets the
// candidate pairs K5 keeps, which ENTER drops); the points are processed in Morton order of
// 0.4 R_p cells over +-6.4 R_p, so that warps that run together stream the same cells.
int nx_density_accumulate(nx_ctx* ctx, long long n, long long npts, const double* pts,
                          const double* radius, double* s1, double* s2,
                          unsigned long long* count) {
  ENTER(ctx);
  if (n < 0 || npts < 0) { ctx->err = "nx_density_accumulate: negative size"; return -1; }
  if (n > resident_rows(ctx)) { ctx->err = "n exceeds resident packets"; return -1; }
  if (n >= (1LL << 32)) { ctx->err = "more than 2^32 packets per GPU"; return -1; }
  if (n == 0 || npts == 0) return 0;
  if (!pts || !radius || !s1 || !s2 || !count) { ctx->err = "nx_density_accumulate: null argument"; return -1; }
  for (long long i = 0; i < npts; ++i) {
    if (!std::isfinite(pts[i]) || !std::isfinite(pts[npts + i]) || !std::isfinite(pts[2 * npts + i]) ||
        !std::isfinite(radius[i]) || !(radius[i] > 0.0)) {
      ctx->err = "nx_density_accumulate: points and radii must be finite, radii > 0";
      return -1;
    }
  }
  { int r0 = materialize(ctx); if (r0) return r0; }
  // Morton order (counting sort of 15-bit keys)
  std::vector<unsigned> key((size_t)npts), order((size_t)npts), hist(NX_LOS_KEY_BINS + 1, 0u);
  for (long long i = 0; i < npts; ++i) {
    unsigned k = 0;
    for (int a = 0; a < 3; ++a) {
      double v = (pts[a * npts + i] + 6.4) / 0.4;
      v = v < 0.0 ? 0.0 : (v > 31.0 ? 31.0 : v);
      const unsigned q = (unsigned)v;
      for (int b = 0; b < 5; ++b) k |= ((q >> b) & 1u) << (3 * b + a);
    }
    key[i] = k;
    ++hist[k + 1];
  }
  for (int k = 0; k < NX_LOS_KEY_BINS; ++k) hist[k + 1] += hist[k];
  for (long long i = 0; i < npts; ++i) order[hist[key[i]]++] = (unsigned)i;

  const size_t np = (size_t)npts;
  const size_t nb = np < (size_t)NX_DENSITY_BATCH ? np : (size_t)NX_DENSITY_BATCH;
  double *d_in = nullptr, *d_out = nullptr;
  unsigned* d_idx = nullptr;
  SCR(SCR_DENS_IN, d_in, 4 * np);                   // x, y, z, radius
  SCR(SCR_DENS_OUT, d_out, 3 * np);                 // s1, s2, count (u64)
  SCR(SCR_DENS_IDX, d_idx, np + 6 * nb + 2 * nb + 2);   // order, box, nitem, item_off, cursor
  unsigned* d_order = d_idx;
  int* d_box = reinterpret_cast<int*>(d_idx + np);
  unsigned* d_nitem = d_idx + np + 6 * nb;
  unsigned* d_off = d_nitem + nb;
  unsigned* d_cursor = d_off + nb + 1;
  double* d_s1 = d_out;
  double* d_s2 = d_out + np;
  unsigned long long* d_cnt = reinterpret_cast<unsigned long long*>(d_out + 2 * np);
  CK(cudaMemcpyAsync(d_in, pts, 3 * np * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaMemcpyAsync(d_in + 3 * np, radius, np * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaMemcpyAsync(d_order, order.data(), np * sizeof(unsigned), cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaMemsetAsync(d_out, 0, 3 * np * sizeof(double), ctx->stream));
  int r = alloc_los_work(ctx, n);
  if (r == 0) r = begin_timed(ctx);
  int nlaunch = 6;
  if (r == 0) {
    LosParams lp{};
    lp.round_f32 = 1;
    lp.skip_dead = 1;
    cudaError_t e = launch_los_grid_build(ctx->stream, ctx->device, state_cols(ctx), n, lp, ctx->losw);
    if (e == cudaSuccess)
      e = launch_density(ctx->stream, ctx->device, ctx->losw, npts, d_in, d_in + 3 * np, d_order,
                         d_box, d_nitem, d_off, d_cursor, d_s1, d_s2, d_cnt, &nlaunch);
    if (e != cudaSuccess) { ctx->err = cudaGetErrorString(e); r = -(int)e; }
  }
  if (r == 0) r = end_timed(ctx, nlaunch);
  if (r == 0) {
    std::vector<double> out(3 * np);
    CK(cudaMemcpyAsync(out.data(), d_out, 3 * np * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    const unsigned long long* c = reinterpret_cast<const unsigned long long*>(out.data() + 2 * np);
    for (size_t i = 0; i < np; ++i) {
      s1[i] += out[i];
      s2[i] += out[np + i];
      count[i] += c[i];
    }
  }
  return r;
}

// ---- resident packet tables (device-side Output.save, Output.py:522-543) -----------------
int nx_compact_state(nx_ctx* ctx, long long n, int skip_dead, int round_f32, nx_packets** out,
                     long long* count) {
  ENTER(ctx);
  if (!out) { ctx->err = "nx_compact_state: null output"; return -1; }
  *out = nullptr;
  ctx->bound = nullptr;
  if (n > ctx->cap) { ctx->err = "n exceeds resident packets"; return -1; }
  nx_packets* h = new nx_packets();
  if (n > 0) {
    const long long nt = compact_tiles(n);
    if (nt + 2 > ctx->cmp_tiles_cap) {
      cudaFree(ctx->cmp_tiles);
      ctx->cmp_tiles = nullptr; ctx->cmp_tiles_cap = 0;
      CK(cudaMalloc(&ctx->cmp_tiles, (size_t)(nt + 2) * sizeof(unsigned)));
      ctx->cmp_tiles_cap = nt + 2;
    }
    StateCols P = in_cols(ctx);
    int r;
    if ((r = begin_timed(ctx))) { delete h; return r; }
    cudaError_t e = launch_compact_count(ctx->stream, P.c[7], n, skip_dead, ctx->cmp_tiles,
                                         ctx->scalars + 4);
    unsigned long long total = 0;
    if (e == cudaSuccess)
      e = cudaMemcpyAsync(&total, ctx->scalars + 4, sizeof(total), cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    if (e == cudaSuccess && total > 0) {
      h->n = (long long)total;
      h->cap = ((h->n + 31) / 32) * 32;
      h->ncols = 9;
      e = table_alloc(h, ctx->stream, 9, false);
      if (e == cudaSuccess)
        e = launch_compact_scatter(ctx->stream, P, n, skip_dead, round_f32,
                                   ctx->fresh ? 0 : 1, ctx->cmp_tiles, h->cols,
                                   (size_t)h->cap, h->index);
    }
    if (e != cudaSuccess) {
      ctx->err = std::string("nx_compact_state: ") + cudaGetErrorString(e);
      free_packets(h, ctx->stream);
      return -(int)e;
    }
    if ((r = end_timed(ctx, total > 0 ? 3 : 2))) { free_packets(h, ctx->stream); return r; }
  }
  *out = h;
  if (count) *count = h->n;
  return 0;
}

int nx_packets_upload(nx_ctx* ctx, long long n, const double* const* cols, const uint32_t* index,
                      nx_packets** out) {
  ENTER(ctx);
  if (!out) { ctx->err = "nx_packets_upload: null output"; return -1; }
  nx_packets* h = new nx_packets();
  h->n = n;
  h->cap = ((std::max(n, 1LL) + 31) / 32) * 32;
  cudaError_t e = table_alloc(h, ctx->stream, 8, false);
  for (int k = 0; k < 8 && e == cudaSuccess && n > 0; ++k)
    e = cudaMemcpyAsync(h->cols + (size_t)k * h->cap, cols[k], (size_t)n * sizeof(double),
                        cudaMemcpyHostToDevice, ctx->stream);
  if (e == cudaSuccess && n > 0 && index)
    e = cudaMemcpyAsync(h->index, index, (size_t)n * sizeof(unsigned), cudaMemcpyHostToDevice, ctx->stream);
  if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
  if (e != cudaSuccess) {
    ctx->err = std::string("nx_packets_upload: ") + cudaGetErrorString(e);
    free_packets(h, ctx->stream);
    return -(int)e;
  }
  *out = h;
  return 0;
}

int nx_packets_bind(nx_ctx* ctx, nx_packets* h) {
  ctx->los_kept.np = 0;
  ctx->bound = h;
  return 0;
}

int nx_packets_count(nx_ctx* ctx, nx_packets* h, long long* count) {
  if (!h) { ctx->err = "null packet table"; return -1; }
  if (count) *count = h->n;
  return 0;
}

int nx_packets_export(nx_ctx* ctx, nx_packets* h, float* const* cols, int32_t* index,
                      uint16_t* step) {
  CK(cudaSetDevice(ctx->device));
  if (!h) { ctx->err = "null packet table"; return -1; }
  if (h->n == 0) return 0;
  bool any = false;
  for (int k = 0; k < h->ncols; ++k) any |= cols && cols[k];
  float* tmp = nullptr;
  cudaError_t e = cudaSuccess;
  if (any) {
    SCR(SCR_TMP, tmp, (size_t)h->ncols * h->n);
    e = launch_to_f32(ctx->stream, h->cols, (size_t)h->cap, h->n, h->ncols, tmp);
  }
  for (int k = 0; any && k < h->ncols && e == cudaSuccess; ++k)
    if (cols[k])
      e = cudaMemcpyAsync(cols[k], tmp + (size_t)k * h->n, (size_t)h->n * sizeof(float),
                          cudaMemcpyDeviceToHost, ctx->stream);
  if (e == cudaSuccess && index)
    e = cudaMemcpyAsync(index, h->index, (size_t)h->n * sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->stream);
  if (e == cudaSuccess && step) {
    if (h->step)
      e = cudaMemcpyAsync(step, h->step, (size_t)h->n * sizeof(uint16_t), cudaMemcpyDeviceToHost, ctx->stream);
    else
      std::memset(step, 0, (size_t)h->n * sizeof(uint16_t));
  }
  if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
  ctx->launches += 1;
  if (e != cudaSuccess) { ctx->err = std::string("nx_packets_export: ") + cudaGetErrorString(e); return -(int)e; }
  return 0;
}

int nx_packets_free(nx_ctx* ctx, nx_packets* h) {
  if (!h) return 0;
  cudaSetDevice(ctx->device);
  ctx->los_kept.np = 0;
  if (ctx->bound == h) ctx->bound = nullptr;
  free_packets(h, ctx->stream);
  return 0;
}

int nx_last_kernel_ms(nx_ctx* ctx, float* ms) {
  CK(cudaSetDevice(ctx->device));
  CK(cudaEventSynchronize(ctx->ev1));
  CK(cudaEventElapsedTime(&ctx->last_ms, ctx->ev0, ctx->ev1));
  if (ms) *ms = ctx->last_ms;
  return 0;
}

int nx_kernel_launches(nx_ctx* ctx, unsigned long long* count) {
  if (count) *count = ctx->launches;
  return 0;
}

int nx_measure_fp64_peak(nx_ctx* ctx, double* tflops) {
  CK(cudaSetDevice(ctx->device));
  int blocks = 0, threads = 0;
  const int iters = 1 << 15;
  double* out = nullptr;
  CK(cudaMalloc(&out, (size_t)148 * 64 * 256 * sizeof(double)));
  float best = 1e30f;
  for (int rep = 0; rep < 6; ++rep) {
    CK(cudaEventRecord(ctx->ev0, ctx->stream));
    CK(launch_fp64_peak(ctx->stream, ctx->device, out, iters, &blocks, &threads));
    CK(cudaEventRecord(ctx->ev1, ctx->stream));
    CK(cudaEventSynchronize(ctx->ev1));
    float ms = 0.f;
    CK(cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1));
    if (rep > 0 && ms < best) best = ms;
    ctx->launches += 1;
  }
  cudaFree(out);
  const double flops = 2.0 * 8.0 * iters * (double)blocks * threads;
  if (tflops) *tflops = flops / (best * 1e-3) / 1e12;
  return 0;
}

int nx_measure_copy_bw(nx_ctx* ctx, long long bytes, double* gbs) {
  CK(cudaSetDevice(ctx->device));
  const long long n = bytes / 8 / 2 * 2;
  double *a = nullptr, *b = nullptr;
  CK(cudaMalloc(&a, n * sizeof(double)));
  CK(cudaMalloc(&b, n * sizeof(double)));
  CK(cudaMemsetAsync(a, 0, n * sizeof(double), ctx->stream));
  float best = 1e30f;
  for (int rep = 0; rep < 6; ++rep) {
    CK(cudaEventRecord(ctx->ev0, ctx->stream));
    CK(launch_copy(ctx->stream, ctx->device, a, b, n));
    CK(cudaEventRecord(ctx->ev1, ctx->stream));
    CK(cudaEventSynchronize(ctx->ev1));
    float ms = 0.f;
    CK(cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1));
    if (rep > 0 && ms < best) best = ms;
    ctx->launches += 1;
  }
  cudaFree(a); cudaFree(b);
  if (gbs) *gbs = 2.0 * n * sizeof(double) / (best * 1e-3) / 1e9;
  return 0;
}

}  // extern "C"
