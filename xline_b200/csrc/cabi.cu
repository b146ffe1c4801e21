// C ABI (include/xline_b200.h) and host-side orchestration of the tracking kernels:
// variant selection, shared-memory ring sizing, turn segmentation with survivor
// compaction between launches, the host-buffer entry point, and the FP64-peak probe.
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include <algorithm>
#include <cmath>
#include <mutex>
#include <string>
#include <type_traits>
#include <vector>

#include "../../include/xline_b200.h"
#include "kargs.h"
#include "launch_plan.h"

namespace xlb {

static thread_local std::string g_err;
static thread_local xlb_track_stats_t g_stats;

static int fail(int code, const std::string &msg) {
  g_err = msg;
  return code;
}
#define XLB_CUDA(call)                                                                     \
  do {                                                                                     \
    cudaError_t e__ = (call);                                                              \
    if (e__ != cudaSuccess) {                                                              \
      return fail(XLB_ECUDA, std::string(#call) + ": " + cudaGetErrorString(e__));         \
    }                                                                                      \
  } while (0)

// ------------------------------------------------------------------ survivor compaction
// Order-preserving stream compaction of {i : state[i]==1} built from warp ballots:
// pass 1 counts per block, pass 2 scans the block totals, pass 3 re-derives the ballots
// and scatters.  Deterministic (no atomics on the output position).
constexpr int CP_THREADS = 512;
constexpr int CP_ITEMS = 8;  // elements per thread

__global__ void __launch_bounds__(CP_THREADS) compact_count(const long long *state, long long n,
                                                            int *block_sums) {
  __shared__ int warp_cnt[CP_THREADS / 32];
  const long long base = static_cast<long long>(blockIdx.x) * (CP_THREADS * CP_ITEMS);
  int cnt = 0;
#pragma unroll
  for (int it = 0; it < CP_ITEMS; ++it) {
    const long long i = base + static_cast<long long>(it) * CP_THREADS + threadIdx.x;
    const bool keep = (i < n) && (state[i] == 1);
    cnt += __popc(__ballot_sync(0xffffffffu, keep));
  }
  if ((threadIdx.x & 31) == 0) warp_cnt[threadIdx.x >> 5] = cnt;
  __syncthreads();
  if (threadIdx.x == 0) {
    int t = 0;
    for (int w = 0; w < CP_THREADS / 32; ++w) t += warp_cnt[w];
    block_sums[blockIdx.x] = t;
  }
}

__global__ void __launch_bounds__(1024) compact_scan(int *block_sums, int nblocks, int *n_out) {
  // exclusive scan of block_sums by one CTA (nblocks <= a few 1e4), warp-shuffle based
  __shared__ int warp_tot[32];
  __shared__ int carry;
  if (threadIdx.x == 0) carry = 0;
  __syncthreads();
  for (int start = 0; start < nblocks; start += 1024) {
    const int i = start + threadIdx.x;
    const int v = (i < nblocks) ? block_sums[i] : 0;
    int incl = v;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const int t = __shfl_up_sync(0xffffffffu, incl, d);
      if ((threadIdx.x & 31) >= d) incl += t;
    }
    if ((threadIdx.x & 31) == 31) warp_tot[threadIdx.x >> 5] = incl;
    __syncthreads();
    if (threadIdx.x < 32) {
      int w = warp_tot[threadIdx.x];
      int wi = w;
#pragma unroll
      for (int d = 1; d < 32; d <<= 1) {
        const int t = __shfl_up_sync(0xffffffffu, wi, d);
        if (threadIdx.x >= d) wi += t;
      }
      warp_tot[threadIdx.x] = wi - w;  // exclusive warp offsets
    }
    __syncthreads();
    const int excl = carry + warp_tot[threadIdx.x >> 5] + incl - v;
    if (i < nblocks) block_sums[i] = excl;
    __syncthreads();
    if (threadIdx.x == 1023) carry = excl + v;
    __syncthreads();
  }
  if (threadIdx.x == 0) *n_out = carry;
}

__global__ void __launch_bounds__(CP_THREADS) compact_scatter(const long long *state, long long n,
                                                              const int *block_offs, int *idx_out) {
  __shared__ int warp_cnt[CP_ITEMS][CP_THREADS / 32];
  const long long base = static_cast<long long>(blockIdx.x) * (CP_THREADS * CP_ITEMS);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  unsigned ballots[CP_ITEMS];
#pragma unroll
  for (int it = 0; it < CP_ITEMS; ++it) {
    const long long i = base + static_cast<long long>(it) * CP_THREADS + threadIdx.x;
    const bool keep = (i < n) && (state[i] == 1);
    ballots[it] = __ballot_sync(0xffffffffu, keep);
    if (lane == 0) warp_cnt[it][warp] = __popc(ballots[it]);
  }
  __syncthreads();
  // output order = increasing i: item-major, then warp, then lane
  int off = block_offs[blockIdx.x];
#pragma unroll
  for (int it = 0; it < CP_ITEMS; ++it) {
    int before = 0;
    for (int w = 0; w < CP_THREADS / 32; ++w) {
      const int c = warp_cnt[it][w];
      if (w < warp) before += c;
    }
    int tot = 0;
    for (int w = 0; w < CP_THREADS / 32; ++w) tot += warp_cnt[it][w];
    const long long i = base + static_cast<long long>(it) * CP_THREADS + threadIdx.x;
    if ((ballots[it] >> lane) & 1u) {
      const int pos = off + before + __popc(ballots[it] & ((1u << lane) - 1u));
      idx_out[pos] = static_cast<int>(i);
    }
    off += tot;
  }
}

// ------------------------------------------------------------------ per-device scratch
struct Scratch {
  int device = -1;
  int *idx = nullptr;         // survivor list
  int *block_sums = nullptr;  // compaction scratch
  long long cap = 0;          // capacity of idx (entries)
  int nblocks_cap = 0;
  unsigned int *queue = nullptr;   // work queue of the persistent kernel: two counters + ring of ready items
  size_t queue_cap = 0;
  unsigned int *n_lost = nullptr;  // device counter
  int *n_active = nullptr;         // device survivor count
  unsigned int *h_pinned = nullptr;  // [0]=n_lost, [1]=n_active (pinned host)
  // host entry point arena
  unsigned char *arena = nullptr;
  size_t arena_bytes = 0;
  cudaStream_t stream = nullptr;  // host entry point stream
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  // One call at a time per device: the queue, the survivor list, the counters and the pinned
  // read-back words above are shared by every xlb_track_* call on this GPU.  Host threads
  // serialise on `call_mu` (recursive: the host entry point calls the device one); work that a
  // previous call left running on ANOTHER stream is ordered before the next call's by `done`,
  // recorded at the end of every call and waited for at the start of the next (CallScope).
  std::recursive_mutex call_mu;
  cudaEvent_t done = nullptr;
  bool have_done = false;
  // launch-length schedule (see track_device_impl): loss rate per turn seen by the last
  // segmented call, and the particle set it belonged to
  const double *sched_x = nullptr;
  long long sched_n = 0;
  double sched_rate = -1.0;
  double *moments = nullptr;  // beam-moment partial sums (moments.cu)
  size_t moments_cap = 0;     // doubles
};

static std::mutex g_mu;
static std::vector<Scratch *> g_scratch;

static int get_scratch(Scratch **out) {
  int dev = 0;
  XLB_CUDA(cudaGetDevice(&dev));
  std::lock_guard<std::mutex> lk(g_mu);
  for (Scratch *s : g_scratch)
    if (s->device == dev) {
      *out = s;
      return XLB_OK;
    }
  Scratch *s = new Scratch();
  s->device = dev;
  XLB_CUDA(cudaMalloc(&s->n_lost, sizeof(unsigned int)));
  XLB_CUDA(cudaMalloc(&s->n_active, sizeof(int)));
  XLB_CUDA(cudaMemset(s->n_lost, 0, sizeof(unsigned int)));
  XLB_CUDA(cudaMallocHost(&s->h_pinned, 2 * sizeof(unsigned int)));
  XLB_CUDA(cudaStreamCreateWithFlags(&s->stream, cudaStreamNonBlocking));
  XLB_CUDA(cudaEventCreate(&s->ev0));
  XLB_CUDA(cudaEventCreate(&s->ev1));
  XLB_CUDA(cudaEventCreateWithFlags(&s->done, cudaEventDisableTiming));
  g_scratch.push_back(s);
  *out = s;
  return XLB_OK;
}

namespace {
// The scope of one call on the current device: holds its Scratch's `call_mu`, makes `st` wait for
// what the previous call enqueued and, whatever way the call ends, records `done` on `st` so that
// the next call waits for what this one enqueued.
class CallScope {
 public:
  Scratch *s = nullptr;
  int open(cudaStream_t st) {
    int rc;
    if ((rc = get_scratch(&s)) != XLB_OK) return rc;
    lock_ = std::unique_lock<std::recursive_mutex>(s->call_mu);
    st_ = st;
    if (s->have_done) XLB_CUDA(cudaStreamWaitEvent(st, s->done, 0));
    return XLB_OK;
  }
  ~CallScope() {
    if (lock_.owns_lock() && cudaEventRecord(s->done, st_) == cudaSuccess) s->have_done = true;
  }

 private:
  std::unique_lock<std::recursive_mutex> lock_;
  cudaStream_t st_ = nullptr;
};
}  // namespace

// Grows the device buffer `*buf` to at least `count` elements; what it held is not kept.
template <typename T, typename N>
static int grow(T **buf, N *cap, N count) {
  if (count <= *cap) return XLB_OK;
  if (*buf) cudaFree(*buf);
  *buf = nullptr;
  *cap = 0;
  XLB_CUDA(cudaMalloc(buf, static_cast<size_t>(count) * sizeof(T)));
  *cap = count;
  return XLB_OK;
}

// The address of a pointer field, as the slot a device pointer is written to.
template <typename T>
static void **slot(T **field) {
  return reinterpret_cast<void **>(const_cast<std::remove_const_t<T> **>(field));
}

// One beam-moment store of slots 0..n-1 into out[0..XLB_MOMENT_WORDS), enqueued on `st`.
static int beam_moments(Scratch *s, const xlb_particles_t *p, double *out, cudaStream_t st) {
  int rc;
  if ((rc = grow(&s->moments, &s->moments_cap, beam_moments_scratch_words(p->n))) != XLB_OK) return rc;
  XLB_CUDA(beam_moments_launch(p->x, p->px, p->y, p->py, p->zeta, p->delta,
                               reinterpret_cast<const long long *>(p->state), p->n, s->moments, out, st));
  return XLB_OK;
}

// The stores of one xlb_track_device_moments call: store k after t_k = start + k * skip turns.
struct MomentStores {
  xlb_moments_spec_t spec;
  double *out;
  long long k = 0;  // next store
  long long next_turn(long long num_turns) const { return moment_store_turn(spec, k, num_turns); }
  // takes every store due after `done` turns (t_k <= done <= num_turns)
  int take(Scratch *s, const xlb_particles_t *p, long long done, long long num_turns, cudaStream_t st) {
    int rc;
    while (next_turn(num_turns) <= done) {
      if ((rc = beam_moments(s, p, out + static_cast<size_t>(k) * XLB_MOMENT_WORDS, st)) != XLB_OK) return rc;
      ++k;
    }
    return XLB_OK;
  }
};

// Survivor list of slots 0..n-1 into idx_out and its length into *n_out, enqueued on `st`.
static int compact_alive(Scratch *s, const long long *state, long long n, int *idx_out, int *n_out,
                         cudaStream_t st) {
  if (n <= 0) {
    XLB_CUDA(cudaMemsetAsync(n_out, 0, sizeof(int), st));
    return XLB_OK;
  }
  const int nblocks = static_cast<int>((n + CP_THREADS * CP_ITEMS - 1) / (CP_THREADS * CP_ITEMS));
  int rc;
  if ((rc = grow(&s->block_sums, &s->nblocks_cap, nblocks)) != XLB_OK) return rc;
  compact_count<<<nblocks, CP_THREADS, 0, st>>>(state, n, s->block_sums);
  compact_scan<<<1, 1024, 0, st>>>(s->block_sums, nblocks, n_out);
  compact_scatter<<<nblocks, CP_THREADS, 0, st>>>(state, n, s->block_sums, idx_out);
  XLB_CUDA(cudaGetLastError());
  return XLB_OK;
}

// Re-compacts the survivors of slots 0..n-1 into s->idx and waits for their number.
static int recompact(Scratch *s, const long long *state, long long n, cudaStream_t st, long long *n_alive) {
  int rc;
  if ((rc = grow(&s->idx, &s->cap, n)) != XLB_OK) return rc;
  if ((rc = compact_alive(s, state, n, s->idx, s->n_active, st)) != XLB_OK) return rc;
  XLB_CUDA(cudaMemcpyAsync(&s->h_pinned[1], s->n_active, sizeof(int), cudaMemcpyDeviceToHost, st));
  XLB_CUDA(cudaStreamSynchronize(st));
  g_stats.compactions += 1;
  *n_alive = static_cast<int>(s->h_pinned[1]);
  return XLB_OK;
}

// ------------------------------------------------------------------ variant selection
// All kernel families (one variant table per translation unit), most specialised first.
typedef const Variant *(*TableFn)(int *);
static const TableFn kTables[] = {fast_lean_nc_lo_variants, fast_lean_nc_variants, fast_lean_variants,
                                  fast_bf_nc_lo_variants,   fast_bf_variants,      fast_bf6_variants,
                                  strict_variants,          strict_bf_variants};
static const int kNumTables = static_cast<int>(sizeof(kTables) / sizeof(kTables[0]));

// What a call asks of a kernel family.
struct Need {
  bool strict, beamfields, bb6d, chi, trace, polygons;
  int max_order;  // highest multipole order the lattice may hold (255 = unknown)
  bool radiation;
};
static bool admits(const Variant &v, const Need &q) {
  if ((v.strict != 0) != q.strict) return false;
  if ((v.radiation != 0) != q.radiation) return false;  // the twins with the MULTIPOLE_RAD case
  // the twins with the LIMIT_POLYGON and EXCITER cases (the radiation twins carry them as well)
  if (!q.radiation && (v.polygons != 0) != q.polygons) return false;
  if (q.strict) return (v.beamfields != 0) == q.beamfields;
  const int bf = q.beamfields ? (q.bb6d ? 2 : 1) : 0;
  if (v.beamfields != bf) return false;
  if (v.nochi && q.chi) return false;
  if (v.maxorder && q.max_order > v.maxorder) return false;
  return true;
}
// The first (most specialised) admissible family that has the requested particles-per-thread;
// failing that, the closest particles-per-thread of the most specialised admissible family.
// Within a family: the variant with the smallest launch-bounds ceiling that still admits
// `threads` (tighter ceilings allow more registers).
static const Variant *pick_variant(const Need &q, int ppt, int threads) {
  const Variant *fallback = nullptr;
  for (int t = 0; t < kNumTables; ++t) {
    int n = 0;
    const Variant *tab = kTables[t](&n);
    const Variant *best = nullptr;
    for (int i = 0; i < n; ++i) {
      const Variant &v = tab[i];
      if (!admits(v, q)) continue;
      if (q.trace) {
        if (v.trace) return &v;
        continue;
      }
      if (v.trace) continue;
      if (!best) { best = &v; continue; }
      const int dv = std::abs(v.ppt - ppt), db = std::abs(best->ppt - ppt);
      if (dv < db) { best = &v; continue; }
      if (dv > db) continue;
      const bool vfit = v.threads >= threads, bfit = best->threads >= threads;
      if (vfit && (!bfit || v.threads < best->threads)) best = &v;
      if (!vfit && !bfit && v.threads > best->threads) best = &v;
    }
    if (!best) continue;
    if (best->ppt == ppt && best->threads >= threads) return best;
    if (!fallback) fallback = best;
  }
  return fallback;
}

// A variant, its CTA size, the CTAs the device holds at once and its registers per thread.
struct Shape {
  const Variant *v;
  int threads, resident, regs;
};
// The shape of a launch over the `n_now` particles still in the beam: a small (or scraped-down)
// beam is spread over all SMs first -- fewer particles per thread as long as the CTAs of the
// preferred shape would leave CTA slots empty (strong scaling, C1, the heavy-loss C2 beam).  All
// variants give the same bits, so the choice is invisible in the results.
static int choose(const Need &q, const xlb_track_options_t &o, int sms, size_t smem, long long n_now,
                  Shape *out) {
  const LaunchRequest r =
      launch_request(o.particles_per_thread, o.threads_per_block, q.strict, q.beamfields, q.chi, n_now, sms);
  const Variant *v = pick_variant(q, r.ppt, r.threads);
  if (!v) return fail(XLB_EINVAL, "no kernel variant compiled for this lattice");
  const int threads =
      q.trace ? v->threads : (o.threads_per_block > 0 ? o.threads_per_block : std::min(v->threads, r.threads));
  if (threads % 32 || threads > v->threads)
    return fail(XLB_EINVAL, "threads_per_block must be a multiple of 32 and <= the variant's limit");
  XLB_CUDA(cudaFuncSetAttribute(v->func, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
  cudaFuncAttributes fa;
  XLB_CUDA(cudaFuncGetAttributes(&fa, v->func));
  int occ = 1;
  XLB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, v->func, threads, smem));
  *out = {v, threads, std::max(1, occ) * sms, fa.numRegs};
  return XLB_OK;
}

static int launch(const Variant &v, const KArgs &a, int grid, int threads, size_t smem, cudaStream_t st) {
  void *args[] = {const_cast<KArgs *>(&a)};
  XLB_CUDA(cudaLaunchKernel(v.func, dim3(grid), dim3(threads), args, smem, st));
  return XLB_OK;
}

static int check_lattice_header(const xlb_lattice_t *lat) {
  if (!lat || !lat->words) return fail(XLB_EINVAL, "lattice is null");
  if (lat->chunk_words < 4 || (lat->chunk_words & 1))
    return fail(XLB_ELATTICE, "chunk_words must be even and >= 4");
  if (static_cast<long long>(lat->chunk_words) * 8 > 96 * 1024)
    return fail(XLB_ELATTICE, "chunk larger than 96 KiB");
  if (lat->n_chunks < 1) return fail(XLB_ELATTICE, "n_chunks < 1");
  const int64_t chunk_region = static_cast<int64_t>(lat->chunk_words) * lat->n_chunks;
  if (lat->flags & XLB_F_EXCITER) {  // the chunks, then the exciters' data region
    if (lat->n_words < chunk_region) return fail(XLB_ELATTICE, "n_words < chunk_words * n_chunks");
  } else if (lat->n_words != chunk_region) {
    return fail(XLB_ELATTICE, "n_words != chunk_words * n_chunks");
  }
  if (reinterpret_cast<uintptr_t>(lat->words) & 15)
    return fail(XLB_ELATTICE, "lattice words must be 16-byte aligned");
  if (lat->n_segments < 0 || (lat->n_segments > 0 && !lat->segments))
    return fail(XLB_ELATTICE, "bad segment table");
  int next = 0;
  for (int k = 0; k < lat->n_segments; ++k) {
    const int32_t *sg = lat->segments + 3 * k;
    if (sg[0] != next || sg[1] < 1) return fail(XLB_ELATTICE, "segments must tile the chunks in order");
    if (sg[2] != XLB_SEG_MAIN && sg[2] != XLB_SEG_BB6D) return fail(XLB_ELATTICE, "unknown segment kind");
    if (sg[2] == XLB_SEG_BB6D && (sg[1] != 1 || !(lat->flags & XLB_F_BB6D) || (lat->flags & XLB_F_STRICT)))
      return fail(XLB_ELATTICE, "a 6D-lens segment is one chunk of a fast lattice flagged XLB_F_BB6D");
    next += sg[1];
  }
  if (lat->n_segments > 0) {
    if (next != lat->n_chunks) return fail(XLB_ELATTICE, "segments do not cover all chunks");
    if (lat->segments[3 * (lat->n_segments - 1) + 2] != XLB_SEG_MAIN)
      return fail(XLB_ELATTICE, "the last segment must be a MAIN segment");
  }
  return XLB_OK;
}

static int check_particles(const xlb_particles_t *p) {
  if (!p) return fail(XLB_EINVAL, "particles is null");
  if (p->n < 0) return fail(XLB_EINVAL, "negative particle count");
  if (p->n > 2147483647LL) return fail(XLB_EINVAL, "more than 2^31-1 particles per call");
  if (p->n == 0) return XLB_OK;
  if (!p->x || !p->px || !p->y || !p->py || !p->zeta || !p->delta || !p->rpp || !p->rvv ||
      !p->s || !p->state || !p->at_element || !p->at_turn || !p->particle_id)
    return fail(XLB_EINVAL, "a required particle column is null");
  if (!(p->beta0 > 0) || !(p->energy0 > 0) || !(p->p0c > 0))
    return fail(XLB_EINVAL, "reference particle (p0c, beta0, energy0) must be positive");
  return XLB_OK;
}

// The arguments of a tracking call; a call without particles or turns has nothing more to check.
static int check_call(const xlb_lattice_t *lat, const xlb_particles_t *p, const xlb_track_options_t *o,
                      const MomentStores *stores) {
  int rc;
  if ((rc = check_lattice_header(lat)) != XLB_OK) return rc;
  if ((rc = check_particles(p)) != XLB_OK) return rc;
  if (!o) return fail(XLB_EINVAL, "options is null");
  if (o->num_turns < 0) return fail(XLB_EINVAL, "num_turns < 0");
  if (stores && o->trace) return fail(XLB_EINVAL, "beam-moment stores do not combine with a trace");
  if (p->n == 0 || o->num_turns == 0) return XLB_OK;
  if (o->trace && (o->num_turns != 1 || o->trace_particles < 1))
    return fail(XLB_EINVAL, "element-by-element trace needs num_turns == 1 and trace_particles >= 1");
  if (lat->n_segments > 1 && (o->trace || (lat->flags & XLB_F_STRICT)))
    return fail(XLB_EINVAL, "segmented lattices are for the fast kernels without trace");
  if ((lat->flags & XLB_F_EXCITER) && ((lat->flags & XLB_F_STRICT) || lat->n_segments > 0))
    return fail(XLB_ELATTICE, "exciter: a strict or segmented lattice cannot carry exciters");
  if (lat->flags & XLB_F_RADIATION) {
    if (lat->flags & (XLB_F_STRICT | XLB_F_BEAMFIELDS | XLB_F_BB6D))
      return fail(XLB_ELATTICE, "radiation: a strict or beam-field lattice cannot carry radiating multipoles");
    if (p->chi) return fail(XLB_EINVAL, "radiation: one species only (a chi column was given)");
    if (o->element_index_offset < 0 ||
        o->element_index_offset + static_cast<int64_t>(lat->n_elements) > XLB_RAD_MAX_ELEMENTS)
      return fail(XLB_EINVAL, "radiation: element_index_offset + n_elements exceeds 2^24");
  }
  return XLB_OK;
}

// The kernel arguments of a call, over all its particles (a launch over the survivors sets a.n and
// a.idx).
static KArgs kernel_args(const xlb_lattice_t *lat, const xlb_particles_t *p, const xlb_track_options_t *o,
                         unsigned int *n_lost) {
  KArgs a;
  memset(&a, 0, sizeof(a));
  a.lat = lat->words;
  a.chunk_words = lat->chunk_words;
  a.n_chunks = lat->n_chunks;
  a.n = p->n;
  a.x = p->x; a.px = p->px; a.y = p->y; a.py = p->py; a.zeta = p->zeta; a.delta = p->delta;
  a.rpp = p->rpp; a.rvv = p->rvv; a.s = p->s; a.chi = p->chi; a.qr = p->charge_ratio;
  a.state = reinterpret_cast<long long *>(p->state);
  a.at_element = reinterpret_cast<long long *>(p->at_element);
  a.at_turn = reinterpret_cast<long long *>(p->at_turn);
  a.pid = reinterpret_cast<const long long *>(p->particle_id);
  a.q0 = p->q0; a.p0c = p->p0c; a.beta0 = p->beta0; a.energy0 = p->energy0;
  a.sc_common = p->q0 * p->q0 * (1.0 - p->beta0 * p->beta0) / (p->p0c * p->beta0);
  a.loss_tally = reinterpret_cast<long long *>(o->loss_tally);
  a.mon = o->monitor_data;
  a.mon_words = o->monitor_words;
  a.n_lost = n_lost;
  a.trace = o->trace;
  a.trace_n = o->trace_particles;
  a.elem_off = static_cast<int>(o->element_index_offset);
  a.count_turns = (o->flags & XLB_OPT_NO_TURN_COUNT) ? 0 : 1;
  return a;
}

// Enqueues `turns` turns of the a.n particles (survivor list a.idx) in the shape `sh`, and sets
// the launch stats.  `tpi`: turns per work item of the persistent queue, <= 0 = no queue.
static int enqueue_turns(const xlb_lattice_t *lat, KArgs a, const Shape &sh, int turns, int tpi, size_t smem,
                         int sms, Scratch *s, cudaStream_t st) {
  const long long per_block = static_cast<long long>(sh.threads) * sh.v->ppt;
  const int blocks = static_cast<int>((a.n + per_block - 1) / per_block);
  g_stats.blocks = blocks;
  g_stats.threads = sh.threads;
  a.num_turns = turns;
  a.queue = nullptr;
  a.n_blocks = static_cast<unsigned int>(blocks);
  a.n_items = static_cast<unsigned int>(blocks);
  a.turns_per_item = turns;
  if (lat->n_segments > 1) {
    // turn by turn, segment by segment: tracking kernel up to the next 6D lens, the lens
    // kernel, and so on; the closing MAIN segment counts the turn
    const int count_turns = a.count_turns;
    a.num_turns = 1;
    a.turns_per_item = 1;
    const int lens_threads = 128;
    const int lens_blocks = static_cast<int>((a.n + lens_threads - 1) / lens_threads);
    int rc;
    for (int t = 0; t < turns; ++t) {
      for (int k = 0; k < lat->n_segments; ++k) {
        const int32_t *sg = lat->segments + 3 * k;
        const uint64_t *first = lat->words + static_cast<size_t>(sg[0]) * lat->chunk_words;
        if (sg[2] == XLB_SEG_BB6D) {
          fast_bb6d_launch(a, reinterpret_cast<const unsigned long long *>(first), lens_blocks, lens_threads, st);
        } else {
          a.lat = first;
          a.n_chunks = sg[1];
          a.count_turns = (k == lat->n_segments - 1) ? count_turns : 0;
          if ((rc = launch(*sh.v, a, blocks, sh.threads, smem, st)) != XLB_OK) return rc;
        }
        g_stats.kernel_launches += 1;
      }
    }
    XLB_CUDA(cudaGetLastError());
    return XLB_OK;
  }
  int grid = blocks;
  if (tpi > 0 && turns > tpi && blocks > sms) {
    // persistent CTAs + a device-side ring of ready (block, turn segment) items (track_impl.cuh).
    // Also when every CTA could be resident at once (sms < blocks <= resident): SMs would hold
    // different numbers of CTAs, a CTA on a fuller SM runs slower, and with one item per CTA
    // the launch lasts as long as its slowest CTA.
    const long long segs = (turns + tpi - 1) / tpi;
    if (static_cast<long long>(blocks) * segs < (1LL << 26)) {  // ring of at most 512 MiB
      // two counters + one 64-bit ready entry per item beyond the first segment of every block
      const size_t qwords = 2 + 2 * static_cast<size_t>(blocks) * static_cast<size_t>(segs - 1);
      int rc;
      if ((rc = grow(&s->queue, &s->queue_cap, qwords)) != XLB_OK) return rc;
      XLB_CUDA(cudaMemsetAsync(s->queue, 0, qwords * sizeof(unsigned int), st));
      a.queue = s->queue;
      a.n_items = static_cast<unsigned int>(blocks * segs);
      a.turns_per_item = tpi;
      grid = persistent_grid(blocks, sh.resident, sms);
    }
  }
  g_stats.kernel_launches += 1;
  return launch(*sh.v, a, grid, sh.threads, smem, st);
}

// `stores` (optional): beam-moment stores taken on the stream after the launch that ends on their
// turn; launches are cut at the store turns.
static int track_device_impl(const xlb_lattice_t *lat, xlb_particles_t *p,
                             const xlb_track_options_t *o, cudaStream_t st, bool timed,
                             MomentStores *stores = nullptr) {
  memset(&g_stats, 0, sizeof(g_stats));
  int rc;
  if ((rc = check_call(lat, p, o, stores)) != XLB_OK) return rc;
  const bool empty = p->n == 0 || o->num_turns == 0;
  if (empty && !stores) return XLB_OK;
  const bool split = lat->n_segments > 1;  // 6D lenses run as kernels of their own
  const Need need{(lat->flags & XLB_F_STRICT) != 0, (lat->flags & XLB_F_BEAMFIELDS) != 0,
                  (lat->flags & XLB_F_BB6D) != 0 && !split, p->chi != nullptr, o->trace != nullptr,
                  (lat->flags & (XLB_F_POLYGONS | XLB_F_EXCITER)) != 0, (lat->flags & XLB_F_LOW_ORDER) ? 3 : 255,
                  (lat->flags & XLB_F_RADIATION) != 0};
  const size_t smem = XLB_STAGES * static_cast<size_t>(lat->chunk_words) * 8 +
                      (2 * XLB_STAGES + 2) * sizeof(unsigned long long);
  int dev = 0, sms = 0;
  Shape shape{};
  if (!empty) {
    XLB_CUDA(cudaGetDevice(&dev));
    XLB_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    if ((rc = choose(need, *o, sms, smem, p->n, &shape)) != XLB_OK) return rc;  // validates the caller's shape
  }
  CallScope call;
  if ((rc = call.open(st)) != XLB_OK) return rc;
  Scratch *s = call.s;
  if (empty) return stores->take(s, p, o->num_turns, o->num_turns, st);

  KArgs a = kernel_args(lat, p, o, s->n_lost);
  // Work-item length.  An item costs a load and a store of its block's particles and a ticket
  // (microseconds); a shorter item leaves a shorter tail at the end of a launch (the last, partly
  // filled round of items) and rotates the blocks faster.  Automatic: one turn when a turn streams
  // 16 chunks or more (LHC: 121, C2 at 250 k particles +3 %, at 1 M +1 % over five turns), else
  // as many turns as make 16 chunks (PS Booster: 6).
  const int tpi = (o->turns_per_item == 0) ? std::max(1, (16 + lat->n_chunks - 1) / lat->n_chunks)
                                           : o->turns_per_item;
  const int seg = launch_cap(o->turns_per_launch, o->num_turns, lat->n_chunks);
  const double thr = (o->compact_threshold > 0) ? o->compact_threshold : (1.0 / 128.0);
  long long n_active = p->n;
  long long lost_since_compact = 0;
  const bool segmented = seg < o->num_turns;
  if (segmented || stores) XLB_CUDA(cudaMemsetAsync(s->n_lost, 0, sizeof(unsigned int), st));
  // Launch-length ramp: a beam that is scraped hard in its first turns (SURVEY 8(d): 80 % of the
  // C2 beam within a few turns) would keep those lanes idle for a whole launch.  A segmented job
  // on a particle set not seen before starts with a launch of ONE turn; after every launch the
  // loss rate per turn just measured sets the next length (at most twice the previous one, at
  // most `seg`), and survivors are re-compacted as before.  A call that continues with the
  // particle set of the previous call starts from the rate that call ended with.  The schedule
  // never changes results (a launch boundary is invisible to the particles).
  const bool ramp = segmented && p->n >= 32768;
  int cur_len = seg;
  if (ramp) {
    const bool continuing = (s->sched_x == p->x && s->sched_n == p->n && s->sched_rate >= 0.0);
    cur_len = continuing ? launch_length_for_rate(s->sched_rate, seg) : 1;
  }
  double last_rate = -1.0;

  if (timed) XLB_CUDA(cudaEventRecord(s->ev0, st));
  if (o->turns_per_launch > 0 || segmented) {
    // particles lost in earlier calls still sit in the caller's arrays (state 0): start from
    // the compacted survivor list so they do not occupy lanes
    long long alive = 0;
    if ((rc = recompact(s, a.state, p->n, st, &alive)) != XLB_OK) return rc;
    if (alive < p->n) {
      a.n = n_active = alive;
      a.idx = s->idx;
    }
  }
  long long lost_before_launch = 0;
  if (stores && (rc = stores->take(s, p, 0, o->num_turns, st)) != XLB_OK) return rc;
  for (int done = 0; done < o->num_turns && n_active > 0;) {
    int turns = std::min(ramp ? cur_len : seg, o->num_turns - done);
    if (stores) turns = static_cast<int>(std::min<long long>(turns, stores->next_turn(o->num_turns) - done));
    if ((rc = choose(need, *o, sms, smem, n_active, &shape)) != XLB_OK) return rc;
    if ((rc = enqueue_turns(lat, a, shape, turns, tpi, smem, sms, s, st)) != XLB_OK) return rc;
    done += turns;
    if (stores && (rc = stores->take(s, p, done, o->num_turns, st)) != XLB_OK) return rc;
    if (done >= o->num_turns) break;
    // survivors: read the loss counter; re-compact when enough lanes went idle
    XLB_CUDA(cudaMemcpyAsync(&s->h_pinned[0], s->n_lost, sizeof(unsigned int), cudaMemcpyDeviceToHost, st));
    XLB_CUDA(cudaStreamSynchronize(st));
    const long long lost_total = s->h_pinned[0];
    if (ramp) {
      last_rate = static_cast<double>(lost_total - lost_before_launch) /
                  (static_cast<double>(n_active) * static_cast<double>(turns));
      cur_len = ramp_step(last_rate, seg, cur_len);
    }
    lost_before_launch = lost_total;
    const long long newly = lost_total - lost_since_compact;
    if (newly > 0 && static_cast<double>(newly) >= thr * static_cast<double>(n_active)) {
      if ((rc = recompact(s, a.state, p->n, st, &n_active)) != XLB_OK) return rc;
      a.n = n_active;
      a.idx = s->idx;
      lost_since_compact = lost_total;
    }
  }
  // a beam lost entirely before num_turns: the remaining stores see it empty
  if (stores && (rc = stores->take(s, p, o->num_turns, o->num_turns, st)) != XLB_OK) return rc;
  float total_ms = 0.f;
  if (timed) {
    XLB_CUDA(cudaEventRecord(s->ev1, st));
    XLB_CUDA(cudaEventSynchronize(s->ev1));
    XLB_CUDA(cudaEventElapsedTime(&total_ms, s->ev0, s->ev1));
  }
  if (ramp) {
    s->sched_x = p->x;
    s->sched_n = p->n;
    if (last_rate >= 0.0) s->sched_rate = last_rate;
    else if (!(s->sched_rate >= 0.0)) s->sched_rate = 0.0;
  }
  g_stats.kernel_ms = total_ms;
  g_stats.regs_per_thread = shape.regs;
  g_stats.smem_bytes = static_cast<int>(smem);
  g_stats.n_alive_in = p->n;
  g_stats.n_alive_out = n_active;
  return XLB_OK;
}

// ------------------------------------------------------------------ FP64 peak probe
template <int CHAINS>
__global__ void __launch_bounds__(256) dfma_peak_kernel(double *out, int iters, double a, double b) {
  double acc[CHAINS];
#pragma unroll
  for (int c = 0; c < CHAINS; ++c) acc[c] = threadIdx.x * 1e-3 + c;
  for (int i = 0; i < iters; ++i) {
#pragma unroll
    for (int c = 0; c < CHAINS; ++c) acc[c] = fma(acc[c], a, b);
  }
  double t = 0;
#pragma unroll
  for (int c = 0; c < CHAINS; ++c) t += acc[c];
  if (t == 123.456) out[0] = t;  // keep the chains alive
}

// One warp, CHAINS independent dependent-DFMA chains: cycles per DFMA (clock64).  CHAINS = 1
// gives the dependent-issue latency, larger CHAINS the single-warp throughput.
template <int CHAINS>
__global__ void dfma_latency_kernel(double *out, long long *cycles, int iters, double a, double b) {
  double acc[CHAINS];
#pragma unroll
  for (int c = 0; c < CHAINS; ++c) acc[c] = threadIdx.x * 1e-3 + c;
  const long long t0 = clock64();
  for (int i = 0; i < iters; ++i) {
#pragma unroll
    for (int c = 0; c < CHAINS; ++c) acc[c] = fma(acc[c], a, b);
  }
  const long long t1 = clock64();
  double t = 0;
#pragma unroll
  for (int c = 0; c < CHAINS; ++c) t += acc[c];
  if (threadIdx.x == 0) *cycles = t1 - t0;
  if (t == 123.456) out[0] = t;
}

template <int CHAINS>
static int run_latency(double *d, long long *dc, double *cyc_per_dfma) {
  const int iters = 1 << 14;
  dfma_latency_kernel<CHAINS><<<1, 32>>>(d, dc, iters, 1.0000001, 1e-9);
  dfma_latency_kernel<CHAINS><<<1, 32>>>(d, dc, iters, 1.0000001, 1e-9);
  long long h = 0;
  XLB_CUDA(cudaMemcpy(&h, dc, sizeof(h), cudaMemcpyDeviceToHost));
  *cyc_per_dfma = static_cast<double>(h) / (static_cast<double>(iters) * CHAINS);
  return XLB_OK;
}

}  // namespace xlb

using namespace xlb;

extern "C" {

int xlb_abi_version(void) { return XLB_ABI_VERSION; }
const char *xlb_last_error(void) { return g_err.c_str(); }

int xlb_get_stats(xlb_track_stats_t *out) {
  if (!out) return fail(XLB_EINVAL, "out is null");
  *out = g_stats;
  return XLB_OK;
}

int xlb_lattice_validate(const xlb_lattice_t *lat) {
  int rc = check_lattice_header(lat);
  if (rc != XLB_OK) return rc;
  bool saw_end_turn = false;
  // last chunk of every segment (of the lattice when it is not segmented) and the chunks
  // that belong to 6D-lens segments
  std::vector<char> seg_last(lat->n_chunks, 0), lens_chunk(lat->n_chunks, 0);
  seg_last[lat->n_chunks - 1] = 1;
  for (int k = 0; k < lat->n_segments; ++k) {
    const int32_t *sg = lat->segments + 3 * k;
    seg_last[sg[0] + sg[1] - 1] = 1;
    if (sg[2] == XLB_SEG_BB6D) lens_chunk[sg[0]] = 1;
  }
  for (int c = 0; c < lat->n_chunks; ++c) {
    const uint64_t *w = lat->words + static_cast<size_t>(c) * lat->chunk_words;
    int pos = 0;
    bool closed = false;
    while (pos < lat->chunk_words) {
      const uint64_t hdr = w[pos];
      const int tag = static_cast<int>(hdr & 0xff);
      const int aux = static_cast<int>((hdr >> 8) & 0xff);
      const int pairs = static_cast<int>((hdr >> 16) & 0x3fff);
      const bool hdr_a1 = (hdr & XLB_HDR_HAS_A1) != 0;
      const bool hx_only = ((hdr >> 31) & 1) != 0;  // XLB_HDR_HX_ONLY
      int want = -1;  // expected record length in pairs, -1 = variable
      switch (tag) {
        case XLB_T_END_TURN:
          if (!seg_last[c]) return fail(XLB_ELATTICE, "END_TURN before the last chunk");
          saw_end_turn = true;
          closed = true;
          break;
        case XLB_T_END_CHUNK:
          if (seg_last[c]) return fail(XLB_ELATTICE, "last chunk must end with END_TURN");
          closed = true;
          break;
        case XLB_T_DRIFT:
        case XLB_T_DRIFT_EXACT: want = 1; break;
        case XLB_T_MULTIPOLE:
        case XLB_T_MULTIPOLE_CURVED:
          want = (tag == XLB_T_MULTIPOLE ? 1 : 3) + aux + 1;
          if ((lat->flags & XLB_F_LOW_ORDER) && aux > 3)
            return fail(XLB_ELATTICE, "XLB_F_LOW_ORDER set but a multipole has order > 3");
          break;
        case XLB_T_CAVITY:
        case XLB_T_SAWTOOTH_CAVITY:
        case XLB_T_XYSHIFT:
        case XLB_T_SROTATION:
        case XLB_T_DIPOLE_EDGE: want = 2; break;
        case XLB_T_RFMULTIPOLE: want = 2 + 2 * (aux + 1); break;
        case XLB_T_LIMIT_RECT:
        case XLB_T_LIMIT_ELLIPSE: want = 3 + ((aux & XLB_AUX_DRIFT) ? 1 : 0); break;
        case XLB_T_LIMIT_RECT_ELLIPSE: want = 4 + ((aux & XLB_AUX_DRIFT) ? 1 : 0); break;
        case XLB_T_LIMIT_POLYGON: {  // [hdr,n_edges][s_here,drift] then [y_lo,y_hi][x_lo,slope] per edge
          const int64_t n_edges = static_cast<int64_t>(w[pos + 1]);
          if (!(lat->flags & XLB_F_POLYGONS)) return fail(XLB_ELATTICE, "polygon record without XLB_F_POLYGONS");
          if (n_edges < 1 || n_edges > lat->chunk_words || 2 + 2 * n_edges != pairs)
            return fail(XLB_ELATTICE, "polygon record: n_edges < 1 or size != 2 + 2 * n_edges pairs");
          if (pos + 2 * pairs + 2 > lat->chunk_words)
            return fail(XLB_ELATTICE, "record runs past the end of its chunk");
          for (int64_t e = 0; e < n_edges; ++e) {
            double v[4];
            memcpy(v, &w[pos + 4 + 4 * e], sizeof v);
            if (!(std::isfinite(v[0]) && std::isfinite(v[1]) && std::isfinite(v[2]) && std::isfinite(v[3])))
              return fail(XLB_ELATTICE, "polygon record: non-finite edge word");
            if (!(v[0] < v[1])) return fail(XLB_ELATTICE, "polygon record: edge with y_lo >= y_hi");
          }
          want = pairs;
          break;
        }
        case XLB_T_MULTIPOLE_RAD: {  // [hdr,mode][L,1/L][K_e,hbar_c][alpha,seed] + MULTIPOLE(_CURVED) record
          if (!(lat->flags & XLB_F_RADIATION)) return fail(XLB_ELATTICE, "radiating multipole without XLB_F_RADIATION");
          if ((lat->flags & XLB_F_LOW_ORDER) && aux > 3)
            return fail(XLB_ELATTICE, "XLB_F_LOW_ORDER set but a multipole has order > 3");
          if (pos + 10 > lat->chunk_words) return fail(XLB_ELATTICE, "record runs past the end of its chunk");
          const int64_t mode = static_cast<int64_t>(w[pos + 1]);
          if (mode != XLB_RAD_MEAN && mode != XLB_RAD_QUANTUM) return fail(XLB_ELATTICE, "radiating multipole: bad mode");
          double v[5];
          memcpy(v, &w[pos + 2], sizeof v);  // L, 1/L, K_e, hbar_c, alpha
          for (double x : v)
            if (!(std::isfinite(x) && x > 0)) return fail(XLB_ELATTICE, "radiating multipole: L, 1/L and the constants must be finite and > 0");
          const uint64_t sub = w[pos + 8];
          const int st = static_cast<int>(sub & 0xff), saux = static_cast<int>((sub >> 8) & 0xff);
          const int spairs = static_cast<int>((sub >> 16) & 0x3fff);
          if ((st != XLB_T_MULTIPOLE && st != XLB_T_MULTIPOLE_CURVED) || saux != aux ||
              spairs != (st == XLB_T_MULTIPOLE ? 1 : 3) + aux + 1 || (sub & 0xc0000000u))
            return fail(XLB_ELATTICE, "radiating multipole: the embedded record is not a multipole of the same order");
          want = 4 + spairs;
          break;
        }
        case XLB_T_EXCITER: {  // [hdr,A][B,start_turn][n_samples,data_offset] + (kn_i,ks_i) i=order..0
          if (!(lat->flags & XLB_F_EXCITER)) return fail(XLB_ELATTICE, "exciter record without XLB_F_EXCITER");
          if ((lat->flags & XLB_F_LOW_ORDER) && aux > 3)
            return fail(XLB_ELATTICE, "XLB_F_LOW_ORDER set but an exciter has order > 3");
          if (pos + 6 > lat->chunk_words) return fail(XLB_ELATTICE, "record runs past the end of its chunk");
          double ab[2];
          memcpy(&ab[0], &w[pos + 1], sizeof(double));
          memcpy(&ab[1], &w[pos + 2], sizeof(double));
          if (!(std::isfinite(ab[0]) && std::isfinite(ab[1]))) return fail(XLB_ELATTICE, "exciter: A or B not finite");
          const int64_t n_samples = static_cast<int64_t>(w[pos + 4]), off = static_cast<int64_t>(w[pos + 5]);
          const int64_t chunk_region = static_cast<int64_t>(lat->chunk_words) * lat->n_chunks;
          if (n_samples < 0 || off < chunk_region || off > lat->n_words || n_samples > lat->n_words - off)
            return fail(XLB_ELATTICE, "exciter: the samples are not inside the data region");
          for (int64_t k = 0; k < n_samples; ++k) {
            double v;
            memcpy(&v, &lat->words[off + k], sizeof v);
            if (!std::isfinite(v)) return fail(XLB_ELATTICE, "exciter: non-finite sample");
          }
          want = 3 + aux + 1;
          break;
        }
        case XLB_T_MONITOR: want = 5; break;
        case XLB_T_BEAMBEAM4D:
        case XLB_T_SPACECHARGE:
        case XLB_T_BEAMBEAM6D:
          if (lens_chunk[c]) {
            if (tag != XLB_T_BEAMBEAM6D || pos != 0)
              return fail(XLB_ELATTICE, "a 6D-lens segment holds exactly one BEAMBEAM6D record");
          } else {
            if (!(lat->flags & XLB_F_BEAMFIELDS))
              return fail(XLB_ELATTICE, "beam-field record without XLB_F_BEAMFIELDS");
            if (tag == XLB_T_BEAMBEAM6D && lat->n_segments > 1)
              return fail(XLB_ELATTICE, "BEAMBEAM6D record in a MAIN segment of a segmented lattice");
          }
          if (tag == XLB_T_BEAMBEAM6D && !(lat->flags & XLB_F_BB6D))
            return fail(XLB_ELATTICE, "BeamBeam6D record without XLB_F_BB6D");
          if (pairs < 6) return fail(XLB_ELATTICE, "bad beam-field record length");
          break;
        default: {
          if ((tag & 0xc0) == XLB_T_EDGE_BLOCK) {
            want = 2;
            break;
          }
          if ((tag & 0xc0) == XLB_T_THIN_BLOCK && (lat->flags & XLB_F_LOW_ORDER) && aux > 3)
            return fail(XLB_ELATTICE, "XLB_F_LOW_ORDER set but a block record has order > 3");
          if ((tag & 0xe0) == XLB_T_THIN_BLOCK) {
            want = 2 + aux + 1 + ((tag & 4) ? 2 : 0) + ((tag & 3) ? 2 : 0);
            break;
          }
          if ((tag & 0xe0) == XLB_T_MERGED_BLOCK) {
            if (lat->flags & XLB_F_STRICT) return fail(XLB_ELATTICE, "merged block in a strict lattice");
            const int64_t f = static_cast<int64_t>(w[pos + 3]);
            if ((((f >> 8) & 1) != 0) != hdr_a1)
              return fail(XLB_ELATTICE, "merged block: XLB_HDR_HAS_A1 disagrees with the record");
            want = 2 + aux + 1 + ((tag & 4) ? 3 : 0) + (((f >> 8) & 1) ? 2 : 0) + ((tag & 3) ? 2 : 0) +
                   static_cast<int>(f & 0xff) + 1 + 1;  // ... K1's pairs, [path length, 0]
            break;
          }
          char buf[96];
          snprintf(buf, sizeof buf, "unknown tag %d in chunk %d at word %d", tag, c, pos);
          return fail(XLB_ELATTICE, buf);
        }
      }
      if (hdr_a1 && (tag & 0xe0) != XLB_T_MERGED_BLOCK)
        return fail(XLB_ELATTICE, "XLB_HDR_HAS_A1 on a record that is not a merged block");
      if (hx_only) {  // only on curved block records of the fast encoding, and only when hyl == 0
        const bool block = (tag & 0xc0) == XLB_T_THIN_BLOCK && (tag & 4);
        if (!block || (lat->flags & XLB_F_STRICT))
          return fail(XLB_ELATTICE, "XLB_HDR_HX_ONLY on a record that is not a curved block of the fast encoding");
        double hyl;
        memcpy(&hyl, &w[pos + 2 * (2 + aux + 1) + 1], sizeof hyl);
        if (hyl != 0.0) return fail(XLB_ELATTICE, "XLB_HDR_HX_ONLY set but hyl != 0");
      }
      if (lens_chunk[c] && tag != XLB_T_BEAMBEAM6D && tag != XLB_T_END_TURN)
        return fail(XLB_ELATTICE, "a 6D-lens segment holds exactly one BEAMBEAM6D record");
      if (!closed && (pairs < 1 || (want >= 0 && pairs != want))) {
        char buf[112];
        snprintf(buf, sizeof buf, "record of tag %d in chunk %d at word %d has size %d, expected %d",
                 tag, c, pos, pairs, want);
        return fail(XLB_ELATTICE, buf);
      }
      if (!closed && pos + 2 * pairs + 2 > lat->chunk_words)
        return fail(XLB_ELATTICE, "record runs past the end of its chunk");
      if (closed) break;
      pos += 2 * pairs;
    }
    if (!closed) return fail(XLB_ELATTICE, "chunk not terminated by END_CHUNK/END_TURN");
  }
  if (!saw_end_turn) return fail(XLB_ELATTICE, "no END_TURN record");
  if ((lat->flags & XLB_F_EXCITER) && ((lat->flags & XLB_F_STRICT) || lat->n_segments > 0))
    return fail(XLB_ELATTICE, "exciter: a strict or segmented lattice cannot carry exciters");
  if (lat->flags & XLB_F_RADIATION) {
    if (lat->flags & XLB_F_STRICT) return fail(XLB_ELATTICE, "radiation: the strict encoding has no radiating multipoles");
    if (lat->flags & (XLB_F_BEAMFIELDS | XLB_F_BB6D))
      return fail(XLB_ELATTICE, "radiation: beam-field lattices cannot carry radiating multipoles");
    if (lat->n_elements > XLB_RAD_MAX_ELEMENTS) return fail(XLB_ELATTICE, "radiation: more than 2^24 elements");
  }
  return XLB_OK;
}

int xlb_track_device(const xlb_lattice_t *lattice, xlb_particles_t *particles,
                     const xlb_track_options_t *opts, void *stream) {
  return track_device_impl(lattice, particles, opts, static_cast<cudaStream_t>(stream), false);
}

int xlb_track_device_timed(const xlb_lattice_t *lattice, xlb_particles_t *particles,
                           const xlb_track_options_t *opts, void *stream) {
  return track_device_impl(lattice, particles, opts, static_cast<cudaStream_t>(stream), true);
}

int xlb_track_device_moments(const xlb_lattice_t *lattice, xlb_particles_t *particles,
                             const xlb_track_options_t *opts, const xlb_moments_spec_t *spec, double *out,
                             void *stream) {
  if (!spec) return fail(XLB_EINVAL, "moments spec is null");
  if (spec->num_stores < 0 || spec->start < 0 || spec->skip < 1)
    return fail(XLB_EINVAL, "moments spec needs num_stores >= 0, start >= 0, skip >= 1");
  if (spec->num_stores > 0 && !out) return fail(XLB_EINVAL, "moments out is null");
  MomentStores stores{*spec, out};
  return track_device_impl(lattice, particles, opts, static_cast<cudaStream_t>(stream), false, &stores);
}

int xlb_beam_moments_device(const xlb_particles_t *particles, double *out, void *stream) {
  int rc;
  if ((rc = check_particles(particles)) != XLB_OK) return rc;
  if (!out) return fail(XLB_EINVAL, "out is null");
  CallScope call;
  if ((rc = call.open(static_cast<cudaStream_t>(stream))) != XLB_OK) return rc;
  return beam_moments(call.s, particles, out, static_cast<cudaStream_t>(stream));
}

int xlb_naff_device(const double *u, const double *pu, int64_t n, int64_t num_turns, int64_t stride,
                    double beta, double alpha, double *tune_out, double *amplitude_out, void *stream) {
  if (n < 0) return fail(XLB_EINVAL, "n < 0");
  if (num_turns < XLB_NAFF_MIN_TURNS || num_turns > XLB_NAFF_MAX_TURNS)
    return fail(XLB_EINVAL, "num_turns outside [XLB_NAFF_MIN_TURNS, XLB_NAFF_MAX_TURNS]");
  if (stride < n) return fail(XLB_EINVAL, "stride < n");
  if (n > 0 && (!u || !tune_out || !amplitude_out)) return fail(XLB_EINVAL, "null pointer");
  if (pu && !(std::isfinite(beta) && beta > 0.0 && std::isfinite(alpha)))
    return fail(XLB_EINVAL, "beta must be finite and > 0, alpha finite");
  if (n > 2147483647LL) return fail(XLB_EINVAL, "n too large");
  if (n == 0) return XLB_OK;
  CallScope call;
  int rc;
  if ((rc = call.open(static_cast<cudaStream_t>(stream))) != XLB_OK) return rc;
  XLB_CUDA(naff_launch(u, pu, n, static_cast<int>(num_turns), stride, beta, alpha, tune_out, amplitude_out,
                       static_cast<cudaStream_t>(stream)));
  return XLB_OK;
}

// The argument checks of the tangent-map entry points (`what` names the call in messages).
// `radiation`: mean-mode radiating multipoles are allowed.
static int tangent_checks(const xlb_lattice_t *lat, xlb_particles_t *p, const xlb_track_options_t *o, bool radiation,
                          const char *what, int *threads) {
  int rc;
  if ((rc = check_call(lat, p, o, nullptr)) != XLB_OK) return rc;
  char buf[160];
  if (o->trace) {
    snprintf(buf, sizeof buf, "%s does not combine with a trace", what);
    return fail(XLB_EINVAL, buf);
  }
  if (!radiation && (lat->flags & XLB_F_RADIATION))
    return fail(XLB_EINVAL, "tangent tracking: radiating multipoles are not in the tangent map");
  if (lat->flags & XLB_F_STRICT) {
    snprintf(buf, sizeof buf, "%s needs a lattice in the fast encoding", what);
    return fail(XLB_EINVAL, buf);
  }
  if (lat->n_segments > 0) {
    snprintf(buf, sizeof buf, "%s needs an unsegmented lattice", what);
    return fail(XLB_EINVAL, buf);
  }
  if (o->particles_per_thread != 0 && o->particles_per_thread != 1) {
    snprintf(buf, sizeof buf, "%s runs one particle per thread", what);
    return fail(XLB_EINVAL, buf);
  }
  *threads = o->threads_per_block > 0 ? o->threads_per_block : 128;
  if (*threads % 32 || *threads > XLB_TANGENT_MAX_THREADS)
    return fail(XLB_EINVAL, "threads_per_block must be a multiple of 32 and <= XLB_TANGENT_MAX_THREADS");
  return XLB_OK;
}

// The kernels know one record per element: refuse the block records and the 6D lens (and, with
// radiation, quantum-mode radiating multipoles) up front, naming the element.
static int tangent_scan(const xlb_lattice_t *lat, bool radiation, const char *what, cudaStream_t st) {
  std::vector<uint64_t> w(static_cast<size_t>(lat->n_words));
  XLB_CUDA(cudaMemcpyAsync(w.data(), lat->words, w.size() * 8, cudaMemcpyDefault, st));
  XLB_CUDA(cudaStreamSynchronize(st));
  for (int c = 0; c < lat->n_chunks; ++c) {
    for (size_t pos = static_cast<size_t>(c) * lat->chunk_words; pos < static_cast<size_t>(c + 1) * lat->chunk_words;) {
      const uint64_t hdr = w[pos];
      const int tag = static_cast<int>(hdr & 0xff), pairs = static_cast<int>((hdr >> 16) & 0x3fff);
      if (tag == XLB_T_END_TURN || tag == XLB_T_END_CHUNK) break;
      if (tag == XLB_T_BEAMBEAM6D || tag >= XLB_T__COUNT) {
        char buf[160];
        snprintf(buf, sizeof buf, "%s: element %d is %s", what, static_cast<int>(hdr >> 32),
                 tag == XLB_T_BEAMBEAM6D ? "a BeamBeam6D lens (its Jacobian is not implemented)"
                 : tag == XLB_T_EXCITER  ? "an Exciter (a turn-dependent map has no tangent map or closed orbit)"
                                         : "a fused block record (pack one record per element)");
        return fail(XLB_EINVAL, buf);
      }
      if (radiation && tag == XLB_T_MULTIPOLE_RAD && static_cast<int64_t>(w[pos + 1]) != XLB_RAD_MEAN) {
        char buf[160];
        snprintf(buf, sizeof buf, "%s: element %d radiates in quantum mode (the tangent map and the envelope "
                 "take mean-mode records)", what, static_cast<int>(hdr >> 32));
        return fail(XLB_EINVAL, buf);
      }
      if (pairs < 1) return fail(XLB_ELATTICE, "record of size 0");
      pos += 2 * static_cast<size_t>(pairs);
    }
  }
  return XLB_OK;
}

// The three tangent-map entry points: the kernel of `mode` over the particles of p.  `jac` is J, or
// Sigma for the envelope; log2_scale and fli go with J, energy_loss with Sigma.
static int track_tangent_impl(const xlb_lattice_t *lat, xlb_particles_t *p, const xlb_track_options_t *o,
                              tangent::Mode mode, double *jac, int64_t *log2_scale, double *fli,
                              double *energy_loss, void *stream) {
  memset(&g_stats, 0, sizeof(g_stats));
  const bool envelope = mode == tangent::ENVELOPE, radiation = mode != tangent::TANGENT;
  const char *what = envelope ? "envelope tracking" : "tangent tracking";
  int rc, threads;
  if ((rc = tangent_checks(lat, p, o, radiation, what, &threads)) != XLB_OK) return rc;
  if (p->n == 0 || o->num_turns == 0) return XLB_OK;
  if (envelope && (!jac || !energy_loss)) return fail(XLB_EINVAL, "cov and energy_loss must not be null");
  if (!envelope && (!jac || !log2_scale || !fli))
    return fail(XLB_EINVAL, "jac, log2_scale and fli must not be null");
  const cudaStream_t st = static_cast<cudaStream_t>(stream);
  CallScope call;
  if ((rc = call.open(st)) != XLB_OK) return rc;
  if ((rc = tangent_scan(lat, radiation, what, st)) != XLB_OK) return rc;
  KArgs a = kernel_args(lat, p, o, call.s->n_lost);
  a.num_turns = o->num_turns;
  XLB_CUDA(tangent_launch(mode, a, jac, reinterpret_cast<long long *>(log2_scale), fli, energy_loss, threads, st));
  g_stats.kernel_launches = 1;
  g_stats.threads = threads;
  g_stats.blocks = static_cast<int>((p->n + threads - 1) / threads);
  g_stats.n_alive_in = p->n;
  return XLB_OK;
}

int xlb_track_tangent_device(const xlb_lattice_t *lat, xlb_particles_t *p, const xlb_track_options_t *o,
                             double *jac, int64_t *log2_scale, double *fli, void *stream) {
  return track_tangent_impl(lat, p, o, tangent::TANGENT, jac, log2_scale, fli, nullptr, stream);
}

int xlb_track_tangent_radiation_device(const xlb_lattice_t *lat, xlb_particles_t *p, const xlb_track_options_t *o,
                                       double *jac, int64_t *log2_scale, double *fli, void *stream) {
  return track_tangent_impl(lat, p, o, tangent::TANGENT_R, jac, log2_scale, fli, nullptr, stream);
}

int xlb_track_envelope_device(const xlb_lattice_t *lat, xlb_particles_t *p, const xlb_track_options_t *o,
                              double *cov, double *energy_loss, void *stream) {
  return track_tangent_impl(lat, p, o, tangent::ENVELOPE, cov, nullptr, nullptr, energy_loss, stream);
}

int xlb_compact_alive_device(const int64_t *state, int64_t n, int32_t *idx_out, int32_t *n_out,
                             void *stream) {
  if (n < 0 || (n > 0 && (!state || !idx_out)) || !n_out) return fail(XLB_EINVAL, "bad argument");
  if (n > 2147483647LL) return fail(XLB_EINVAL, "n too large");
  CallScope call;
  int rc;
  if ((rc = call.open(static_cast<cudaStream_t>(stream))) != XLB_OK) return rc;
  return compact_alive(call.s, reinterpret_cast<const long long *>(state), n, idx_out, n_out,
                       static_cast<cudaStream_t>(stream));
}

int xlb_track_host(const xlb_lattice_t *hl, xlb_particles_t *hp, const xlb_track_options_t *o) {
  int rc;
  if ((rc = check_lattice_header(hl)) != XLB_OK) return rc;
  if ((rc = check_particles(hp)) != XLB_OK) return rc;
  if (!o) return fail(XLB_EINVAL, "options is null");
  if ((rc = xlb_lattice_validate(hl)) != XLB_OK) return rc;
  if (o->trace) return fail(XLB_EINVAL, "element-by-element trace is a device-entry-point feature");
  const long long n = hp->n;
  if (n == 0 || o->num_turns == 0) return XLB_OK;
  Scratch *s = nullptr;
  if ((rc = get_scratch(&s)) != XLB_OK) return rc;
  const cudaStream_t st = s->stream;
  CallScope call;
  if ((rc = call.open(st)) != XLB_OK) return rc;

  xlb_particles_t dp = *hp;
  xlb_track_options_t od = *o;
  // a chi column of ones is the one-species case: not uploaded, and the kernels without a chi
  // register serve the call (see xlb_particles_t)
  bool chi_trivial = true;
  if (hp->chi)
    for (long long i = 0; i < n; ++i)
      if (hp->chi[i] != 1.0) { chi_trivial = false; break; }
  if (chi_trivial) dp.chi = nullptr;

  // The arrays of the call: host array (NULL = none), the field of the device-side call that
  // receives its device address, its size, and whether the tracking writes it.  The particle
  // columns come first.
  struct Column {
    const void *host;
    void **dev;
    size_t bytes;
    bool back;
  };
  const size_t col = static_cast<size_t>(n) * 8;
  const Column cols[] = {
      {hp->x, slot(&dp.x), col, true},
      {hp->px, slot(&dp.px), col, true},
      {hp->y, slot(&dp.y), col, true},
      {hp->py, slot(&dp.py), col, true},
      {hp->zeta, slot(&dp.zeta), col, true},
      {hp->delta, slot(&dp.delta), col, true},
      {hp->rpp, slot(&dp.rpp), col, true},
      {hp->rvv, slot(&dp.rvv), col, true},
      {hp->s, slot(&dp.s), col, true},
      {hp->state, slot(&dp.state), col, true},
      {hp->at_element, slot(&dp.at_element), col, true},
      {hp->at_turn, slot(&dp.at_turn), col, true},
      {hp->particle_id, slot(&dp.particle_id), col, false},
      {dp.chi, slot(&dp.chi), col, false},
      {hp->charge_ratio, slot(&dp.charge_ratio), col, false},
      {o->loss_tally, slot(&od.loss_tally), static_cast<size_t>(hl->n_elements) * 8, true},
      {o->monitor_data, slot(&od.monitor_data), static_cast<size_t>(o->monitor_words) * 8, true},
  };
  const int n_cols = static_cast<int>(sizeof(cols) / sizeof(cols[0])), n_particle_cols = 15;

  // Small single-launch calls on PINNED host buffers (C1: 10 000 particles x 100 turns): the
  // kernel reads and writes the caller's arrays in place through their device aliases -- the
  // particle state crosses the bus once each way inside the kernel's own entry and exit, instead
  // of 26 separate DMA transfers of 80 kB whose set-up latencies dominate a 0.3 ms call.
  auto alias = [](const void *h, void **d) {
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, h) != cudaSuccess) {
      cudaGetLastError();
      return false;
    }
    if (at.type != cudaMemoryTypeHost || !at.devicePointer) return false;
    *d = at.devicePointer;
    return true;
  };
  bool in_place = n <= 16384 && launch_cap(o->turns_per_launch, o->num_turns, hl->n_chunks) >= o->num_turns;
  for (int c = 0; c < n_particle_cols && in_place; ++c)
    in_place = !cols[c].host || alias(cols[c].host, cols[c].dev);
  const int first = in_place ? n_particle_cols : 0;  // the arrays copied to and from the device

  // device arena: lattice | copied arrays
  auto al = [](size_t v) { return (v + 255) & ~static_cast<size_t>(255); };
  const size_t lat_bytes = al(static_cast<size_t>(hl->n_words) * 8);
  size_t need = lat_bytes;
  for (int c = first; c < n_cols; ++c)
    if (cols[c].host) need += al(cols[c].bytes);
  if ((rc = grow(&s->arena, &s->arena_bytes, need)) != XLB_OK) return rc;
  xlb_lattice_t dl = *hl;
  dl.words = reinterpret_cast<const uint64_t *>(s->arena);
  XLB_CUDA(cudaMemcpyAsync(s->arena, hl->words, static_cast<size_t>(hl->n_words) * 8, cudaMemcpyHostToDevice, st));
  unsigned char *cur = s->arena + lat_bytes;
  for (int c = first; c < n_cols; ++c) {
    if (!cols[c].host) continue;
    *cols[c].dev = cur;
    cur += al(cols[c].bytes);
    XLB_CUDA(cudaMemcpyAsync(*cols[c].dev, cols[c].host, cols[c].bytes, cudaMemcpyHostToDevice, st));
  }
  if ((rc = track_device_impl(&dl, &dp, &od, st, !in_place)) != XLB_OK) return rc;
  for (int c = first; c < n_cols; ++c)
    if (cols[c].host && cols[c].back)  // the caller's writable arrays
      XLB_CUDA(cudaMemcpyAsync(const_cast<void *>(cols[c].host), *cols[c].dev, cols[c].bytes,
                               cudaMemcpyDeviceToHost, st));
  XLB_CUDA(cudaStreamSynchronize(st));
  return XLB_OK;
}

int xlb_measure_fp64_peak(int repeats, double *flops_out, double *ms_out) {
  if (!flops_out) return fail(XLB_EINVAL, "flops_out is null");
  int dev = 0;
  XLB_CUDA(cudaGetDevice(&dev));
  cudaDeviceProp prop;
  XLB_CUDA(cudaGetDeviceProperties(&prop, dev));
  constexpr int CHAINS = 8;
  const int iters = 1 << 15;
  const int blocks = prop.multiProcessorCount * 8;
  double *d = nullptr;
  XLB_CUDA(cudaMalloc(&d, 64));
  cudaEvent_t e0, e1;
  XLB_CUDA(cudaEventCreate(&e0));
  XLB_CUDA(cudaEventCreate(&e1));
  float best = 1e30f;
  if (repeats < 1) repeats = 1;
  for (int r = 0; r < repeats + 2; ++r) {
    XLB_CUDA(cudaEventRecord(e0));
    dfma_peak_kernel<CHAINS><<<blocks, 256>>>(d, iters, 1.0000001, 1e-9);
    XLB_CUDA(cudaEventRecord(e1));
    XLB_CUDA(cudaEventSynchronize(e1));
    float ms = 0;
    XLB_CUDA(cudaEventElapsedTime(&ms, e0, e1));
    if (r >= 2 && ms < best) best = ms;  // first two are warm-up
  }
  XLB_CUDA(cudaGetLastError());
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  cudaFree(d);
  const double flops = 2.0 * CHAINS * static_cast<double>(iters) * 256.0 * blocks;
  *flops_out = flops / (best * 1e-3);
  if (ms_out) *ms_out = best;
  return XLB_OK;
}

int xlb_measure_dfma_latency(double *cycles_per_dfma, int n) {
  if (!cycles_per_dfma || n < 4) return fail(XLB_EINVAL, "need room for 4 results");
  double *d = nullptr;
  long long *dc = nullptr;
  XLB_CUDA(cudaMalloc(&d, 64));
  XLB_CUDA(cudaMalloc(&dc, 8));
  int rc = run_latency<1>(d, dc, &cycles_per_dfma[0]);
  if (rc == XLB_OK) rc = run_latency<2>(d, dc, &cycles_per_dfma[1]);
  if (rc == XLB_OK) rc = run_latency<4>(d, dc, &cycles_per_dfma[2]);
  if (rc == XLB_OK) rc = run_latency<8>(d, dc, &cycles_per_dfma[3]);
  cudaFree(d);
  cudaFree(dc);
  return rc;
}

int xlb_selftest_exact_division(const double *divisors, int n_divisors, int mode, int samples_per_thread,
                                uint64_t seed, int exponent_span, uint64_t *mismatches, uint64_t *samples) {
  if (!divisors || n_divisors < 1 || !mismatches || samples_per_thread < 1 || exponent_span < 0 ||
      exponent_span > 900 || (mode != 0 && mode != 1))
    return fail(XLB_EINVAL, "bad argument");
  for (int i = 0; i < n_divisors; ++i) {
    const double b = divisors[i];
    if (mode == 0 && !(b >= 1 && b <= 255 && b == static_cast<double>(static_cast<int>(b))))
      return fail(XLB_EINVAL, "mode 0 takes integer divisors 1..255");
    if (!(b > 0) || b > 1e150 || b < 1e-150) return fail(XLB_EINVAL, "divisor out of range");
  }
  double *d = nullptr;
  unsigned long long *dm = nullptr;
  XLB_CUDA(cudaMalloc(&d, sizeof(double) * n_divisors));
  XLB_CUDA(cudaMalloc(&dm, sizeof(unsigned long long)));
  XLB_CUDA(cudaMemcpy(d, divisors, sizeof(double) * n_divisors, cudaMemcpyHostToDevice));
  XLB_CUDA(cudaMemset(dm, 0, sizeof(unsigned long long)));
  const int rc = strict_selftest_division(d, n_divisors, mode, samples_per_thread, seed, exponent_span, dm, nullptr);
  if (rc != 0) return fail(XLB_ECUDA, cudaGetErrorString(static_cast<cudaError_t>(rc)));
  unsigned long long h = 0;
  XLB_CUDA(cudaMemcpy(&h, dm, sizeof(h), cudaMemcpyDeviceToHost));
  cudaFree(d);
  cudaFree(dm);
  *mismatches = h;
  if (samples) *samples = 148ull * 4 * 256 * static_cast<unsigned long long>(samples_per_thread) * n_divisors;
  return XLB_OK;
}

int xlb_kernel_variant_count(void) {
  int total = 0;
  for (int t = 0; t < kNumTables; ++t) {
    int n = 0;
    kTables[t](&n);
    total += n;
  }
  return total;
}

int xlb_kernel_variant_info(int i, char *name, int name_len, int *regs, int *max_threads) {
  for (int t = 0; t < kNumTables; ++t) {
    int n = 0;
    const Variant *tab = kTables[t](&n);
    if (i < n) {
      const Variant &v = tab[i];
      if (name && name_len > 0) {
        strncpy(name, v.name, name_len - 1);
        name[name_len - 1] = 0;
      }
      cudaFuncAttributes fa;
      cudaError_t e = cudaFuncGetAttributes(&fa, v.func);
      if (regs) *regs = (e == cudaSuccess) ? fa.numRegs : -1;
      if (max_threads) *max_threads = v.threads;
      if (e != cudaSuccess) cudaGetLastError();
      return XLB_OK;
    }
    i -= n;
  }
  return fail(XLB_EINVAL, "variant index out of range");
}

}  // extern "C"
