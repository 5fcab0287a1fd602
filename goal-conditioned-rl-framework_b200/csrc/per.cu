// Device-resident uniform and prioritised replay (sm_100a).
//
// Replaces ReplayBuffer (reference src/buffer.py:8-35) and PERBuffer (src/buffer.py:38-89): the two buffers
// behind agent.update() besides HERBuffer.  Both are bounded FIFO deques of (s, a, r, s', d); the prioritised
// one carries a float32 priority per entry, draws B positions with numpy.random.choice(N, B, p=P) and hands
// back importance weights.
//
// HBM layout:
//   rows[cap][row_f]  : s[D] | a[A] | r | ns[D] | d | pad   (fp32, row stride a multiple of 16 B), a ring:
//                       deque position p lives in slot (total - len + p) mod cap
//   prio[cap]         : float32 priority per slot (1.0 on append, src/buffer.py:48)
//   pnorm[cap]        : P of the last sample() in deque order (src/buffer.py:54-59)
//   cdf[cap]          : the float64 table RandomState.choice searches, in deque order
//
// Exactness.  The positions a sample returns are index work, so every float operation that feeds them is
// reproduced bit for bit:
//   * P.sum(): NumPy's float32 pairwise summation tree (leaves of <= 128 elements with 8 strided accumulators,
//     halves rounded down to a multiple of 8) -- the host builds the leaf / node table for the current N, one
//     8-lane group per leaf sums it, one CTA folds the tree level by level;
//   * P /= sum: IEEE float32 division;
//   * cdf = cumsum(float64(P)): a LEFT-TO-RIGHT chain of float64 additions in the reference.  A parallel scan
//     reorders the additions, which is only harmless when no addition rounds.  Every P[i] is a float32, so
//     when all of them are integer multiples of 2^-52 (true whenever P[i] >= 2^-29, i.e. for all but extreme
//     priority ratios) and the total is below 2, every partial sum in ANY order is exactly representable: the
//     kernels then scan the values as int64 fixed point (units of 2^-52) and the result provably equals the
//     sequential one.  If one element fails the test, a flag routes the call to the general path further down
//     (the rounding of every addition tracked exactly, still in parallel);
//   * cdf /= cdf[-1]: IEEE float64 division; searchsorted(side="right"): count of entries <= u.
// float32 power (importance weights, new priorities) is computed as float(pow(double)) -- within an ulp of
// any libm / SIMD powf the reference may run on (DESIGN.md, prioritised replay).
#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstring>
#include <functional>
#include <vector>

#include "common.cuh"
#include "graphs.cuh"

namespace gcrl {
namespace {

constexpr int kScanThreads = 256;
constexpr int kScanItems = 8;
constexpr int kScanTile = kScanThreads * kScanItems;
constexpr double kTwo52 = 4503599627370496.0;          // 2^52
constexpr double kTwo53 = 9007199254740992.0;

// Per-call scalars of a prioritised draw, read from device memory so that the captured graph of the draw can be
// replayed while the ring keeps turning (start moves with every push) and beta anneals.
struct PerCall {
  int64_t start;
  float neg_beta;
  int pad;
};

struct ReplayGeom {
  float *rows;
  float *prio;
  int64_t cap;
  int D, A, row_f;
};

__device__ __forceinline__ int64_t slot_of(int64_t start, int64_t pos, int64_t cap) {
  int64_t s = start + pos;
  return s >= cap ? s - cap : s;
}

__global__ void fill_kernel(float *p, int64_t start, int64_t n, int64_t cap, float v) {
  for (int64_t i = blockIdx.x * int64_t(blockDim.x) + threadIdx.x; i < n; i += int64_t(gridDim.x) * blockDim.x)
    p[slot_of(start, i, cap)] = v;
}

__global__ void fill_i32_kernel(int *p, int64_t n, int v) {
  for (int64_t i = blockIdx.x * int64_t(blockDim.x) + threadIdx.x; i < n; i += int64_t(gridDim.x) * blockDim.x) p[i] = v;
}

// ---- P.sum() ---------------------------------------------------------------------------------
// One 8-lane group per leaf [leaf_off[l], leaf_off[l+1]) of NumPy's pairwise tree.
__global__ void __launch_bounds__(256)
leaf_sum_kernel(const float *__restrict__ prio, const PerCall *__restrict__ call, int64_t cap,
                const int *__restrict__ leaf_off, int n_leaves, float *__restrict__ vals, int *__restrict__ flags) {
  if (blockIdx.x == 0 && threadIdx.x == 0) *flags = 0;       // the inexact-cumsum flag of this sample() call
  const int64_t start = call->start;
  const int lane8 = threadIdx.x & 7;
  const int leaf = (blockIdx.x * blockDim.x + threadIdx.x) >> 3;
  const bool live = leaf < n_leaves;
  const int lo = live ? leaf_off[leaf] : 0;
  const int n = live ? leaf_off[leaf + 1] - lo : 0;
  const bool big = n >= 8;                                  // n < 8 only when the whole vector is that short
  const int end = n - (n & 7);
  float r = 0.0f;
  if (big) {
    r = prio[slot_of(start, lo + lane8, cap)];
    for (int i = 8; i < end; i += 8) r = __fadd_rn(r, prio[slot_of(start, lo + i + lane8, cap)]);
  }
  // ((r0 + r1) + (r2 + r3)) + ((r4 + r5) + (r6 + r7)); every lane of the warp takes part in the shuffles
  r = __fadd_rn(r, __shfl_xor_sync(0xffffffffu, r, 1));
  r = __fadd_rn(r, __shfl_xor_sync(0xffffffffu, r, 2));
  r = __fadd_rn(r, __shfl_xor_sync(0xffffffffu, r, 4));
  if (live && lane8 == 0) {
    float res = big ? r : 0.0f;
    for (int i = big ? end : 0; i < n; ++i) res = __fadd_rn(res, prio[slot_of(start, lo + i, cap)]);
    vals[leaf] = res;
  }
}

// Folds the tree: nodes are grouped by height, children precede parents; one CTA, one barrier per level.
// SMEM: the node values live in shared memory (a level costs a barrier instead of an L2 round trip);
// used whenever leaves + internal nodes fit (up to ~3M priorities), else the values stay in global memory.
template <bool SMEM>
__global__ void __launch_bounds__(1024)
tree_fold_kernel(float *__restrict__ vals, const int *__restrict__ node_l, const int *__restrict__ node_r,
                 const int *__restrict__ group_off, int n_groups, int n_leaves, float *__restrict__ psum) {
  extern __shared__ float sv[];
  float *v = SMEM ? sv : vals;
  if (SMEM) {
    for (int j = threadIdx.x; j < n_leaves; j += blockDim.x) sv[j] = vals[j];
    __syncthreads();
  }
  for (int g = 0; g < n_groups; ++g) {
    for (int j = group_off[g] + threadIdx.x; j < group_off[g + 1]; j += blockDim.x)
      v[n_leaves + j] = __fadd_rn(v[node_l[j]], v[node_r[j]]);
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    const int n_internal = group_off[n_groups];
    // np.add.reduce seeds with the identity: 0.0f + tree
    *psum = __fadd_rn(0.0f, v[n_internal > 0 ? n_leaves + n_internal - 1 : 0]);
  }
}

// ---- P /= sum, fixed-point conversion, per-tile inclusive scan ---------------------------------
__device__ __forceinline__ int64_t shfl_up_i64(int64_t v, int d) {
  int lo = int(uint32_t(uint64_t(v))), hi = int(uint32_t(uint64_t(v) >> 32));
  lo = __shfl_up_sync(0xffffffffu, lo, d);
  hi = __shfl_up_sync(0xffffffffu, hi, d);
  return int64_t((uint64_t(uint32_t(hi)) << 32) | uint32_t(lo));
}

__global__ void __launch_bounds__(kScanThreads)
normalise_scan_kernel(const float *__restrict__ prio, const PerCall *__restrict__ call, int64_t cap, int64_t n,
                      const float *__restrict__ psum, float *__restrict__ pnorm, int64_t *__restrict__ fixed,
                      int64_t *__restrict__ tile_sum, int *__restrict__ flags) {
  const int64_t start = call->start;
  __shared__ float sp[kScanTile];
  __shared__ int64_t warp_tot[kScanThreads / 32];
  const int64_t base = int64_t(blockIdx.x) * kScanTile;
  const float s = *psum;
  const bool positive = s > 0.0f;
  const float uniform = float(1.0 / double(n));              // P[:] = 1.0 / N  (src/buffer.py:59)
  for (int k = threadIdx.x; k < kScanTile; k += kScanThreads) {
    const int64_t i = base + k;
    float p = 0.0f;
    if (i < n) {
      p = positive ? __fdiv_rn(prio[slot_of(start, i, cap)], s) : uniform;
      pnorm[i] = p;
    }
    sp[k] = p;
  }
  __syncthreads();
  int64_t v[kScanItems];
  int64_t run = 0;
  bool inexact = false;
#pragma unroll
  for (int j = 0; j < kScanItems; ++j) {
    const double x = double(sp[threadIdx.x * kScanItems + j]) * kTwo52;
    inexact |= !(x == rint(x)) || !(x < kTwo53);
    run += int64_t(x);
    v[j] = run;
  }
  // inclusive scan of the per-thread totals over the CTA
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  int64_t incl = run;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const int64_t o = shfl_up_i64(incl, d);
    if (lane >= d) incl += o;
  }
  if (lane == 31) warp_tot[warp] = incl;
  __syncthreads();
  int64_t warp_base = 0;
  for (int w = 0; w < warp; ++w) warp_base += warp_tot[w];
  const int64_t excl = warp_base + incl - run;
#pragma unroll
  for (int j = 0; j < kScanItems; ++j) {
    const int64_t i = base + threadIdx.x * kScanItems + j;
    if (i < n) fixed[i] = excl + v[j];
  }
  if (threadIdx.x == kScanThreads - 1) tile_sum[blockIdx.x] = warp_base + incl;
  if (__syncthreads_or(inexact) && threadIdx.x == 0) atomicOr(flags, 1);
}

// exclusive scan of the tile totals (one CTA), grand total -> total_out
__global__ void __launch_bounds__(1024)
tile_scan_kernel(int64_t *__restrict__ tile_sum, int n_tiles, int64_t *__restrict__ total_out, int *__restrict__ flags) {
  __shared__ int64_t sm[1024];
  __shared__ int64_t carry;
  if (threadIdx.x == 0) carry = 0;
  __syncthreads();
  for (int b0 = 0; b0 < n_tiles; b0 += 1024) {
    const int i = b0 + threadIdx.x;
    const int64_t x = i < n_tiles ? tile_sum[i] : 0;
    sm[threadIdx.x] = x;
    __syncthreads();
    for (int d = 1; d < 1024; d <<= 1) {
      const int64_t o = int(threadIdx.x) >= d ? sm[threadIdx.x - d] : 0;
      __syncthreads();
      sm[threadIdx.x] += o;
      __syncthreads();
    }
    if (i < n_tiles) tile_sum[i] = carry + sm[threadIdx.x] - x;
    __syncthreads();
    if (threadIdx.x == 0) carry += sm[1023];
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    *total_out = carry;
    if (!(double(carry) < kTwo53) || carry <= 0) atomicOr(flags, 1);
  }
}

// exact path: cdf[i] = F_i / F_last  (F in units of 2^-52; the power of two cancels in the quotient)
__global__ void __launch_bounds__(kScanThreads)
cdf_from_fixed_kernel(int64_t *__restrict__ fixed, const int64_t *__restrict__ tile_off,
                      const int64_t *__restrict__ total, int64_t n, const int *__restrict__ flags) {
  if (*flags & 1) return;
  const double tot = double(*total);
  double *cdf = reinterpret_cast<double *>(fixed);
  const int64_t base = int64_t(blockIdx.x) * kScanTile;
  const int64_t off = tile_off[blockIdx.x];
  for (int k = threadIdx.x; k < kScanTile; k += kScanThreads) {
    const int64_t i = base + k;
    if (i < n) cdf[i] = __ddiv_rn(double(fixed[i] + off), tot);
  }
}

// ---- inexact case: the reference's left-to-right float64 chain, reproduced in parallel ---------------
// c_i = RN(c_{i-1} + p_i).  While c stays inside one binade [2^k, 2^(k+1)) it is an integer multiple of
// u = 2^(k-52), and adding p = (a + f) u  (a integer, 0 <= f < 1) rounds to c + a u (f < 1/2), c + (a + 1) u
// (f > 1/2) or, on a tie (f == 1/2 -- by far the most common inexact case for float32 inputs), to whichever of
// the two is an even multiple of u.  So one element is a function {parity of c / u} -> (increment in units of
// u, new parity), these functions compose associatively, and a chunk of elements collapses to two integer
// increments and two outgoing parities.  Phase A summarises every 512-element chunk for the binade its
// incoming value is expected in (from the truncated fixed-point scan); phase B walks the chunk summaries in
// order with the true running value -- one exact addition per chunk -- and processes the few chunks the
// summary does not cover (binade crossings, about one per power of two) element by element; phase C expands
// the summarised chunks in parallel.  Every value written is exactly the sequential one.
constexpr int kChunk = 512;
constexpr int kChunkPerLane = kChunk / 32;

struct __align__(8) ChunkSum {
  int64_t d0, d1;      // increment in units of u for incoming parity 0 / 1
  int k;               // binade of the incoming value the summary was built for
  int bits;            // bit0 / bit1: outgoing parity for incoming parity 0 / 1; bit2: summary valid
};

struct ParityFn {
  int64_t d0, d1;
  int o;               // bit0: outgoing parity for incoming parity 0, bit1: for incoming parity 1
};

__device__ __forceinline__ ParityFn fn_compose(const ParityFn &A, const ParityFn &B) {   // A first, then B
  ParityFn r;
  const bool a0 = A.o & 1, a1 = (A.o >> 1) & 1;
  r.d0 = A.d0 + (a0 ? B.d1 : B.d0);
  r.d1 = A.d1 + (a1 ? B.d1 : B.d0);
  const int o0 = a0 ? (B.o >> 1) & 1 : B.o & 1;
  const int o1 = a1 ? (B.o >> 1) & 1 : B.o & 1;
  r.o = o0 | (o1 << 1);
  return r;
}

// p = q u with q = p * scale (scale = 1 / u, a power of two: exact); q has at most 24 significant bits
__device__ __forceinline__ ParityFn fn_element(float p, double scale, bool &bad) {
  const double q = double(p) * scale;
  ParityFn r;
  if (!(q < kTwo53)) { bad = true; r.d0 = r.d1 = 0; r.o = 2; return r; }
  const double a = floor(q), f = q - a;
  const int64_t ai = int64_t(a);
  if (f == 0.5) {                    // tie: the even neighbour, whatever it takes
    r.d0 = ai + (ai & 1);
    r.d1 = ai + ((ai + 1) & 1);
    r.o = 0;
  } else {
    const int64_t d = ai + (f > 0.5 ? 1 : 0);
    r.d0 = r.d1 = d;
    r.o = int(d & 1) | (int((d + 1) & 1) << 1);
  }
  return r;
}

__device__ __forceinline__ int64_t shfl_i64(int64_t v, int src) {
  int lo = int(uint32_t(uint64_t(v))), hi = int(uint32_t(uint64_t(v) >> 32));
  lo = __shfl_sync(0xffffffffu, lo, src);
  hi = __shfl_sync(0xffffffffu, hi, src);
  return int64_t((uint64_t(uint32_t(hi)) << 32) | uint32_t(lo));
}

__device__ __forceinline__ double pow2(int e) { return __longlong_as_double(int64_t(1023 + e) << 52); }
__device__ __forceinline__ int binade_of(double c) { return int((__double_as_longlong(c) >> 52) & 0x7ff) - 1023; }

// lane-local fold of the lane's 16 elements + inclusive scan over the warp; returns the lane's inclusive
// function, *excl = the function of everything before the lane's first element
__device__ __forceinline__ ParityFn chunk_scan(const float (&p)[kChunkPerLane], double scale, int lane, ParityFn *excl,
                                               bool *bad_out) {
  bool bad = false;
  ParityFn acc = fn_element(p[0], scale, bad);
#pragma unroll
  for (int j = 1; j < kChunkPerLane; ++j) acc = fn_compose(acc, fn_element(p[j], scale, bad));
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    ParityFn o;
    o.d0 = shfl_up_i64(acc.d0, d);
    o.d1 = shfl_up_i64(acc.d1, d);
    o.o = __shfl_up_sync(0xffffffffu, acc.o, d);
    if (lane >= d) acc = fn_compose(o, acc);
  }
  ParityFn e;
  e.d0 = shfl_up_i64(acc.d0, 1);
  e.d1 = shfl_up_i64(acc.d1, 1);
  e.o = __shfl_up_sync(0xffffffffu, acc.o, 1);
  if (lane == 0) { e.d0 = e.d1 = 0; e.o = 2; }
  *excl = e;
  *bad_out = __any_sync(0xffffffffu, bad);
  return acc;
}

__device__ __forceinline__ void load_chunk(const float *__restrict__ pnorm, int64_t i0, int64_t n, int lane,
                                           float (&p)[kChunkPerLane]) {
  const int64_t base = i0 + lane * kChunkPerLane;
#pragma unroll
  for (int j = 0; j < kChunkPerLane; ++j) p[j] = base + j < n ? pnorm[base + j] : 0.0f;
}

__global__ void __launch_bounds__(256)
chunk_summary_kernel(const float *__restrict__ pnorm, const int64_t *__restrict__ fixed,
                     const int64_t *__restrict__ tile_off, int64_t n, int n_chunks, ChunkSum *__restrict__ sums,
                     const int *__restrict__ flags) {
  if (!(*flags & 1)) return;
  const int lane = threadIdx.x & 31;
  const int j = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (j >= n_chunks) return;
  const int64_t i0 = int64_t(j) * kChunk;
  double approx = 0.0;                               // truncated fixed-point prefix: the binade guess only
  if (i0 > 0) approx = double(fixed[i0 - 1] + tile_off[(i0 - 1) / kScanTile]) / kTwo52;
  ChunkSum s;
  s.d0 = s.d1 = 0; s.k = 0; s.bits = 0;
  const int k = approx > 0.0 ? binade_of(approx) : -2000;
  if (k > -900 && k < 900) {
    float p[kChunkPerLane];
    load_chunk(pnorm, i0, n, lane, p);
    ParityFn excl;
    bool bad;
    const ParityFn incl = chunk_scan(p, pow2(52 - k), lane, &excl, &bad);
    s.d0 = shfl_i64(incl.d0, 31);
    s.d1 = shfl_i64(incl.d1, 31);
    s.k = k;
    s.bits = __shfl_sync(0xffffffffu, incl.o, 31) | (bad ? 0 : 4);
  }
  if (lane == 0) sums[j] = s;
}

constexpr int kWalkBatch = 512;       // chunk summaries staged in shared memory per refill

// One warp.  Up to 32 chunk summaries at a time: a warp scan of the composed parity functions gives every chunk's
// incoming value in one step, and the longest prefix that keeps the running value inside its binade is
// accepted; the chunk in which the value crosses a power of two (about one per binade) is chained element by
// element through the lanes' registers.
__global__ void __launch_bounds__(32)
chunk_walk_kernel(const float *__restrict__ pnorm, double *__restrict__ cdf, int64_t n, int n_chunks,
                  const ChunkSum *__restrict__ sums, double *__restrict__ cin, unsigned char *__restrict__ expand,
                  double *__restrict__ last, const int *__restrict__ flags) {
  if (!(*flags & 1)) return;
  __shared__ ChunkSum ssum[kWalkBatch];
  __shared__ double scin[kWalkBatch];
  __shared__ unsigned char sexp[kWalkBatch];
  const int lane = threadIdx.x;
  double c = 0.0;                                    // every lane carries the same running value
  for (int j0 = 0; j0 < n_chunks; j0 += kWalkBatch) {
    const int nb = min(kWalkBatch, n_chunks - j0);
    for (int t = lane; t < nb; t += 32) ssum[t] = sums[j0 + t];
    __syncwarp();
    for (int g0 = 0; g0 < nb;) {
      // ---- fast: the longest run of chunks (up to 32) that keeps c inside its current binade ----
      const bool live = g0 + lane < nb;
      const ChunkSum q = ssum[min(g0 + lane, nb - 1)];
      const int k0 = __shfl_sync(0xffffffffu, q.k, 0);
      const double lo = pow2(k0), hi = pow2(k0 + 1), u = pow2(k0 - 52);
      const unsigned same = __ballot_sync(0xffffffffu, live && (q.bits & 4) && q.k == k0);
      int m = 0;
      ParityFn acc;
      acc.d0 = q.d0; acc.d1 = q.d1; acc.o = q.bits & 3;
      if (!((same >> lane) & 1)) { acc.d0 = acc.d1 = 0; acc.o = 2; }   // never accepted; keeps the scan defined
#pragma unroll
      for (int d = 1; d < 32; d <<= 1) {
        ParityFn o;
        o.d0 = shfl_up_i64(acc.d0, d);
        o.d1 = shfl_up_i64(acc.d1, d);
        o.o = __shfl_up_sync(0xffffffffu, acc.o, d);
        if (lane >= d) acc = fn_compose(o, acc);
      }
      const bool odd = __double_as_longlong(c) & 1;                    // parity of c / u
      const int64_t d_incl = odd ? acc.d1 : acc.d0;
      int64_t d_excl = shfl_up_i64(d_incl, 1);
      if (lane == 0) d_excl = 0;
      const double c_out = __dadd_rn(c, double(d_incl) * u);          // exact while below hi (increments >= 0)
      const unsigned inside = __ballot_sync(0xffffffffu, c_out < hi);
      if ((same & 1) && k0 > -900 && c >= lo && c < hi) m = __ffs(~(same & inside)) - 1;   // leading ones
      if (m < 0) m = 32;
      if (m > 0) {
        if (lane < m) { scin[g0 + lane] = __dadd_rn(c, double(d_excl) * u); sexp[g0 + lane] = 1; }
        c = __shfl_sync(0xffffffffu, c_out, m - 1);
        g0 += m;
        continue;
      }
      // ---- the chunk in which c leaves its binade (or the very first one): the plain chain ----
      // lane l holds elements [16 l, 16 l + 16) in registers; the running value visits the lanes in order
      // (one shuffle per lane), so the dependent chain is 512 register-to-register additions
      {
        const int jj = g0;
        if (lane == 0) { scin[jj] = c; sexp[jj] = 0; }
        const int64_t i0 = int64_t(j0 + jj) * kChunk;
        float p[kChunkPerLane];
        load_chunk(pnorm, i0, n, lane, p);
        double v[kChunkPerLane];
#pragma unroll 1
        for (int l = 0; l < 32; ++l) {
          double t = c;
#pragma unroll
          for (int e = 0; e < kChunkPerLane; ++e) {
            t = __dadd_rn(t, double(p[e]));
            if (lane == l) v[e] = t;
          }
          c = __shfl_sync(0xffffffffu, t, l);
        }
        const int64_t base = i0 + lane * kChunkPerLane;
#pragma unroll
        for (int e = 0; e < kChunkPerLane; ++e)
          if (base + e < n) cdf[base + e] = v[e];
        g0 += 1;
      }
    }
    __syncwarp();
    for (int t = lane; t < nb; t += 32) { cin[j0 + t] = scin[t]; expand[j0 + t] = sexp[t]; }
    __syncwarp();
  }
  if (lane == 0) *last = c;
}

__global__ void __launch_bounds__(256)
chunk_expand_kernel(const float *__restrict__ pnorm, double *__restrict__ cdf, int64_t n, int n_chunks,
                    const ChunkSum *__restrict__ sums, const double *__restrict__ cin,
                    const unsigned char *__restrict__ expand, const int *__restrict__ flags) {
  if (!(*flags & 1)) return;
  const int lane = threadIdx.x & 31;
  const int j = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (j >= n_chunks || !expand[j]) return;
  const int64_t i0 = int64_t(j) * kChunk;
  const int k = sums[j].k;
  const double c0 = cin[j], scale = pow2(52 - k), u = pow2(k - 52);
  float p[kChunkPerLane];
  load_chunk(pnorm, i0, n, lane, p);
  ParityFn excl;
  bool bad;
  chunk_scan(p, scale, lane, &excl, &bad);
  const bool odd_in = __double_as_longlong(c0) & 1;
  int64_t off = odd_in ? excl.d1 : excl.d0;                          // units of u before the lane's first element
  int par = odd_in ? (excl.o >> 1) & 1 : excl.o & 1;
  const int64_t base = i0 + lane * kChunkPerLane;
#pragma unroll
  for (int t = 0; t < kChunkPerLane; ++t) {
    bool b2 = false;
    const ParityFn f = fn_element(p[t], scale, b2);
    off += par ? f.d1 : f.d0;
    par = par ? (f.o >> 1) & 1 : f.o & 1;
    if (base + t < n) cdf[base + t] = __dadd_rn(c0, double(off) * u);
  }
}

__global__ void cdf_divide_kernel(double *__restrict__ cdf, int64_t n, const double *__restrict__ last,
                                  const int *__restrict__ flags) {
  if (!(*flags & 1)) return;
  const double t = *last;
  for (int64_t i = blockIdx.x * int64_t(blockDim.x) + threadIdx.x; i < n; i += int64_t(gridDim.x) * blockDim.x)
    cdf[i] = __ddiv_rn(cdf[i], t);
}

// ---- draw + gather ------------------------------------------------------------------------------
// number of table entries <= u (np.searchsorted(cdf, u, side="right")), one warp, 32-way
__device__ __forceinline__ int64_t warp_upper_bound(const double *__restrict__ cdf, int64_t n, double u, int lane) {
  int64_t lo = 0, hi = n;                                      // entries [lo, hi) undecided; answer in [lo, hi]
  while (hi - lo > 32) {
    const int64_t step = (hi - lo + 31) >> 5;
    const int64_t probe = lo + (lane + 1) * step - 1;
    const bool le = probe < hi ? (cdf[probe] <= u) : false;
    const int cnt = __popc(__ballot_sync(0xffffffffu, le));    // monotone table: a prefix of the lanes
    lo += cnt * step;                                          // entries below are <= u
    hi = min(hi, lo + step - 1);                               // the next probe (if any) was > u
  }
  const bool le = lo + lane < hi ? (cdf[lo + lane] <= u) : false;
  return lo + __popc(__ballot_sync(0xffffffffu, le));
}

__device__ __forceinline__ void scatter_row(const ReplayGeom &g, int64_t slot, int64_t b, int lane,
                                            float *s, float *a, float *r, float *ns, float *d) {
  const float *row = g.rows + slot * g.row_f;
  const int D = g.D, A = g.A;
  for (int k = lane; k < 2 * D + A + 2; k += 32) {
    const float v = row[k];
    if (k < D) s[b * D + k] = v;
    else if (k < D + A) a[b * A + (k - D)] = v;
    else if (k == D + A) r[b] = v;
    else if (k < 2 * D + A + 1) ns[b * D + (k - D - A - 1)] = v;
    else d[b] = v;
  }
}

__global__ void __launch_bounds__(256)
per_draw_kernel(ReplayGeom g, const PerCall *__restrict__ call, int64_t n, const double *__restrict__ cdf,
                const float *__restrict__ pnorm, const double *__restrict__ u, int B, float *s, float *a, float *r,
                float *ns, float *d, float *__restrict__ w_raw, int64_t *__restrict__ pos_out,
                int64_t *__restrict__ slot_out) {
  const int64_t start = call->start;
  const float neg_beta = call->neg_beta;
  const int lane = threadIdx.x & 31;
  const int64_t b = (blockIdx.x * int64_t(blockDim.x) + threadIdx.x) >> 5;
  if (b >= B) return;
  int64_t pos = warp_upper_bound(cdf, n, u[b], lane);
  if (pos >= n) pos = n - 1;                                   // unreachable: u < 1 == cdf[n-1]
  const int64_t slot = slot_of(start, pos, g.cap);
  scatter_row(g, slot, b, lane, s, a, r, ns, d);
  if (lane == 0) {
    const float x = __fmul_rn(float(n), pnorm[pos]);           // N * P[i]                (src/buffer.py:65)
    float w;
    if (neg_beta == -1.0f) w = __fdiv_rn(1.0f, x);             // NumPy's scalar-exponent fast paths
    else if (neg_beta == 0.0f) w = 1.0f;
    else w = float(pow(double(x), double(neg_beta)));
    w_raw[b] = w;
    pos_out[b] = pos;
    slot_out[b] = slot;
  }
}

// weights /= weights.max()   (src/buffer.py:66)
__global__ void __launch_bounds__(1024) weight_norm_kernel(const float *__restrict__ w_raw, float *__restrict__ w, int B) {
  __shared__ float sm[1024];
  float m = -INFINITY;
  for (int i = threadIdx.x; i < B; i += 1024) m = fmaxf(m, w_raw[i]);
  sm[threadIdx.x] = m;
  __syncthreads();
  for (int s2 = 512; s2 >= 1; s2 >>= 1) {
    if (int(threadIdx.x) < s2) sm[threadIdx.x] = fmaxf(sm[threadIdx.x], sm[threadIdx.x + s2]);
    __syncthreads();
  }
  m = sm[0];
  for (int i = threadIdx.x; i < B; i += 1024) w[i] = __fdiv_rn(w_raw[i], m);
}

// call != nullptr: the ring start is read from device memory (a replayed n-update graph follows the pushes made
// between two calls); else `start` by value (gcrl_replay_sample)
__global__ void __launch_bounds__(256)
uniform_gather_kernel(ReplayGeom g, int64_t start, const PerCall *__restrict__ call, const int64_t *__restrict__ pos,
                      int B, float *s, float *a, float *r, float *ns, float *d) {
  const int lane = threadIdx.x & 31;
  const int64_t b = (blockIdx.x * int64_t(blockDim.x) + threadIdx.x) >> 5;
  if (b >= B) return;
  scatter_row(g, slot_of(call != nullptr ? call->start : start, pos[b], g.cap), b, lane, s, a, r, ns, d);
}

// ---- update_priorities (src/buffer.py:86-89): in draw order, so the LAST duplicate of a position wins ----
__global__ void prio_winner_kernel(const int64_t *__restrict__ slot, int B, int *__restrict__ winner) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b < B) atomicMax(&winner[slot[b]], b);
}

__global__ void prio_write_kernel(const int64_t *__restrict__ slot, const float *__restrict__ td, int B, float alpha,
                                  float eps, float *__restrict__ prio, int *__restrict__ winner) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  const int64_t sl = slot[b];
  if (winner[sl] != b) return;
  const float x = __fadd_rn(fabsf(td[b]), eps);
  prio[sl] = alpha == 1.0f ? x : float(pow(double(x), double(alpha)));
  winner[sl] = -1;
}

inline int blocks_for(int64_t n, int per_block) { return int(std::max<int64_t>(1, (n + per_block - 1) / per_block)); }

}  // namespace
}  // namespace gcrl

using namespace gcrl;

struct gcrl_replay {
  int device = 0;
  ReplayGeom g{};
  bool prioritized = false;
  double alpha = 0.0;
  int64_t total = 0, len = 0;
  float *pnorm = nullptr;
  int64_t *fixed = nullptr;          // int64 fixed point, then the float64 table in place
  int64_t *tile_sum = nullptr, *d_total = nullptr;
  double *d_last = nullptr;
  void *d_chunk_sums = nullptr;      // ChunkSum[n_chunks]
  double *d_chunk_in = nullptr;
  unsigned char *d_chunk_expand = nullptr;
  float *d_psum = nullptr;
  int *d_flags = nullptr, *winner = nullptr;
  // pairwise-sum tree of the current N
  int64_t tree_n = -1;
  bool fold_smem_set = false;
  // the draw as a captured graph: (n, B, output pointers) -> exec; recaptured when the key repeats
  PerCall *d_call = nullptr;
  struct DrawKey {
    int64_t n = -1, B = -1;
    const void *ptr[6] = {};
    bool operator==(const DrawKey &o) const {
      return n == o.n && B == o.B && std::memcmp(ptr, o.ptr, sizeof(ptr)) == 0;
    }
  } graph_key, last_key;
  GraphRec graph{nullptr, 0};
  cudaStream_t cap_stream = nullptr;
  bool use_graphs = true;
  int n_leaves = 0, n_groups = 0;
  size_t tree_cap = 0;
  int *d_leaf_off = nullptr, *d_node_l = nullptr, *d_node_r = nullptr, *d_group_off = nullptr;
  float *d_vals = nullptr;
  // per-batch scratch
  int64_t batch_cap = 0, last_B = 0;
  double *d_u = nullptr;
  float *d_wraw = nullptr;
  int64_t *d_pos = nullptr, *d_slot = nullptr;
  PinnedRing stage;
  // n-update calls (gcrl_agent_update_many_replay, gcrl_sac_update_many_replay): PerCall[n], then the uniforms
  // (prioritised) or the positions (uniform) [n][B], 8 bytes each; many_n = the length the call draws from
  char *d_many = nullptr;
  size_t many_cap = 0;
  int64_t many_n = 0;
  // changes whenever a device array a captured n-update graph reads is reallocated (and differs between handles)
  uint64_t epoch = 0;
  int64_t start() const { return (total - len) % g.cap; }
};

namespace {

std::atomic<uint64_t> g_epoch{0};
void new_epoch(gcrl_replay *h) { h->epoch = ++g_epoch; }

void ensure_batch(gcrl_replay *h, int64_t B, cudaStream_t st) {
  if (B <= h->batch_cap) return;
  GCRL_CUDA(cudaStreamSynchronize(st));
  if (h->graph.exec) { cudaGraphExecDestroy(h->graph.exec); h->graph.exec = nullptr; }
  new_epoch(h);
  for (void *p : {(void *)h->d_u, (void *)h->d_wraw, (void *)h->d_pos, (void *)h->d_slot})
    if (p) GCRL_CUDA(cudaFree(p));
  h->batch_cap = std::max<int64_t>(B, 1024);
  h->d_u = dev_alloc<double>(size_t(h->batch_cap));
  h->d_wraw = dev_alloc<float>(size_t(h->batch_cap));
  h->d_pos = dev_alloc<int64_t>(size_t(h->batch_cap));
  h->d_slot = dev_alloc<int64_t>(size_t(h->batch_cap));
}

// NumPy's pairwise tree for n elements: leaves left to right, internal nodes grouped by height.
void build_tree(gcrl_replay *h, int64_t n, cudaStream_t st) {
  if (h->tree_n == n) return;
  GCRL_REQUIRE(n < (int64_t(1) << 31), "prioritised replay holds at most 2^31 - 1 entries");
  std::vector<int> leaf_off;
  struct Node { int l, r, height; };
  std::vector<Node> nodes;
  // returns a node reference: leaf i -> i, internal node j -> -(j + 1); second = height
  std::function<std::pair<int, int>(int64_t, int64_t)> rec = [&](int64_t lo, int64_t m) -> std::pair<int, int> {
    if (m <= 128) {
      leaf_off.push_back(int(lo));
      return {int(leaf_off.size()) - 1, 0};
    }
    int64_t m2 = m / 2;
    m2 -= m2 % 8;
    const auto l = rec(lo, m2);
    const auto r = rec(lo + m2, m - m2);
    nodes.push_back({l.first, r.first, std::max(l.second, r.second) + 1});
    return {-int(nodes.size()), nodes.back().height};
  };
  const int max_h = rec(0, n).second;
  leaf_off.push_back(int(n));
  const int L = int(leaf_off.size()) - 1, I = int(nodes.size());
  // stable order by height (children before parents; the root comes last); group g holds height g + 1
  std::vector<int> counts(max_h + 2, 0), group_off(max_h + 1, 0);
  for (auto &nd : nodes) counts[nd.height]++;
  for (int g = 0; g < max_h; ++g) group_off[g + 1] = group_off[g] + counts[g + 1];
  std::vector<int> cursor(group_off.begin(), group_off.end()), new_id(I), order(I);
  for (int j = 0; j < I; ++j) { new_id[j] = cursor[nodes[j].height - 1]++; order[new_id[j]] = j; }
  std::vector<int> node_l(std::max(I, 1)), node_r(std::max(I, 1));
  auto ref = [&](int c) { return c >= 0 ? c : L + new_id[-c - 1]; };
  for (int k = 0; k < I; ++k) { node_l[k] = ref(nodes[order[k]].l); node_r[k] = ref(nodes[order[k]].r); }

  const size_t need = size_t(L) + 2;
  if (need > h->tree_cap) {
    GCRL_CUDA(cudaStreamSynchronize(st));
    if (h->graph.exec) { cudaGraphExecDestroy(h->graph.exec); h->graph.exec = nullptr; }   // it holds the old tables
    new_epoch(h);
    for (void *p : {(void *)h->d_leaf_off, (void *)h->d_node_l, (void *)h->d_node_r, (void *)h->d_vals})
      if (p) GCRL_CUDA(cudaFree(p));
    h->tree_cap = need * 2;
    h->d_leaf_off = dev_alloc<int>(h->tree_cap);
    h->d_node_l = dev_alloc<int>(h->tree_cap);
    h->d_node_r = dev_alloc<int>(h->tree_cap);
    h->d_vals = dev_alloc<float>(h->tree_cap * 2);
  }
  if (!h->d_group_off) h->d_group_off = dev_alloc<int>(128);
  GCRL_REQUIRE(max_h + 1 <= 128, "summation tree too deep");
  // table uploads are synchronous pageable copies: N changes only while the buffer is filling
  GCRL_CUDA(cudaStreamSynchronize(st));
  GCRL_CUDA(cudaMemcpy(h->d_leaf_off, leaf_off.data(), size_t(L + 1) * sizeof(int), cudaMemcpyHostToDevice));
  if (I > 0) {
    GCRL_CUDA(cudaMemcpy(h->d_node_l, node_l.data(), size_t(I) * sizeof(int), cudaMemcpyHostToDevice));
    GCRL_CUDA(cudaMemcpy(h->d_node_r, node_r.data(), size_t(I) * sizeof(int), cudaMemcpyHostToDevice));
  }
  GCRL_CUDA(cudaMemcpy(h->d_group_off, group_off.data(), size_t(max_h + 1) * sizeof(int), cudaMemcpyHostToDevice));
  h->n_leaves = L;
  h->n_groups = max_h;
  h->tree_n = n;
  if (!h->fold_smem_set) {      // outside any capture: the fold's shared-memory form may need up to 200 KB
    GCRL_CUDA(cudaFuncSetAttribute(tree_fold_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    h->fold_smem_set = true;
  }
}

// The 11 launches of one prioritised draw from the first n entries: per-call scalars and uniforms from `call` / `u`
void issue_draw(gcrl_replay *h, int64_t n, int64_t B, const PerCall *call, const double *u, float *s, float *a, float *r,
                float *ns, float *d, float *weights_dev, cudaStream_t st) {
  const int64_t cap = h->g.cap;
  leaf_sum_kernel<<<blocks_for(int64_t(h->n_leaves) * 8, 256), 256, 0, st>>>(h->g.prio, call, cap, h->d_leaf_off,
                                                                           h->n_leaves, h->d_vals, h->d_flags);
  GCRL_LAUNCHED();
  {
    const size_t fold_smem = size_t(2 * h->n_leaves) * sizeof(float);
    if (fold_smem <= size_t(200) * 1024) {
      tree_fold_kernel<true><<<1, 1024, fold_smem, st>>>(h->d_vals, h->d_node_l, h->d_node_r, h->d_group_off,
                                                         h->n_groups, h->n_leaves, h->d_psum);
    } else {
      tree_fold_kernel<false><<<1, 1024, 0, st>>>(h->d_vals, h->d_node_l, h->d_node_r, h->d_group_off, h->n_groups,
                                                  h->n_leaves, h->d_psum);
    }
    GCRL_LAUNCHED();
  }
  const int tiles = blocks_for(n, kScanTile);
  normalise_scan_kernel<<<tiles, kScanThreads, 0, st>>>(h->g.prio, call, cap, n, h->d_psum, h->pnorm, h->fixed,
                                                        h->tile_sum, h->d_flags);
  GCRL_LAUNCHED();
  tile_scan_kernel<<<1, 1024, 0, st>>>(h->tile_sum, tiles, h->d_total, h->d_flags);
  GCRL_LAUNCHED();
  cdf_from_fixed_kernel<<<tiles, kScanThreads, 0, st>>>(h->fixed, h->tile_sum, h->d_total, n, h->d_flags);
  GCRL_LAUNCHED();
  double *cdf = reinterpret_cast<double *>(h->fixed);
  {   // inexact additions: summarise the chunks, walk them in order, expand (all three return at once otherwise)
    const int n_chunks = blocks_for(n, kChunk);
    ChunkSum *sums = static_cast<ChunkSum *>(h->d_chunk_sums);
    chunk_summary_kernel<<<blocks_for(int64_t(n_chunks) * 32, 256), 256, 0, st>>>(h->pnorm, h->fixed, h->tile_sum, n, n_chunks,
                                                                               sums, h->d_flags);
    GCRL_LAUNCHED();
    chunk_walk_kernel<<<1, 32, 0, st>>>(h->pnorm, cdf, n, n_chunks, sums, h->d_chunk_in, h->d_chunk_expand, h->d_last,
                                        h->d_flags);
    GCRL_LAUNCHED();
    chunk_expand_kernel<<<blocks_for(int64_t(n_chunks) * 32, 256), 256, 0, st>>>(h->pnorm, cdf, n, n_chunks, sums,
                                                                              h->d_chunk_in, h->d_chunk_expand, h->d_flags);
    GCRL_LAUNCHED();
  }
  cdf_divide_kernel<<<std::min(tiles, sm_count() * 8), 256, 0, st>>>(cdf, n, h->d_last, h->d_flags);
  GCRL_LAUNCHED();
  per_draw_kernel<<<blocks_for(B * 32, 256), 256, 0, st>>>(h->g, call, n, cdf, h->pnorm, u, int(B), s, a, r, ns, d,
                                                          h->d_wraw, h->d_pos, h->d_slot);
  GCRL_LAUNCHED();
  weight_norm_kernel<<<1, 1024, 0, st>>>(h->d_wraw, weights_dev, int(B));
  GCRL_LAUNCHED();
}

// update_priorities of the positions the preceding draw left in d_slot (winner is back to -1 after each write)
void issue_write_back(gcrl_replay *h, int64_t B, const float *td_dev, cudaStream_t st) {
  prio_winner_kernel<<<blocks_for(B, 256), 256, 0, st>>>(h->d_slot, int(B), h->winner);
  GCRL_LAUNCHED();
  prio_write_kernel<<<blocks_for(B, 256), 256, 0, st>>>(h->d_slot, td_dev, int(B), float(h->alpha), 1e-6f, h->g.prio,
                                                       h->winner);
  GCRL_LAUNCHED();
}

void require_outputs(const float *s, const float *a, const float *r, const float *ns, const float *d) {
  GCRL_REQUIRE(s && a && r && ns && d, "NULL batch pointer");
}

const PerCall *many_call(const gcrl_replay *h, int i) { return reinterpret_cast<const PerCall *>(h->d_many) + i; }
const void *many_payload(const gcrl_replay *h, int n, int64_t B, int i) {
  return h->d_many + size_t(n) * sizeof(PerCall) + size_t(i) * size_t(B) * 8;
}

}  // namespace

// ---- graph-safe pieces of n-update calls (agent.cu, sac.cu) ------------------------------------------------------
// The agent stages the call once (host), then records or issues, per update i, sample(i) -> its update ->
// write_back(td) (prioritised).  Every launch reads what changes between calls -- ring start, beta, uniforms or
// positions -- from the staged slots, and the priorities carry over from one update to the next in stream order.
namespace gcrl {

bool replay_prioritized(const gcrl_replay *h) { return h->prioritized; }
int replay_state_dim(const gcrl_replay *h) { return h->g.D; }
int replay_act_dim(const gcrl_replay *h) { return h->g.A; }
int replay_device(const gcrl_replay *h) { return h->device; }
uint64_t replay_epoch(const gcrl_replay *h) { return h->epoch; }
int64_t replay_many_n(const gcrl_replay *h) { return h->many_n; }

// Checks the call (moving nothing when it is refused), then moves every update's PerCall {ring start, -beta[i]} and
// its uniforms u_host[i] (prioritised) or positions pos_host[i] (uniform) to the device in ONE pinned copy.  The
// summation tree for the current length is built here, outside any capture.
void replay_many_stage(gcrl_replay *h, int64_t B, int n, const int64_t *pos_host, const double *u_host,
                       const double *beta, cudaStream_t st) {
  GCRL_REQUIRE(n >= 1 && n <= GCRL_MAX_MANY_STEPS, "n must be in [1, GCRL_MAX_MANY_STEPS]");
  if (h->prioritized) GCRL_REQUIRE(u_host != nullptr && beta != nullptr, "a prioritised buffer needs the uniforms and beta");
  else GCRL_REQUIRE(pos_host != nullptr, "a uniform buffer needs the positions");
  if (h->len < B) throw Error(GCRL_ERR_UNDERFILLED, "[ERROR] Not enough in buffer to sample");
  if (!h->prioritized)
    for (int64_t i = 0; i < int64_t(n) * B; ++i)
      if (pos_host[i] < 0 || pos_host[i] >= h->len) throw Error(GCRL_ERR_INVALID, "sample index out of range [0, len)");
  const size_t calls = size_t(n) * sizeof(PerCall), payload = size_t(n) * size_t(B) * 8;
  if (calls + payload > h->many_cap) {
    GCRL_CUDA(cudaStreamSynchronize(st));
    if (h->d_many) GCRL_CUDA(cudaFree(h->d_many));
    h->d_many = nullptr;
    h->many_cap = 0;
    new_epoch(h);
    h->d_many = dev_alloc<char>((calls + payload) * 2);
    h->many_cap = (calls + payload) * 2;
  }
  if (h->prioritized) {
    ensure_batch(h, B, st);
    build_tree(h, h->len, st);
  }
  int sl;
  char *p = h->stage.acquire(calls + payload, &sl);
  for (int i = 0; i < n; ++i) {
    const PerCall c{h->start(), h->prioritized ? float(-beta[i]) : 0.f, 0};
    std::memcpy(p + size_t(i) * sizeof(PerCall), &c, sizeof(PerCall));
  }
  std::memcpy(p + calls, h->prioritized ? static_cast<const void *>(u_host) : static_cast<const void *>(pos_host), payload);
  GCRL_CUDA(cudaMemcpyAsync(h->d_many, p, calls + payload, cudaMemcpyHostToDevice, st));
  h->stage.release(sl, st);
  h->many_n = h->len;
  if (h->prioritized) h->last_B = B;          // last_positions / update_priorities_last refer to this batch afterwards
}

// The batch of update i of the staged call into s .. d; the importance weights into weights_dev (prioritised)
void replay_many_sample(gcrl_replay *h, int64_t B, int n, int i, float *s, float *a, float *r, float *ns, float *d,
                        float *weights_dev, cudaStream_t st) {
  if (h->prioritized) {
    issue_draw(h, h->many_n, B, many_call(h, i), static_cast<const double *>(many_payload(h, n, B, i)), s, a, r, ns, d,
               weights_dev, st);
  } else {
    uniform_gather_kernel<<<blocks_for(B * 32, 256), 256, 0, st>>>(
        h->g, 0, many_call(h, i), static_cast<const int64_t *>(many_payload(h, n, B, i)), int(B), s, a, r, ns, d);
    GCRL_LAUNCHED();
  }
}

// update_priorities of update i's positions with its per-sample TD errors (prioritised)
void replay_many_write_back(gcrl_replay *h, int64_t B, const float *td_dev, cudaStream_t st) {
  issue_write_back(h, B, td_dev, st);
}

}  // namespace gcrl

extern "C" {

int gcrl_replay_create(gcrl_replay **out, int device, int64_t capacity, int state_dim, int act_dim,
                       int prioritized, double alpha) {
  GCRL_API_BEGIN
  GCRL_REQUIRE(out != nullptr, "out is NULL");
  GCRL_REQUIRE(capacity >= 1 && capacity < (int64_t(1) << 31), "capacity must be in [1, 2^31)");
  GCRL_REQUIRE(state_dim >= 1 && act_dim >= 1, "bad state_dim / act_dim");
  GCRL_REQUIRE(!prioritized || alpha >= 0.0, "alpha must be >= 0");
  GCRL_CUDA(cudaSetDevice(device));
  auto *h = new gcrl_replay();
  try {
    h->device = device;
    h->prioritized = prioritized != 0;
    h->alpha = alpha;
    h->g.cap = capacity;
    h->g.D = state_dim;
    h->g.A = act_dim;
    h->g.row_f = (2 * state_dim + act_dim + 2 + 3) & ~3;
    h->g.rows = dev_alloc<float>(size_t(capacity) * h->g.row_f);
    if (h->prioritized) {
      h->g.prio = dev_alloc<float>(size_t(capacity));
      h->pnorm = dev_alloc<float>(size_t(capacity));
      h->fixed = dev_alloc<int64_t>(size_t(capacity));
      h->tile_sum = dev_alloc<int64_t>(size_t(capacity / kScanTile + 2));
      h->d_total = dev_alloc<int64_t>(1);
      h->d_last = dev_alloc<double>(1);
      {
        const size_t nc = size_t(capacity / kChunk + 2);
        h->d_chunk_sums = dev_alloc<ChunkSum>(nc);
        h->d_chunk_in = dev_alloc<double>(nc);
        h->d_chunk_expand = dev_alloc<unsigned char>(nc);
      }
      h->d_psum = dev_alloc<float>(1);
      h->d_flags = dev_alloc<int>(1);
      h->d_call = dev_alloc<PerCall>(1);
      GCRL_CUDA(cudaStreamCreateWithFlags(&h->cap_stream, cudaStreamNonBlocking));
      h->use_graphs = graphs_enabled();
      h->winner = dev_alloc<int>(size_t(capacity));
      fill_i32_kernel<<<blocks_for(capacity, 256 * 8), 256>>>(h->winner, capacity, -1);
      GCRL_LAUNCHED();
      GCRL_CUDA(cudaMemset(h->d_flags, 0, sizeof(int)));
      GCRL_CUDA(cudaDeviceSynchronize());
    }
    h->stage.init(size_t(1) << 16);
    new_epoch(h);
  } catch (...) {
    delete h;
    throw;
  }
  *out = h;
  GCRL_API_END
}

int gcrl_replay_destroy(gcrl_replay *h) {
  GCRL_API_BEGIN
  if (h == nullptr) return GCRL_OK;
  cudaSetDevice(h->device);
  cudaDeviceSynchronize();
  for (void *p : {(void *)h->g.rows, (void *)h->g.prio, (void *)h->pnorm, (void *)h->fixed, (void *)h->tile_sum,
                  (void *)h->d_total, (void *)h->d_last, h->d_chunk_sums, (void *)h->d_chunk_in, (void *)h->d_chunk_expand, (void *)h->d_psum, (void *)h->d_flags, (void *)h->winner,
                  (void *)h->d_leaf_off, (void *)h->d_node_l, (void *)h->d_node_r, (void *)h->d_group_off,
                  (void *)h->d_vals, (void *)h->d_u, (void *)h->d_wraw, (void *)h->d_pos, (void *)h->d_slot})
    if (p) cudaFree(p);
  if (h->graph.exec) cudaGraphExecDestroy(h->graph.exec);
  if (h->cap_stream) cudaStreamDestroy(h->cap_stream);
  if (h->d_call) cudaFree(h->d_call);
  if (h->d_many) cudaFree(h->d_many);
  h->stage.destroy();
  delete h;
  GCRL_API_END
}

int64_t gcrl_replay_len(gcrl_replay *h) { return h ? h->len : -1; }
int64_t gcrl_replay_total(gcrl_replay *h) { return h ? h->total : -1; }

int gcrl_replay_push(gcrl_replay *h, int64_t n, const float *rows_host, void *stream) {
  GCRL_API_BEGIN
  GCRL_REQUIRE(h != nullptr && rows_host != nullptr && n >= 0, "bad argument");
  GCRL_CUDA(cudaSetDevice(h->device));
  cudaStream_t st = as_stream(stream);
  const int wf = 2 * h->g.D + h->g.A + 2, rf = h->g.row_f;
  const int64_t cap = h->g.cap;
  int64_t skip = std::max<int64_t>(0, n - cap);            // a deque(maxlen) keeps only the newest `cap`
  h->total += skip;
  h->len = std::max<int64_t>(0, h->len - skip);
  for (int64_t done = skip; done < n;) {
    const int64_t slot = h->total % cap;
    const int64_t m = std::min<int64_t>({n - done, cap - slot, int64_t(16384)});
    int sl;
    char *p = h->stage.acquire(size_t(m) * wf * 4, &sl);
    std::memcpy(p, rows_host + done * wf, size_t(m) * wf * 4);
    GCRL_CUDA(cudaMemcpy2DAsync(h->g.rows + slot * rf, size_t(rf) * 4, p, size_t(wf) * 4, size_t(wf) * 4, size_t(m),
                                cudaMemcpyHostToDevice, st));
    h->stage.release(sl, st);
    if (h->prioritized) {
      fill_kernel<<<blocks_for(m, 256), 256, 0, st>>>(h->g.prio, slot, m, cap, 1.0f);
      GCRL_LAUNCHED();
    }
    h->total += m;
    h->len = std::min(cap, h->len + m);
    done += m;
  }
  GCRL_API_END
}

int gcrl_replay_sample(gcrl_replay *h, int64_t B, const int64_t *idx_host, float *s, float *a, float *r, float *ns,
                       float *d, void *stream) {
  GCRL_API_BEGIN
  GCRL_REQUIRE(h != nullptr && idx_host != nullptr && B >= 1, "bad argument");
  require_outputs(s, a, r, ns, d);
  GCRL_REQUIRE(h->len >= B, "Not enough in buffer to sample");
  for (int64_t i = 0; i < B; ++i) GCRL_REQUIRE(idx_host[i] >= 0 && idx_host[i] < h->len, "position outside the buffer");
  GCRL_CUDA(cudaSetDevice(h->device));
  cudaStream_t st = as_stream(stream);
  ensure_batch(h, B, st);
  int sl;
  char *p = h->stage.acquire(size_t(B) * 8, &sl);
  std::memcpy(p, idx_host, size_t(B) * 8);
  GCRL_CUDA(cudaMemcpyAsync(h->d_pos, p, size_t(B) * 8, cudaMemcpyHostToDevice, st));
  h->stage.release(sl, st);
  uniform_gather_kernel<<<blocks_for(B * 32, 256), 256, 0, st>>>(h->g, h->start(), nullptr, h->d_pos, int(B), s, a, r,
                                                                 ns, d);
  GCRL_LAUNCHED();
  GCRL_API_END
}

int gcrl_replay_sample_prioritized(gcrl_replay *h, int64_t B, const double *u_host, double beta, float *s, float *a,
                                   float *r, float *ns, float *d, float *weights_dev, int64_t *idx_host_out,
                                   void *stream) {
  GCRL_API_BEGIN
  GCRL_REQUIRE(h != nullptr && h->prioritized, "not a prioritised buffer");
  GCRL_REQUIRE(u_host != nullptr && weights_dev != nullptr && B >= 1, "bad argument");
  require_outputs(s, a, r, ns, d);
  GCRL_REQUIRE(h->len >= B, "Not enough in buffer to sample");
  GCRL_CUDA(cudaSetDevice(h->device));
  cudaStream_t st = as_stream(stream);
  ensure_batch(h, B, st);
  const int64_t n = h->len, start = h->start();
  build_tree(h, n, st);
  {   // per-call scalars + the B uniforms: one pinned slot, two small copies
    int sl;
    char *p = h->stage.acquire(size_t(B) * 8 + sizeof(PerCall), &sl);
    PerCall hc{start, float(-beta), 0};
    std::memcpy(p, &hc, sizeof(PerCall));
    std::memcpy(p + sizeof(PerCall), u_host, size_t(B) * 8);
    GCRL_CUDA(cudaMemcpyAsync(h->d_call, p, sizeof(PerCall), cudaMemcpyHostToDevice, st));
    GCRL_CUDA(cudaMemcpyAsync(h->d_u, p + sizeof(PerCall), size_t(B) * 8, cudaMemcpyHostToDevice, st));
    h->stage.release(sl, st);
  }
  auto launch_all = [&](cudaStream_t st) {
    issue_draw(h, n, B, h->d_call, h->d_u, s, a, r, ns, d, weights_dev, st);
  };
  // The draw is 11 small launches: replayed as one graph once the same (length, batch, outputs) repeats -- i.e.
  // as soon as the ring is full; while it is still filling every call has a new length and launches directly.
  gcrl_replay::DrawKey key;
  key.n = n; key.B = B;
  const void *ptrs[6] = {s, a, r, ns, d, weights_dev};
  std::memcpy(key.ptr, ptrs, sizeof(ptrs));
  if (h->use_graphs && h->graph.exec != nullptr && key == h->graph_key) {
    launch_graph(h->graph, st);
  } else if (h->use_graphs && key == h->last_key) {
    if (h->graph.exec) { cudaGraphExecDestroy(h->graph.exec); h->graph.exec = nullptr; }
    h->graph = capture_graph(h->cap_stream, launch_all);
    h->graph_key = key;
    launch_graph(h->graph, st);
  } else {
    launch_all(st);
  }
  h->last_key = key;
  h->last_B = B;
  if (idx_host_out != nullptr) {
    GCRL_CUDA(cudaMemcpyAsync(idx_host_out, h->d_pos, size_t(B) * 8, cudaMemcpyDeviceToHost, st));
    GCRL_CUDA(cudaStreamSynchronize(st));
  }
  GCRL_API_END
}

int gcrl_replay_update_priorities(gcrl_replay *h, int64_t B, const int64_t *idx_host, const float *td_dev,
                                  void *stream) {
  GCRL_API_BEGIN
  GCRL_REQUIRE(h != nullptr && h->prioritized && td_dev != nullptr && B >= 1, "bad argument");
  GCRL_CUDA(cudaSetDevice(h->device));
  cudaStream_t st = as_stream(stream);
  if (idx_host != nullptr) {                       // explicit deque positions (any caller-held index list)
    ensure_batch(h, B, st);
    int sl;
    int64_t *p = reinterpret_cast<int64_t *>(h->stage.acquire(size_t(B) * 8, &sl));
    const int64_t start = h->start(), cap = h->g.cap;
    for (int64_t i = 0; i < B; ++i) {
      GCRL_REQUIRE(idx_host[i] >= 0 && idx_host[i] < h->len, "position outside the buffer");
      p[i] = (start + idx_host[i]) % cap;
    }
    GCRL_CUDA(cudaMemcpyAsync(h->d_slot, p, size_t(B) * 8, cudaMemcpyHostToDevice, st));
    h->stage.release(sl, st);
  } else {
    GCRL_REQUIRE(B == h->last_B, "update_priorities without positions must follow the sample() of the same batch");
  }
  issue_write_back(h, B, td_dev, st);
  h->last_B = idx_host != nullptr ? 0 : h->last_B;
  GCRL_API_END
}

int gcrl_replay_get_priorities(gcrl_replay *h, float *prio_host, void *stream) {
  GCRL_API_BEGIN
  GCRL_REQUIRE(h != nullptr && h->prioritized && prio_host != nullptr, "bad argument");
  GCRL_CUDA(cudaSetDevice(h->device));
  cudaStream_t st = as_stream(stream);
  const int64_t start = h->start(), first = std::min(h->len, h->g.cap - start);
  GCRL_CUDA(cudaMemcpyAsync(prio_host, h->g.prio + start, size_t(first) * 4, cudaMemcpyDeviceToHost, st));
  if (h->len > first)
    GCRL_CUDA(cudaMemcpyAsync(prio_host + first, h->g.prio, size_t(h->len - first) * 4, cudaMemcpyDeviceToHost, st));
  GCRL_CUDA(cudaStreamSynchronize(st));
  GCRL_API_END
}

int gcrl_replay_set_priorities(gcrl_replay *h, const float *prio_host, int64_t n, void *stream) {
  GCRL_API_BEGIN
  GCRL_REQUIRE(h != nullptr && h->prioritized && prio_host != nullptr && n == h->len, "bad argument");
  GCRL_CUDA(cudaSetDevice(h->device));
  cudaStream_t st = as_stream(stream);
  const int64_t start = h->start(), first = std::min(h->len, h->g.cap - start);
  GCRL_CUDA(cudaStreamSynchronize(st));
  GCRL_CUDA(cudaMemcpy(h->g.prio + start, prio_host, size_t(first) * 4, cudaMemcpyHostToDevice));
  if (h->len > first)
    GCRL_CUDA(cudaMemcpy(h->g.prio, prio_host + first, size_t(h->len - first) * 4, cudaMemcpyHostToDevice));
  GCRL_API_END
}

int gcrl_replay_get_rows(gcrl_replay *h, int64_t first, int64_t n, float *rows_host, void *stream) {
  GCRL_API_BEGIN
  GCRL_REQUIRE(h != nullptr && rows_host != nullptr && first >= 0 && n >= 0 && first + n <= h->len, "bad range");
  GCRL_CUDA(cudaSetDevice(h->device));
  cudaStream_t st = as_stream(stream);
  const int wf = 2 * h->g.D + h->g.A + 2, rf = h->g.row_f;
  const int64_t cap = h->g.cap;
  for (int64_t done = 0; done < n;) {
    const int64_t slot = (h->start() + first + done) % cap;
    const int64_t m = std::min(n - done, cap - slot);
    GCRL_CUDA(cudaMemcpy2DAsync(rows_host + done * wf, size_t(wf) * 4, h->g.rows + slot * rf, size_t(rf) * 4,
                                size_t(wf) * 4, size_t(m), cudaMemcpyDeviceToHost, st));
    done += m;
  }
  GCRL_CUDA(cudaStreamSynchronize(st));
  GCRL_API_END
}

int gcrl_replay_last_sample_info(gcrl_replay *h, float *priority_sum, int *sequential_cumsum, void *stream) {
  GCRL_API_BEGIN
  GCRL_REQUIRE(h != nullptr && h->prioritized, "bad argument");
  GCRL_CUDA(cudaSetDevice(h->device));
  GCRL_CUDA(cudaStreamSynchronize(as_stream(stream)));
  if (priority_sum) GCRL_CUDA(cudaMemcpy(priority_sum, h->d_psum, 4, cudaMemcpyDeviceToHost));
  if (sequential_cumsum) {
    int f = 0;
    GCRL_CUDA(cudaMemcpy(&f, h->d_flags, 4, cudaMemcpyDeviceToHost));
    *sequential_cumsum = f & 1;
  }
  GCRL_API_END
}

int gcrl_replay_last_positions(gcrl_replay *h, int64_t B, int64_t *idx_host, void *stream) {
  GCRL_API_BEGIN
  GCRL_REQUIRE(h != nullptr && h->prioritized && idx_host != nullptr, "bad argument");
  GCRL_REQUIRE(B >= 1 && B == h->last_B, "no prioritised sample of this batch size to report");
  GCRL_CUDA(cudaSetDevice(h->device));
  cudaStream_t st = as_stream(stream);
  GCRL_CUDA(cudaMemcpyAsync(idx_host, h->d_pos, size_t(B) * 8, cudaMemcpyDeviceToHost, st));
  GCRL_CUDA(cudaStreamSynchronize(st));
  GCRL_API_END
}

int gcrl_replay_last_tables(gcrl_replay *h, float *pnorm_host, double *cdf_host, void *stream) {
  GCRL_API_BEGIN
  GCRL_REQUIRE(h != nullptr && h->prioritized, "bad argument");
  GCRL_CUDA(cudaSetDevice(h->device));
  GCRL_CUDA(cudaStreamSynchronize(as_stream(stream)));
  const int64_t n = h->tree_n;
  GCRL_REQUIRE(n >= 1 && n == h->len, "no sample() at the current length");
  if (pnorm_host) GCRL_CUDA(cudaMemcpy(pnorm_host, h->pnorm, size_t(n) * 4, cudaMemcpyDeviceToHost));
  if (cdf_host) GCRL_CUDA(cudaMemcpy(cdf_host, h->fixed, size_t(n) * 8, cudaMemcpyDeviceToHost));
  GCRL_API_END
}

}  // extern "C"
