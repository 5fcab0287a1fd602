// Device-side view of the HER episode store (csrc/her.cu), shared with the row-slab update kernel (fused.cu), which
// samples its own rows: position -> (episode, t, j) -> packed row + relabel goal, the mapping SURVEY.md 8(a-3) proves
// equal to apply_her entry for entry (reference src/buffer.py:143-179).  Online relabelling (online_k > 0, a store
// with K = 0) draws the relabel coin and goal step per sampled row instead (DESIGN.md section 2).
#pragma once
#include "common.cuh"

namespace gcrl {

constexpr int kBucketShift = 6;
constexpr int kSamplesPerBlock = 128;
constexpr int kSampleThreads = 256;

struct __align__(16) EpRec {
  int64_t entry_start;
  uint32_t tr_slot;
  uint32_t T;
};

struct __align__(32) BucketRec {     // the episode that holds entry (bucket << kBucketShift)
  int64_t entry_start;
  uint32_t tr_slot;
  uint32_t T;
  int64_t eid;
  int64_t pad;
};

struct HerHeader {
  int64_t total_entries;
  int64_t len;
  int64_t ep_first;
  int64_t ep_last;
  unsigned long long draw_epoch;
  unsigned int ticket;
  unsigned int pad;
};

struct HerGeom {
  float *rows;
  float *ag;
  EpRec *eps;
  BucketRec *buckets;
  HerHeader *hdr;
  uint32_t cap_tr, ep_mask, bucket_mask;
  int D, G, A, K, row_f, gpad;
  int off_ns, off_a, off_r, off_d, off_ag, off_fut;
  FastDiv div_k1, div_D, div_A, div_rf4;
  uint64_t seed;
  float threshold;          // sparse reward: -(||ag - g|| > threshold), 0.05 for the Panda tasks
  int strategy;             // goal selection: GCRL_HER_FUTURE / _FINAL / _EPISODE
  int online_k;             // > 0: online relabelling, each sampled row relabelled with probability k / (k + 1)
};

// totals by value (or through a small device struct for graph-captured consumers): the host mirrors the deque
// counters and counts the device-stream draws, so no thread waits on a header load before it can compute anything
struct SampleScalars {
  int64_t total_entries, len;
  unsigned long long draw_epoch;
  long long use_idx;          // != 0: positions come from the index buffer (the host's random.sample stream)
};

// ---------------------------------------------------------------------------------------
// on-device index stream: keyed 4-round Feistel permutation of [0, n) with cycle walking.
// Position i of call `epoch` is perm_epoch(i): B distinct, uniformly spread positions,
// i.e. sampling WITHOUT replacement like random.sample (reference src/buffer.py:124).
// ---------------------------------------------------------------------------------------
__host__ __device__ inline int64_t feistel_position(uint64_t x, uint64_t n, uint64_t seed,
                                                    uint64_t epoch) {
  if (n <= 1) return 0;
  int b = 0;
  while (b < 63 && (1ull << b) < n) ++b;
  if (b < 2) b = 2;
  b += (b & 1);
  const int half = b >> 1;
  const uint32_t mask = half >= 32 ? 0xffffffffu : ((1u << half) - 1u);
  const uint64_t k0 = splitmix64(seed ^ (epoch * 0xD1B54A32D192ED03ull));
  const uint64_t k1 = splitmix64(k0);
  const uint32_t keys[4] = {uint32_t(k0), uint32_t(k0 >> 32), uint32_t(k1), uint32_t(k1 >> 32)};
  do {
    uint32_t L = uint32_t(x >> half) & mask, R = uint32_t(x) & mask;
#ifdef __CUDA_ARCH__   // (the host compiler does not know the pragma and warns)
#pragma unroll
#endif
    for (int r = 0; r < 4; ++r) {
      uint32_t nl = R;
      R = L ^ (mix32(R ^ keys[r]) & mask);
      L = nl;
    }
    x = (uint64_t(L) << half) | R;
  } while (x >= n);
  return int64_t(x);
}

// Online relabelling: the 64-bit hash of (buffer seed, draw epoch, batch row i).  Row i is relabelled iff
// h % (k + 1) != 0, to goal step lo + (h >> 32) % (T - lo) (lo = t + 1 for `future`, 0 for `episode`).
__host__ __device__ inline uint64_t her_relabel_hash(uint64_t seed, uint64_t epoch, uint64_t i) {
  return splitmix64(splitmix64(seed ^ 0x6A09E667F3BCC909ull ^ (epoch * 0xD1B54A32D192ED03ull)) + i);
}

// One sample: deque position -> bucket record -> (episode, t, j) -> ring slot.  `futw` receives the 4 packed
// future offsets that contain this relabel's (j > 0), loaded here so that it travels with the row gather.  Where
// the goal step f is known without that load (online mode, eager `final`), futw carries f in every byte instead
// (online mode: j = 1 and f in the low byte), so her_future_slot reads it the same way.
struct SampleRef {
  uint32_t slot, ep0, j, futw;
};

// The n-step sampler also needs the sample's step t and its episode's length T (the window is t .. t+k-1).
struct SampleRefN {
  SampleRef r;
  uint32_t t, T;
};

__device__ __forceinline__ SampleRefN her_resolve_n(const HerGeom &g, const SampleScalars &sc, int64_t i,
                                                    const int64_t *__restrict__ idx, int64_t *__restrict__ idx_out) {
  int64_t p;
  if (idx != nullptr) {
    p = idx[i];
    p = p < 0 ? 0 : (p >= sc.len ? sc.len - 1 : p);
  } else {
    p = feistel_position(uint64_t(i), uint64_t(sc.len), g.seed, sc.draw_epoch);
  }
  if (idx_out != nullptr) idx_out[i] = p;
  const int64_t ge = sc.total_entries - sc.len + p;  // global entry id
  const int4 *bp = reinterpret_cast<const int4 *>(g.buckets + ((ge >> kBucketShift) & g.bucket_mask));
  const int4 b0 = __ldg(bp), b1 = __ldg(bp + 1);
  int64_t entry_start = (int64_t(uint32_t(b0.y)) << 32) | uint32_t(b0.x);
  uint32_t tr_slot = uint32_t(b0.z), T = uint32_t(b0.w);
  int64_t eid = (int64_t(uint32_t(b1.y)) << 32) | uint32_t(b1.x);
  // the bucket's episode holds entry (bucket << 6); the position may belong to a later one (an episode of 50
  // steps spans 246 entries = ~4 buckets, so usually it does not): walk forward over the episode records
  while (ge >= entry_start + int64_t(T - 1) * (g.K + 1) + 1) {
    ++eid;
    const EpRec r2 = g.eps[eid & g.ep_mask];
    entry_start = r2.entry_start; tr_slot = r2.tr_slot; T = r2.T;
  }
  const uint32_t o = uint32_t(ge - entry_start);
  uint32_t t = g.div_k1.div(o);
  uint32_t j = o - t * uint32_t(g.K + 1);
  if (t >= T - 1) { t = T - 1; j = 0; }  // last step carries no relabels
  uint32_t slot = tr_slot + t;
  if (slot >= g.cap_tr) slot -= g.cap_tr;
  SampleRef r{slot, tr_slot, j, 0u};
  if (g.online_k > 0) {            // K == 0 store: j == 0 above; the goal's slot is known after this round trip
    const uint64_t h = her_relabel_hash(g.seed, sc.draw_epoch, uint64_t(i));
    const uint32_t lo = g.strategy == GCRL_HER_EPISODE ? 0u : t + 1;
    if (lo < T && h % uint64_t(g.online_k + 1) != 0) {
      r.j = 1;
      r.futw = g.strategy == GCRL_HER_FINAL ? T - 1 : lo + uint32_t(h >> 32) % (T - lo);
    }
  } else if (j > 0) {
    r.futw = g.strategy == GCRL_HER_FINAL
                 ? (T - 1) * 0x01010101u
                 : __ldg(reinterpret_cast<const uint32_t *>(g.rows + size_t(slot) * g.row_f + g.off_fut) + ((j - 1) >> 2));
  }
  return SampleRefN{r, t, T};
}

__device__ __forceinline__ SampleRef her_resolve(const HerGeom &g, const SampleScalars &sc, int64_t i,
                                                 const int64_t *__restrict__ idx, int64_t *__restrict__ idx_out) {
  return her_resolve_n(g, sc, i, idx, idx_out).r;
}

// n-step returns (gcrl_her_set_n_step): fixed for the buffer's lifetime, passed beside HerGeom so that the row-slab
// kernel, which embeds HerGeom in its arguments, keeps its parameter layout
struct NStepArgs {
  int n;          // 1: one-step rows
  float gamma;
};

// ring slot of the transition whose achieved goal relabels this sample (j > 0)
__device__ __forceinline__ uint32_t her_future_slot(const HerGeom &g, const SampleRef &r) {
  uint32_t fs = r.ep0 + ((r.futw >> (8 * ((r.j - 1) & 3))) & 0xffu);
  if (fs >= g.cap_tr) fs -= g.cap_tr;
  return fs;
}

// Relabel one packed row in place (shared memory): goal columns of s and s' <- future achieved goal, reward <-
// sparse rule in unfused IEEE fp32 (left-to-right sum, no FMA), done <- 0.
__device__ __forceinline__ void her_relabel_row(const HerGeom &g, float *row, const float *gf /* [G] */) {
  float acc = 0.f;
  for (int c = 0; c < g.G; ++c) {
    const float diff = __fsub_rn(row[g.off_ag + c], gf[c]);    // achieved(t) - future goal
    const float sq = __fmul_rn(diff, diff);
    acc = (c == 0) ? sq : __fadd_rn(acc, sq);
    row[g.D - g.G + c] = gf[c];
    row[g.off_ns + g.D - g.G + c] = gf[c];
  }
  const float dist = __fsqrt_rn(acc);
  // -(d > threshold) as float32: -1.0f, or -0.0f with the SIGN BIT SET on success
  // (-np.array(False, float32)).  Written as an INTEGER word: with a float-typed select
  // nvcc 12.9 rewrites {-1.0f, -0.0f} into int->float(-(int)pred), which yields +0.0f.
  reinterpret_cast<uint32_t *>(row)[g.off_r] = 0x80000000u | ((dist > g.threshold) ? 0x3F800000u : 0u);
  row[g.off_d] = 0.0f;                                        // new_done = False
}

}  // namespace gcrl
