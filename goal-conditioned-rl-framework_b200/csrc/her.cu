// Device-resident HER episode store + lazy future-relabelling sampler (sm_100a).
//
// Replaces HERBuffer (reference src/buffer.py:92-179).  The reference materialises
// every relabelled copy into a Python deque at episode end; here only the T raw
// transitions of an episode are stored (one packed row each) and sample() maps a deque
// position -> (episode, t, j) -> relabelled transition on the fly.  The mapping is the
// one SURVEY.md 8(a-3) proves entry-for-entry equal to apply_her.
//
// HBM layout (all fp32 words, row stride a multiple of 16 B):
//   rows[cap_tr][row_f] : s[D] | ns[D] | a[A] | r | d | ag[G] | fut[k] (uint8, packed) | pad
//   ag  [cap_tr][gpad]  : compact copy of ag so the future-goal gather touches a 12-16 B
//                         row of a small (L2-resident at 1M transitions) array
//   eps [cap_ep]        : {entry_start, tr_slot, T} per live episode (ring, pow2)
//   buckets[nb]         : the RECORD {entry_start, tr_slot, T, id} of the episode holding entry (b << 6)
//                         (ring, pow2, 32 B): position -> episode in ONE load for the common case (the position
//                         falls into that episode), else a short forward walk over eps
//   hdr                 : totals, maintained by the commit kernel (diagnostics; the sampler gets them by value)
//
// The sampler is a chain of dependent gathers, so its latency is the number of HBM round trips on that chain:
// bucket record -> (packed row || future-offset word) -> future goal = 3 (round 1: header -> bucket -> episode
// record -> binary search -> two rounds of row loads -> future goal = 6-7).  Online relabelling and eager `final`
// know the goal step after the bucket record, so there the goal gather runs beside the row gather: 2.
#include <algorithm>
#include <cstring>
#include <deque>
#include <vector>

#include "her_device.cuh"

namespace gcrl {

struct __align__(16) CommitHdr {
  int64_t entry_start, eid, total_entries, len, ep_first, first_bucket;
  uint32_t n_buckets, tr_slot, T, pad;
};
static_assert(sizeof(CommitHdr) == 64, "CommitHdr must be 64 bytes");

// ---------------------------------------------------------------------------------------
// commit: scatter one staged episode blob into the rings
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) her_commit_kernel(HerGeom g, const char *__restrict__ blob) {
  const CommitHdr h = *reinterpret_cast<const CommitHdr *>(blob);
  const float4 *src_rows = reinterpret_cast<const float4 *>(blob + sizeof(CommitHdr));
  const int rf4 = g.row_f >> 2, g4 = g.gpad >> 2;
  const float4 *src_ag = src_rows + size_t(h.T) * rf4;
  float4 *rows4 = reinterpret_cast<float4 *>(g.rows);
  float4 *ag4 = reinterpret_cast<float4 *>(g.ag);
  const int tid = blockIdx.x * blockDim.x + threadIdx.x;
  const int nth = gridDim.x * blockDim.x;
  for (int e = tid; e < int(h.T) * rf4; e += nth) {
    uint32_t t = g.div_rf4.div(e), q = e - t * rf4;
    uint32_t slot = h.tr_slot + t;
    if (slot >= g.cap_tr) slot -= g.cap_tr;
    rows4[size_t(slot) * rf4 + q] = src_rows[e];
  }
  for (int e = tid; e < int(h.T) * g4; e += nth) {
    uint32_t t = e / g4, q = e - t * g4;
    uint32_t slot = h.tr_slot + t;
    if (slot >= g.cap_tr) slot -= g.cap_tr;
    ag4[size_t(slot) * g4 + q] = src_ag[e];
  }
  for (int b = tid; b < int(h.n_buckets); b += nth) {
    BucketRec br;
    br.entry_start = h.entry_start; br.tr_slot = h.tr_slot; br.T = h.T; br.eid = h.eid; br.pad = 0;
    g.buckets[(h.first_bucket + b) & g.bucket_mask] = br;
  }
  if (tid == 0) {
    EpRec rec;
    rec.entry_start = h.entry_start;
    rec.tr_slot = h.tr_slot;
    rec.T = h.T;
    g.eps[h.eid & g.ep_mask] = rec;
    g.hdr->total_entries = h.total_entries;
    g.hdr->len = h.len;
    g.hdr->ep_first = h.ep_first;
    g.hdr->ep_last = h.eid;
  }
}

// ---------------------------------------------------------------------------------------
// sample: gather + relabel + reward, 128 samples per CTA staged through shared memory so
// both the row gathers (16 B vectors, 13 per Push row) and the five output streams are
// coalesced.
// ---------------------------------------------------------------------------------------
template <bool VEC>
__device__ __forceinline__ void write_field(float *__restrict__ out, const float *tile, int n,
                                            int width, int off, int row_f, const FastDiv &dw,
                                            int tid) {
  const int total = n * width;
  if (VEC) {
    for (int q = tid * 4; q < total; q += kSampleThreads * 4) {
      uint32_t i = dw.div(q), c = q - i * width;
      if (q + 3 < total) {
        float v[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          v[u] = tile[i * row_f + off + c];
          if (++c == uint32_t(width)) { c = 0; ++i; }
        }
        stg_stream4(reinterpret_cast<float4 *>(out + q), make_float4(v[0], v[1], v[2], v[3]));
      } else {
        for (int e = q; e < total; ++e) {
          out[e] = tile[i * row_f + off + c];
          if (++c == uint32_t(width)) { c = 0; ++i; }
        }
      }
    }
  } else {
    for (int q = tid; q < total; q += kSampleThreads) {
      uint32_t i = dw.div(q), c = q - i * width;
      out[q] = tile[i * row_f + off + c];
    }
  }
}

// sparse reward of achieved goal `a` against goal `gf` (her_relabel_row's rule): -1.0f, or -0.0f on success
__device__ __forceinline__ float her_sparse_reward(const HerGeom &g, const float *a, const float *gf) {
  float acc = 0.f;
  for (int c = 0; c < g.G; ++c) {
    const float diff = __fsub_rn(a[c], gf[c]);
    const float sq = __fmul_rn(diff, diff);
    acc = (c == 0) ? sq : __fadd_rn(acc, sq);
  }
  // the word goes through an opaque move: seen as a float select of {-1.0f, -0.0f}, nvcc 12.9 rewrites it into
  // int->float(-(int)pred), which yields +0.0f (see her_relabel_row)
  const uint32_t w = 0x80000000u | ((__fsqrt_rn(acc) > g.threshold) ? 0x3F800000u : 0u);
  float r;
  asm("mov.b32 %0, %1;" : "=f"(r) : "r"(w));
  return r;
}

// window steps whose reward word / achieved goal one thread has in flight at once: n <= 7 takes one round of loads
// (a chunk of 8 spills in the 16 B-store instantiation, 6 uses 82 registers and none)
constexpr int kNStepChunk = 6;

// ring slot of window step t+i (i < T - t <= cap_tr: one wrap at most)
__device__ __forceinline__ uint32_t her_window_slot(const HerGeom &g, const SampleRef &r, uint32_t i) {
  uint32_t s = r.slot + i;
  if (s >= g.cap_tr) s -= g.cap_tr;
  return s;
}

// what window step t+i contributes to an n-step reward: its stored reward word (j = 0, in .x), or its achieved goal
// from the compact copy (relabelled, G <= 4; wider goals are read column by column where they are used)
__device__ __forceinline__ float4 her_window_load(const HerGeom &g, const SampleRef &r, uint32_t i) {
  const uint32_t s = her_window_slot(g, r, i);
  if (r.j == 0) return make_float4(__ldg(g.rows + size_t(s) * g.row_f + g.off_r), 0.f, 0.f, 0.f);
  if (g.G <= 4) return __ldg(reinterpret_cast<const float4 *>(g.ag + size_t(s) * g.gpad));
  return make_float4(0.f, 0.f, 0.f, 0.f);
}

// NSTEP: n-step rows (DESIGN.md section 2).  Sample i at step t of an episode of T steps takes the window
// t .. t+k-1, k = min(n, T - t): r <- r_t + gamma (r_{t+1} + gamma (... + gamma r_{t+k-1})) (unfused fp32, from the
// back), s' <- ns of row t+k-1 (goal columns <- the sample's goal), d <- 1 - gamma^(k-1) (1 - done_{t+k-1}), so that
// gamma (1 - d) is the bootstrap weight gamma^k (1 - done).  Relabelled rows recompute every r_{t+i} for their goal
// from the compact ag array and take done = 0.  k = 1 rows are the one-step rows.
template <bool VEC, int SPB, bool NSTEP>
__global__ void __launch_bounds__(kSampleThreads)
her_sample_kernel(const __grid_constant__ HerGeom g, const SampleScalars sc_arg, const SampleScalars *__restrict__ sc_dev,
                  int64_t B, const int64_t *__restrict__ idx,
                  float *__restrict__ out_s, float *__restrict__ out_a, float *__restrict__ out_r,
                  float *__restrict__ out_ns, float *__restrict__ out_d, int64_t *__restrict__ idx_out,
                  const NStepArgs nst) {
  // sc_dev: the totals and draw epoch of this launch's update, written by the host before a replayed graph runs
  // (a value captured into the graph would freeze them); otherwise they come by value
  const SampleScalars sc = sc_dev != nullptr ? *sc_dev : sc_arg;
  extern __shared__ float4 smem4[];
  float *tile = reinterpret_cast<float *>(smem4);
  uint32_t *m_row = reinterpret_cast<uint32_t *>(tile + SPB * g.row_f);
  uint32_t *m_last = m_row + SPB;                                  // NSTEP: ring slot of row t+k-1
  float *tile_ns = reinterpret_cast<float *>(m_last + SPB);        // NSTEP: [SPB][D] s' of row t+k-1

  const int tid = threadIdx.x;
  const int64_t base = int64_t(blockIdx.x) * SPB;
  const int n = int(min(int64_t(SPB), B - base));

  // ---- round trip 1: deque position -> bucket record -> (episode, t, j) -> ring slot (her_device.cuh) ----
  SampleRef ref{0u, 0u, 0u, 0u};
  uint32_t k = 1;
  if (tid < n) {
    if constexpr (NSTEP) {
      const SampleRefN rn = her_resolve_n(g, sc, base + tid, sc.use_idx ? idx : nullptr, idx_out);
      ref = rn.r;
      k = min(uint32_t(nst.n), rn.T - rn.t);
      uint32_t last = ref.slot + k - 1;
      if (last >= g.cap_tr) last -= g.cap_tr;
      m_last[tid] = last;
    } else {
      ref = her_resolve(g, sc, base + tid, sc.use_idx ? idx : nullptr, idx_out);
    }
    m_row[tid] = ref.slot;
  }
  __syncthreads();

  // ---- round trip 2: coalesced 16 B gathers of the packed rows into shared memory, all loads of a thread in flight
  {
    const int rf4 = g.row_f >> 2;
    const int nchunks = n * rf4;
    const float4 *rows4 = reinterpret_cast<const float4 *>(g.rows);
    constexpr int U = 8;
    for (int c0 = tid; c0 < nchunks; c0 += kSampleThreads * U) {
      float4 v[U];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const int c = c0 + u * kSampleThreads;
        if (c < nchunks) {
          const uint32_t i = g.div_rf4.div(c), q = c - i * rf4;
          v[u] = ldg_stream4(rows4 + size_t(m_row[i]) * rf4 + q);
        }
      }
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const int c = c0 + u * kSampleThreads;
        if (c < nchunks) smem4[c] = v[u];
      }
    }
    if constexpr (NSTEP) {       // s' segment of row t+k-1, into its own tile
      const int total = n * g.D;
      for (int e0 = tid; e0 < total; e0 += kSampleThreads * U) {
        float v[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
          const int e = e0 + u * kSampleThreads;
          if (e < total) {
            const uint32_t i = g.div_D.div(e), c = e - i * g.D;
            v[u] = __ldg(g.rows + size_t(m_last[i]) * g.row_f + g.off_ns + c);
          }
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
          const int e = e0 + u * kSampleThreads;
          if (e < total) tile_ns[e] = v[u];
        }
      }
    }
  }
  // ---- round trip 3: the relabel goal (issued before the barrier: it overlaps the tail of the gather; where
  //      her_resolve knew the goal step without the offset word, it does not depend on round trip 2)
  float gf[4] = {0.f, 0.f, 0.f, 0.f};
  const float *agf = nullptr;
  if (tid < n && ref.j > 0) {
    agf = g.ag + size_t(her_future_slot(g, ref)) * g.gpad;
    if (g.G <= 4) {
      const float4 v = __ldg(reinterpret_cast<const float4 *>(agf));
      gf[0] = v.x; gf[1] = v.y; gf[2] = v.z; gf[3] = v.w;
    }
  }
  // NSTEP: the last kNStepChunk window steps' reward words (or, relabelled, achieved goals) and the done word of row
  // t+k-1 ride with the goal: none of them depends on it
  float4 wv[NSTEP ? kNStepChunk : 1];
  float done_last = 0.f;
  if constexpr (NSTEP) {
    if (tid < n && k > 1) {
      if (ref.j == 0) done_last = __ldg(g.rows + size_t(m_last[tid]) * g.row_f + g.off_d);
#pragma unroll
      for (int u = 0; u < kNStepChunk; ++u) {
        const int i = int(k) - 1 - u;
        if (i >= 1) wv[u] = her_window_load(g, ref, uint32_t(i));
      }
    }
  }
  __syncthreads();

  // ---- relabel + sparse reward (bit-exact fp32, no FMA) --------------------------------------------------
  if (tid < n && ref.j > 0) {
    float *row = tile + tid * g.row_f;
    if (g.G <= 4) {
      her_relabel_row(g, row, gf);
    } else {                       // wide goals: read from the compact copy one column at a time
      float acc = 0.f;
      for (int c = 0; c < g.G; ++c) {
        const float gfc = __ldg(agf + c);
        const float diff = __fsub_rn(row[g.off_ag + c], gfc);
        const float sq = __fmul_rn(diff, diff);
        acc = (c == 0) ? sq : __fadd_rn(acc, sq);
        row[g.D - g.G + c] = gfc;
        row[g.off_ns + g.D - g.G + c] = gfc;
      }
      const float dist = __fsqrt_rn(acc);
      reinterpret_cast<uint32_t *>(row)[g.off_r] = 0x80000000u | ((dist > g.threshold) ? 0x3F800000u : 0u);
      row[g.off_d] = 0.0f;
    }
  }
  if constexpr (NSTEP) {
    if (tid < n) {
      float *row = tile + tid * g.row_f;
      if (ref.j > 0)
        for (int c = 0; c < g.G; ++c) tile_ns[tid * g.D + g.D - g.G + c] = g.G <= 4 ? gf[c] : __ldg(agf + c);
      if (k > 1) {
        // window steps k-1 .. 1, from the back, kNStepChunk per round of loads (the first round was issued above)
        float acc = 0.f;
        for (int hi = int(k) - 1; hi >= 1; hi -= kNStepChunk) {
          if (hi != int(k) - 1) {
#pragma unroll
            for (int u = 0; u < kNStepChunk; ++u)
              if (hi - u >= 1) wv[u] = her_window_load(g, ref, uint32_t(hi - u));
          }
#pragma unroll
          for (int u = 0; u < kNStepChunk; ++u) {
            const int i = hi - u;
            if (i < 1) break;
            float ri;
            if (ref.j == 0) {
              ri = wv[u].x;
            } else if (g.G <= 4) {
              const float a4[4] = {wv[u].x, wv[u].y, wv[u].z, wv[u].w};
              ri = her_sparse_reward(g, a4, gf);
            } else {
              ri = her_sparse_reward(g, g.ag + size_t(her_window_slot(g, ref, uint32_t(i))) * g.gpad, agf);
            }
            acc = (i == int(k) - 1) ? ri : __fadd_rn(ri, __fmul_rn(nst.gamma, acc));
          }
        }
        float p = 1.f;                                    // gamma^(k-1), k-1 rounded products
        for (uint32_t i = 1; i < k; ++i) p = __fmul_rn(p, nst.gamma);
        row[g.off_r] = __fadd_rn(row[g.off_r], __fmul_rn(nst.gamma, acc));
        row[g.off_d] = __fsub_rn(1.f, __fmul_rn(p, __fsub_rn(1.f, ref.j > 0 ? 0.f : done_last)));
      }
    }
  }
  __syncthreads();

  // ---- coalesced write-out of the five output tensors ---------------------------------------------------
  const FastDiv one(1);
  write_field<VEC>(out_s + base * g.D, tile, n, g.D, 0, g.row_f, g.div_D, tid);
  if constexpr (NSTEP)
    write_field<VEC>(out_ns + base * g.D, tile_ns, n, g.D, 0, g.D, g.div_D, tid);
  else
    write_field<VEC>(out_ns + base * g.D, tile, n, g.D, g.off_ns, g.row_f, g.div_D, tid);
  write_field<VEC>(out_a + base * g.A, tile, n, g.A, g.off_a, g.row_f, g.div_A, tid);
  write_field<VEC>(out_r + base, tile, n, 1, g.off_r, g.row_f, one, tid);
  write_field<VEC>(out_d + base, tile, n, 1, g.off_d, g.row_f, one, tid);
}

}  // namespace gcrl

// ---------------------------------------------------------------------------------------
// host object
// ---------------------------------------------------------------------------------------
using namespace gcrl;

struct gcrl_her {
  int device = 0;
  int64_t max_entries = 0, cap_tr = 0, cap_ep = 0, nb = 0;
  HerGeom g{};
  // host bookkeeping (mirrors the reference deque's counters)
  int64_t total_entries = 0, total_tr = 0, next_eid = 0, ep_first = 0, tr_live_first = 0;
  std::deque<std::pair<int64_t, int>> live;  // (entry_end, T) of live episodes, oldest first
  uint64_t seed = 0, host_ctr = 0;
  unsigned long long draw_epoch = 0;         // one per launch that draws its own positions; online store: every launch
  PinnedRing stage;
  char *d_stage[PinnedRing::kSlots] = {};
  size_t blob_max = 0;
  PinnedRing idx_stage;
  int64_t *d_idx = nullptr;
  size_t idx_cap = 0;
  // device scratch for the host-output path
  float *d_out = nullptr;
  int64_t *d_idx_out = nullptr;
  size_t out_cap = 0;
  size_t smem_bytes = 0;
  NStepArgs nstep{1, 1.f};                   // gcrl_her_set_n_step

  int64_t len() const { return std::min(total_entries, max_entries); }
};

namespace gcrl {
SampleScalars her_next_scalars(gcrl_her *h, bool positions_given) {
  SampleScalars sc;
  sc.total_entries = h->total_entries;
  sc.len = h->len();
  sc.draw_epoch = h->draw_epoch;
  sc.use_idx = positions_given ? 1 : 0;
  // device index stream: one epoch per draw; online relabelling draws its coins from the epoch on every call
  if (!positions_given || h->g.online_k > 0) h->draw_epoch += 1;
  return sc;
}
const HerGeom &her_geom(const gcrl_her *h) { return h->g; }
int64_t her_len(const gcrl_her *h) { return h->len(); }
}  // namespace gcrl

static constexpr int kSmallTile = 32;      // samples per CTA while the batch is too small to fill the SMs with 128
static size_t sample_smem(const gcrl_her *h, int spb) { return size_t(spb) * h->g.row_f * 4 + size_t(spb) * 4; }
// the n-step tile adds the slot of each sample's last window row and that row's s'
static size_t sample_smem_nstep(const gcrl_her *h, int spb) { return sample_smem(h, spb) + size_t(spb) * (4 + h->g.D * 4); }

// sc_dev == nullptr: this call draws the scalars (her_next_scalars) and passes them by value
static void her_launch_sample(gcrl_her *h, int64_t B, const int64_t *idx_dev, float *s, float *a,
                              float *r, float *ns, float *d, int64_t *idx_out, cudaStream_t st,
                              const SampleScalars *sc_dev = nullptr) {
  auto aligned = [](const void *p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; };
  const bool vec = aligned(s) && aligned(a) && aligned(r) && aligned(ns) && aligned(d);
  const SampleScalars sc = sc_dev != nullptr ? SampleScalars{} : her_next_scalars(h, idx_dev != nullptr);
  // small batches: 32 samples per CTA (4x the CTAs, each row gather a single round of loads)
  const bool small = B <= int64_t(sm_count()) * 4 * kSmallTile;
  const int spb = small ? kSmallTile : kSamplesPerBlock;
  const unsigned blocks = unsigned((B + spb - 1) / spb);
  const bool nstep = h->nstep.n > 1;
  const size_t smem = nstep ? sample_smem_nstep(h, spb) : sample_smem(h, spb);
  const NStepArgs nst = h->nstep;
  auto kernel = small ? (nstep ? (vec ? her_sample_kernel<true, kSmallTile, true> : her_sample_kernel<false, kSmallTile, true>)
                               : (vec ? her_sample_kernel<true, kSmallTile, false> : her_sample_kernel<false, kSmallTile, false>))
                      : (nstep ? (vec ? her_sample_kernel<true, kSamplesPerBlock, true> : her_sample_kernel<false, kSamplesPerBlock, true>)
                               : (vec ? her_sample_kernel<true, kSamplesPerBlock, false> : her_sample_kernel<false, kSamplesPerBlock, false>));
  kernel<<<blocks, kSampleThreads, smem, st>>>(h->g, sc, sc_dev, B, idx_dev, s, a, r, ns, d, idx_out, nst);
  GCRL_LAUNCHED();
}

static const int64_t *her_stage_indices(gcrl_her *h, int64_t B, const int64_t *idx_host,
                                        cudaStream_t st) {
  if (idx_host == nullptr) return nullptr;
  const int64_t len = h->len();
  for (int64_t i = 0; i < B; ++i)
    if (idx_host[i] < 0 || idx_host[i] >= len)
      throw Error(GCRL_ERR_INVALID, "sample index out of range [0, len)");
  if (size_t(B) > h->idx_cap) {
    GCRL_CUDA(cudaStreamSynchronize(st));
    if (h->d_idx) GCRL_CUDA(cudaFree(h->d_idx));
    h->idx_cap = size_t(B) * 2;
    h->d_idx = dev_alloc<int64_t>(h->idx_cap);
  }
  int slot;
  char *p = h->idx_stage.acquire(size_t(B) * sizeof(int64_t), &slot);
  std::memcpy(p, idx_host, size_t(B) * sizeof(int64_t));
  GCRL_CUDA(cudaMemcpyAsync(h->d_idx, p, size_t(B) * sizeof(int64_t), cudaMemcpyHostToDevice, st));
  h->idx_stage.release(slot, st);
  return h->d_idx;
}

// Exposed to the agent translation unit (fused sample + update path).
namespace gcrl {
void her_sample_into(gcrl_her *h, int64_t B, const int64_t *idx_host, float *s, float *a, float *r,
                     float *ns, float *d, int64_t *idx_out, cudaStream_t st) {
  GCRL_REQUIRE(B >= 0, "negative batch size");
  if (h->len() < B)
    throw Error(GCRL_ERR_UNDERFILLED, "[ERROR] Not enough in buffer to sample");
  if (B == 0) return;
  const int64_t *idx_dev = her_stage_indices(h, B, idx_host, st);
  her_launch_sample(h, B, idx_dev, s, a, r, ns, d, idx_out, st);
}
// The sampler as a node of a captured graph: totals, draw epoch and index-buffer switch are read from `sc_dev`
// (filled from her_next_scalars by the caller before every replay), positions from `idx_dev` when sc_dev->use_idx.
void her_sample_graphed(gcrl_her *h, int64_t B, const SampleScalars *sc_dev, const int64_t *idx_dev, float *s,
                        float *a, float *r, float *ns, float *d, cudaStream_t st) {
  her_launch_sample(h, B, idx_dev, s, a, r, ns, d, nullptr, st, sc_dev);
}
unsigned long long &her_draw_epoch(gcrl_her *h) { return h->draw_epoch; }
int her_state_dim(const gcrl_her *h) { return h->g.D; }
int her_act_dim(const gcrl_her *h) { return h->g.A; }
int her_device(const gcrl_her *h) { return h->device; }
int her_n_step(const gcrl_her *h) { return h->nstep.n; }
}  // namespace gcrl

static int64_t next_pow2(int64_t x) {
  int64_t p = 1;
  while (p < x) p <<= 1;
  return p;
}

extern "C" {

int gcrl_her_create(gcrl_her **out, int device, int64_t max_entries, int64_t cap_transitions,
                    int state_dim, int goal_dim, int act_dim, int k_future, uint64_t seed) {
  GCRL_API_BEGIN
  GCRL_REQUIRE(out != nullptr, "out is NULL");
  GCRL_REQUIRE(max_entries >= 1, "max_entries must be >= 1");
  GCRL_REQUIRE(goal_dim >= 1 && state_dim > goal_dim, "need state_dim > goal_dim >= 1");
  GCRL_REQUIRE(act_dim >= 1 && k_future >= 0 && k_future <= 64, "bad act_dim / k_future");
  // the live window holds at most max_entries - 1 entries besides the oldest live episode's, which may keep up to
  // 254 transitions whose entries are already evicted (a K = 0 / online store has one entry per transition)
  if (cap_transitions <= 0) cap_transitions = max_entries + 254;
  GCRL_REQUIRE(cap_transitions < (int64_t(1) << 31), "cap_transitions must be < 2^31");
  GCRL_CUDA(cudaSetDevice(device));
  auto *h = new gcrl_her();
  try {
    h->device = device;
    h->max_entries = max_entries;
    h->cap_tr = cap_transitions;
    h->cap_ep = next_pow2(cap_transitions);
    h->nb = next_pow2((max_entries >> kBucketShift) + 4);
    h->seed = seed;
    HerGeom &g = h->g;
    g.D = state_dim; g.G = goal_dim; g.A = act_dim; g.K = k_future;
    g.off_ns = state_dim;
    g.off_a = 2 * state_dim;
    g.off_r = g.off_a + act_dim;
    g.off_d = g.off_r + 1;
    g.off_ag = g.off_d + 1;
    g.off_fut = g.off_ag + goal_dim;
    g.row_f = (g.off_fut + (k_future + 3) / 4 + 3) & ~3;
    g.gpad = (goal_dim + 3) & ~3;
    g.cap_tr = uint32_t(h->cap_tr);
    g.ep_mask = uint32_t(h->cap_ep - 1);
    g.bucket_mask = uint32_t(h->nb - 1);
    g.div_k1 = FastDiv(uint32_t(k_future + 1));
    g.div_D = FastDiv(uint32_t(state_dim));
    g.div_A = FastDiv(uint32_t(act_dim));
    g.div_rf4 = FastDiv(uint32_t(g.row_f / 4));
    g.seed = seed;
    g.threshold = 0.05f;
    h->smem_bytes = sample_smem(h, kSamplesPerBlock);
    GCRL_REQUIRE(h->smem_bytes <= 227 * 1024, "transition row too wide for the sampler tile");
    g.rows = dev_alloc<float>(size_t(h->cap_tr) * g.row_f);
    g.ag = dev_alloc<float>(size_t(h->cap_tr) * g.gpad);
    g.eps = dev_alloc<EpRec>(size_t(h->cap_ep));
    g.buckets = dev_alloc<BucketRec>(size_t(h->nb));
    g.hdr = dev_alloc<HerHeader>(1);
    GCRL_CUDA(cudaMemset(g.hdr, 0, sizeof(HerHeader)));
    GCRL_CUDA(cudaMemset(g.buckets, 0, size_t(h->nb) * sizeof(BucketRec)));
    GCRL_CUDA(cudaMemset(g.eps, 0, size_t(h->cap_ep) * sizeof(EpRec)));
    h->blob_max = sizeof(CommitHdr) + size_t(255) * (g.row_f + g.gpad) * 4;
    h->stage.init(h->blob_max);
    for (int i = 0; i < PinnedRing::kSlots; ++i) h->d_stage[i] = dev_alloc<char>(h->blob_max);
    h->idx_stage.init(size_t(1) << 16);
    GCRL_CUDA(cudaFuncSetAttribute(her_sample_kernel<true, kSamplesPerBlock, false>,
                                   cudaFuncAttributeMaxDynamicSharedMemorySize, int(h->smem_bytes)));
    GCRL_CUDA(cudaFuncSetAttribute(her_sample_kernel<false, kSamplesPerBlock, false>,
                                   cudaFuncAttributeMaxDynamicSharedMemorySize, int(h->smem_bytes)));
    GCRL_CUDA(cudaFuncSetAttribute(her_sample_kernel<true, kSmallTile, false>,
                                   cudaFuncAttributeMaxDynamicSharedMemorySize, int(sample_smem(h, kSmallTile))));
    GCRL_CUDA(cudaFuncSetAttribute(her_sample_kernel<false, kSmallTile, false>,
                                   cudaFuncAttributeMaxDynamicSharedMemorySize, int(sample_smem(h, kSmallTile))));
  } catch (...) {
    delete h;
    throw;
  }
  *out = h;
  GCRL_API_END
}

int gcrl_her_destroy(gcrl_her *h) {
  GCRL_API_BEGIN
  if (h == nullptr) return GCRL_OK;
  cudaSetDevice(h->device);
  cudaDeviceSynchronize();
  cudaFree(h->g.rows); cudaFree(h->g.ag); cudaFree(h->g.eps); cudaFree(h->g.buckets);
  cudaFree(h->g.hdr);
  for (auto p : h->d_stage) cudaFree(p);
  if (h->d_idx) cudaFree(h->d_idx);
  if (h->d_out) cudaFree(h->d_out);
  if (h->d_idx_out) cudaFree(h->d_idx_out);
  h->stage.destroy();
  h->idx_stage.destroy();
  delete h;
  GCRL_API_END
}

int gcrl_her_push_episode(gcrl_her *h, int T, const float *s, const float *a, const float *ns,
                          const float *r, const float *d, const float *ag, const uint8_t *fut,
                          void *stream) {
  GCRL_API_BEGIN
  GCRL_NVTX("gcrl_her_push_episode");
  GCRL_REQUIRE(h != nullptr, "handle is NULL");
  GCRL_REQUIRE(T >= 1 && T <= 255, "episode length must be in [1, 255]");
  GCRL_REQUIRE(s && a && ns && r && d && ag, "NULL episode array");
  GCRL_REQUIRE(fut == nullptr || h->g.online_k == 0, "an online-relabelling store draws its goals at sample time (fut must be NULL)");
  GCRL_CUDA(cudaSetDevice(h->device));
  const HerGeom &g = h->g;
  const int k = g.K;
  const int64_t E = int64_t(T - 1) * (k + 1) + 1;
  // ---- eviction accounting (per-entry FIFO of deque(maxlen), src/buffer.py:101) ----
  const int64_t new_total = h->total_entries + E;
  const int64_t new_len = std::min(new_total, h->max_entries);
  const int64_t first_live = new_total - new_len;
  int64_t ep_first = h->ep_first, tr_live_first = h->tr_live_first;
  size_t drop = 0;
  while (drop < h->live.size() && h->live[drop].first <= first_live) {
    tr_live_first += h->live[drop].second;
    ++ep_first;
    ++drop;
  }
  if (h->total_tr + T - tr_live_first > h->cap_tr)
    throw Error(GCRL_ERR_CAPACITY, "transition ring too small for the live window");
  if (h->next_eid + 1 - ep_first > h->cap_ep)
    throw Error(GCRL_ERR_CAPACITY, "episode ring too small for the live window");
  // ---- stage the blob ----
  const size_t bytes = sizeof(CommitHdr) + size_t(T) * (g.row_f + g.gpad) * 4;
  int slot;
  char *blob = h->stage.acquire(bytes, &slot);
  auto *ch = reinterpret_cast<CommitHdr *>(blob);
  ch->entry_start = h->total_entries;
  ch->eid = h->next_eid;
  ch->total_entries = new_total;
  ch->len = new_len;
  ch->ep_first = ep_first;
  const int64_t b0 = (h->total_entries + (1 << kBucketShift) - 1) >> kBucketShift;
  const int64_t b1 = (new_total + (1 << kBucketShift) - 1) >> kBucketShift;  // exclusive
  ch->first_bucket = b0;
  ch->n_buckets = uint32_t(b1 - b0);
  ch->tr_slot = uint32_t(h->total_tr % h->cap_tr);
  ch->T = uint32_t(T);
  ch->pad = 0;
  float *rows = reinterpret_cast<float *>(blob + sizeof(CommitHdr));
  float *agc = rows + size_t(T) * g.row_f;
  for (int t = 0; t < T; ++t) {
    float *row = rows + size_t(t) * g.row_f;
    std::memset(row, 0, size_t(g.row_f) * 4);
    std::memcpy(row, s + size_t(t) * g.D, size_t(g.D) * 4);
    std::memcpy(row + g.off_ns, ns + size_t(t) * g.D, size_t(g.D) * 4);
    std::memcpy(row + g.off_a, a + size_t(t) * g.A, size_t(g.A) * 4);
    row[g.off_r] = r[t];
    row[g.off_d] = d[t];
    std::memcpy(row + g.off_ag, ag + size_t(t) * g.G, size_t(g.G) * 4);
    uint8_t *fb = reinterpret_cast<uint8_t *>(row + g.off_fut);
    if (t < T - 1) {
      // the strategy's goal range [lo, T-1]: future [t+1, T-1], final {T-1}, episode [0, T-1]
      const int lo = g.strategy == GCRL_HER_EPISODE ? 0 : (g.strategy == GCRL_HER_FINAL ? T - 1 : t + 1);
      for (int j = 0; j < k; ++j) {
        int f;
        if (fut != nullptr) {
          f = fut[size_t(t) * k + j];
          if (f < lo || f >= T) throw Error(GCRL_ERR_INVALID, "relabel goal index outside the strategy's range");
        } else if (lo == T - 1) {
          f = lo;
        } else {
          f = lo + int(splitmix64(h->seed ^ (0xA5A5A5A5ull + h->host_ctr++)) % uint64_t(T - lo));
        }
        fb[j] = uint8_t(f);
      }
    }
    float *agr = agc + size_t(t) * g.gpad;
    std::memset(agr, 0, size_t(g.gpad) * 4);
    std::memcpy(agr, ag + size_t(t) * g.G, size_t(g.G) * 4);
  }
  cudaStream_t st = as_stream(stream);
  GCRL_CUDA(cudaMemcpyAsync(h->d_stage[slot], blob, bytes, cudaMemcpyHostToDevice, st));
  h->stage.release(slot, st);
  const int work = T * (g.row_f / 4);
  const int blocks = std::max(1, std::min(32, (work + 255) / 256));
  her_commit_kernel<<<blocks, 256, 0, st>>>(g, h->d_stage[slot]);
  GCRL_LAUNCHED();
  // ---- commit host counters ----
  h->live.erase(h->live.begin(), h->live.begin() + drop);
  h->live.emplace_back(new_total, T);
  h->ep_first = ep_first;
  h->tr_live_first = tr_live_first;
  h->total_entries = new_total;
  h->total_tr += T;
  h->next_eid += 1;
  GCRL_API_END
}

int gcrl_her_set_threshold(gcrl_her *h, float threshold) {
  GCRL_API_BEGIN
  GCRL_REQUIRE(h != nullptr, "handle is NULL");
  GCRL_REQUIRE(threshold >= 0.f, "the distance threshold must be >= 0");
  h->g.threshold = threshold;
  GCRL_API_END
}

int gcrl_her_set_goal_selection(gcrl_her *h, int strategy, int online_k) {
  GCRL_API_BEGIN
  GCRL_REQUIRE(h != nullptr, "handle is NULL");
  GCRL_REQUIRE(strategy == GCRL_HER_FUTURE || strategy == GCRL_HER_FINAL || strategy == GCRL_HER_EPISODE,
               "unknown goal-selection strategy");
  GCRL_REQUIRE(online_k >= 0 && online_k <= 64, "online_k must be in [0, 64]");
  GCRL_REQUIRE(online_k == 0 || h->g.K == 0, "online relabelling needs a store created with k_future = 0");
  GCRL_REQUIRE(h->next_eid == 0, "the goal selection cannot change once an episode has been committed");
  h->g.strategy = strategy;
  h->g.online_k = online_k;
  GCRL_API_END
}

int gcrl_her_set_n_step(gcrl_her *h, int n, float gamma) {
  GCRL_API_BEGIN
  GCRL_REQUIRE(h != nullptr, "handle is NULL");
  GCRL_REQUIRE(n >= 1 && n <= 255, "n_step must be in [1, 255]");
  GCRL_REQUIRE(n == 1 || (gamma > 0.f && gamma <= 1.f), "n-step returns need a discount gamma in (0, 1]");
  GCRL_REQUIRE(h->next_eid == 0, "n_step cannot change once an episode has been committed");
  GCRL_REQUIRE(n == 1 || sample_smem_nstep(h, kSamplesPerBlock) <= 227 * 1024,
               "transition row too wide for the n-step sampler tile");
  if (n > 1) {
    GCRL_CUDA(cudaSetDevice(h->device));
    GCRL_CUDA(cudaFuncSetAttribute(her_sample_kernel<true, kSamplesPerBlock, true>,
                                   cudaFuncAttributeMaxDynamicSharedMemorySize, int(sample_smem_nstep(h, kSamplesPerBlock))));
    GCRL_CUDA(cudaFuncSetAttribute(her_sample_kernel<false, kSamplesPerBlock, true>,
                                   cudaFuncAttributeMaxDynamicSharedMemorySize, int(sample_smem_nstep(h, kSamplesPerBlock))));
    GCRL_CUDA(cudaFuncSetAttribute(her_sample_kernel<true, kSmallTile, true>,
                                   cudaFuncAttributeMaxDynamicSharedMemorySize, int(sample_smem_nstep(h, kSmallTile))));
    GCRL_CUDA(cudaFuncSetAttribute(her_sample_kernel<false, kSmallTile, true>,
                                   cudaFuncAttributeMaxDynamicSharedMemorySize, int(sample_smem_nstep(h, kSmallTile))));
  }
  h->nstep = NStepArgs{n, n > 1 ? gamma : 1.f};
  GCRL_API_END
}

uint64_t gcrl_her_get_draw_epoch(const gcrl_her *h) { return h ? h->draw_epoch : 0; }

int gcrl_her_set_draw_epoch(gcrl_her *h, uint64_t epoch) {
  GCRL_API_BEGIN
  GCRL_REQUIRE(h != nullptr, "handle is NULL");
  h->draw_epoch = epoch;
  GCRL_API_END
}

int gcrl_her_index_tables(gcrl_her *h, const void **eps_dev, int64_t *eps_bytes, const void **buckets_dev,
                          int64_t *bucket_bytes) {
  GCRL_API_BEGIN
  GCRL_REQUIRE(h != nullptr, "handle is NULL");
  if (eps_dev) *eps_dev = h->g.eps;
  if (eps_bytes) *eps_bytes = h->cap_ep * int64_t(sizeof(EpRec));
  if (buckets_dev) *buckets_dev = h->g.buckets;
  if (bucket_bytes) *bucket_bytes = h->nb * int64_t(sizeof(BucketRec));
  GCRL_API_END
}

int64_t gcrl_her_len(const gcrl_her *h) { return h ? h->len() : 0; }
int64_t gcrl_her_total_entries(const gcrl_her *h) { return h ? h->total_entries : 0; }
int64_t gcrl_her_live_transitions(const gcrl_her *h) {
  return h ? h->total_tr - h->tr_live_first : 0;
}

// ---- export of the live window (true resume): episodes oldest first, exactly as committed ----------
int64_t gcrl_her_live_episodes(const gcrl_her *h) { return h ? int64_t(h->live.size()) : 0; }

int gcrl_her_get_episode(gcrl_her *h, int64_t i, int *T_out, float *s, float *a, float *ns, float *r, float *d,
                         float *ag, uint8_t *fut, void *stream) {
  GCRL_API_BEGIN
  GCRL_REQUIRE(h != nullptr && T_out != nullptr, "NULL argument");
  GCRL_REQUIRE(i >= 0 && i < int64_t(h->live.size()), "episode index outside the live window");
  const HerGeom &g = h->g;
  int64_t first = h->tr_live_first;
  for (int64_t e = 0; e < i; ++e) first += h->live[size_t(e)].second;
  const int T = h->live[size_t(i)].second;
  *T_out = T;
  if (s == nullptr) return GCRL_OK;                      // length query only
  GCRL_REQUIRE(a && ns && r && d && ag && (fut || g.K == 0), "NULL episode array");
  GCRL_CUDA(cudaSetDevice(h->device));
  cudaStream_t st = as_stream(stream);
  std::vector<float> rows(size_t(T) * g.row_f);
  const int64_t slot0 = first % h->cap_tr;
  const int64_t n0 = std::min<int64_t>(T, h->cap_tr - slot0);       // the ring may wrap inside the episode
  GCRL_CUDA(cudaMemcpyAsync(rows.data(), g.rows + size_t(slot0) * g.row_f, size_t(n0) * g.row_f * 4,
                            cudaMemcpyDeviceToHost, st));
  if (n0 < T)
    GCRL_CUDA(cudaMemcpyAsync(rows.data() + size_t(n0) * g.row_f, g.rows, size_t(T - n0) * g.row_f * 4,
                              cudaMemcpyDeviceToHost, st));
  GCRL_CUDA(cudaStreamSynchronize(st));
  for (int t = 0; t < T; ++t) {
    const float *row = rows.data() + size_t(t) * g.row_f;
    std::memcpy(s + size_t(t) * g.D, row, size_t(g.D) * 4);
    std::memcpy(ns + size_t(t) * g.D, row + g.off_ns, size_t(g.D) * 4);
    std::memcpy(a + size_t(t) * g.A, row + g.off_a, size_t(g.A) * 4);
    r[t] = row[g.off_r];
    d[t] = row[g.off_d];
    std::memcpy(ag + size_t(t) * g.G, row + g.off_ag, size_t(g.G) * 4);
    if (g.K > 0) std::memcpy(fut + size_t(t) * g.K, row + g.off_fut, size_t(g.K));
  }
  GCRL_API_END
}

int gcrl_her_clear(gcrl_her *h) {
  GCRL_API_BEGIN
  GCRL_REQUIRE(h != nullptr, "handle is NULL");
  GCRL_CUDA(cudaSetDevice(h->device));
  GCRL_CUDA(cudaDeviceSynchronize());
  GCRL_CUDA(cudaMemset(h->g.hdr, 0, sizeof(HerHeader)));
  h->total_entries = h->total_tr = h->next_eid = h->ep_first = h->tr_live_first = 0;
  h->draw_epoch = 0;
  h->live.clear();
  GCRL_API_END
}

int gcrl_her_sample(gcrl_her *h, int64_t B, const int64_t *idx_host, float *states_dev,
                    float *actions_dev, float *rewards_dev, float *next_states_dev,
                    float *dones_dev, int64_t *idx_out_dev, void *stream) {
  GCRL_API_BEGIN
  GCRL_NVTX("gcrl_her_sample");
  GCRL_REQUIRE(h != nullptr, "handle is NULL");
  GCRL_REQUIRE(B == 0 || (states_dev && actions_dev && rewards_dev && next_states_dev && dones_dev),
               "NULL output");
  GCRL_CUDA(cudaSetDevice(h->device));
  her_sample_into(h, B, idx_host, states_dev, actions_dev, rewards_dev, next_states_dev, dones_dev,
                  idx_out_dev, as_stream(stream));
  GCRL_API_END
}

int gcrl_her_sample_dev_idx(gcrl_her *h, int64_t B, const int64_t *idx_dev, float *states_dev,
                            float *actions_dev, float *rewards_dev, float *next_states_dev,
                            float *dones_dev, void *stream) {
  GCRL_API_BEGIN
  GCRL_REQUIRE(h != nullptr && idx_dev != nullptr, "NULL handle / indices");
  GCRL_CUDA(cudaSetDevice(h->device));
  if (h->len() < B) throw Error(GCRL_ERR_UNDERFILLED, "[ERROR] Not enough in buffer to sample");
  if (B > 0)
    her_launch_sample(h, B, idx_dev, states_dev, actions_dev, rewards_dev, next_states_dev,
                      dones_dev, nullptr, as_stream(stream));
  GCRL_API_END
}

int gcrl_her_sample_host(gcrl_her *h, int64_t B, const int64_t *idx_host, float *states,
                         float *actions, float *rewards, float *next_states, float *dones,
                         int64_t *idx_out, void *stream) {
  GCRL_API_BEGIN
  GCRL_NVTX("gcrl_her_sample_host");
  GCRL_REQUIRE(h != nullptr, "handle is NULL");
  GCRL_CUDA(cudaSetDevice(h->device));
  cudaStream_t st = as_stream(stream);
  const HerGeom &g = h->g;
  const size_t per = size_t(2 * g.D + g.A + 2);
  const size_t Bp = (size_t(B) + 3) & ~size_t(3);  // keep every field 16 B aligned
  if (Bp > h->out_cap) {
    GCRL_CUDA(cudaStreamSynchronize(st));
    if (h->d_out) GCRL_CUDA(cudaFree(h->d_out));
    if (h->d_idx_out) GCRL_CUDA(cudaFree(h->d_idx_out));
    h->out_cap = Bp * 2;
    h->d_out = dev_alloc<float>(h->out_cap * per);
    h->d_idx_out = dev_alloc<int64_t>(h->out_cap);
  }
  float *ds = h->d_out, *dns = ds + Bp * g.D, *da = dns + Bp * g.D, *dr = da + Bp * g.A,
        *dd = dr + Bp;
  her_sample_into(h, B, idx_host, ds, da, dr, dns, dd, idx_out ? h->d_idx_out : nullptr, st);
  if (B > 0) {
    GCRL_CUDA(cudaMemcpyAsync(states, ds, size_t(B) * g.D * 4, cudaMemcpyDeviceToHost, st));
    GCRL_CUDA(cudaMemcpyAsync(next_states, dns, size_t(B) * g.D * 4, cudaMemcpyDeviceToHost, st));
    GCRL_CUDA(cudaMemcpyAsync(actions, da, size_t(B) * g.A * 4, cudaMemcpyDeviceToHost, st));
    GCRL_CUDA(cudaMemcpyAsync(rewards, dr, size_t(B) * 4, cudaMemcpyDeviceToHost, st));
    GCRL_CUDA(cudaMemcpyAsync(dones, dd, size_t(B) * 4, cudaMemcpyDeviceToHost, st));
    if (idx_out)
      GCRL_CUDA(cudaMemcpyAsync(idx_out, h->d_idx_out, size_t(B) * 8, cudaMemcpyDeviceToHost, st));
    GCRL_CUDA(cudaStreamSynchronize(st));
  }
  GCRL_API_END
}

}  // extern "C"
