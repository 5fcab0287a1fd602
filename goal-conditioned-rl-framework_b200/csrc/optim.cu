// Gradient reduction, global-norm clipping, Adam / AdamW and Polyak kernels.
//
// Replaces (reference src/agent.py): clip_grad_norm_ (:1295,:1331), get_gradient_norm
// (:1279-1286, 8 host syncs per call -> one device scalar), torch.optim.Adam.step (:1297,
// :1333; AdamW for TD3 :46-48) and the per-parameter Polyak loop (:1259-1271).  Each network
// is one flat fp32 buffer, so an optimiser step is two launches: a fixed-order reduction of
// the split-batch partial gradients (+ sum of squares) and one fused clip + Adam (+ Polyak)
// pass.  Bound: HBM traffic of 7 fp32 words per parameter (g, m, v, p read; m, v, p write).
#include <algorithm>
#include <cstdlib>

#include "mlp.cuh"

namespace gcrl {

long long p2p_timeout_cycles();
constexpr int kOptThreads = 256;

int reduce_grid(int total) {
  return std::max(1, std::min((total + kOptThreads - 1) / kOptThreads, sm_count() * 4));
}

__device__ __forceinline__ float block_sum_fixed(float v, float *scratch /*[32]*/) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int s = 16; s >= 1; s >>= 1) v += __shfl_xor_sync(0xffffffffu, v, s);
  if (lane == 0) scratch[warp] = v;
  __syncthreads();
  float r = 0.f;
  if (warp == 0) {
    r = lane < (blockDim.x >> 5) ? scratch[lane] : 0.f;
#pragma unroll
    for (int s = 16; s >= 1; s >>= 1) r += __shfl_xor_sync(0xffffffffu, r, s);
  }
  return r;  // valid in warp 0
}

__device__ __forceinline__ void reduce_grads_body(const ReduceArgs &a) {
  __shared__ float scratch[32];
  float sq = 0.f;
  for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < a.total; e += gridDim.x * blockDim.x) {
    float g = 0.f;
    bool found = false;
#pragma unroll 4
    for (int s = 0; s < a.nseg; ++s) {
      const SegDesc &sd = a.seg[s];
      if (e >= sd.begin && e < sd.begin + sd.count) {
        found = true;
        if (sd.partials != nullptr) {
          const float *src = sd.partials + sd.offset + (e - sd.begin);
          for (int k = 0; k < sd.splits; ++k) g += src[int64_t(k) * sd.split_stride];
        } else {
          g = a.grad[e];
        }
      }
    }
    if (!found) g = 0.f;  // alignment padding between segments
    a.grad[e] = g;
    sq = fmaf(g, g, sq);
  }
  const float tot = block_sum_fixed(sq, scratch);
  if (threadIdx.x == 0) a.sumsq_partials[blockIdx.x] = tot;
  if (blockIdx.x == 0 && a.metric_partials != nullptr && threadIdx.x < 3) {
    float s = 0.f;
    for (int k = 0; k < a.metric_splits; ++k) s += a.metric_partials[size_t(k) * 4 + threadIdx.x];
    const int slot = threadIdx.x == 0 ? a.slot_loss : (threadIdx.x == 1 ? a.slot_td : a.slot_q);
    if (slot >= 0) a.metrics[slot] = s * a.metric_scale;
  }
}

__global__ void __launch_bounds__(kOptThreads) reduce_grads_kernel(ReduceArgs a) {
  pdl_wait();
  pdl_launch_dependents();
  reduce_grads_body(a);
}

void launch_reduce_grads(const ReduceArgs &a, cudaStream_t st) {
  launch_pdl<PDL_OPTIM>(reduce_grads_kernel, dim3(reduce_grid(a.total)), dim3(kOptThreads), 0, st, a);
  GCRL_LAUNCHED();
}

// ---- data-parallel gradient averaging over NVLink peer memory (one process per GPU) ----------------
// Every rank maps the flat gradient buffers of all its peers (CUDA IPC) and averages them itself, in rank
// order 0..world-1 on every rank -> bit-identical replicas, no NCCL launch on the critical path (a 0.55 MB
// all-reduce is pure latency: 32 us through NCCL at 8 GPUs, measured).  Cross-GPU ordering is a flag barrier:
// rank r bumps slot r of every peer's flag array, then spins on its own array.
__global__ void __launch_bounds__(32)
p2p_barrier_kernel(unsigned int *const *peer_flags, unsigned int *epoch, int rank, int world, int *err,
                   long long timeout_cycles) {
  __shared__ unsigned int e_s;
  if (threadIdx.x == 0) e_s = *epoch + 1u;
  __syncwarp();
  const unsigned int e = e_s;
  if (int(threadIdx.x) < world) {
    __threadfence_system();                                   // my gradients are visible before the flag is
    volatile unsigned int *dst = peer_flags[threadIdx.x] + rank;
    *dst = e;
    volatile unsigned int *src = peer_flags[rank] + threadIdx.x;
    const long long t0 = clock64();
    while (*src < e) {
      if (clock64() - t0 > timeout_cycles) {                  // a peer died; fail loudly instead of hanging
        *err = 1 + int(threadIdx.x) + 16 * rank;
        break;
      }
      __nanosleep(40);
    }
    __threadfence_system();
  }
  __syncwarp();
  if (threadIdx.x == 0) *epoch = e;
}

// watchdog of every cross-GPU wait: 60 s by default, GCRL_P2P_TIMEOUT_MS overrides (tests, debugging)
long long p2p_timeout_cycles() {
  static long long cyc = 0;
  if (cyc == 0) {
    const char *e = getenv("GCRL_P2P_TIMEOUT_MS");
    const double ms = e ? atof(e) : 60000.0;
    cyc = (long long)(ms * 2.0e6);        // ~2 GHz SM clock
  }
  return cyc;
}

void launch_p2p_barrier(unsigned int *const *peer_flags, unsigned int *epoch, int rank, int world, int *err,
                        cudaStream_t st) {
  p2p_barrier_kernel<<<1, 32, 0, st>>>(peer_flags, epoch, rank, world, err, p2p_timeout_cycles());
  GCRL_LAUNCHED();
}

// ---- barrier + average in ONE launch ---------------------------------------------------------------------
// CTA 0 publishes this rank's batch-mean metrics and tells every peer "my gradient of this network is complete"
// (stream order: the weight-gradient kernel has finished); EVERY CTA then polls the rank's own flag words, which the
// peers write over NVLink, and reads all ranks' buffers for its elements -- all loads of a thread in flight
// together (an NVLink round trip is ~2 us; a load-add-load-add chain over 8 ranks would be 8 of them) -- summing
// in rank order 0..N-1 on every rank: bit-identical replicas by construction.  The batch-mean metrics ride on
// the same barrier (double-buffered outbox, rank-order mean).  The last CTA to finish advances the epoch word
// the next barrier starts from.  Reuse of a gradient buffer is safe without a second barrier: a rank overwrites
// it two barriers later, which its peers can only have reached after finishing these reads.
struct P2PReduceArgs {
  const float *const *peers;            // [world] flat gradient of this network on every rank
  unsigned int *const *peer_flags;      // [world] flag arrays (8 words each)
  const float *const *peer_outbox;      // [world] metric outboxes (2 x 8 floats each)
  unsigned int *epoch, *ticket, *go;
  int *err;
  long long timeout_cycles;
  int rank, world, n;
  float inv_world;
  float *out, *sumsq_partials;
  const float *local_metrics;
  float *outbox, *metrics_avg;
  unsigned int metric_mask;             // slots averaged over the ranks at this barrier
  int debug;                            // timing experiments only (GCRL_P2P_DEBUG): 1 no flag wait, 2 local reads only
  int signalled;                        // this rank's flag was raised by the kernel that produced the gradient
};

template <int WORLD>
__global__ void __launch_bounds__(kOptThreads) p2p_reduce_kernel(const __grid_constant__ P2PReduceArgs a) {
  __shared__ float scratch[32];
  __shared__ unsigned int e_s;
  pdl_wait();      // (no early launch of the dependent optimiser kernel: its CTAs would sit on the SMs while this one polls)
  const int tid = threadIdx.x;
  if (tid == 0) e_s = *a.epoch + 1u;
  __syncthreads();
  const unsigned int e = e_s;
  if (blockIdx.x == 0 && !a.signalled) {
    if (tid < 8) a.outbox[(e & 1u) * 8 + tid] = a.local_metrics[tid];
    __syncthreads();
    if (tid < a.world) {
      __threadfence_system();                                  // gradient + outbox visible before the flag is
      volatile unsigned int *dst = a.peer_flags[tid] + a.rank;
      *dst = e;
    }
  }
  // Only ONE warp of the grid polls the flag words the peers write over NVLink (system-scope acquire loads, with
  // back-off); the other CTAs wait on a local "go" word that CTA 0 releases at GPU scope.  (Every CTA polling
  // the NVLink-written line itself -- 8 x 135 spinning threads at 8 ranks -- starved the incoming writes: the
  // 8-GPU run of this round hung in exactly that variant, 2 and 4 GPUs did not.)
  if (!(a.debug & 1)) {
    if (blockIdx.x == 0) {
      if (tid < a.world) {
        const unsigned int *src = a.peer_flags[a.rank] + tid;
        const long long t0 = clock64();
        unsigned int seen;
        for (;;) {
          asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(seen) : "l"(src) : "memory");
          if (seen >= e) break;
          if (clock64() - t0 > a.timeout_cycles) {             // a peer died: fail loudly instead of hanging
            atomicExch(a.err, 1 + tid + 16 * a.rank);
            break;
          }
          __nanosleep(40);
        }
      }
      __syncthreads();
      if (tid == 0) asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(a.go), "r"(e) : "memory");
    } else {
      if (tid == 0) {
        const long long t0 = clock64();
        unsigned int seen;
        for (;;) {
          asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(seen) : "l"(a.go) : "memory");
          if (seen >= e || clock64() - t0 > 2 * a.timeout_cycles) break;
          __nanosleep(20);
        }
      }
      __syncthreads();
    }
  }
  float sq = 0.f;
  const int n4 = a.n >> 2;                                     // flat buffers are 16-byte granular
  for (int q = blockIdx.x * blockDim.x + tid; q < n4; q += gridDim.x * blockDim.x) {
    float4 v[WORLD];
#pragma unroll
    for (int r = 0; r < WORLD; ++r)
      if (r < a.world) v[r] = __ldcv(reinterpret_cast<const float4 *>(a.peers[(a.debug & 2) ? a.rank : r]) + q);   // never a stale L1 line
    float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int r = 0; r < WORLD; ++r)
      if (r < a.world) { s.x += v[r].x; s.y += v[r].y; s.z += v[r].z; s.w += v[r].w; }
    s.x *= a.inv_world; s.y *= a.inv_world; s.z *= a.inv_world; s.w *= a.inv_world;
    reinterpret_cast<float4 *>(a.out)[q] = s;
    sq = fmaf(s.x, s.x, sq); sq = fmaf(s.y, s.y, sq); sq = fmaf(s.z, s.z, sq); sq = fmaf(s.w, s.w, sq);
  }
  const float tot = block_sum_fixed(sq, scratch);
  if (tid == 0) a.sumsq_partials[blockIdx.x] = tot;
  if (blockIdx.x == 0 && tid < 8 && ((a.metric_mask >> tid) & 1u)) {
    float s = 0.f;
    for (int r = 0; r < a.world; ++r) s += __ldcv(a.peer_outbox[r] + (e & 1u) * 8 + tid);
    a.metrics_avg[tid] = s * a.inv_world;
  }
  if (tid == 0) {
    __threadfence();
    const unsigned int t = atomicAdd(a.ticket, 1u);
    if (t == gridDim.x - 1) {
      *a.ticket = 0;
      *a.epoch = e;
    }
  }
}

int p2p_reduce_grid(int n) { return std::max(1, std::min(((n >> 2) + kOptThreads - 1) / kOptThreads, sm_count())); }

void launch_p2p_reduce(const P2PReduceHost &h, cudaStream_t st) {
  P2PReduceArgs a{};
  a.peers = h.peers; a.peer_flags = h.peer_flags; a.peer_outbox = h.peer_outbox;
  a.epoch = h.epoch; a.ticket = h.ticket; a.go = h.go; a.err = h.err;
  a.timeout_cycles = p2p_timeout_cycles();
  a.rank = h.rank; a.world = h.world; a.n = h.n; a.inv_world = 1.0f / float(h.world);
  a.out = h.out; a.sumsq_partials = h.sumsq_partials;
  a.local_metrics = h.local_metrics; a.outbox = h.outbox; a.metrics_avg = h.metrics_avg; a.metric_mask = h.metric_mask;
  GCRL_REQUIRE(h.world >= 1 && h.world <= 8 && (h.n & 3) == 0, "p2p reduce: 1 <= world <= 8, 16-byte granular buffers");
  static const int debug = getenv("GCRL_P2P_DEBUG") ? atoi(getenv("GCRL_P2P_DEBUG")) : 0;
  a.debug = debug;
  a.signalled = h.signalled;
  const dim3 grid(p2p_reduce_grid(h.n)), block(kOptThreads);
  if (h.world <= 2) launch_pdl<PDL_P2P>(p2p_reduce_kernel<2>, grid, block, 0, st, a);
  else if (h.world <= 4) launch_pdl<PDL_P2P>(p2p_reduce_kernel<4>, grid, block, 0, st, a);
  else launch_pdl<PDL_P2P>(p2p_reduce_kernel<8>, grid, block, 0, st, a);
  GCRL_LAUNCHED();
}

// torch.optim.Adam(W) single-tensor semantics (betas 0.9/0.999, eps 1e-8):
//   p *= 1 - lr*wd (AdamW only);  m += (1-b1)(g-m);  v = v*b2 + (1-b2) g g;
//   p -= (lr/bc1) * m / (sqrt(v)/sqrt(bc2) + eps)
// preceded by clip_grad_norm_: g *= min(1, max_norm / (||g|| + 1e-6)).
//
// Only g and the sums of squares come from the kernel this one depends on (weight-gradient kernel, gradient
// reduction, sums-of-squares kernel or peer average -- p2p_reduce_kernel writes gavg and sumsq).  p, m, v, tmap,
// target and the step scalars of a thread's first element are loaded BEFORE pdl_wait(), so that their DRAM round
// trip overlaps the tail of that kernel:
//   - p, m, v and pT are written only by this kernel, and the target it blends only by this kernel's own Polyak
//     (polyak_kernel writes the DDPG actor target, which no Adam launch blends, and the targets in
//     gcrl_agent_soft_update, which no Adam launch follows directly).  The actor-target Polyak that may directly
//     precede the DDPG critic step writes nothing the critic step reads.  tmap never changes; the step scalars are
//     a host copy made before the update.
//   - Every kernel launched with the PDL attribute executes pdl_launch_dependents() only after its own pdl_wait()
//     (p2p_reduce_kernel not at all: it releases this one when it exits), and a kernel launched without it starts
//     after its predecessor has completed.  So when this kernel starts, every launch two or more back has completed
//     and its writes are visible: the other critic's step (TD3), the previous update's steps (update_many).
//     Keep pdl_launch_dependents() below pdl_wait() everywhere, or these loads may read stale values.
// At B = 256 one grid-stride pass covers every element; later passes load after the wait as before.
__device__ __forceinline__ void adam_body(const AdamArgs &a) {
  __shared__ float s_coef, s_norm;
  const int e0 = blockIdx.x * blockDim.x + threadIdx.x, stride = gridDim.x * blockDim.x;
  float p0 = 0.f, m0 = 0.f, v0 = 0.f, t0 = 0.f;
  int tm0 = -1;
  if (e0 < a.n) {
    p0 = a.p[e0]; m0 = a.m[e0]; v0 = a.v[e0];
    if (a.tmap != nullptr) tm0 = a.tmap[e0];
    if (a.polyak) t0 = a.target[e0];
  }
  const float step_size = a.which == 0 ? a.sc->step_size_c : a.sc->step_size_a;
  const float bc2_sqrt = a.which == 0 ? a.sc->bc2_sqrt_c : a.sc->bc2_sqrt_a;
  const float decay = a.which == 0 ? a.sc->decay_c : a.sc->decay_a;
  pdl_wait();
  pdl_launch_dependents();
  if (threadIdx.x < 32) {
    float s = 0.f;
    for (int i = threadIdx.x; i < a.nsumsq; i += 32) s += a.sumsq_partials[i];
#pragma unroll
    for (int k = 16; k >= 1; k >>= 1) s += __shfl_xor_sync(0xffffffffu, s, k);
    if (threadIdx.x == 0) {
      const float norm = sqrtf(s);
      float coef = 1.0f;
      if (a.max_norm >= 0.f) coef = fminf(a.max_norm / (norm + 1e-6f), 1.0f);
      s_coef = coef;
      s_norm = norm;
    }
  }
  __syncthreads();
  const float coef = s_coef;
  // scalar arguments exactly as torch narrows them: float(1 - 0.9), float(0.999), float(1 - 0.999)
  const float omb1 = float(1.0 - 0.9), b2 = float(0.999), omb2 = float(1.0 - 0.999), eps = 1e-8f;
  // the roundings spelled out (the contractions the compiler chose for this kernel before its loads were hoisted),
  // so that moving a load cannot change which products are fused
  auto step = [&](int e, float p, float m, float v, int tm, float tgt) {
    const float g = __fmul_rn(a.g[e], coef);
    if (a.weight_decay != 0.f) p = __fmul_rn(p, decay);
    m = __fmaf_rn(__fsub_rn(g, m), omb1, m);
    v = __fmaf_rn(__fmul_rn(omb2, g), g, __fmul_rn(v, b2));
    const float denom = __fadd_rn(sqrtf(v) / bc2_sqrt, eps);
    p = __fmaf_rn(-step_size, m / denom, p);
    a.m[e] = m;
    a.v[e] = v;
    a.p[e] = p;
    if (tm >= 0) a.pT[tm] = p;
    if (a.polyak) {
      const float t = __fmaf_rn(a.tau, p, __fmul_rn(a.one_minus_tau, tgt));
      a.target[e] = t;
      if (tm >= 0 && a.targetT != nullptr) a.targetT[tm] = t;     // (SAC / TQC targets keep no W^T)
    }
  };
  if (e0 < a.n) step(e0, p0, m0, v0, tm0, t0);
  for (int e = e0 + stride; e < a.n; e += stride)
    step(e, a.p[e], a.m[e], a.v[e], a.tmap != nullptr ? a.tmap[e] : -1, a.polyak ? a.target[e] : 0.f);
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    const float post = s_norm * coef;         // norm after clipping (src/agent.py:1332,:1300)
    if (a.metrics != nullptr && a.slot_norm >= 0) a.metrics[a.slot_norm] = post;
    if (a.publish != nullptr) {
      // every other slot was written by earlier kernels of this update; the norm slot just above by this thread
      for (int i = 0; i < 8; ++i) a.publish[i] = (a.publish_src == a.metrics && i == a.slot_norm) ? post : __ldcg(a.publish_src + i);
      reinterpret_cast<int *>(a.publish)[9] = a.publish_err != nullptr ? __ldcg(a.publish_err) : 0;
      __threadfence_system();
      reinterpret_cast<volatile unsigned int *>(a.publish)[8] = a.sc->seq;
    }
  }
}

__global__ void __launch_bounds__(kOptThreads) adam_kernel(AdamArgs a) { adam_body(a); }

void launch_adam(const AdamArgs &a, cudaStream_t st) {
  launch_pdl<PDL_OPTIM>(adam_kernel, dim3(reduce_grid(a.n)), dim3(kOptThreads), 0, st, a);
  GCRL_LAUNCHED();
}

__global__ void __launch_bounds__(kOptThreads)
polyak_kernel(float *__restrict__ target, const float *__restrict__ src, int n, float tau, float omt,
              const int *__restrict__ tmap, float *__restrict__ targetT) {
  pdl_wait();
  pdl_launch_dependents();
  for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < n; e += gridDim.x * blockDim.x) {
    const float t = tau * src[e] + omt * target[e];
    target[e] = t;
    if (tmap != nullptr) {
      const int tm = tmap[e];
      if (tm >= 0) targetT[tm] = t;
    }
  }
}

void launch_polyak(float *target, const float *src, int n, float tau, float one_minus_tau,
                   const int *tmap, float *targetT, cudaStream_t st) {
  launch_pdl<PDL_OPTIM>(polyak_kernel, dim3(reduce_grid(n)), dim3(kOptThreads), 0, st, target, src, n, tau, one_minus_tau, tmap, targetT);
  GCRL_LAUNCHED();
}

__global__ void __launch_bounds__(kOptThreads)
sync_transposed_kernel(const float *__restrict__ p, float *__restrict__ pT, const int *__restrict__ tmap, int n) {
  for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < n; e += gridDim.x * blockDim.x) {
    const int tm = tmap[e];
    if (tm >= 0) pT[tm] = p[e];
  }
}

void launch_sync_transposed(const float *p, float *pT, const int *tmap, int n, cudaStream_t st) {
  sync_transposed_kernel<<<reduce_grid(n), kOptThreads, 0, st>>>(p, pT, tmap, n);
  GCRL_LAUNCHED();
}

}  // namespace gcrl
