// fp32 (FFMA) forward / backward kernels for the 64..512-wide actor / critic MLPs.
//
// Replaces the torch library calls behind Actor/Critic (reference src/model.py:7-83) and
// autograd in DDPG.critic_update / actor_update (src/agent.py:1288-1343): nn.Linear,
// LeakyReLU(0.01), Tanh, torch.cat (folded: the producers write straight into the
// [state | action] rows), mse / smooth-l1 and the backward GEMMs.  This is the
// parity-exact path (plain fp32 fused multiply-add, deterministic fixed-order
// reductions).
#include <algorithm>

#include "mlp.cuh"

namespace gcrl {

enum : int { OP_FWD = 0, OP_DGRAD = 1, OP_WGRAD = 2 };

struct GemmParams {
  const float *A; int lda;
  const float *B; int ldb;
  float *C; int ldc;
  const float *bias;
  const float *act; int ldact;
  float *Cb;
  int M, N, K;
  int act_mode;
  int k_chunk;
  int64_t c_split_stride, cb_split_stride;
};

constexpr int BK = 16;
constexpr int SPAD = 4;

// ---- tile loaders ------------------------------------------------------------------------
// RC: element (i, r) at base[i * ld + r]  (reduction index contiguous)
template <int BT, int NT>
__device__ __forceinline__ void load_rc(const float *__restrict__ base, int ld, int i0, int imax, int r0,
                                        int rmax, float4 (&reg)[BT * 4 / NT], int tid) {
#pragma unroll
  for (int u = 0; u < BT * 4 / NT; ++u) {
    const int c = tid + u * NT;
    const int i = c >> 2, q = c & 3;
    const int gi = i0 + i, gr = r0 + q * 4;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (gi < imax && gr < rmax) {
      const float *ptr = base + size_t(gi) * ld + gr;
      if (gr + 3 < rmax) {
        v = *reinterpret_cast<const float4 *>(ptr);
      } else {
        v.x = ptr[0];
        if (gr + 1 < rmax) v.y = ptr[1];
        if (gr + 2 < rmax) v.z = ptr[2];
      }
    }
    reg[u] = v;
  }
}
template <int BT, int NT>
__device__ __forceinline__ void store_rc(float (*S)[BT + SPAD], const float4 (&reg)[BT * 4 / NT], int tid) {
#pragma unroll
  for (int u = 0; u < BT * 4 / NT; ++u) {
    const int c = tid + u * NT;
    const int i = c >> 2, q = c & 3;
    S[q * 4 + 0][i] = reg[u].x;
    S[q * 4 + 1][i] = reg[u].y;
    S[q * 4 + 2][i] = reg[u].z;
    S[q * 4 + 3][i] = reg[u].w;
  }
}
// IC: element (i, r) at base[r * ld + i]  (output index contiguous)
template <int BT, int NT>
__device__ __forceinline__ void load_ic(const float *__restrict__ base, int ld, int i0, int imax, int r0,
                                        int rmax, float4 (&reg)[BT * 4 / NT], int tid) {
#pragma unroll
  for (int u = 0; u < BT * 4 / NT; ++u) {
    const int c = tid + u * NT;
    const int r = c / (BT / 4), q = c % (BT / 4);
    const int gr = r0 + r, gi = i0 + q * 4;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (gr < rmax && gi < imax) {
      const float *ptr = base + size_t(gr) * ld + gi;
      if (gi + 3 < imax) {
        v = *reinterpret_cast<const float4 *>(ptr);
      } else {
        v.x = ptr[0];
        if (gi + 1 < imax) v.y = ptr[1];
        if (gi + 2 < imax) v.z = ptr[2];
      }
    }
    reg[u] = v;
  }
}
template <int BT, int NT>
__device__ __forceinline__ void store_ic(float (*S)[BT + SPAD], const float4 (&reg)[BT * 4 / NT], int tid) {
#pragma unroll
  for (int u = 0; u < BT * 4 / NT; ++u) {
    const int c = tid + u * NT;
    const int r = c / (BT / 4), q = c % (BT / 4);
    *reinterpret_cast<float4 *>(&S[r][q * 4]) = reg[u];
  }
}

// ---- tiled SGEMM: C[M,N] = sum_r A(m,r) B(r,n) with op-specific operand layouts -----------
//   OP_FWD  : A = X  (RC),  B = W  (RC),  epilogue + bias, LeakyReLU
//   OP_DGRAD: A = dZ (RC),  B = W  (IC),  epilogue * LeakyReLU'(act)
//   OP_WGRAD: A = dZ (IC),  B = X  (IC),  reduction = batch, split over blockIdx.z; the CTAs
//             of the first tile column also emit the bias gradient (column sums of dZ)
template <int BM, int BN, int TM, int TN, int OP>
__device__ __forceinline__ void gemm_body(const GemmParams &p, const int bx, const int by, const int bz) {
  constexpr int NT = (BM / TM) * (BN / TN);
  constexpr int TXN = BN / TN;
  static_assert((BM * 4) % NT == 0 && (BN * 4) % NT == 0, "tile/threads mismatch");
  static_assert(TM == 4 || TM == 8, "TM");
  static_assert(TN == 4 || TN == 8, "TN");
  __shared__ __align__(16) float As[2][BK][BM + SPAD];
  __shared__ __align__(16) float Bs[2][BK][BN + SPAD];

  const int tid = threadIdx.x;
  const int tx = tid % TXN, ty = tid / TXN;
  const int m0 = by * BM, n0 = bx * BN;
  int rbeg = 0, rend = p.K;
  if (OP == OP_WGRAD) {
    rbeg = bz * p.k_chunk;
    rend = min(p.K, rbeg + p.k_chunk);
  }
  const int nk = (rend - rbeg + BK - 1) / BK;

  float4 ra[BM * 4 / NT], rb[BN * 4 / NT];
  float acc[TM][TN];
#pragma unroll
  for (int i = 0; i < TM; ++i)
#pragma unroll
    for (int j = 0; j < TN; ++j) acc[i][j] = 0.f;
  float bsum = 0.f;

  auto gload = [&](int t) {
    const int r0 = rbeg + t * BK;
    if (OP == OP_WGRAD) load_ic<BM, NT>(p.A, p.lda, m0, p.M, r0, rend, ra, tid);
    else                load_rc<BM, NT>(p.A, p.lda, m0, p.M, r0, rend, ra, tid);
    if (OP == OP_FWD)   load_rc<BN, NT>(p.B, p.ldb, n0, p.N, r0, rend, rb, tid);
    else                load_ic<BN, NT>(p.B, p.ldb, n0, p.N, r0, rend, rb, tid);
  };
  auto sstore = [&](int buf) {
    if (OP == OP_WGRAD) store_ic<BM, NT>(As[buf], ra, tid); else store_rc<BM, NT>(As[buf], ra, tid);
    if (OP == OP_FWD)   store_rc<BN, NT>(Bs[buf], rb, tid); else store_ic<BN, NT>(Bs[buf], rb, tid);
  };

  if (nk > 0) {
    gload(0);
    sstore(0);
  }
  __syncthreads();
  for (int t = 0; t < nk; ++t) {
    const int buf = t & 1;
    if (t + 1 < nk) gload(t + 1);
#pragma unroll
    for (int k = 0; k < BK; ++k) {
      float a[TM], b[TN];
      {
        const float4 v = *reinterpret_cast<const float4 *>(&As[buf][k][ty * 4]);
        a[0] = v.x; a[1] = v.y; a[2] = v.z; a[3] = v.w;
        if (TM == 8) {
          const float4 w = *reinterpret_cast<const float4 *>(&As[buf][k][BM / 2 + ty * 4]);
          a[TM - 4] = w.x; a[TM - 3] = w.y; a[TM - 2] = w.z; a[TM - 1] = w.w;
        }
      }
      {
        const float4 v = *reinterpret_cast<const float4 *>(&Bs[buf][k][tx * 4]);
        b[0] = v.x; b[1] = v.y; b[2] = v.z; b[3] = v.w;
        if (TN == 8) {
          const float4 w = *reinterpret_cast<const float4 *>(&Bs[buf][k][BN / 2 + tx * 4]);
          b[TN - 4] = w.x; b[TN - 3] = w.y; b[TN - 2] = w.z; b[TN - 1] = w.w;
        }
      }
#pragma unroll
      for (int i = 0; i < TM; ++i)
#pragma unroll
        for (int j = 0; j < TN; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
    }
    if (OP == OP_WGRAD && bx == 0 && tid < BM) {
#pragma unroll
      for (int k = 0; k < BK; ++k) bsum += As[buf][k][tid];
    }
    if (t + 1 < nk) sstore(buf ^ 1);
    __syncthreads();
  }

  // ---- epilogue ----
  float *C = p.C;
  if (OP == OP_WGRAD) C += int64_t(bz) * p.c_split_stride;
#pragma unroll
  for (int i = 0; i < TM; ++i) {
    const int m = m0 + ((TM == 8 && i >= 4) ? (BM / 2 + ty * 4 + i - 4) : (ty * 4 + i));
    if (m >= p.M) continue;
#pragma unroll
    for (int jh = 0; jh < TN / 4; ++jh) {
      const int n = n0 + (jh == 0 ? tx * 4 : BN / 2 + tx * 4);
      float v[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        float x = acc[i][jh * 4 + j];
        const int nn = n + j;
        if (nn < p.N) {
          if (OP == OP_FWD) {
            x += p.bias[nn];
            if (p.act_mode == ACT_LEAKY) x = x > 0.f ? x : x * kLeakySlope;
          } else if (OP == OP_DGRAD) {
            if (p.act != nullptr) {
              const float h = p.act[size_t(m) * p.ldact + nn];
              x = h > 0.f ? x : x * kLeakySlope;
            }
          }
        }
        v[j] = x;
      }
      // weight-gradient slabs are written over the full padded row (zeros beyond N) so the
      // fixed-order reduction never reads an unwritten word
      const int nbound = (OP == OP_WGRAD) ? p.ldc : p.N;
      float *dst = C + size_t(m) * p.ldc + n;
      if (n + 3 < nbound) {
        *reinterpret_cast<float4 *>(dst) = make_float4(v[0], v[1], v[2], v[3]);
      } else {
#pragma unroll
        for (int j = 0; j < 4; ++j)
          if (n + j < nbound) dst[j] = v[j];
      }
    }
  }
  if (OP == OP_WGRAD && bx == 0 && tid < BM && m0 + tid < p.M)
    p.Cb[int64_t(bz) * p.cb_split_stride + m0 + tid] = bsum;
}

template <int BM, int BN, int TM, int TN, int OP>
__global__ void __launch_bounds__((BM / TM) * (BN / TN)) gemm_kernel(GemmParams p) {
  gemm_body<BM, BN, TM, TN, OP>(p, blockIdx.x, blockIdx.y, blockIdx.z);
}

// Same-shape problems in one launch (the n critics of an ensemble): blockIdx.z enumerates the problems.
struct BatchedGemm {
  GemmParams p[kMaxBatchedLinear];
};

template <int BM, int BN, int TM, int TN, int OP>
__global__ void __launch_bounds__((BM / TM) * (BN / TN)) batched_gemm_kernel(BatchedGemm bg) {
  gemm_body<BM, BN, TM, TN, OP>(bg.p[blockIdx.z], blockIdx.x, blockIdx.y, 0);
}

template <int OP>
static void launch_batched_gemm(const BatchedGemm &bg, int n, cudaStream_t st) {
  const GemmParams &p = bg.p[0];
  const int sms = sm_count();
  auto tiles = [&](int bm, int bn) { return ((p.M + bm - 1) / bm) * ((p.N + bn - 1) / bn) * n; };
  if (tiles(128, 128) >= sms) {
    dim3 grid((p.N + 127) / 128, (p.M + 127) / 128, n);
    batched_gemm_kernel<128, 128, 8, 8, OP><<<grid, 256, 0, st>>>(bg);
  } else if (tiles(64, 64) >= sms / 2) {
    dim3 grid((p.N + 63) / 64, (p.M + 63) / 64, n);
    batched_gemm_kernel<64, 64, 4, 4, OP><<<grid, 256, 0, st>>>(bg);
  } else {
    dim3 grid((p.N + 31) / 32, (p.M + 31) / 32, n);
    batched_gemm_kernel<32, 32, 4, 4, OP><<<grid, 64, 0, st>>>(bg);
  }
  GCRL_LAUNCHED();
}

void launch_linear_fwd_batched(const LinearFwdProblem *pr, int n, int M, int N, int K, int act, cudaStream_t st) {
  GCRL_REQUIRE(n >= 1 && n <= kMaxBatchedLinear, "too many batched problems");
  BatchedGemm bg{};
  for (int i = 0; i < n; ++i) {
    GemmParams &p = bg.p[i];
    p.A = pr[i].X; p.lda = pr[i].ldx; p.B = pr[i].W; p.ldb = pr[i].ldw; p.C = pr[i].Y; p.ldc = pr[i].ldy;
    p.bias = pr[i].bias;
    p.M = M; p.N = N; p.K = K; p.act_mode = act;
  }
  launch_batched_gemm<OP_FWD>(bg, n, st);
}

void launch_linear_dgrad_batched(const LinearDgradProblem *pr, int n, int M, int N, int K, cudaStream_t st) {
  GCRL_REQUIRE(n >= 1 && n <= kMaxBatchedLinear, "too many batched problems");
  BatchedGemm bg{};
  for (int i = 0; i < n; ++i) {
    GemmParams &p = bg.p[i];
    p.A = pr[i].dZ; p.lda = pr[i].lddz; p.B = pr[i].W; p.ldb = pr[i].ldw; p.C = pr[i].dX; p.ldc = pr[i].lddx;
    p.act = pr[i].Xact; p.ldact = pr[i].ldxa;
    p.M = M; p.N = K; p.K = N;  // output [M, K_layer], reduction over the layer's N outputs
  }
  launch_batched_gemm<OP_DGRAD>(bg, n, st);
}

// Multi-problem weight-gradient launches: blockIdx.x enumerates the 32 x 32 output tiles of all problems.
struct MultiGemm {
  GemmParams p[kMaxWgradProblems];
  float *gW[kMaxWgradProblems], *gB[kMaxWgradProblems];   // complete-gradient destinations (wgrad_tile_kernel)
  int tile_begin[kMaxWgradProblems + 1];
  int tiles_x[kMaxWgradProblems];
  int nprob;
  WgradFinal fin;
};

__device__ __forceinline__ void locate_tile(const MultiGemm &mg, int &i, int &bx, int &by) {
  i = 0;
  while (i + 1 < mg.nprob && int(blockIdx.x) >= mg.tile_begin[i + 1]) ++i;
  const int local = blockIdx.x - mg.tile_begin[i];
  bx = local % mg.tiles_x[i];
  by = local / mg.tiles_x[i];
}

// split-batch partial slabs (blockIdx.z), summed later by reduce_grads_kernel: the ensemble path of sac.cu
template <int BM, int BN, int TM, int TN>
__global__ void __launch_bounds__((BM / TM) * (BN / TN)) multi_wgrad_kernel(const __grid_constant__ MultiGemm mg) {
  int i, bx, by;
  locate_tile(mg, i, bx, by);
  gemm_body<BM, BN, TM, TN, OP_WGRAD>(mg.p[i], bx, by, blockIdx.z);
}

// ---- complete weight gradients in one launch (row-slab path, batch <= 1024) -------------------------------
// One CTA per 32 x 32 output tile, GROUPS groups of 64 threads; group g reduces batch rows [g chunk, (g+1) chunk)
// with the 4 x 4 register tiles of gemm_body (own shared-memory stage, own named barrier), then the groups'
// tiles are summed through shared memory in group order -- a fixed order -- straight into the flat gradient,
// together with the tile's sum of squares for the global-norm clip.  No partial slabs in HBM, no reduction
// launch, no atomics.  Tile 0 also finalises the batch-mean metrics of the phase.
constexpr int kWgThreads = 64, kWgTile = 32, kWgFinish = 256;
constexpr int kWgMaxMetricSlabs = 256;                       // row-slab kernels run <= 256 CTAs (fused_supported)
constexpr int kWgStageFloats = 2 * 2 * BK * (kWgTile + SPAD);      // As[2][BK][36] + Bs[2][BK][36] per group

__device__ __forceinline__ void bar_group(int grp) { asm volatile("bar.sync %0, %1;" ::"r"(grp + 1), "n"(kWgThreads) : "memory"); }

// sum of squares of one finished tile: thread t < 256 owns the 16-byte group t of the tile (+ bias row t for
// t < 32 in the first tile column); 8 warp trees, then the 8 warp sums in order.  Shared by both kernels below.
__device__ __forceinline__ void tile_sumsq_store(float sq, float *s_sq, float *dst) {
  const int tid = threadIdx.x;
  if (tid < kWgFinish) {
#pragma unroll
    for (int s = 16; s >= 1; s >>= 1) sq += __shfl_xor_sync(0xffffffffu, sq, s);
    if ((tid & 31) == 0) s_sq[tid >> 5] = sq;
  }
  __syncthreads();
  if (tid == 0) {
    float t = 0.f;
#pragma unroll
    for (int w = 0; w < kWgFinish / 32; ++w) t += s_sq[w];
    *dst = t;
  }
}

template <int GROUPS>
__global__ void __launch_bounds__(kWgThreads * GROUPS) wgrad_tile_kernel(const __grid_constant__ MultiGemm mg) {
  constexpr int BM = kWgTile, BN = kWgTile, NT = kWgThreads, TXN = BN / 4;
  static_assert(GROUPS * kWgThreads >= kWgFinish && GROUPS <= 8, "finish mapping / named barriers");
  extern __shared__ float4 wg_sm4[];
  __shared__ float s_sq[kWgFinish / 32];
  float *sm = reinterpret_cast<float *>(wg_sm4);
  __shared__ __align__(16) float s_met[kWgMaxMetricSlabs * 4];
  pdl_wait();
  pdl_launch_dependents();
  // tile 0 sums the row-slab kernel's metric partials slab after slab at the end; copied here in one round trip,
  // they are no longer a chain of loads at the end of the kernel (B = 256: 128 slabs, 8 round trips of 16 loads)
  const bool metrics_here = blockIdx.x == 0 && mg.fin.metric_partials != nullptr;
  if (metrics_here && int(threadIdx.x) < mg.fin.metric_splits) {
    const unsigned int d = static_cast<unsigned int>(__cvta_generic_to_shared(s_met + threadIdx.x * 4));
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(d), "l"(mg.fin.metric_partials + threadIdx.x * 4) : "memory");
  }
  int pi, bx, by;
  locate_tile(mg, pi, bx, by);
  const GemmParams &p = mg.p[pi];
  const int grp = threadIdx.x / NT, tid = threadIdx.x % NT;
  const int tx = tid % TXN, ty = tid / TXN;
  const int m0 = by * BM, n0 = bx * BN;
  float(*As)[BK][BM + SPAD] = reinterpret_cast<float(*)[BK][BM + SPAD]>(sm + size_t(grp) * kWgStageFloats);
  float(*Bs)[BK][BN + SPAD] = reinterpret_cast<float(*)[BK][BN + SPAD]>(sm + size_t(grp) * kWgStageFloats + 2 * BK * (BM + SPAD));
  const int rbeg = min(p.K, grp * p.k_chunk), rend = min(p.K, rbeg + p.k_chunk);
  const int nk = (rend - rbeg + BK - 1) / BK;
  float4 ra[BM * 4 / NT], rb[BN * 4 / NT];
  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
  float bsum = 0.f;
  auto gload = [&](int t) {
    const int r0 = rbeg + t * BK;
    load_ic<BM, NT>(p.A, p.lda, m0, p.M, r0, rend, ra, tid);
    load_ic<BN, NT>(p.B, p.ldb, n0, p.N, r0, rend, rb, tid);
  };
  auto sstore = [&](int buf) {
    store_ic<BM, NT>(As[buf], ra, tid);
    store_ic<BN, NT>(Bs[buf], rb, tid);
  };
  if (nk > 0) {
    gload(0);
    sstore(0);
  }
  bar_group(grp);
  for (int t = 0; t < nk; ++t) {
    const int buf = t & 1;
    if (t + 1 < nk) gload(t + 1);
#pragma unroll
    for (int k = 0; k < BK; ++k) {
      const float4 av = *reinterpret_cast<const float4 *>(&As[buf][k][ty * 4]);
      const float4 bv = *reinterpret_cast<const float4 *>(&Bs[buf][k][tx * 4]);
      const float a[4] = {av.x, av.y, av.z, av.w}, b[4] = {bv.x, bv.y, bv.z, bv.w};
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
    }
    if (bx == 0 && tid < BM) {
#pragma unroll
      for (int k = 0; k < BK; ++k) bsum += As[buf][k][tid];
    }
    if (t + 1 < nk) sstore(buf ^ 1);
    bar_group(grp);
  }
  // ---- the groups' tiles -> shared memory (each group reuses its own stage), then the ordered sum ----
  float *red = sm + size_t(grp) * kWgStageFloats;          // [32][32] tile, then [32] bias sums
#pragma unroll
  for (int i = 0; i < 4; ++i)
    *reinterpret_cast<float4 *>(red + (ty * 4 + i) * BN + tx * 4) = make_float4(acc[i][0], acc[i][1], acc[i][2], acc[i][3]);
  if (tid < BM) red[BM * BN + tid] = bsum;
  asm volatile("cp.async.wait_all;" ::: "memory");           // (the metric partials)
  __syncthreads();
  float sq = 0.f;
  const int t = threadIdx.x;
  if (t < kWgFinish) {
    const int r = t / (BN / 4), c = (t % (BN / 4)) * 4;
    float4 g = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int z = 0; z < GROUPS; ++z) {
      const float4 v = *reinterpret_cast<const float4 *>(sm + size_t(z) * kWgStageFloats + r * BN + c);
      g.x += v.x; g.y += v.y; g.z += v.z; g.w += v.w;
    }
    // rows are written over the full padded width (zeros beyond the layer's input width)
    if (m0 + r < p.M && n0 + c < p.ldc) {
      *reinterpret_cast<float4 *>(mg.gW[pi] + size_t(m0 + r) * p.ldc + n0 + c) = g;
      sq = fmaf(g.x, g.x, sq); sq = fmaf(g.y, g.y, sq); sq = fmaf(g.z, g.z, sq); sq = fmaf(g.w, g.w, sq);
    }
    if (bx == 0 && t < BM && m0 + t < p.M) {
      float gb = 0.f;
#pragma unroll
      for (int z = 0; z < GROUPS; ++z) gb += sm[size_t(z) * kWgStageFloats + BM * BN + t];
      mg.gB[pi][m0 + t] = gb;
      sq = fmaf(gb, gb, sq);
    }
  }
  if (metrics_here && t < 3) {
    float s = 0.f;
    for (int k = 0; k < mg.fin.metric_splits; ++k) s += s_met[k * 4 + t];
    const int slot = t == 0 ? mg.fin.slot_loss : (t == 1 ? mg.fin.slot_td : mg.fin.slot_q);
    if (slot >= 0) mg.fin.metrics[slot] = s * mg.fin.metric_scale;
  }
  tile_sumsq_store(sq, s_sq, mg.fin.sumsq_partials + blockIdx.x);
  if (mg.fin.peer_flags != nullptr) {
    // every CTA: gradient tile (and tile 0's metrics) ordered before its ticket; the last one raises the flags
    __shared__ int s_last;
    __syncthreads();
    if (t == 0) {
      __threadfence();
      const unsigned int k = atomicAdd(mg.fin.ticket, 1u);
      s_last = k == gridDim.x - 1;
      if (s_last) *mg.fin.ticket = 0;
    }
    __syncthreads();
    if (s_last) {
      const unsigned int e = *mg.fin.epoch + 1u;
      if (t < 8) mg.fin.outbox[(e & 1u) * 8 + t] = __ldcg(mg.fin.metrics + t);
      __syncthreads();
      if (t < mg.fin.world) {
        __threadfence_system();
        volatile unsigned int *dst = mg.fin.peer_flags[t] + mg.fin.rank;
        *dst = e;
      }
    }
  }
}

// sums of squares of a complete flat gradient, tile by tile, bit-identical to what wgrad_tile_kernel leaves
// for the same values (the data-parallel phases, after the cross-rank average replaced the gradient)
__global__ void __launch_bounds__(kWgFinish) wgrad_sumsq_kernel(const __grid_constant__ MultiGemm mg) {
  constexpr int BM = kWgTile, BN = kWgTile;
  __shared__ float s_sq[kWgFinish / 32];
  pdl_wait();
  pdl_launch_dependents();
  int pi, bx, by;
  locate_tile(mg, pi, bx, by);
  const GemmParams &p = mg.p[pi];
  const int m0 = by * BM, n0 = bx * BN, t = threadIdx.x;
  const int r = t / (BN / 4), c = (t % (BN / 4)) * 4;
  float sq = 0.f;
  if (m0 + r < p.M && n0 + c < p.ldc) {
    const float4 g = __ldcg(reinterpret_cast<const float4 *>(mg.gW[pi] + size_t(m0 + r) * p.ldc + n0 + c));
    sq = fmaf(g.x, g.x, sq); sq = fmaf(g.y, g.y, sq); sq = fmaf(g.z, g.z, sq); sq = fmaf(g.w, g.w, sq);
  }
  if (bx == 0 && t < BM && m0 + t < p.M) {
    const float gb = __ldcg(mg.gB[pi] + m0 + t);
    sq = fmaf(gb, gb, sq);
  }
  tile_sumsq_store(sq, s_sq, mg.fin.sumsq_partials + blockIdx.x);
}

static int fill_multi(MultiGemm &mg, const WgradProblem *probs, int nprob, int M, int64_t split_stride, int chunk,
                      bool need_dest) {
  GCRL_REQUIRE(nprob >= 1 && nprob <= kMaxWgradProblems, "too many wgrad problems");
  mg.nprob = nprob;
  int tiles = 0;
  for (int i = 0; i < nprob; ++i) {
    GemmParams &p = mg.p[i];
    p.A = probs[i].dZ; p.lda = probs[i].lddz; p.B = probs[i].X; p.ldb = probs[i].ldx;
    p.C = probs[i].pW; p.ldc = probs[i].ldw; p.Cb = probs[i].pB;
    p.M = probs[i].N; p.N = probs[i].K; p.K = M;
    p.k_chunk = chunk;
    p.c_split_stride = split_stride;
    p.cb_split_stride = split_stride;
    mg.gW[i] = probs[i].gW; mg.gB[i] = probs[i].gB;
    GCRL_REQUIRE(!need_dest || (probs[i].gW != nullptr && probs[i].gB != nullptr), "fused wgrad needs gradient destinations");
    mg.tile_begin[i] = tiles;
    mg.tiles_x[i] = (p.N + 31) / 32;
    tiles += mg.tiles_x[i] * ((p.M + 31) / 32);
  }
  mg.tile_begin[nprob] = tiles;
  return tiles;
}

int launch_multi_wgrad(const WgradProblem *probs, int nprob, int M, int64_t split_stride, int max_splits,
                       cudaStream_t st) {
  int splits = std::max(1, std::min(max_splits, M / 64));
  int chunk = (M + splits - 1) / splits;
  chunk = (chunk + BK - 1) / BK * BK;
  splits = (M + chunk - 1) / chunk;
  MultiGemm mg{};
  const int tiles = fill_multi(mg, probs, nprob, M, split_stride, chunk, false);
  multi_wgrad_kernel<32, 32, 4, 4><<<dim3(tiles, 1, splits), 64, 0, st>>>(mg);
  GCRL_LAUNCHED();
  return splits;
}

template <int GROUPS>
static void launch_wgrad_tiles(const MultiGemm &mg, int tiles, cudaStream_t st) {
  static bool attr_set = false;
  const size_t smem = size_t(GROUPS) * kWgStageFloats * sizeof(float);
  if (!attr_set && smem > 48 * 1024) {
    GCRL_CUDA(cudaFuncSetAttribute(wgrad_tile_kernel<GROUPS>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem)));
    attr_set = true;
  }
  // no early launch: the small CTAs would pile onto the SMs the preceding row-slab kernel leaves free.  Measured again
  // with the metric partials prefetched (profiles/r04_update_tail.json, B = 256 flushed step on one B200 at 1000 W):
  // PDL_WGRAD on 0.1209 ms, off 0.1147 ms; each weight-gradient launch adds 10.6-11.0 instead of 7.2-7.3 us
  launch_pdl<PDL_WGRAD>(wgrad_tile_kernel<GROUPS>, dim3(tiles), dim3(kWgThreads * GROUPS), smem, st, mg);
}

int launch_wgrad_complete(const WgradProblem *probs, int nprob, int M, const WgradFinal &fin, cudaStream_t st) {
  // 4 or 8 groups per CTA (the ordered sum needs >= 256 threads; named barriers 1..8 + the CTA barrier)
  const int groups = M > 256 ? 8 : 4;
  int chunk = (M + groups - 1) / groups;
  chunk = (chunk + BK - 1) / BK * BK;
  GCRL_REQUIRE(fin.metric_partials == nullptr ||
                   (fin.metric_splits <= kWgMaxMetricSlabs && (reinterpret_cast<uintptr_t>(fin.metric_partials) & 15) == 0),
               "wgrad metrics: at most 256 16-byte aligned partial slabs");
  MultiGemm mg{};
  mg.fin = fin;
  const int tiles = fill_multi(mg, probs, nprob, M, 0, chunk, true);
  if (groups == 8) launch_wgrad_tiles<8>(mg, tiles, st);
  else launch_wgrad_tiles<4>(mg, tiles, st);
  GCRL_LAUNCHED();
  return tiles;
}

int launch_wgrad_sumsq(const WgradProblem *probs, int nprob, float *sumsq_partials, cudaStream_t st) {
  MultiGemm mg{};
  mg.fin.sumsq_partials = sumsq_partials;
  const int tiles = fill_multi(mg, probs, nprob, 0, 0, 0, true);
  launch_pdl<PDL_WGRAD>(wgrad_sumsq_kernel, dim3(tiles), dim3(kWgFinish), 0, st, mg);
  GCRL_LAUNCHED();
  return tiles;
}

template <int OP>
static void launch_gemm(const GemmParams &p, int splits, cudaStream_t st) {
  const int sms = sm_count();
  // weight-gradient slabs: the column tiles span the whole padded row (ldc), so that the epilogue writes its zeros
  // beyond N even where ldc reaches past the last tile of the N columns
  const int ncols = OP == OP_WGRAD ? std::max(p.N, p.ldc) : p.N;
  auto tiles = [&](int bm, int bn) { return ((p.M + bm - 1) / bm) * ((ncols + bn - 1) / bn) * splits; };
  if (tiles(128, 128) >= sms) {
    dim3 grid((ncols + 127) / 128, (p.M + 127) / 128, splits);
    gemm_kernel<128, 128, 8, 8, OP><<<grid, 256, 0, st>>>(p);
  } else if (tiles(64, 64) >= sms / 2) {
    dim3 grid((ncols + 63) / 64, (p.M + 63) / 64, splits);
    gemm_kernel<64, 64, 4, 4, OP><<<grid, 256, 0, st>>>(p);
  } else {
    dim3 grid((ncols + 31) / 32, (p.M + 31) / 32, splits);
    gemm_kernel<32, 32, 4, 4, OP><<<grid, 64, 0, st>>>(p);
  }
  GCRL_LAUNCHED();
}

void launch_linear_fwd(const float *X, int ldx, const float *W, int ldw, const float *bias, float *Y,
                       int ldy, int M, int N, int K, int act, cudaStream_t st) {
  GemmParams p{};
  p.A = X; p.lda = ldx; p.B = W; p.ldb = ldw; p.C = Y; p.ldc = ldy; p.bias = bias;
  p.M = M; p.N = N; p.K = K; p.act_mode = act;
  launch_gemm<OP_FWD>(p, 1, st);
}

void launch_linear_dgrad(const float *dZ, int lddz, const float *W, int ldw, const float *Xact,
                         int ldxa, float *dX, int lddx, int M, int N, int K, cudaStream_t st) {
  GemmParams p{};
  p.A = dZ; p.lda = lddz; p.B = W; p.ldb = ldw; p.C = dX; p.ldc = lddx;
  p.act = Xact; p.ldact = ldxa;
  p.M = M; p.N = K; p.K = N;  // output [M, K_layer], reduction over the layer's N outputs
  launch_gemm<OP_DGRAD>(p, 1, st);
}

int launch_linear_wgrad(const float *dZ, int lddz, const float *X, int ldx, float *pW, int ldw,
                        int64_t w_split_stride, float *pB, int64_t b_split_stride, int M, int N, int K,
                        int max_splits, cudaStream_t st) {
  // output [N, K] (+ bias [N]); reduction over the M batch rows, split into slabs
  const int sms = sm_count();
  const int base_tiles = ((N + 63) / 64) * ((K + 63) / 64);
  int splits = std::max(1, std::min(max_splits, (2 * sms + base_tiles - 1) / base_tiles));
  int chunk = (M + splits - 1) / splits;
  chunk = std::max(64, (chunk + BK - 1) / BK * BK);
  splits = (M + chunk - 1) / chunk;
  GemmParams p{};
  p.A = dZ; p.lda = lddz; p.B = X; p.ldb = ldx; p.C = pW; p.ldc = ldw; p.Cb = pB;
  p.M = N; p.N = K; p.K = M;
  p.k_chunk = chunk;
  p.c_split_stride = w_split_stride;
  p.cb_split_stride = b_split_stride;
  launch_gemm<OP_WGRAD>(p, splits, st);
  return splits;
}

// ---- skinny output layer ---------------------------------------------------------------------
template <int NOUT>
__global__ void __launch_bounds__(256)
head_fwd_kernel(const float *__restrict__ H, int ldh, const float *__restrict__ W, int ldw,
                const float *__restrict__ bias, float *__restrict__ out, int ldo, int col0, int M, int K,
                int tanh_out) {
  // One warp per row, kRows rows of a warp in flight at once (the loads of all of them are issued before the first
  // FMA): with one row at a time a warp had 1 KB in flight and the 64 MB read of a B = 65 536 batch ran at 2 TB/s.
  // Per row the arithmetic and its order are those of the one-row loop (lane-strided partial sums, xor-shuffle tree).
  constexpr int kRows = 4;
  const int lane = threadIdx.x & 31;
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int nwarps = (gridDim.x * blockDim.x) >> 5;
  const int K4 = K >> 2;
  for (int m0 = warp * kRows; m0 < M; m0 += nwarps * kRows) {
    float acc[kRows][NOUT];
#pragma unroll
    for (int r = 0; r < kRows; ++r)
#pragma unroll
      for (int n = 0; n < NOUT; ++n) acc[r][n] = 0.f;
    for (int k4 = lane; k4 < K4; k4 += 32) {
      float4 hv[kRows];
#pragma unroll
      for (int r = 0; r < kRows; ++r)
        hv[r] = m0 + r < M ? *reinterpret_cast<const float4 *>(H + size_t(m0 + r) * ldh + k4 * 4)
                           : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
      for (int n = 0; n < NOUT; ++n) {
        const float4 wv = *reinterpret_cast<const float4 *>(W + size_t(n) * ldw + k4 * 4);
#pragma unroll
        for (int r = 0; r < kRows; ++r) {
          acc[r][n] = fmaf(hv[r].x, wv.x, acc[r][n]);
          acc[r][n] = fmaf(hv[r].y, wv.y, acc[r][n]);
          acc[r][n] = fmaf(hv[r].z, wv.z, acc[r][n]);
          acc[r][n] = fmaf(hv[r].w, wv.w, acc[r][n]);
        }
      }
    }
    for (int k = K4 * 4 + lane; k < K; k += 32) {
#pragma unroll
      for (int r = 0; r < kRows; ++r)
        if (m0 + r < M) {
#pragma unroll
          for (int n = 0; n < NOUT; ++n) acc[r][n] = fmaf(H[size_t(m0 + r) * ldh + k], W[size_t(n) * ldw + k], acc[r][n]);
        }
    }
#pragma unroll
    for (int r = 0; r < kRows; ++r)
#pragma unroll
      for (int n = 0; n < NOUT; ++n)
#pragma unroll
        for (int s = 16; s >= 1; s >>= 1) acc[r][n] += __shfl_xor_sync(0xffffffffu, acc[r][n], s);
    if (lane < kRows && m0 + lane < M) {               // lane r stores row m0 + r
#pragma unroll
      for (int n = 0; n < NOUT; ++n) {
        float v = 0.f;
#pragma unroll
        for (int r = 0; r < kRows; ++r) v = lane == r ? acc[r][n] : v;
        v += bias[n];
        if (tanh_out) v = tanhf(v);
        out[size_t(m0 + lane) * ldo + col0 + n] = v;
      }
    }
  }
}

// scalar heads of several same-shape networks in one launch: blockIdx.y enumerates the networks
struct HeadFwdBatch {
  HeadFwdProblem p[kMaxBatchedLinear];
};

__global__ void __launch_bounds__(256) head_fwd_batched_kernel(HeadFwdBatch hb, int ldh, int ldw, int M, int K) {
  const HeadFwdProblem &pr = hb.p[blockIdx.y];
  const int lane = threadIdx.x & 31;
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int nwarps = (gridDim.x * blockDim.x) >> 5;
  const int K4 = K >> 2;
  for (int m = warp; m < M; m += nwarps) {          // same arithmetic order as head_fwd_kernel<1>
    const float *h = pr.Hact + size_t(m) * ldh;
    float acc = 0.f;
    for (int k4 = lane; k4 < K4; k4 += 32) {
      const float4 hv = *reinterpret_cast<const float4 *>(h + k4 * 4);
      const float4 wv = *reinterpret_cast<const float4 *>(pr.W + k4 * 4);
      acc = fmaf(hv.x, wv.x, acc);
      acc = fmaf(hv.y, wv.y, acc);
      acc = fmaf(hv.z, wv.z, acc);
      acc = fmaf(hv.w, wv.w, acc);
    }
    for (int k = K4 * 4 + lane; k < K; k += 32) acc = fmaf(h[k], pr.W[k], acc);
#pragma unroll
    for (int s = 16; s >= 1; s >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, s);
    if (lane == 0) pr.out[m] = acc + pr.bias[0];
  }
}

void launch_head_fwd_batched(const HeadFwdProblem *pr, int n, int ldh, int ldw, int M, int K, cudaStream_t st) {
  GCRL_REQUIRE(n >= 1 && n <= kMaxBatchedLinear, "too many batched problems");
  HeadFwdBatch hb{};
  for (int i = 0; i < n; ++i) hb.p[i] = pr[i];
  const int blocks = std::max(1, std::min((M + 7) / 8, sm_count() * 8));
  head_fwd_batched_kernel<<<dim3(blocks, n), 256, 0, st>>>(hb, ldh, ldw, M, K);
  GCRL_LAUNCHED();
}

void launch_head_fwd(const float *Hact, int ldh, const float *W, int ldw, const float *bias, float *out,
                     int ldo, int col0, int M, int K, int nout, int tanh_out, cudaStream_t st) {
  const int blocks = std::max(1, std::min((M + 31) / 32, sm_count() * 8));       // 8 warps x 4 rows per block
  switch (nout) {
    case 1: head_fwd_kernel<1><<<blocks, 256, 0, st>>>(Hact, ldh, W, ldw, bias, out, ldo, col0, M, K, tanh_out); break;
    case 2: head_fwd_kernel<2><<<blocks, 256, 0, st>>>(Hact, ldh, W, ldw, bias, out, ldo, col0, M, K, tanh_out); break;
    case 3: head_fwd_kernel<3><<<blocks, 256, 0, st>>>(Hact, ldh, W, ldw, bias, out, ldo, col0, M, K, tanh_out); break;
    case 4: head_fwd_kernel<4><<<blocks, 256, 0, st>>>(Hact, ldh, W, ldw, bias, out, ldo, col0, M, K, tanh_out); break;
    default: throw Error(GCRL_ERR_INVALID, "head width must be 1..4");
  }
  GCRL_LAUNCHED();
}

// ---- loss + backward through the skinny output layer ------------------------------------------
constexpr int kHeadSlabMax = 512;
constexpr int kHeadColBlock = 64;

template <int NOUT>
__device__ __forceinline__ void head_bwd_body(const HeadBwdArgs &a, int rows_per_slab) {
  __shared__ float dz_s[kHeadSlabMax][NOUT];
  __shared__ float met_s[kHeadSlabMax][3];
  const int tid = threadIdx.x;
  const int r0 = blockIdx.x * rows_per_slab;
  const int nrows = min(rows_per_slab, a.M - r0);
  const float invM = 1.0f / float(a.M);

  for (int i = tid; i < nrows; i += blockDim.x) {
    const int m = r0 + i;
    if (a.mode == 0) {
      float y;
      if (a.y_in != nullptr) {
        y = a.y_in[m];
      } else {
        float qt = a.qt1[m];
        if (a.qt2 != nullptr) qt = fminf(qt, a.qt2[m]);
        y = a.r[m] + a.gamma * (1.0f - a.d[m]) * qt;
        if (a.clamp_y) y = fminf(fmaxf(y, a.y_lo), 0.0f);
      }
      if (a.y_out != nullptr) a.y_out[m] = y;
      const float q = a.q[m];
      const float diff = q - y;
      float loss, g;
      if (a.loss_kind == 0) {            // mse_loss
        loss = diff * diff;
        g = 2.0f * diff;
      } else {                           // smooth_l1_loss, beta = 1
        const float ad = fabsf(diff);
        loss = ad < 1.0f ? 0.5f * diff * diff : ad - 0.5f;
        g = ad < 1.0f ? diff : (diff > 0.f ? 1.0f : -1.0f);
      }
      const float w = a.is_w != nullptr ? a.is_w[m] : 1.0f;   // (weights * loss).mean(), src/agent.py:1322-1324
      dz_s[i][0] = g * invM * w;
      met_s[i][0] = loss * w;
      if (a.q_other != nullptr) {        // TD3: mean(max(td1, td2)), mean over both critics' q
        const float qo = a.q_other[m];
        met_s[i][1] = fmaxf(fabsf(q - y), fabsf(qo - y));
        met_s[i][2] = 0.5f * (q + qo);
      } else {
        met_s[i][1] = fabsf(y - q);
        met_s[i][2] = q;
      }
      if (a.td_out != nullptr && blockIdx.y == 0) a.td_out[m] = met_s[i][1];
    } else if (a.mode == 1) {
      dz_s[i][0] = -invM;
      met_s[i][0] = -a.q[m];             // actor loss = -mean(q)
      met_s[i][1] = 0.f;
      met_s[i][2] = a.q[m];
    } else {
#pragma unroll
      for (int n = 0; n < NOUT; ++n) dz_s[i][n] = a.dz_in[size_t(m) * 4 + n];
    }
  }
  __syncthreads();

  if (blockIdx.y == 0) {
    if (a.mode != 2 && tid < 3) {          // fixed-order partial sums of the slab's metrics
      float s = 0.f;
      for (int i = 0; i < nrows; ++i) s += met_s[i][tid];
      a.metric_partials[size_t(blockIdx.x) * 4 + tid] = s;
    }
    if (a.pB != nullptr && tid >= 32 && tid < 32 + NOUT) {
      const int n = tid - 32;
      float s = 0.f;
      for (int i = 0; i < nrows; ++i) s += dz_s[i][n];
      a.pB[int64_t(blockIdx.x) * a.b_split_stride + n] = s;
    }
  }

  // column block blockIdx.y (64 columns): 16 column groups of 4 x 16 row groups; every access is a
  // 16-byte vector; the per-row-group weight-gradient partials are combined in a fixed order
  __shared__ float red_s[16][NOUT][kHeadColBlock];
  const int cgp = tid & 15, rg = tid >> 4;
  const int k0 = blockIdx.y * kHeadColBlock + cgp * 4;
  float w[NOUT][4], acc[NOUT][4];
  bool valid[4];
#pragma unroll
  for (int u = 0; u < 4; ++u) valid[u] = k0 + u < a.K;
#pragma unroll
  for (int n = 0; n < NOUT; ++n)
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      w[n][u] = valid[u] ? a.W[size_t(n) * a.ldw + k0 + u] : 0.f;
      acc[n][u] = 0.f;
    }
  if (valid[0]) {
#pragma unroll 4
    for (int i = rg; i < nrows; i += 16) {
      const size_t m = size_t(r0 + i);
      const float4 hv = *reinterpret_cast<const float4 *>(a.Hact + m * a.ldh + k0);
      const float h[4] = {valid[0] ? hv.x : 0.f, valid[1] ? hv.y : 0.f, valid[2] ? hv.z : 0.f, valid[3] ? hv.w : 0.f};
      float dh[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
      for (int n = 0; n < NOUT; ++n) {
        const float dz = dz_s[i][n];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          dh[u] = fmaf(dz, w[n][u], dh[u]);
          acc[n][u] = fmaf(dz, h[u], acc[n][u]);
        }
      }
#pragma unroll
      for (int u = 0; u < 4; ++u) dh[u] = h[u] > 0.f ? dh[u] : dh[u] * kLeakySlope;
      *reinterpret_cast<float4 *>(a.dZprev + m * a.lddz + k0) = make_float4(dh[0], dh[1], dh[2], dh[3]);
    }
  }
  if (a.pW != nullptr) {
#pragma unroll
    for (int n = 0; n < NOUT; ++n)
#pragma unroll
      for (int u = 0; u < 4; ++u) red_s[rg][n][cgp * 4 + u] = acc[n][u];
    __syncthreads();
    for (int idx = tid; idx < NOUT * kHeadColBlock; idx += blockDim.x) {
      const int n = idx / kHeadColBlock, c = idx - n * kHeadColBlock;
      const int k = blockIdx.y * kHeadColBlock + c;
      if (k < a.ldw) {                    // columns K .. ldw-1 (row padding of the slab) receive exact zeros
        float s = 0.f;
#pragma unroll
        for (int g = 0; g < 16; ++g) s += red_s[g][n][c];
        a.pW[int64_t(blockIdx.x) * a.w_split_stride + size_t(n) * a.ldw + k] = s;
      }
    }
  }
}

template <int NOUT>
__global__ void __launch_bounds__(256) head_bwd_kernel(HeadBwdArgs a, int rows_per_slab) {
  head_bwd_body<NOUT>(a, rows_per_slab);
}

// the same for several same-shape networks (scalar heads of a critic ensemble): blockIdx.z = network
struct HeadBwdBatch {
  HeadBwdArgs a[kMaxBatchedLinear];
};
__global__ void __launch_bounds__(256) head_bwd_batched_kernel(HeadBwdBatch hb, int rows_per_slab) {
  head_bwd_body<1>(hb.a[blockIdx.z], rows_per_slab);
}

int launch_head_bwd_batched(const HeadBwdArgs *a, int n, int max_splits, cudaStream_t st) {
  GCRL_REQUIRE(n >= 1 && n <= kMaxBatchedLinear, "too many batched problems");
  HeadBwdBatch hb{};
  for (int i = 0; i < n; ++i) {
    GCRL_REQUIRE(a[i].nout == 1 && a[i].M == a[0].M && a[i].K == a[0].K, "batched heads must share their shape");
    hb.a[i] = a[i];
  }
  int rows = (a[0].M + max_splits - 1) / max_splits;
  rows = std::min(kHeadSlabMax, std::max(rows, 16));
  const int slabs = (a[0].M + rows - 1) / rows;
  if (slabs > max_splits) throw Error(GCRL_ERR_INVALID, "batch too large for head_bwd partial buffers");
  const dim3 grid(slabs, (a[0].K + kHeadColBlock - 1) / kHeadColBlock, n);
  head_bwd_batched_kernel<<<grid, 256, 0, st>>>(hb, rows);
  GCRL_LAUNCHED();
  return slabs;
}

int launch_head_bwd(const HeadBwdArgs &a, int max_splits, cudaStream_t st) {
  int rows = (a.M + max_splits - 1) / max_splits;
  rows = std::min(kHeadSlabMax, std::max(rows, 16));
  const int slabs = (a.M + rows - 1) / rows;
  if (slabs > max_splits) throw Error(GCRL_ERR_INVALID, "batch too large for head_bwd partial buffers");
  const dim3 grid(slabs, (a.K + kHeadColBlock - 1) / kHeadColBlock);
  switch (a.nout) {
    case 1: head_bwd_kernel<1><<<grid, 256, 0, st>>>(a, rows); break;
    case 2: head_bwd_kernel<2><<<grid, 256, 0, st>>>(a, rows); break;
    case 3: head_bwd_kernel<3><<<grid, 256, 0, st>>>(a, rows); break;
    case 4: head_bwd_kernel<4><<<grid, 256, 0, st>>>(a, rows); break;
    default: throw Error(GCRL_ERR_INVALID, "head width must be 1..4");
  }
  GCRL_LAUNCHED();
  return slabs;
}

// ---- d(actor loss)/d(action) through critic layer 1, fused with tanh' ---------------------------
__global__ void __launch_bounds__(256)
action_grad_kernel(const float *__restrict__ dZ1, int lddz, const float *__restrict__ W1, int ldw,
                   const float *__restrict__ sa, int ldsa, int col0, float *__restrict__ dz_out, int M, int N,
                   int nact, int staged) {
  // the [N][4] action-column block of W1 is staged once per CTA (a strided gather otherwise: every lane
  // would touch a different row of W1 for every element of dZ1); very wide layers read it in place
  extern __shared__ float4 w_s[];
  if (staged) {
    for (int n = threadIdx.x; n < N; n += blockDim.x) {
      const float *w = W1 + size_t(n) * ldw + col0;
      w_s[n] = make_float4(w[0], nact > 1 ? w[1] : 0.f, nact > 2 ? w[2] : 0.f, nact > 3 ? w[3] : 0.f);
    }
    __syncthreads();
  }
  const int lane = threadIdx.x & 31;
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int nwarps = (gridDim.x * blockDim.x) >> 5;
  for (int m = warp; m < M; m += nwarps) {
    float acc[4] = {0.f, 0.f, 0.f, 0.f};
    for (int n = lane; n < N; n += 32) {
      const float g = dZ1[size_t(m) * lddz + n];
      float4 w;
      if (staged) {
        w = w_s[n];
      } else {
        const float *wp = W1 + size_t(n) * ldw + col0;
        w = make_float4(wp[0], nact > 1 ? wp[1] : 0.f, nact > 2 ? wp[2] : 0.f, nact > 3 ? wp[3] : 0.f);
      }
      acc[0] = fmaf(g, w.x, acc[0]);
      acc[1] = fmaf(g, w.y, acc[1]);
      acc[2] = fmaf(g, w.z, acc[2]);
      acc[3] = fmaf(g, w.w, acc[3]);
    }
#pragma unroll
    for (int j = 0; j < 4; ++j)
#pragma unroll
      for (int s = 16; s >= 1; s >>= 1) acc[j] += __shfl_xor_sync(0xffffffffu, acc[j], s);
    if (lane < 4) {
      float v = 0.f;
      if (lane < nact) {
        const float act = sa[size_t(m) * ldsa + col0 + lane];
        const float g = lane == 0 ? acc[0] : (lane == 1 ? acc[1] : (lane == 2 ? acc[2] : acc[3]));
        v = g * (1.0f - act * act);
      }
      dz_out[size_t(m) * 4 + lane] = v;
    }
  }
}

void launch_action_grad(const float *dZ1, int lddz, const float *W1, int ldw, const float *sa, int ldsa,
                        int col0, float *dz_out, int M, int N, int nact, cudaStream_t st) {
  GCRL_REQUIRE(nact >= 1 && nact <= 4, "act_dim must be 1..4");
  const int blocks = std::max(1, std::min((M + 7) / 8, sm_count() * 8));
  const int staged = size_t(N) * 16 <= 48 * 1024 ? 1 : 0;
  action_grad_kernel<<<blocks, 256, staged ? size_t(N) * 16 : 0, st>>>(dZ1, lddz, W1, ldw, sa, ldsa, col0, dz_out, M,
                                                                        N, nact, staged);
  GCRL_LAUNCHED();
}

// ---- batch ingest: all packed operand rows in one launch ---------------------------------------
__global__ void __launch_bounds__(256)
ingest_batch_kernel(const float *__restrict__ s, const float *__restrict__ a, const float *__restrict__ r,
                    const float *__restrict__ ns, const float *__restrict__ d, int D, int A, int M,
                    float *__restrict__ sa, float *__restrict__ nsa, float *__restrict__ spi, int ldc,
                    float *__restrict__ r_out, float *__restrict__ d_out, FastDiv dl) {
  const int total = M * ldc;
  for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < total; e += gridDim.x * blockDim.x) {
    const int m = int(dl.div(uint32_t(e)));
    const int c = e - m * ldc;
    float vs = 0.f, vsa = 0.f, vns = 0.f;
    if (c < D) {
      vs = s[size_t(m) * D + c];
      vsa = vs;
      vns = ns[size_t(m) * D + c];
    } else if (c < D + A) {
      vsa = a[size_t(m) * A + (c - D)];
    }
    sa[e] = vsa;
    nsa[e] = vns;
    spi[e] = vs;
    if (c == 0) {
      r_out[m] = r[m];
      d_out[m] = d[m];
    }
  }
}

void launch_ingest_batch(const float *s, const float *a, const float *r, const float *ns, const float *d,
                         int D, int A, int M, float *sa, float *nsa, float *spi, int ldc, float *r_out,
                         float *d_out, cudaStream_t st) {
  const int total = M * ldc;
  if (total == 0) return;
  const int blocks = std::min((total + 255) / 256, sm_count() * 8);
  ingest_batch_kernel<<<blocks, 256, 0, st>>>(s, a, r, ns, d, D, A, M, sa, nsa, spi, ldc, r_out, d_out,
                                             FastDiv(uint32_t(ldc)));
  GCRL_LAUNCHED();
}

__global__ void __launch_bounds__(256)
td3_smooth_kernel(float *__restrict__ x, int ldx, int col0, const float *__restrict__ noise, int A, int M,
                  float sigma, float clampv) {
  const int total = M * A;
  for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < total; e += gridDim.x * blockDim.x) {
    const int m = e / A, j = e - m * A;
    float n = noise[e] * sigma;
    n = fminf(fmaxf(n, -clampv), clampv);
    float *p = x + size_t(m) * ldx + col0 + j;
    *p = fminf(fmaxf(*p + n, -1.0f), 1.0f);
  }
}

void launch_td3_smooth(float *x, int ldx, int col0, const float *noise, int A, int M, float sigma,
                       float clampv, cudaStream_t st) {
  const int total = M * A;
  if (total == 0) return;
  td3_smooth_kernel<<<std::min((total + 255) / 256, sm_count() * 8), 256, 0, st>>>(x, ldx, col0, noise, A,
                                                                                  M, sigma, clampv);
  GCRL_LAUNCHED();
}

// ---- [s | a | 0] row packing ------------------------------------------------------------------
__global__ void __launch_bounds__(256)
pack_rows_kernel(const float *__restrict__ s, int D, const float *__restrict__ a, int A, float *__restrict__ out,
                 int ldo, int64_t total, FastDiv dl) {
  for (int64_t e = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; e < total;
       e += int64_t(gridDim.x) * blockDim.x) {
    const int64_t m = (total < (int64_t(1) << 31)) ? int64_t(dl.div(uint32_t(e))) : e / ldo;
    const int c = int(e - m * ldo);
    float v = 0.f;
    if (c < D) v = s[m * D + c];
    else if (a != nullptr && c < D + A) v = a[m * A + (c - D)];
    out[e] = v;
  }
}

void launch_pack_rows(const float *s, int D, const float *a, int A, float *out, int ldo, int M,
                      cudaStream_t st) {
  const int64_t total = int64_t(M) * ldo;
  if (total == 0) return;
  const int blocks = int(std::min<int64_t>((total + 255) / 256, int64_t(sm_count()) * 8));
  pack_rows_kernel<<<blocks, 256, 0, st>>>(s, D, a, A, out, ldo, total, FastDiv(uint32_t(ldo)));
  GCRL_LAUNCHED();
}

}  // namespace gcrl
