// Row-slab fused DDPG update kernels (small / medium batch regime).
//
// Every network pass of the update is independent per batch row; only the weight gradients
// reduce over rows.  So one CTA takes a slab of R batch rows and carries it through ALL layers:
//   critic phase (reference src/agent.py:1302-1329):
//     a' = target_actor(s')  ->  q' = target_critic(s', a')  ->  y = clamp(r + gamma (1-d) q')
//     q = critic(s, a)       ->  dL/dq = 2 (q - y) / B       ->  backward through the critic
//   actor phase (src/agent.py:1288-1294):
//     a = actor(s) -> q = critic(s, a) (stepped critic) -> d(-mean q)/da -> backward through the actor
// with activations in shared memory ([feature][row] layout, so a thread's R row values are one
// 16/32-byte broadcast load) and weights streamed from L2 with coalesced 16-byte loads.  The
// forward uses a transposed copy Wt[in][out] of every weight (maintained by the Adam / Polyak
// kernels), the input-gradient pass uses W[out][in] as stored: in both the reduction index is the
// row index of the matrix, so one routine serves both.  Warps split the reduction range
// (K-split) and combine in shared memory in a fixed order -> deterministic.
// The kernels leave the per-layer activations and pre-activation gradients in global memory; the
// weight-gradient GEMMs of all layers then run as ONE multi-problem launch (mlp.cu).
// Launches per update: 57 -> 9.
#include <cooperative_groups.h>

#include <algorithm>
#include <cstdlib>

#include "mlp.cuh"

namespace gcrl {

constexpr int kFusedThreads = 512;
constexpr int kFusedWarps = kFusedThreads / 32;

enum : int { EPI_BIAS_LEAKY = 0, EPI_DLEAKY = 1 };

template <int R>
struct RowVec {
  float v[R];
};

template <int R>
__device__ __forceinline__ void load_rows(const float *p, float (&x)[R]) {
  if constexpr (R == 2) {
    const float2 t = *reinterpret_cast<const float2 *>(p);
    x[0] = t.x; x[1] = t.y;
  } else {
    const float4 *q = reinterpret_cast<const float4 *>(p);
#pragma unroll
    for (int i = 0; i < R / 4; ++i) {
      const float4 t = q[i];
      x[4 * i] = t.x; x[4 * i + 1] = t.y; x[4 * i + 2] = t.z; x[4 * i + 3] = t.w;
    }
  }
}

// yT[j][r] = epi( sum_i xT[i][r] * M[i * ldm + j] ),  i in [0, K), j in [0, N)
//   EPI_BIAS_LEAKY: leaky(acc + bias[j])          (forward layer; M = Wt)
//   EPI_DLEAKY    : acc * leaky'(refT[j][r])      (input gradient;  M = W)
// xT, refT, yT: shared memory [feature][R]; red: shared scratch of 2048 * R floats.
// NC / KC > 0 fix N / K at compile time (the arguments are then ignored): the column split, the K-split and the trip
// counts become constants.  The sums are the same either way.
// All threads of the CTA must call; ends with a __syncthreads().
template <int R, int EPI, int NC = 0, int KC = 0>
__device__ __forceinline__ void slab_matmul(const float *xT, int K_, const float *__restrict__ M, int ldm, int N_,
                                            const float *__restrict__ bias, const float *refT, float *yT,
                                            float *red) {
  const int K = KC > 0 ? KC : K_, N = NC > 0 ? NC : N_;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int ngroups = (N + 3) >> 2;              // 4 adjacent output columns per thread
  const int ncw = (ngroups + 31) >> 5;           // warps needed to cover the columns
  const int ks_total = kFusedWarps / ncw;        // K-split factor
  const int Np = ncw * 128;
  const int cw = warp % ncw, ks = warp / ncw;
  const int j0 = (cw * 32 + lane) * 4;
  // bias of this thread's first epilogue element, loaded now so that its L2 round trip overlaps the K loop instead
  // of following the barrier (at H = 256, R = 2 that is the thread's only element)
  float bias0 = 0.f;
  if (EPI == EPI_BIAS_LEAKY && int(threadIdx.x) < N * R) bias0 = __ldg(bias + threadIdx.x / R);
  if (ks < ks_total) {
    const int kc = (K + ks_total - 1) / ks_total;
    // every K-split range is full when K divides evenly (a compile-time fact at KC > 0)
    constexpr int kst = NC > 0 ? kFusedWarps / (((NC + 3) / 4 + 31) / 32) : 1;
    const bool full = KC > 0 && NC > 0 && KC % kst == 0;
    const int kbeg = ks * kc, kend = full ? kbeg + kc : min(K, kbeg + kc);
    float acc[4][R];
#pragma unroll
    for (int c = 0; c < 4; ++c)
#pragma unroll
      for (int r = 0; r < R; ++r) acc[c][r] = 0.f;
    if (j0 < N) {
      const float *mp = M + size_t(kbeg) * ldm + j0;
#pragma unroll 8
      for (int i = kbeg; i < kend; ++i, mp += ldm) {
        const float4 w = __ldg(reinterpret_cast<const float4 *>(mp));
        float x[R];
        load_rows<R>(xT + i * R, x);
#pragma unroll
        for (int r = 0; r < R; ++r) {
          acc[0][r] = fmaf(w.x, x[r], acc[0][r]);
          acc[1][r] = fmaf(w.y, x[r], acc[1][r]);
          acc[2][r] = fmaf(w.z, x[r], acc[2][r]);
          acc[3][r] = fmaf(w.w, x[r], acc[3][r]);
        }
      }
    }
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      if constexpr (R == 2) {
        *reinterpret_cast<float2 *>(red + (size_t(ks) * Np + j0 + c) * R) = make_float2(acc[c][0], acc[c][1]);
      } else {
        float4 *dst = reinterpret_cast<float4 *>(red + (size_t(ks) * Np + j0 + c) * R);
#pragma unroll
        for (int q = 0; q < R / 4; ++q)
          dst[q] = make_float4(acc[c][4 * q], acc[c][4 * q + 1], acc[c][4 * q + 2], acc[c][4 * q + 3]);
      }
    }
  }
  __syncthreads();
  for (int e = threadIdx.x; e < N * R; e += kFusedThreads) {
    const int j = e / R, r = e - j * R;
    float s = red[size_t(j) * R + r];
    for (int k2 = 1; k2 < ks_total; ++k2) s += red[(size_t(k2) * Np + j) * R + r];
    if (EPI == EPI_BIAS_LEAKY) {
      s += e == int(threadIdx.x) ? bias0 : bias[j];
      s = s > 0.f ? s : s * kLeakySlope;
    } else {
      s = refT[e] > 0.f ? s : s * kLeakySlope;
    }
    yT[e] = s;
  }
  __syncthreads();
}

// out[j][r] = f( sum_k hT[k][r] * Wh[j * ldw + k] + bh[j] ), j < nout <= 4: one warp per (j, r)
template <int R, int KC = 0>
__device__ __forceinline__ void slab_head(const float *hT, int K_, const float *__restrict__ Wh, int ldw,
                                          const float *__restrict__ bh, int nout, bool tanh_out, float *out) {
  const int K = KC > 0 ? KC : K_;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int p = warp; p < nout * R; p += kFusedWarps) {
    const int j = p / R, r = p - j * R;
    const float bj = __ldg(bh + j);              // issued with the weight loads, not after the shuffle tree
    float acc = 0.f;
#pragma unroll 8
    for (int k = lane; k < K; k += 32) acc = fmaf(hT[k * R + r], __ldg(Wh + size_t(j) * ldw + k), acc);
#pragma unroll
    for (int s = 16; s >= 1; s >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, s);
    if (lane == 0) {
      float v = acc + bj;
      out[p] = tanh_out ? tanhf(v) : v;
    }
  }
  __syncthreads();
}

// smem [feature][R] -> global [row0 + r][ld] (rows >= B skipped)
template <int R, int NC = 0>
__device__ __forceinline__ void store_rows(const float *yT, int N_, float *__restrict__ out, int ld, int row0,
                                           int B) {
  const int N = NC > 0 ? NC : N_;
  for (int e = threadIdx.x; e < N * R; e += kFusedThreads) {
    const int r = e / N, j = e - r * N;
    if (row0 + r < B) out[size_t(row0 + r) * ld + j] = yT[j * R + r];
  }
}

// Pull a network's parameters into L2 before the layer chain starts.  After an L2 flush (or any other traffic
// that evicted them) every layer step would otherwise begin with a DRAM round trip that all CTAs wait on, since
// they walk the weights in the same order; one 128-byte line per thread, spread over the grid.
__device__ __forceinline__ void prefetch_l2(const float *p, int n, int gtid, int gthreads) {
  for (int e = gtid * 32; e < n; e += gthreads * 32) asm volatile("prefetch.global.L2 [%0];" ::"l"(p + e));
}
__device__ __forceinline__ void prefetch_net(const FusedNet &n, bool forward, bool backward, int gtid, int gthreads) {
  prefetch_l2(n.flat, n.nflat, gtid, gthreads);              // biases, head, W[out][in] (input gradient)
  if (forward) prefetch_l2(n.flatT, n.nflatT, gtid, gthreads);
  (void)backward;
}

struct SmemPlan {
  float *xa, *xb, *t0, *t1, *keep1, *keep2, *red, *small;   // keep1 / keep2: L layers of H * R each
};

template <int R>
__device__ __forceinline__ SmemPlan carve(float *base, int KinP, int H, int L, bool two_keeps) {
  SmemPlan p;
  p.xa = base; base += KinP * R;
  p.xb = base; base += KinP * R;
  p.t0 = base; base += H * R;
  p.t1 = base; base += H * R;
  p.keep1 = base; base += L * H * R;
  p.keep2 = two_keeps ? base : nullptr; if (two_keeps) base += L * H * R;
  p.red = base; base += 2048 * R;
  p.small = base;
  return p;
}

size_t fused_smem_bytes(int R, int D, int A, int H, int L, bool two_keeps) {
  const int KinP = (D + A + 3) & ~3;
  size_t f = size_t(2) * KinP * R + size_t(2) * H * R + size_t(L) * H * R * (two_keeps ? 2 : 1) +
             size_t(2048) * R + 24 * R;
  return f * sizeof(float);
}

// ---------------------------------------------------------------------------------------------
// step table
// ---------------------------------------------------------------------------------------------
// Each kernel is a chain of layer steps.  Written out as calls, every step would be its own inlined copy of the
// layer routine, and after an L2 flush each copy's instructions come from DRAM the one time the chain reaches them.
// So the chain is a table, built at kernel start (one entry per thread), and one loop runs it through a single
// copy of each body: the narrow first layer (K = D or D + A), the H-wide hidden layer, the H-wide input-gradient
// layer and the head.  The elementwise work between the steps runs after the step that flags it (`post`).
enum : int { STEP_FIRST = 0, STEP_HIDDEN = 1, STEP_DGRAD = 2, STEP_HEAD = 3 };
enum : int {
  POST_ANEXT = 1,    // critic phase: a' (+ TD3 smoothing noise) into x_ns
  POST_QMIN = 2,     // critic phase, TD3: q' = min of the two target critics
  POST_LOSS = 4,     // critic phase: Bellman target, loss, dL/dq, seed of the critic's backward pass
  POST_ACT = 8,      // actor phase: a into x_sa
  POST_QSEED = 16,   // actor phase: metrics, seed of the critic's backward pass
  POST_DQDA = 32,    // actor phase: dq/da through the critic's first layer, backward through the actor head
};
constexpr int kMaxSteps = 4 * (kFusedMaxL + 1) + kFusedMaxL - 1;   // critic phase with two target critics

struct SlabStep {
  const float *M, *bias, *x, *ref;   // HEAD: M = Wh, bias = bh
  float *y, *gout;                   // gout: global [B][ldh] copy of y, or nullptr
  int K, ldm, kind, post, nout, tanh_out;
};

template <int R, int HC>
__device__ __forceinline__ void run_step(const SlabStep &st, int H, float *red, int ldh, int row0, int B) {
  if (st.kind == STEP_HEAD) {
    slab_head<R, HC>(st.x, H, st.M, st.ldm, st.bias, st.nout, st.tanh_out != 0, st.y);
    return;
  }
  if (st.kind == STEP_DGRAD)
    slab_matmul<R, EPI_DLEAKY, HC, HC>(st.x, H, st.M, st.ldm, H, nullptr, st.ref, st.y, red);
  else if (HC > 0 && st.kind == STEP_HIDDEN)
    slab_matmul<R, EPI_BIAS_LEAKY, HC, HC>(st.x, H, st.M, st.ldm, H, st.bias, nullptr, st.y, red);
  else
    slab_matmul<R, EPI_BIAS_LEAKY, HC, 0>(st.x, st.K, st.M, st.ldm, H, st.bias, nullptr, st.y, red);
  if (st.gout != nullptr) store_rows<R, HC>(st.y, H, st.gout, ldh, row0, B);
}

// layer l (l == L: the head) of a network's forward pass; activations in `keep` (all layers kept) or ping-pong
// between t0 / t1
__device__ __forceinline__ SlabStep forward_step(const FusedNet &n, int l, int L, int H, int R, const float *in,
                                                 int K0, float *keep, float *t0, float *t1, float *gout) {
  SlabStep st;
  const int l1 = l - 1;
  const float *prev = keep ? keep + l1 * H * R : ((l1 & 1) ? t1 : t0);
  st.x = l == 0 ? in : prev;
  st.ref = nullptr;
  st.post = 0; st.nout = 0; st.tanh_out = 0;
  if (l < L) {
    st.kind = l == 0 ? STEP_FIRST : STEP_HIDDEN;
    st.M = n.Wt[l]; st.ldm = n.ldt[l]; st.bias = n.b[l];
    st.K = l == 0 ? K0 : H;
    st.y = keep ? keep + l * H * R : ((l & 1) ? t1 : t0);
    st.gout = gout;
  } else {
    st.kind = STEP_HEAD;
    st.M = n.Wh; st.ldm = n.ldwh; st.bias = n.bh;
    st.K = H;
    st.y = nullptr;
    st.gout = nullptr;
  }
  return st;
}

// input-gradient step through hidden layer l >= 1 of a network: x -> y, leaky' of the kept activation of layer l - 1
__device__ __forceinline__ SlabStep dgrad_step(const FusedNet &n, int l, int H, int R, const float *x, float *y,
                                               const float *keep, float *gout) {
  SlabStep st;
  st.kind = STEP_DGRAD;
  st.M = n.W[l]; st.ldm = n.ldw[l]; st.bias = nullptr;
  st.x = x; st.y = y; st.ref = keep + (l - 1) * H * R; st.gout = gout;
  st.K = H; st.post = 0; st.nout = 0; st.tanh_out = 0;
  return st;
}

// ---------------------------------------------------------------------------------------------
// critic phase
// ---------------------------------------------------------------------------------------------
// TD3 = false compiles the smoothing noise / second target critic / given-target / smooth-L1 branches out.
// SPLIT: the slab is carried by a 2-CTA cluster.  The target path (a' = pi_t(s'), q' = Q_t(s', a'): 2L + 2 layer
// steps) and the critic forward (L + 1 steps) do not depend on each other, so CTA 0 runs the former while CTA 1
// runs the latter; CTA 0 drops q' into CTA 1's shared memory (DSMEM), one cluster barrier, and CTA 1 goes on
// with the loss and the backward pass.  Critical path 3L + 3 -> 2L + 2 + (L - 1) layer steps; used when both
// CTAs of every slab fit in one wave (by default only at R = 8, see fused_rows_per_cta).
// HC > 0: H == HC, a compile-time constant of the H-wide steps (HC = 0: any H).
template <int R, bool TD3, bool SPLIT, int HC>
__device__ __forceinline__ void critic_phase(const FusedCriticArgs &a) {
  extern __shared__ float4 fsm4[];
  __shared__ SlabStep steps[kMaxSteps];
  const int D = a.D, A = a.A, H = HC > 0 ? HC : a.H, L = a.L, B = a.B;
  const int KinP = (D + A + 3) & ~3;
  SmemPlan sp = carve<R>(reinterpret_cast<float *>(fsm4), KinP, H, L, false);
  pdl_wait();
  pdl_launch_dependents();
  {
    const int gtid = blockIdx.x * kFusedThreads + threadIdx.x, gth = gridDim.x * kFusedThreads;
    if (!TD3 || a.y_in == nullptr) {
      prefetch_net(a.ta, true, false, gtid, gth);
      prefetch_net(a.tc, true, false, gtid, gth);
      if (TD3 && a.has_tc2) prefetch_net(a.tc2, true, false, gtid, gth);
    }
    prefetch_net(a.c, true, true, gtid, gth);
  }
  float *x_ns = sp.xa, *x_sa = sp.xb;
  float *qn = sp.small, *q = qn + R, *yv = q + R, *dzh = yv + R, *rr = dzh + R, *dd = rr + R;
  float *anext = dd + R;                          // [A][R], A <= 4
  const int slab = SPLIT ? int(blockIdx.x >> 1) : int(blockIdx.x);
  const int role = SPLIT ? int(blockIdx.x & 1) : 2;      // 0: target path, 1: critic path, 2: both
  const int row0 = slab * R, tid = threadIdx.x;

  // ---- the step table: target nets (a' = pi_t(s'), q' = Q_t(s', a') [, Q_t2]), critic forward, critic backward
  const int nt = (!TD3 || a.y_in == nullptr) ? ((TD3 && a.has_tc2) ? 3 : 2) : 0;
  const int nsteps = (nt + 1) * (L + 1) + (L - 1);
  if (tid < nsteps) {
    SlabStep st;
    const int n = tid / (L + 1), l = tid - n * (L + 1);
    if (n < nt) {                                   // target actor / target critic(s), activations ping-pong
      const FusedNet &net = n == 0 ? a.ta : (n == 1 ? a.tc : a.tc2);
      st = forward_step(net, l, L, H, R, x_ns, n == 0 ? D : D + A, nullptr, sp.t0, sp.t1, nullptr);
      if (l == L) {
        st.nout = n == 0 ? A : 1;
        st.tanh_out = n == 0;
        st.y = n == 0 ? anext : (n == 1 ? qn : anext);          // Q_t2's q' goes to anext: a' already sits in x_ns
        st.post = n == 0 ? POST_ANEXT : (n == 2 ? POST_QMIN : 0);
      }
    } else if (n == nt) {                           // critic, activations kept for the backward pass
      st = forward_step(a.c, l, L, H, R, x_sa, D + A, sp.keep1, sp.t0, sp.t1, l < L ? a.h_out[l] : nullptr);
      if (l == L) { st.nout = 1; st.y = q; st.post = POST_LOSS; }
    } else {                                        // backward: dz (t0 first) -> pre-activation gradient of layer l-1
      const int b = tid - (nt + 1) * (L + 1), lb = L - 1 - b;
      st = dgrad_step(a.c, lb, H, R, (b & 1) ? sp.t1 : sp.t0, (b & 1) ? sp.t0 : sp.t1, sp.keep1, a.dz_out[lb - 1]);
    }
    steps[tid] = st;
  }

  // ---- 0a. (sample) draw this slab's rows from the HER episode store: 3 dependent gathers (bucket record ->
  //          packed row || future offsets -> future goal), relabel + reward in shared memory ----
  const float *tile = nullptr;
  if (a.sample) {
    const HerGeom &g = a.geom;
    float *tl = sp.red;                              // R packed rows (row_f <= 2048 floats each)
    __shared__ uint32_t s_slot[8];
    const SampleScalars sc = *a.sample_sc;
    const int nrows = min(R, B - row0);
    SampleRef ref{0u, 0u, 0u, 0u};
    if (tid < nrows) {
      ref = her_resolve(g, sc, row0 + tid, sc.use_idx ? a.sample_idx : nullptr, nullptr);
      s_slot[tid] = ref.slot;
    }
    __syncthreads();
    const int rf4 = g.row_f >> 2;
    const float4 *rows4 = reinterpret_cast<const float4 *>(g.rows);
    for (int c = tid; c < nrows * rf4; c += kFusedThreads) {
      const int i = c / rf4, q = c - i * rf4;
      reinterpret_cast<float4 *>(tl)[c] = ldg_stream4(rows4 + size_t(s_slot[i]) * rf4 + q);
    }
    float *gfs = sp.small + 16 * R;                  // behind the per-row scalars: [R][8] future goals (G <= 8)
    if (tid < nrows && ref.j > 0) {
      const float *agf = g.ag + size_t(her_future_slot(g, ref)) * g.gpad;
      for (int c = 0; c < g.G; ++c) gfs[tid * 8 + c] = __ldg(agf + c);
    }
    __syncthreads();
    if (tid < nrows && ref.j > 0) her_relabel_row(g, tl + tid * g.row_f, gfs + tid * 8);
    __syncthreads();
    if (role != 0) {                                 // the dense batch, for the actor phase and the second critic
      for (int e = tid; e < nrows * D; e += kFusedThreads) {
        const int i = e / D, k = e - i * D;
        a.bs[size_t(row0 + i) * D + k] = tl[i * g.row_f + k];
        a.bns[size_t(row0 + i) * D + k] = tl[i * g.row_f + g.off_ns + k];
      }
      for (int e = tid; e < nrows * A; e += kFusedThreads) {
        const int i = e / A, k = e - i * A;
        a.ba[size_t(row0 + i) * A + k] = tl[i * g.row_f + g.off_a + k];
      }
      if (tid < nrows) {
        a.br[row0 + tid] = tl[tid * g.row_f + g.off_r];
        a.bd[row0 + tid] = tl[tid * g.row_f + g.off_d];
      }
    }
    tile = tl;
  }
  // ---- 0. stage the slab's rows: x_ns = [s' | (a')], x_sa = [s | a]; also emit [s | a | 0] rows ----
  for (int e = tid; e < KinP * R; e += kFusedThreads) {
    const int k = e / R, r = e - k * R, row = row0 + r;
    float vns = 0.f, vsa = 0.f;
    if (row < B) {
      if (tile != nullptr) {
        const float *t = tile + r * a.geom.row_f;
        if (k < D) { vns = t[a.geom.off_ns + k]; vsa = t[k]; }
        else if (k < D + A) vsa = t[a.geom.off_a + (k - D)];
      } else {
        if (k < D) { vns = a.ns[size_t(row) * D + k]; vsa = a.s[size_t(row) * D + k]; }
        else if (k < D + A) vsa = a.a[size_t(row) * A + (k - D)];
      }
    }
    x_ns[e] = vns;
    x_sa[e] = vsa;
  }
  if (tid < R) {
    const int row = row0 + tid;
    if (tile != nullptr) {
      rr[tid] = row < B ? tile[tid * a.geom.row_f + a.geom.off_r] : 0.f;
      dd[tid] = row < B ? tile[tid * a.geom.row_f + a.geom.off_d] : 0.f;
    } else {
      rr[tid] = row < B ? a.r[row] : 0.f;
      dd[tid] = row < B ? a.d[row] : 0.f;
    }
  }
  __syncthreads();
  if (a.sa_out != nullptr && role != 0) {
    for (int e = tid; e < a.ldc * R; e += kFusedThreads) {
      const int r = e / a.ldc, k = e - r * a.ldc;
      if (row0 + r < B) a.sa_out[size_t(row0 + r) * a.ldc + k] = k < KinP ? x_sa[k * R + r] : 0.f;
    }
  }
  // head weight of this thread's first element of the dz seed (POST_LOSS), loaded ahead of the layer chain so that
  // the seed starts from a register instead of an L2 round trip (SPLIT: under the wait for q')
  float wh0 = !SPLIT && tid < H * R ? __ldg(a.c.Wh + tid / R) : 0.f;

  const int s_begin = role == 1 ? nt * (L + 1) : 0, s_end = role == 0 ? nt * (L + 1) : nsteps;
  for (int s = s_begin; s < s_end; ++s) {
    const SlabStep st = steps[s];
    run_step<R, HC>(st, H, sp.red, a.ldh, row0, B);
    if (st.post == POST_ANEXT) {
      // ---- a' = target_actor(s') (:1312); TD3: + clamp(noise * sigma, +-c), clamped to [-1, 1] (:174-179) ----
      for (int e = tid; e < A * R; e += kFusedThreads) {
        float v = anext[e];
        if (TD3 && a.noise != nullptr) {
          const int j = e / R, row = row0 + (e - j * R);
          float n = row < B ? a.noise[size_t(row) * A + j] * a.policy_noise : 0.f;
          n = fminf(fmaxf(n, -a.noise_clamp), a.noise_clamp);
          v = fminf(fmaxf(v + n, -1.0f), 1.0f);
        }
        x_ns[D * R + e] = v;
      }
      __syncthreads();
    } else if (TD3 && st.post == POST_QMIN) {
      // ---- TD3: q' = min over the two target critics (:181-183) ----
      if (tid < R) qn[tid] = fminf(qn[tid], anext[tid]);
      __syncthreads();
    } else if (st.post == POST_LOSS) {
      if (SPLIT) {
        wh0 = tid < H * R ? __ldg(a.c.Wh + tid / R) : 0.f;
        cooperative_groups::this_cluster().sync();                // q' has arrived
      }
      // ---- 4. Bellman target, loss, dL/dq (:1316-1326) ----
      if (tid == 0) {
        float ls = 0.f, ts = 0.f, qs = 0.f;
        const float invB = 1.0f / float(B);
        for (int r = 0; r < R; ++r) {
          const int row = row0 + r;
          float g = 0.f;
          if (row < B) {
            float y;
            if (TD3 && a.y_in != nullptr) {
              y = a.y_in[row];
            } else {
              y = rr[r] + a.gamma * (1.0f - dd[r]) * qn[r];
              if (a.clamp_y) y = fminf(fmaxf(y, a.y_lo), 0.0f);
            }
            const float diff = q[r] - y;
            const float w = a.is_w != nullptr ? a.is_w[row] : 1.0f;     // (weights * loss).mean(), :1322-1324
            if (!TD3 || a.loss_kind == 0) {               // mse_loss
              ls += w * (diff * diff);
              g = 2.0f * diff * invB * w;
            } else {                                      // smooth_l1_loss, beta = 1 (TD3, :189-197)
              const float ad = fabsf(diff);
              ls += w * (ad < 1.0f ? 0.5f * diff * diff : ad - 0.5f);
              g = (ad < 1.0f ? diff : (diff > 0.f ? 1.0f : -1.0f)) * invB * w;
            }
            float td;
            if (TD3 && a.q_other != nullptr) {            // TD3 critic 2: max of both TD errors, mean of both Q
              const float qo = a.q_other[row];
              td = fmaxf(fabsf(q[r] - y), fabsf(qo - y));
              qs += 0.5f * (q[r] + qo);
            } else {
              td = fabsf(y - q[r]);
              qs += q[r];
            }
            ts += td;
            if (a.td_out != nullptr) a.td_out[row] = td;
            a.dzh_out[row] = g;
            if (a.y_out && (!TD3 || a.y_in == nullptr)) a.y_out[row] = y;
            if (a.q_out) a.q_out[row] = q[r];
          }
          dzh[r] = g;
        }
        float *mp = a.metric_partials + size_t(slab) * 4;
        mp[0] = ls; mp[1] = ts; mp[2] = qs; mp[3] = 0.f;
      }
      __syncthreads();
      // ---- 5. backward through the critic (the DGRAD steps that follow): seed with the head's gradient ----
      float *dz = sp.t0;
      const float *keep_last = sp.keep1 + (L - 1) * H * R;
      for (int e = tid; e < H * R; e += kFusedThreads) {
        const int k = e / R, r = e - k * R;
        const float g = dzh[r] * (e == tid ? wh0 : __ldg(a.c.Wh + k));
        dz[e] = keep_last[e] > 0.f ? g : g * kLeakySlope;
      }
      __syncthreads();
      store_rows<R, HC>(dz, H, a.dz_out[L - 1], a.ldh, row0, B);
    }
  }
  if (SPLIT && role == 0) {              // hand q' to the critic CTA and leave
    namespace cg = cooperative_groups;
    cg::cluster_group cluster = cg::this_cluster();
    float *peer_qn = cluster.map_shared_rank(qn, 1);
    if (tid < R) peer_qn[tid] = qn[tid];
    cluster.sync();
  }
}

// ---------------------------------------------------------------------------------------------
// actor phase
// ---------------------------------------------------------------------------------------------
template <int R, int HC>
__device__ __forceinline__ void actor_phase(const FusedActorArgs &a) {
  extern __shared__ float4 fsm4[];
  __shared__ SlabStep steps[4 * kFusedMaxL];
  const int D = a.D, A = a.A, H = HC > 0 ? HC : a.H, L = a.L, B = a.B;
  const int KinP = (D + A + 3) & ~3;
  SmemPlan sp = carve<R>(reinterpret_cast<float *>(fsm4), KinP, H, L, true);
  pdl_wait();
  pdl_launch_dependents();
  {
    const int gtid = blockIdx.x * kFusedThreads + threadIdx.x, gth = gridDim.x * kFusedThreads;
    prefetch_net(a.actor, true, true, gtid, gth);
    prefetch_net(a.c, true, true, gtid, gth);
  }
  float *x_sa = sp.xa;
  float *q = sp.small, *act = q + R, *da = act + 4 * R;   // act, da: [A][R]
  const int row0 = blockIdx.x * R, tid = threadIdx.x;
  // the critic's backward pass starts from t0 and leaves d(-mean q)/dz of its first layer in pc; the actor head's
  // backward writes pa, and the actor's backward pass goes on from there
  float *pc = ((L - 1) & 1) ? sp.t1 : sp.t0, *pa = ((L - 1) & 1) ? sp.t0 : sp.t1;

  // ---- the step table: actor forward, critic forward (stepped critic), critic backward, actor backward
  if (tid < 4 * L) {
    SlabStep st;
    if (tid < 2 * (L + 1)) {
      const int n = tid / (L + 1), l = tid - n * (L + 1);
      if (n == 0) {           // a = actor(s) (:1289); hidden activations kept (smem) and emitted (global, for wgrad)
        st = forward_step(a.actor, l, L, H, R, x_sa, D, sp.keep1, sp.t0, sp.t1, l < L ? a.h_out[l] : nullptr);
        if (l == L) { st.nout = A; st.tanh_out = 1; st.y = act; st.post = POST_ACT; }
      } else {                // q = critic([s, a]) with the stepped critic (:1290)
        st = forward_step(a.c, l, L, H, R, x_sa, D + A, sp.keep2, sp.t0, sp.t1, nullptr);
        if (l == L) { st.nout = 1; st.y = q; st.post = POST_QSEED | (L == 1 ? POST_DQDA : 0); }
      }
    } else if (tid < 2 * (L + 1) + (L - 1)) {      // d(-mean q) / d(critic hidden), down to the critic's first layer
      const int b = tid - 2 * (L + 1), l = L - 1 - b;
      st = dgrad_step(a.c, l, H, R, (b & 1) ? sp.t1 : sp.t0, (b & 1) ? sp.t0 : sp.t1, sp.keep2, nullptr);
      if (b == L - 2) st.post = POST_DQDA;
    } else {                                        // backward through the actor's hidden stack
      const int b = tid - 2 * (L + 1) - (L - 1), l = L - 1 - b;
      st = dgrad_step(a.actor, l, H, R, (b & 1) ? pc : pa, (b & 1) ? pa : pc, sp.keep1, a.dz_out[l - 1]);
    }
    steps[tid] = st;
  }

  for (int e = tid; e < KinP * R; e += kFusedThreads) {
    const int k = e / R, r = e - k * R, row = row0 + r;
    x_sa[e] = (row < B && k < D) ? a.s[size_t(row) * D + k] : 0.f;
  }
  // head weights of this thread's first element of the two backward elementwise steps below, loaded ahead so that
  // those steps start from registers instead of L2 round trips
  const float wh0 = tid < H * R ? __ldg(a.c.Wh + tid / R) : 0.f;
  float awh0[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
  for (int j = 0; j < 4; ++j)
    if (tid < H * R && j < A) awh0[j] = __ldg(a.actor.Wh + size_t(j) * a.actor.ldwh + tid / R);
  __syncthreads();

  for (int s = 0; s < 4 * L; ++s) {
    const SlabStep st = steps[s];
    run_step<R, HC>(st, H, sp.red, a.ldh, row0, B);
    if (st.post & POST_ACT) {
      for (int e = tid; e < A * R; e += kFusedThreads) x_sa[D * R + e] = act[e];
      __syncthreads();
    }
    if (st.post & POST_QSEED) {
      if (tid == 0) {
        float qs = 0.f;
        for (int r = 0; r < R; ++r)
          if (row0 + r < B) qs += q[r];
        float *mp = a.metric_partials + size_t(blockIdx.x) * 4;
        mp[0] = -qs; mp[1] = 0.f; mp[2] = qs; mp[3] = 0.f;     // actor loss = -mean(q) (:1291)
      }
      // ---- d(-mean q) / d(critic hidden): seed of the critic's backward pass ----
      const float invB = 1.0f / float(B);
      const float *keep_last = sp.keep2 + (L - 1) * H * R;
      for (int e = tid; e < H * R; e += kFusedThreads) {
        const int k = e / R, r = e - k * R;
        const float g = (row0 + r < B) ? -invB * (e == tid ? wh0 : __ldg(a.c.Wh + k)) : 0.f;
        sp.t0[e] = keep_last[e] > 0.f ? g : g * kLeakySlope;
      }
      __syncthreads();
    }
    if (st.post & POST_DQDA) {
      // ---- dq/da through the critic's first layer (action columns), times tanh' ----
      const int warp = tid >> 5, lane = tid & 31;
      for (int p = warp; p < A * R; p += kFusedWarps) {
        const int j = p / R, r = p - j * R;
        float acc = 0.f;
#pragma unroll 8
        for (int n = lane; n < H; n += 32) acc = fmaf(pc[n * R + r], __ldg(a.c.W[0] + size_t(n) * a.c.ldw[0] + D + j), acc);
#pragma unroll
        for (int s2 = 16; s2 >= 1; s2 >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, s2);
        if (lane == 0) {
          const float t = act[p];
          const float v = acc * (1.0f - t * t);
          da[p] = v;
          if (row0 + r < B) a.da_out[size_t(row0 + r) * 4 + j] = v;
        }
      }
      for (int p = tid; p < R; p += kFusedThreads)               // zero the unused head columns
        for (int j = A; j < 4; ++j)
          if (row0 + p < B) a.da_out[size_t(row0 + p) * 4 + j] = 0.f;
      __syncthreads();
      // ---- backward through the actor head; the actor's DGRAD steps follow ----
      const float *keep_last = sp.keep1 + (L - 1) * H * R;
      for (int e = tid; e < H * R; e += kFusedThreads) {
        const int k = e / R, r = e - k * R;
        float g = 0.f;
#pragma unroll
        for (int j = 0; j < 4; ++j)
          if (j < A) g = fmaf(da[j * R + r], e == tid ? awh0[j] : __ldg(a.actor.Wh + size_t(j) * a.actor.ldwh + k), g);
        pa[e] = keep_last[e] > 0.f ? g : g * kLeakySlope;
      }
      __syncthreads();
      store_rows<R, HC>(pa, H, a.dz_out[L - 1], a.ldh, row0, B);
    }
  }
}

// The kernels: h256:: for H = 256, anyh:: for every width.  Both keep the names the profiler shows for the
// row-slab kernels (fused_critic_kernel<R, TD3, SPLIT>, fused_actor_kernel<R>).  The arguments are grid constants,
// so the per-layer pointer arrays are read in place with a runtime layer index instead of through a stack copy.
namespace h256 {
template <int R, bool TD3, bool SPLIT>
__global__ void __launch_bounds__(kFusedThreads, 1) fused_critic_kernel(const __grid_constant__ FusedCriticArgs a) {
  critic_phase<R, TD3, SPLIT, 256>(a);
}
template <int R>
__global__ void __launch_bounds__(kFusedThreads, 1) fused_actor_kernel(const __grid_constant__ FusedActorArgs a) {
  actor_phase<R, 256>(a);
}
}  // namespace h256
namespace anyh {
template <int R, bool TD3, bool SPLIT>
__global__ void __launch_bounds__(kFusedThreads, 1) fused_critic_kernel(const __grid_constant__ FusedCriticArgs a) {
  critic_phase<R, TD3, SPLIT, 0>(a);
}
template <int R>
__global__ void __launch_bounds__(kFusedThreads, 1) fused_actor_kernel(const __grid_constant__ FusedActorArgs a) {
  actor_phase<R, 0>(a);
}
}  // namespace anyh

// ---------------------------------------------------------------------------------------------
// launchers
// ---------------------------------------------------------------------------------------------
static int g_fused_smem_set[2][6][3] = {};

template <typename K>
static void ensure_smem(K kernel, size_t bytes, int *flag) {
  if (*flag < int(bytes)) {
    GCRL_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int(bytes)));
    *flag = int(bytes);
  }
}

// Rows per CTA.  The kernels are chains of dependent layer steps whose cost grows with R (16 FMAs per weight
// load at R = 4, 8 at R = 2), so the smallest R whose slabs still fit in ONE wave of CTAs wins: at B = 256,
// R = 2 (128 CTAs) runs the critic phase in 36.9 us and the actor phase in ~37 us, R = 4 (64 CTAs) in 48.9 / 45 us
// (36.9 for the critic phase as 2-CTA clusters, see SPLIT, when forced with GCRL_FUSED_R=4).  The default rule
// splits the critic phase only where both CTAs of every slab fit in one wave, 2 * ceil(B / R) <= SMs: at R = 8 for
// 512 < B <= 4 * SMs (513..592 on 148 SMs); R = 4 starts above 2 * SMs rows, so it never splits.
// GCRL_FUSED_R (experiments) forces R = 2, 4 or 8; any other value is ignored -- there are no other kernels, and
// the grid is sized from R.
int fused_rows_per_cta(int B) {
  if (const char *e = getenv("GCRL_FUSED_R")) {
    const int r = atoi(e);
    if (r == 2 || r == 4 || r == 8) return r;
  }
  if (B <= 2 * sm_count()) return 2;
  return B <= 512 ? 4 : 8;
}

// The kernels are instantiated for H = 256 with the width as a compile-time constant, and for any H.
// GCRL_FUSED_GENERIC=1 (tests) runs the any-H instance at H = 256 too; both give the same bits.
static bool fused_h256(int H) {
  const char *e = getenv("GCRL_FUSED_GENERIC");
  return H == 256 && !(e != nullptr && atoi(e) != 0);
}

// can the critic-phase kernel draw its own rows from this episode store?
bool fused_sample_supported(const HerGeom &g) { return g.G <= 8 && g.row_f <= 2048; }

bool fused_supported(int B, int D, int A, int H, int L) {
  if (B < 1 || B > 1024 || L < 1 || L > kFusedMaxL || A > 4 || H < 4 || H > 2048) return false;
  const int R = fused_rows_per_cta(B);
  if ((B + R - 1) / R > 256) return false;
  return fused_smem_bytes(R, D, A, H, L, true) <= size_t(200) * 1024;
}

template <typename K>
static void launch_critic_kernel(K kernel, int *flag, bool clustered, const FusedCriticArgs &a, int grid, size_t smem,
                                 cudaStream_t st) {
  ensure_smem(kernel, smem, flag);
  if (!clustered) {
    launch_pdl<PDL_FUSED>(kernel, dim3(grid), dim3(kFusedThreads), smem, st, a);
    return;
  }
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(2 * grid);
  cfg.blockDim = dim3(kFusedThreads);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[2];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[1].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = pdl_enabled(PDL_FUSED) ? 2 : 1;
  GCRL_CUDA(cudaLaunchKernelEx(&cfg, kernel, a));
}

template <int R, bool TD3, bool SPLIT>
static auto critic_kernel(bool h) { return h ? h256::fused_critic_kernel<R, TD3, SPLIT> : anyh::fused_critic_kernel<R, TD3, SPLIT>; }
template <int R>
static auto actor_kernel(bool h) { return h ? h256::fused_actor_kernel<R> : anyh::fused_actor_kernel<R>; }

static void launch_critic_variant(const FusedCriticArgs &a, bool h, int R, bool td3, bool split, int grid,
                                  size_t smem, cudaStream_t st) {
  auto &flags = g_fused_smem_set[h];
  auto go = [&](auto kernel, int *flag, bool clustered) { launch_critic_kernel(kernel, flag, clustered, a, grid, smem, st); };
  if (R == 2) {
    if (td3) go(critic_kernel<2, true, false>(h), &flags[2][2], false);
    else go(critic_kernel<2, false, false>(h), &flags[0][2], false);
  } else if (R == 4) {
    if (td3 && split) go(critic_kernel<4, true, true>(h), &flags[5][0], true);
    else if (td3) go(critic_kernel<4, true, false>(h), &flags[2][0], false);
    else if (split) go(critic_kernel<4, false, true>(h), &flags[4][0], true);
    else go(critic_kernel<4, false, false>(h), &flags[0][0], false);
  } else {
    if (td3 && split) go(critic_kernel<8, true, true>(h), &flags[5][1], true);
    else if (td3) go(critic_kernel<8, true, false>(h), &flags[2][1], false);
    else if (split) go(critic_kernel<8, false, true>(h), &flags[4][1], true);
    else go(critic_kernel<8, false, false>(h), &flags[0][1], false);
  }
}

int launch_fused_critic(const FusedCriticArgs &a, cudaStream_t st) {
  const int R = fused_rows_per_cta(a.B);
  const int grid = (a.B + R - 1) / R;
  const size_t smem = fused_smem_bytes(R, a.D, a.A, a.H, a.L, false);
  const bool td3 = a.has_tc2 || a.noise != nullptr || a.y_in != nullptr || a.loss_kind != 0 || a.q_other != nullptr;
  // two CTAs per slab (target path | critic path) when there is a target path and everything fits in one wave
  const bool split = R != 2 && a.y_in == nullptr && 2 * grid <= sm_count();
  launch_critic_variant(a, fused_h256(a.H), R, td3, split, grid, smem, st);
  GCRL_LAUNCHED();
  return grid;
}

static void launch_actor_variant(const FusedActorArgs &a, bool h, int R, int grid, size_t smem, cudaStream_t st) {
  auto &flags = g_fused_smem_set[h][1];
  if (R == 2) {
    ensure_smem(actor_kernel<2>(h), smem, &flags[2]);
    launch_pdl<PDL_FUSED>(actor_kernel<2>(h), dim3(grid), dim3(kFusedThreads), smem, st, a);
  } else if (R == 4) {
    ensure_smem(actor_kernel<4>(h), smem, &flags[0]);
    launch_pdl<PDL_FUSED>(actor_kernel<4>(h), dim3(grid), dim3(kFusedThreads), smem, st, a);
  } else {
    ensure_smem(actor_kernel<8>(h), smem, &flags[1]);
    launch_pdl<PDL_FUSED>(actor_kernel<8>(h), dim3(grid), dim3(kFusedThreads), smem, st, a);
  }
}

int launch_fused_actor(const FusedActorArgs &a, cudaStream_t st) {
  const int R = fused_rows_per_cta(a.B);
  const int grid = (a.B + R - 1) / R;
  const size_t smem = fused_smem_bytes(R, a.D, a.A, a.H, a.L, true);
  launch_actor_variant(a, fused_h256(a.H), R, grid, smem, st);
  GCRL_LAUNCHED();
  return grid;
}

}  // namespace gcrl
