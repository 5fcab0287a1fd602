// SAC and "TQC" learners: stochastic BatchNorm actor + truncated critic ensemble.
//
// Replaces (reference src/agent.py) SACAgent.critic_update :548-639, actor_update :513-530,
// alpha_update :532-546, update_critic :487-498, update :659-699 and TQCAgent.critic_update
// :951-1042, actor_update :912-934, alpha_update :936-949, update_critics :888-896, update
// :1062-1100; and SACActorModel.forward / sample (src/model.py:118-141).
//
// One implementation serves both: n critics, the Bellman target and the actor loss use the mean
// of the (n - drop) smallest critic outputs per sample (SAC: n = 2, drop = 1 == torch.min).
// Dense layers run on the fp32 GEMM kernels of mlp.cu; this file adds the BatchNorm1d
// forward / backward (column reductions over the batch), the tanh-Gaussian policy head with
// its log-probability and analytic backward, the sort-truncate-mean over the critic axis (an
// insertion sort in registers), the scalar AdamW on log_alpha and the orchestration.
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <map>
#include <tuple>
#include <vector>

#include "buffer_api.cuh"
#include "graphs.cuh"
#include "mlp.cuh"
#include "params.cuh"

using namespace gcrl;

namespace {

constexpr int kMaxCritics = 8;
constexpr int kSplits = 128;
constexpr int kEnsembleBatchMax = 4096;   // up to this batch the ensemble's backward passes share their launches
constexpr float kBnEps = 1e-5f;        // nn.BatchNorm1d default
constexpr float kBnMomentum = 0.1f;
constexpr float kLogSqrt2Pi = 0.91893853320467274178f;
constexpr int kMetricFloats = 36;         // the device metrics block [32], then the alpha state [4]
// per-update scalars of an n-update call: critic / actor AdamW, alpha's AdamW, the sampler's totals and draw epoch
constexpr size_t kManyScalBytes = 2 * sizeof(StepScalars) + sizeof(SampleScalars);

// ---- BatchNorm1d -----------------------------------------------------------------------------
// One CTA per 32 feature columns, 32 x 32 threads: threadIdx.x = column (coalesced 128-byte row
// segments), threadIdx.y strides the batch rows; fixed-order reduction over threadIdx.y.
__device__ __forceinline__ float col_reduce(float v, float (*red)[33]) {
  red[threadIdx.y][threadIdx.x] = v;
  __syncthreads();
  if (threadIdx.y == 0) {
    float t = 0.f;
#pragma unroll
    for (int i = 0; i < 32; ++i) t += red[i][threadIdx.x];
    red[32][threadIdx.x] = t;
  }
  __syncthreads();
  const float r = red[32][threadIdx.x];
  __syncthreads();
  return r;
}

// z [B][ld] (pre-BN Linear output) is overwritten by xhat; h = relu(xhat * gamma + beta).
__global__ void __launch_bounds__(1024)
bn_fwd_kernel(float *__restrict__ z, int ld, int B, int H, const float *__restrict__ gamma,
              const float *__restrict__ beta, float *__restrict__ rmean, float *__restrict__ rvar,
              float *__restrict__ invstd_out, float *__restrict__ h, int train) {
  __shared__ float red[33][33];
  const int c = blockIdx.x * 32 + threadIdx.x;
  const bool ok = c < H;
  float mu = 0.f, var = 1.f;
  if (train) {
    float s = 0.f;
    if (ok)
      for (int m = threadIdx.y; m < B; m += 32) s += z[size_t(m) * ld + c];
    mu = col_reduce(s, red) / float(B);
    s = 0.f;
    if (ok)
      for (int m = threadIdx.y; m < B; m += 32) {
        const float d = z[size_t(m) * ld + c] - mu;
        s = fmaf(d, d, s);
      }
    var = col_reduce(s, red) / float(B);
    if (ok && threadIdx.y == 0) {   // running statistics: unbiased variance, momentum 0.1
      rmean[c] = (1.0f - kBnMomentum) * rmean[c] + kBnMomentum * mu;
      rvar[c] = (1.0f - kBnMomentum) * rvar[c] + kBnMomentum * (var * (float(B) / float(B - 1)));
    }
  } else if (ok) {
    mu = rmean[c];
    var = rvar[c];
  }
  if (!ok) return;
  const float invstd = 1.0f / sqrtf(var + kBnEps);
  const float g = gamma[c], b = beta[c];
  for (int m = threadIdx.y; m < B; m += 32) {
    const size_t e = size_t(m) * ld + c;
    const float xh = (z[e] - mu) * invstd;
    z[e] = xh;
    h[e] = fmaxf(xh * g + b, 0.f);
  }
  if (threadIdx.y == 0) invstd_out[c] = invstd;
}

// dh [B][ld] = gradient wrt the post-ReLU output, overwritten by the gradient wrt the Linear
// output z.  dgamma / dbeta are written straight into the flat gradient buffer.
__global__ void __launch_bounds__(1024)
bn_bwd_kernel(float *__restrict__ dh, const float *__restrict__ h, const float *__restrict__ xhat, int ld,
              int B, int H, const float *__restrict__ gamma, const float *__restrict__ invstd,
              float *__restrict__ dgamma, float *__restrict__ dbeta) {
  __shared__ float red[33][33];
  const int c = blockIdx.x * 32 + threadIdx.x;
  const bool ok = c < H;
  float s1 = 0.f, s2 = 0.f;
  if (ok)
    for (int m = threadIdx.y; m < B; m += 32) {
      const size_t e = size_t(m) * ld + c;
      const float dy = h[e] > 0.f ? dh[e] : 0.f;
      s1 += dy;
      s2 = fmaf(dy, xhat[e], s2);
    }
  s1 = col_reduce(s1, red);
  s2 = col_reduce(s2, red);
  if (!ok) return;
  const float g = gamma[c], is = invstd[c], n = float(B);
  const float sum_dxhat = s1 * g, sum_dxhat_xhat = s2 * g;
  for (int m = threadIdx.y; m < B; m += 32) {
    const size_t e = size_t(m) * ld + c;
    const float dy = h[e] > 0.f ? dh[e] : 0.f;
    const float dxhat = dy * g;
    dh[e] = is / n * (n * dxhat - sum_dxhat - xhat[e] * sum_dxhat_xhat);
  }
  if (threadIdx.y == 0) {
    dgamma[c] = s2;
    dbeta[c] = s1;
  }
}

// ---- BatchNorm1d with batch statistics over all data-parallel ranks ("sync-BN") --------------------
// The 1-GPU semantics of nn.BatchNorm1d on the concatenated batch (SURVEY 8(e); reference src/model.py:103-111):
// every rank writes its local per-column (mean, M2 = sum (z - mean)^2) -- or, in the backward pass, (sum dy,
// sum dy xhat) -- into its slot of a [world][2 ldh] buffer, the caller all-gathers the buffer between two graph
// segments, and every rank merges the slots in rank order (Chan's parallel variance; equal local batch sizes), so
// all ranks normalise with bit-identical statistics.  With world = 1 the result equals bn_fwd_kernel / bn_bwd_kernel
// bit for bit.
__global__ void __launch_bounds__(1024)
bn_stats_kernel(const float *__restrict__ z, int ld, int B, int H, float *__restrict__ slot, int ldh) {
  __shared__ float red[33][33];
  const int c = blockIdx.x * 32 + threadIdx.x;
  const bool ok = c < H;
  float s = 0.f;
  if (ok)
    for (int m = threadIdx.y; m < B; m += 32) s += z[size_t(m) * ld + c];
  const float mu = col_reduce(s, red) / float(B);
  s = 0.f;
  if (ok)
    for (int m = threadIdx.y; m < B; m += 32) {
      const float d = z[size_t(m) * ld + c] - mu;
      s = fmaf(d, d, s);
    }
  const float m2 = col_reduce(s, red);
  if (ok && threadIdx.y == 0) {
    slot[c] = mu;
    slot[ldh + c] = m2;
  }
}

__global__ void __launch_bounds__(1024)
bn_fwd_sync_kernel(float *__restrict__ z, int ld, int B, int H, const float *__restrict__ gamma,
                   const float *__restrict__ beta, float *__restrict__ rmean, float *__restrict__ rvar,
                   float *__restrict__ invstd_out, float *__restrict__ h, const float *__restrict__ gather, int world,
                   int ldh) {
  const int c = blockIdx.x * 32 + threadIdx.x;
  if (c >= H) return;
  float msum = gather[c];
  for (int r = 1; r < world; ++r) msum += gather[size_t(r) * 2 * ldh + c];
  const float mu = msum / float(world);
  float m2 = 0.f;
  for (int r = 0; r < world; ++r) {
    const float d = gather[size_t(r) * 2 * ldh + c] - mu;
    m2 += gather[size_t(r) * 2 * ldh + ldh + c] + float(B) * d * d;
  }
  const float n = float(world) * float(B);
  const float var = m2 / n;
  if (threadIdx.y == 0) {
    rmean[c] = (1.0f - kBnMomentum) * rmean[c] + kBnMomentum * mu;
    rvar[c] = (1.0f - kBnMomentum) * rvar[c] + kBnMomentum * (var * (n / (n - 1.0f)));
  }
  const float invstd = 1.0f / sqrtf(var + kBnEps);
  const float g = gamma[c], b = beta[c];
  for (int m = threadIdx.y; m < B; m += 32) {
    const size_t e = size_t(m) * ld + c;
    const float xh = (z[e] - mu) * invstd;
    z[e] = xh;
    h[e] = fmaxf(xh * g + b, 0.f);
  }
  if (threadIdx.y == 0) invstd_out[c] = invstd;
}

__global__ void __launch_bounds__(1024)
bn_bwd_stats_kernel(const float *__restrict__ dh, const float *__restrict__ h, const float *__restrict__ xhat, int ld,
                    int B, int H, float *__restrict__ slot, int ldh) {
  __shared__ float red[33][33];
  const int c = blockIdx.x * 32 + threadIdx.x;
  const bool ok = c < H;
  float s1 = 0.f, s2 = 0.f;
  if (ok)
    for (int m = threadIdx.y; m < B; m += 32) {
      const size_t e = size_t(m) * ld + c;
      const float dy = h[e] > 0.f ? dh[e] : 0.f;
      s1 += dy;
      s2 = fmaf(dy, xhat[e], s2);
    }
  s1 = col_reduce(s1, red);
  s2 = col_reduce(s2, red);
  if (ok && threadIdx.y == 0) {
    slot[c] = s1;
    slot[ldh + c] = s2;
  }
}

// dgamma / dbeta stay the LOCAL sums (the flat gradient is averaged over the ranks afterwards, like every other
// parameter gradient); the input gradient uses the sums over all ranks and n = world * B rows.
__global__ void __launch_bounds__(1024)
bn_bwd_sync_kernel(float *__restrict__ dh, const float *__restrict__ h, const float *__restrict__ xhat, int ld, int B,
                   int H, const float *__restrict__ gamma, const float *__restrict__ invstd,
                   float *__restrict__ dgamma, float *__restrict__ dbeta, const float *__restrict__ gather, int world,
                   int rank, int ldh) {
  const int c = blockIdx.x * 32 + threadIdx.x;
  if (c >= H) return;
  float s1 = gather[c], s2 = gather[ldh + c];
  for (int r = 1; r < world; ++r) {
    s1 += gather[size_t(r) * 2 * ldh + c];
    s2 += gather[size_t(r) * 2 * ldh + ldh + c];
  }
  const float g = gamma[c], is = invstd[c], n = float(world) * float(B);
  const float sum_dxhat = s1 * g, sum_dxhat_xhat = s2 * g;
  for (int m = threadIdx.y; m < B; m += 32) {
    const size_t e = size_t(m) * ld + c;
    const float dy = h[e] > 0.f ? dh[e] : 0.f;
    const float dxhat = dy * g;
    dh[e] = is / n * (n * dxhat - sum_dxhat - xhat[e] * sum_dxhat_xhat);
  }
  if (threadIdx.y == 0) {
    dgamma[c] = gather[size_t(rank) * 2 * ldh + ldh + c];
    dbeta[c] = gather[size_t(rank) * 2 * ldh + c];
  }
}

// ---- tanh-Gaussian policy head -------------------------------------------------------------------
struct PolicyFwdArgs {
  const float *feat; int ldh;            // last hidden activation [M, K]
  const float *Wm, *bm, *Ws, *bs; int ldw;
  const float *eps;                      // [M, A] or nullptr (deterministic tanh(mean))
  float *rows; int ldr, col0;            // action written into rows[m, col0 + j] (folds torch.cat)
  float *act_out; int ld_act;            // optional dense [M, ld_act] copy (select_action)
  float *logp, *act4, *std4, *gate4;     // [M], [M,4] x 3 (backward cache; may be nullptr)
  int M, K, A;
};

__global__ void __launch_bounds__(256) policy_fwd_kernel(PolicyFwdArgs a) {
  const int lane = threadIdx.x & 31;
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int nwarps = (gridDim.x * blockDim.x) >> 5;
  for (int m = warp; m < a.M; m += nwarps) {
    const float *h = a.feat + size_t(m) * a.ldh;
    float am[4] = {0.f, 0.f, 0.f, 0.f}, as[4] = {0.f, 0.f, 0.f, 0.f};
    for (int k = lane; k < a.K; k += 32) {
      const float hv = h[k];
#pragma unroll
      for (int j = 0; j < 4; ++j)
        if (j < a.A) {
          am[j] = fmaf(hv, a.Wm[size_t(j) * a.ldw + k], am[j]);
          as[j] = fmaf(hv, a.Ws[size_t(j) * a.ldw + k], as[j]);
        }
    }
#pragma unroll
    for (int j = 0; j < 4; ++j)
#pragma unroll
      for (int s = 16; s >= 1; s >>= 1) {
        am[j] += __shfl_xor_sync(0xffffffffu, am[j], s);
        as[j] += __shfl_xor_sync(0xffffffffu, as[j], s);
      }
    if (lane == 0) {
      float lp_sum = 0.f;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        if (j >= a.A) {
          if (a.act4) { a.act4[size_t(m) * 4 + j] = 0.f; a.std4[size_t(m) * 4 + j] = 0.f; a.gate4[size_t(m) * 4 + j] = 0.f; }
          continue;
        }
        const float mean = am[j] + a.bm[j];
        const float raw = as[j] + a.bs[j];
        const float ls = fminf(fmaxf(raw, -20.0f), 2.0f);       // src/model.py:122
        const float sd = expf(ls);
        float act;
        if (a.eps == nullptr) {
          act = tanhf(mean);
        } else {
          const float xt = mean + sd * a.eps[size_t(m) * a.A + j];   // rsample, :134
          act = tanhf(xt);
          const float diff = xt - mean;
          float lp = -(diff * diff) / (2.0f * (sd * sd)) - logf(sd) - kLogSqrt2Pi;   // Normal.log_prob
          lp -= logf(1.0f - act * act + 1e-8f);                                     // :138
          lp_sum += lp;
        }
        a.rows[size_t(m) * a.ldr + a.col0 + j] = act;
        if (a.act_out) a.act_out[size_t(m) * a.ld_act + j] = act;
        if (a.act4) {
          a.act4[size_t(m) * 4 + j] = act;
          a.std4[size_t(m) * 4 + j] = sd;
          a.gate4[size_t(m) * 4 + j] = (raw >= -20.0f && raw <= 2.0f) ? 1.0f : 0.f;
        }
      }
      if (a.logp) a.logp[m] = lp_sum;
    }
  }
}

// Bellman target: y = r + gamma (1 - d) (mean of the `keep` smallest target-critic values - coef log pi')
__global__ void __launch_bounds__(256)
sac_target_kernel(const float *__restrict__ qt, int64_t ldq, int n, int keep, const float *__restrict__ logp,
                  const float *__restrict__ r, const float *__restrict__ d, float gamma, float coef_const,
                  const float *__restrict__ alpha_dev, float *__restrict__ y, int M) {
  const float coef = coef_const >= 0.f ? coef_const : *alpha_dev;
  for (int m = blockIdx.x * blockDim.x + threadIdx.x; m < M; m += gridDim.x * blockDim.x) {
    float v[kMaxCritics];
#pragma unroll
    for (int i = 0; i < kMaxCritics; ++i) v[i] = i < n ? qt[int64_t(i) * ldq + m] : 3.4e38f;
#pragma unroll
    for (int i = 1; i < kMaxCritics; ++i) {        // insertion sort, ascending
      const float x = v[i];
      int j = i;
#pragma unroll
      for (int t = 0; t < kMaxCritics; ++t)
        if (j > 0 && v[j - 1] > x) { v[j] = v[j - 1]; --j; }
      v[j] = x;
    }
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < kMaxCritics; ++i)
      if (i < keep) s += v[i];
    float tq = s / float(keep);
    tq = tq - coef * logp[m];
    y[m] = r[m] + gamma * (1.0f - d[m]) * tq;
  }
}

// Single-CTA fixed-order reductions over the batch (metrics only; B floats per critic).
__device__ __forceinline__ float cta_sum_1024(float v, float *sm) {
  sm[threadIdx.x] = v;
  __syncthreads();
  for (int s = 512; s >= 1; s >>= 1) {
    if (int(threadIdx.x) < s) sm[threadIdx.x] += sm[threadIdx.x + s];
    __syncthreads();
  }
  const float r = sm[0];
  __syncthreads();
  return r;
}

// out[0..n) = mean (q_i - y)^2; out[8] = mean max_i |q_i - y|; out[9] = mean over i, m of q_i
__global__ void __launch_bounds__(1024)
critic_metrics_kernel(const float *__restrict__ q, int64_t ldq, int n, const float *__restrict__ y, int M,
                      float *__restrict__ out, int q_only, const float *__restrict__ is_w, float *__restrict__ td_out) {
  __shared__ float sm[1024];
  float loss[kMaxCritics], td = 0.f, qs = 0.f;
#pragma unroll
  for (int i = 0; i < kMaxCritics; ++i) loss[i] = 0.f;
  for (int m = threadIdx.x; m < M; m += 1024) {
    float mx = 0.f;
    const float yy = q_only ? 0.f : y[m];
    const float w = is_w != nullptr ? is_w[m] : 1.0f;      // prioritised replay: (weights * loss).mean() (:577-581)
#pragma unroll
    for (int i = 0; i < kMaxCritics; ++i)
      if (i < n) {
        const float qq = q[int64_t(i) * ldq + m];
        const float df = qq - yy;
        loss[i] = fmaf(w * df, df, loss[i]);
        mx = fmaxf(mx, fabsf(df));
        qs += qq;
      }
    td += mx;
    if (td_out != nullptr) td_out[m] = mx;                 // max over the critics of |q_i - y| (:620-621, :1021-1024)
  }
  const float inv = 1.0f / float(M);
  if (!q_only) {
#pragma unroll
    for (int i = 0; i < kMaxCritics; ++i)
      if (i < n) {
        const float t = cta_sum_1024(loss[i], sm);
        if (threadIdx.x == 0) out[i] = t * inv;
      }
    const float t = cta_sum_1024(td, sm);
    if (threadIdx.x == 0) out[8] = t * inv;
  }
  const float t = cta_sum_1024(qs, sm);
  if (threadIdx.x == 0) out[9] = t / (float(M) * float(n));
}

// Actor phase: per sample, which critics are among the `keep` smallest -> dq_i = -(1/keep)/M
// (written with stride 4 for head_bwd mode 2) and the actor loss mean(coef log pi - qtrunc).
__global__ void __launch_bounds__(1024)
actor_trunc_kernel(const float *__restrict__ q, int64_t ldq, int n, int keep, const float *__restrict__ logp,
                   float coef_const, const float *__restrict__ alpha_dev, float *__restrict__ dq /*[n][ldq*4]*/,
                   float *__restrict__ loss_out, int M) {
  __shared__ float sm[1024];
  const float coef = coef_const >= 0.f ? coef_const : *alpha_dev;
  const float w = 1.0f / float(keep);
  float ls = 0.f;
  for (int m = threadIdx.x; m < M; m += 1024) {
    float v[kMaxCritics];
    int id[kMaxCritics];
#pragma unroll
    for (int i = 0; i < kMaxCritics; ++i) { v[i] = i < n ? q[int64_t(i) * ldq + m] : 3.4e38f; id[i] = i; }
#pragma unroll
    for (int i = 1; i < kMaxCritics; ++i) {        // stable insertion sort carrying the critic index
      const float x = v[i];
      const int xi = id[i];
      int j = i;
#pragma unroll
      for (int t = 0; t < kMaxCritics; ++t)
        if (j > 0 && v[j - 1] > x) { v[j] = v[j - 1]; id[j] = id[j - 1]; --j; }
      v[j] = x;
      id[j] = xi;
    }
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < kMaxCritics; ++i)
      if (i < n) {
        const bool kept = i < keep;
        if (kept) s += v[i];
        dq[(int64_t(id[i]) * ldq + m) * 4] = kept ? -(w / float(M)) : 0.f;
      }
    ls += coef * logp[m] - s / float(keep);
  }
  const float t = cta_sum_1024(ls, sm);
  if (threadIdx.x == 0) *loss_out = t / float(M);
}

// ---- quantile critics (TQC with n_quantiles M per critic) ------------------------------------------------
// Atoms of critic i live at z + i * zstride as rows [B][ldm] (ldm = pad4(M)).  Every reduction below runs in a fixed
// order (warp trees, block trees, serial loops), no atomics.

// Target (sb3-contrib order): the n * M atoms of a row sorted ascending, the K smallest kept,
// y[b][j] = r + gamma (1 - d) (z_(j) - coef log pi').  One warp per row; the 32 * KPL keys (+inf past n * M) sit
// KPL per lane (key e = lane * KPL + r) and go through a bitonic network: partners closer than KPL are registers of
// the same lane, the others one shuffle away.
template <int KPL>
__global__ void __launch_bounds__(256)
quantile_target_kernel(const float *__restrict__ zt, int64_t zstride, int ldm, int n, int M, int keep,
                       const float *__restrict__ logp, const float *__restrict__ r, const float *__restrict__ d,
                       float gamma, float coef_const, const float *__restrict__ alpha_dev, float *__restrict__ y,
                       int ldy, int B) {
  const float coef = coef_const >= 0.f ? coef_const : *alpha_dev;
  const int lane = threadIdx.x & 31;
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int nwarps = (gridDim.x * blockDim.x) >> 5;
  const int total = n * M;
  for (int b = warp; b < B; b += nwarps) {
    float v[KPL];
#pragma unroll
    for (int q = 0; q < KPL; ++q) {
      const int e = lane * KPL + q;
      const int i = e / M;
      v[q] = e < total ? zt[int64_t(i) * zstride + int64_t(b) * ldm + (e - i * M)] : INFINITY;
    }
#pragma unroll
    for (int k = 2; k <= 32 * KPL; k <<= 1) {
#pragma unroll
      for (int j = k >> 1; j > 0; j >>= 1) {
        if (j >= KPL) {
#pragma unroll
          for (int q = 0; q < KPL; ++q) {
            const int e = lane * KPL + q;
            const float o = __shfl_xor_sync(0xffffffffu, v[q], j / KPL);
            const bool up = (e & k) == 0, low = (e & j) == 0;
            v[q] = up == low ? fminf(v[q], o) : fmaxf(v[q], o);
          }
        } else {
#pragma unroll
          for (int q = 0; q < KPL; ++q)
            if ((q & j) == 0) {
              const bool up = ((lane * KPL + q) & k) == 0;
              const float a = v[q], c = v[q + j];
              v[q] = up ? fminf(a, c) : fmaxf(a, c);
              v[q + j] = up ? fmaxf(a, c) : fminf(a, c);
            }
        }
      }
    }
    const float ent = coef * logp[b], rb = r[b], disc = gamma * (1.0f - d[b]);
#pragma unroll
    for (int q = 0; q < KPL; ++q) {
      const int e = lane * KPL + q;
      if (e < keep) y[int64_t(b) * ldy + e] = rb + disc * (v[q] - ent);
    }
  }
}

// Critic loss, forward and backward in one pass: blockIdx.y = critic i, blockIdx.x = a block of `rows` batch rows,
// thread t owns (row t / M, atom k = t % M).  With u = y_j - Z_ik, tau_k = (k + 0.5) / M and Huber kappa = 1:
//   dZ_ik = -w_b sum_j |tau_k - 1{u < 0}| clamp(u, -1, 1) / (B M K)          -> dz (the head's input of the backward)
//   loss partial of the block = sum over its (row, k, j) of w_b |tau_k - 1{u < 0}| h(u)   -> loss_part[i][blockIdx.x]
//   |mean_k Z_ik - mean_j y_j| per row                                       -> td_part[i][b]
constexpr int kQhThreads = 256;
constexpr int kQhMaxTargets = 2048;   // rows * K <= (256 / M) * n M <= 8 * 256
__global__ void __launch_bounds__(kQhThreads)
quantile_huber_kernel(const float *__restrict__ z, int64_t zstride, int ldm, int M, const float *__restrict__ y,
                      int ldy, int K, const float *__restrict__ is_w, float *__restrict__ dz,
                      float *__restrict__ loss_part, float *__restrict__ td_part, int B, int rows) {
  __shared__ float ys[kQhMaxTargets];
  __shared__ float zs[kQhThreads];
  __shared__ float red[kQhThreads];
  const int i = blockIdx.y, b0 = blockIdx.x * rows, tid = threadIdx.x;
  const int nrows = min(rows, B - b0);
  for (int t = tid; t < nrows * K; t += kQhThreads) {
    const int rr = t / K;
    ys[t] = y[int64_t(b0 + rr) * ldy + (t - rr * K)];
  }
  const int rr = tid / M, k = tid - rr * M, b = b0 + rr;
  const bool own = rr < nrows;
  const int64_t at = int64_t(i) * zstride + int64_t(b) * ldm + k;
  const float zv = own ? z[at] : 0.f;
  zs[tid] = zv;
  __syncthreads();
  float l = 0.f;
  if (own) {
    const float tau = (float(k) + 0.5f) / float(M);
    const float *yr = ys + rr * K;
    float g = 0.f;
    for (int j = 0; j < K; ++j) {
      const float u = yr[j] - zv;
      const float wt = u < 0.f ? 1.0f - tau : tau;
      const float au = fabsf(u);
      l = fmaf(wt, au > 1.0f ? au - 0.5f : 0.5f * u * u, l);
      g = fmaf(wt, fminf(fmaxf(u, -1.0f), 1.0f), g);
    }
    const float w = is_w != nullptr ? is_w[b] : 1.0f;
    dz[at] = -(w * g) / (float(B) * float(M) * float(K));
    l *= w;
    if (k == 0) {
      float sz = 0.f, sy = 0.f;
      for (int kk = 0; kk < M; ++kk) sz += zs[rr * M + kk];
      for (int j = 0; j < K; ++j) sy += yr[j];
      td_part[int64_t(i) * B + b] = fabsf(sz / float(M) - sy / float(K));
    }
  }
  red[tid] = l;
  __syncthreads();
  for (int s = kQhThreads / 2; s >= 1; s >>= 1) {
    if (tid < s) red[tid] += red[tid + s];
    __syncthreads();
  }
  if (tid == 0) loss_part[int64_t(i) * gridDim.x + blockIdx.x] = red[0];
}

// out[M_CLOSS + i] = (sum of critic i's loss partials) / (B M K); per row the max over the critics of the td parts
// -> td_out (prioritised replay) and their batch mean -> out[M_TD]
__global__ void __launch_bounds__(1024)
quantile_metrics_kernel(const float *__restrict__ loss_part, int nblk, const float *__restrict__ td_part, int n, int B,
                        float count, float *__restrict__ out, int slot_loss, int slot_td, float *__restrict__ td_out) {
  __shared__ float sm[1024];
  for (int i = 0; i < n; ++i) {
    float s = 0.f;
    for (int t = threadIdx.x; t < nblk; t += 1024) s += loss_part[int64_t(i) * nblk + t];
    const float tot = cta_sum_1024(s, sm);
    if (threadIdx.x == 0) out[slot_loss + i] = tot / count;
  }
  float td = 0.f;
  for (int m = threadIdx.x; m < B; m += 1024) {
    float mx = 0.f;
    for (int i = 0; i < n; ++i) mx = fmaxf(mx, td_part[int64_t(i) * B + m]);
    td += mx;
    if (td_out != nullptr) td_out[m] = mx;
  }
  const float tot = cta_sum_1024(td, sm);
  if (threadIdx.x == 0) out[slot_td] = tot / float(B);
}

// Per row b: the mean of the n * M atoms, or coef log pi_b - that mean (the actor loss's row term) when logp is
// given; with dz != nullptr every atom's gradient slot of the row gets dz_value (the actor's backward through the
// critics: d loss / d Z_ik = -1 / (B n M)).  One warp per row.
__global__ void __launch_bounds__(256)
quantile_row_mean_kernel(const float *__restrict__ z, int64_t zstride, int ldm, int n, int M,
                         const float *__restrict__ logp, float coef_const, const float *__restrict__ alpha_dev,
                         float *__restrict__ row_out, float *__restrict__ dz, float dz_value, int B) {
  const int lane = threadIdx.x & 31;
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int nwarps = (gridDim.x * blockDim.x) >> 5;
  const int total = n * M;
  for (int b = warp; b < B; b += nwarps) {
    float s = 0.f;
    for (int e = lane; e < total; e += 32) {
      const int i = e / M;
      const int64_t at = int64_t(i) * zstride + int64_t(b) * ldm + (e - i * M);
      s += z[at];
      if (dz != nullptr) dz[at] = dz_value;
    }
#pragma unroll
    for (int o = 16; o >= 1; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (lane == 0) {
      const float mean = s / float(total);
      row_out[b] = logp != nullptr ? (coef_const >= 0.f ? coef_const : *alpha_dev) * logp[b] - mean : mean;
    }
  }
}

// dact[m, j] (+)= sum_n dZ0[m, n] W0[n, col0 + j]   (critic layer-1 input gradient, action columns)
__global__ void __launch_bounds__(256)
action_grad_acc_kernel(const float *__restrict__ dZ0, int lddz, const float *__restrict__ W0, int ldw, int col0,
                       float *__restrict__ dact, int M, int N, int nact, int accumulate) {
  const int lane = threadIdx.x & 31;
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int nwarps = (gridDim.x * blockDim.x) >> 5;
  for (int m = warp; m < M; m += nwarps) {
    float acc[4] = {0.f, 0.f, 0.f, 0.f};
    for (int n = lane; n < N; n += 32) {
      const float g = dZ0[size_t(m) * lddz + n];
      const float *w = W0 + size_t(n) * ldw + col0;
#pragma unroll
      for (int j = 0; j < 4; ++j)
        if (j < nact) acc[j] = fmaf(g, w[j], acc[j]);
    }
#pragma unroll
    for (int j = 0; j < 4; ++j)
#pragma unroll
      for (int s = 16; s >= 1; s >>= 1) acc[j] += __shfl_xor_sync(0xffffffffu, acc[j], s);
    if (lane == 0) {
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        float v = j < nact ? acc[j] : 0.f;
        if (accumulate) v += dact[size_t(m) * 4 + j];
        dact[size_t(m) * 4 + j] = v;
      }
    }
  }
}

// dzh[m][0..4) = dL/dmean, dzh[m][4..8) = dL/d(log_std head output); analytic rsample backward:
// the Normal.log_prob term contributes 0 to dmean and -dlogp to dlog_std.
__global__ void __launch_bounds__(256)
policy_bwd_kernel(const float *__restrict__ dact, const float *__restrict__ act4, const float *__restrict__ std4,
                  const float *__restrict__ gate4, const float *__restrict__ eps, int A, float coef_const,
                  const float *__restrict__ alpha_dev, float *__restrict__ dzh, int M) {
  const float coef = coef_const >= 0.f ? coef_const : *alpha_dev;
  const float dlogp = coef / float(M);
  for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < M * 4; e += gridDim.x * blockDim.x) {
    const int m = e >> 2, j = e & 3;
    float dm = 0.f, dr = 0.f;
    if (j < A) {
      const float a = act4[e];
      const float one_m = 1.0f - a * a;
      const float gx = dact[e] * one_m + dlogp * (2.0f * a * one_m / (one_m + 1e-8f));
      dm = gx;
      dr = (gx * eps[size_t(m) * A + j] * std4[e] - dlogp) * gate4[e];
    }
    dzh[size_t(m) * 8 + j] = dm;
    dzh[size_t(m) * 8 + 4 + j] = dr;
  }
}

// Backward through both policy heads: partial weight / bias gradients per row slab and
// dfeat[m, k] = sum_j dzh[m, j] W[j, k]  (no activation factor: the ReLU mask is applied by bn_bwd).
constexpr int kHeadRows = 256;
__global__ void __launch_bounds__(256)
policy_head_bwd_kernel(const float *__restrict__ dzh, const float *__restrict__ feat, int ldh,
                       const float *__restrict__ Wm, const float *__restrict__ Ws, int ldw, int A,
                       float *__restrict__ dfeat, int lddf, float *__restrict__ pWm, float *__restrict__ pBm,
                       float *__restrict__ pWs, float *__restrict__ pBs, int64_t split_stride, int M, int K,
                       int rows_per_slab) {
  __shared__ float dz_s[kHeadRows][8];
  const int tid = threadIdx.x;
  const int r0 = blockIdx.x * rows_per_slab;
  const int nrows = min(rows_per_slab, M - r0);
  for (int i = tid; i < nrows * 8; i += blockDim.x) dz_s[i >> 3][i & 7] = dzh[size_t(r0) * 8 + i];
  __syncthreads();
  if (tid < 8) {
    const int j = tid & 3;
    if (j < A) {
      float s = 0.f;
      for (int i = 0; i < nrows; ++i) s += dz_s[i][tid];
      (tid < 4 ? pBm : pBs)[int64_t(blockIdx.x) * split_stride + j] = s;
    }
  }
  for (int k = tid; k < ldw; k += blockDim.x) {
    float w[8], acc[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int jj = j & 3;
      w[j] = (k < K && jj < A) ? (j < 4 ? Wm : Ws)[size_t(jj) * ldw + k] : 0.f;
      acc[j] = 0.f;
    }
    if (k < K) {
      for (int i = 0; i < nrows; ++i) {
        const size_t m = size_t(r0 + i);
        const float h = feat[m * ldh + k];
        float dh = 0.f;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const float dz = dz_s[i][j];
          dh = fmaf(dz, w[j], dh);
          acc[j] = fmaf(dz, h, acc[j]);
        }
        dfeat[m * lddf + k] = dh;
      }
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int jj = j & 3;
      if (jj < A) (j < 4 ? pWm : pWs)[int64_t(blockIdx.x) * split_stride + size_t(jj) * ldw + k] = acc[j];
    }
  }
}

// alpha_update (src/agent.py:532-546): AdamW (wd 0.01, betas 0.9/0.999, eps 1e-8) on the scalar
// log_alpha with gradient -mean(log pi + target_entropy); alpha = exp(log_alpha).  Two kernels so that the
// batch mean can be averaged across data-parallel ranks in between (it sits right behind the actor's
// flat gradient).  st: [0] log_alpha, [1] alpha, [2] m, [3] v
__global__ void __launch_bounds__(1024)
alpha_mean_kernel(const float *__restrict__ logp, int M, float target_entropy, float *__restrict__ mean_out) {
  __shared__ float sm[1024];
  float s = 0.f;
  for (int m = threadIdx.x; m < M; m += 1024) s += logp[m] + target_entropy;
  const float tot = cta_sum_1024(s, sm);
  if (threadIdx.x == 0) *mean_out = tot / float(M);
}

// sc: [0] lr / (1 - b1^t), [1] sqrt(1 - b2^t), [2] 1 - lr * wd  (device scalars, so the update can be a graph)
__global__ void alpha_step_kernel(const float *__restrict__ mean_in, const float *__restrict__ sc,
                                  float *__restrict__ st, float *__restrict__ loss_out) {
  const float step_size = sc[0], bc2_sqrt = sc[1], decay = sc[2];
  const float mean = *mean_in;
  float la = st[0];
  *loss_out = -(la * mean);
  const float g = -mean;
  la *= decay;
  float m1 = st[2], v = st[3];
  m1 = m1 + float(1.0 - 0.9) * (g - m1);
  v = v * float(0.999) + float(1.0 - 0.999) * g * g;
  const float denom = sqrtf(v) / bc2_sqrt + 1e-8f;
  la = la - step_size * (m1 / denom);
  st[0] = la;
  st[1] = expf(la);
  st[2] = m1;
  st[3] = v;
}


// ---- actor parameters ----------------------------------------------------------------------------
// A layout of its own (BatchNorm parameters, two heads); the critics are MlpParams (params.cuh).
struct ActorNet {
  int L = 0, D = 0, H = 0, A = 0, ldh = 0;
  std::vector<int> ldw, w_off, b_off, gam_off, bet_off;     // hidden layers
  int wm_off = 0, bm_off = 0, ws_off = 0, bs_off = 0;       // mean / log_std heads [A][ldh]
  int total = 0;
  float *p = nullptr, *g = nullptr, *m = nullptr, *v = nullptr;
  float *rmean = nullptr, *rvar = nullptr;                  // [L][ldh]
  WeightCopies copies;
  void init_copies() {                                      // W^T of the hidden Linears 1..L-1 (input gradients)
    std::vector<WeightCopies::Linear> tr;
    for (int l = 1; l < L; ++l) tr.push_back({l, w_off[l], H, H, ldw[l]});
    copies.init(total, L, tr, true);
  }
  void init(int D_, int H_, int A_, int L_) {
    L = L_; D = D_; H = H_; A = A_; ldh = pad4(H);
    int off = 0;
    for (int l = 0; l < L; ++l) {
      ldw.push_back(pad4(l == 0 ? D : H));
      w_off.push_back(off); off += H * ldw[l];
      b_off.push_back(off); off += ldh;
      gam_off.push_back(off); off += ldh;
      bet_off.push_back(off); off += ldh;
    }
    wm_off = off; off += A * ldh;
    bm_off = off; off += 4;
    ws_off = off; off += A * ldh;
    bs_off = off; off += 4;
    total = off;
    for (float **q : {&p, &g, &m, &v}) {      // g[total] holds mean(log pi + target_entropy) for alpha_update
      *q = dev_alloc<float>(total + 4);
      GCRL_CUDA(cudaMemset(*q, 0, size_t(total + 4) * 4));
    }
    rmean = dev_alloc<float>(size_t(2) * L * ldh);   // running mean | running var, one buffer (data-parallel average)
    rvar = rmean + size_t(L) * ldh;
    std::vector<float> ones(size_t(L) * ldh, 1.0f);
    GCRL_CUDA(cudaMemset(rmean, 0, ones.size() * 4));
    GCRL_CUDA(cudaMemcpy(rvar, ones.data(), ones.size() * 4, cudaMemcpyHostToDevice));
    for (int l = 0; l < L; ++l)   // BatchNorm weight = 1 (torch default)
      GCRL_CUDA(cudaMemcpy(p + gam_off[l], ones.data(), size_t(H) * 4, cudaMemcpyHostToDevice));
  }
  void destroy() { for (float *q : {p, g, m, v, rmean}) if (q) cudaFree(q); copies.destroy(); }
};

}  // namespace

struct gcrl_sac {
  uint32_t magic = 0x54434153u;   // handle type tag: the two agent families share the Python base class
  int device = 0;
  gcrl_sac_config cfg{};
  int D = 0, A = 0, H = 0, L = 0, n = 0, keep = 0, ldh = 0, ldc = 0;
  int64_t maxB = 0;
  ActorNet actor;
  MlpParams critic[kMaxCritics], target[kMaxCritics];
  int adam_t_c = 0, adam_t_a = 0, adam_t_alpha = 0;
  int dp_B = -1, dp_flags = -1;                  // the update the data-parallel phases belong to
  bool dp_open = false;                          // a phase-wise data-parallel update: phase 0 issued, phase 3 not yet
  bool tc_update = false;                        // the update being recorded / issued runs on the tensor-core engine
  bool use_graphs = true;
  cudaStream_t cap_stream = nullptr;             // capture-only stream (the caller's may be the legacy one)
  std::map<std::tuple<int, int, int>, GraphRec> graphs;   // (B, flags, phase mask)
  // n consecutive updates in one graph (gcrl_sac_update_many): everything a captured update reads that changes from
  // one update to the next has one slot per update, in one device allocation laid out for the call's (n, B):
  // scalars [n] x kManyScalBytes | positions [n][B] int64 | eps_next [n][B][A] | eps_cur [n][B][A] | metrics [n][36]
  // | TD errors [n][B] (prioritised replay; read back with the metric rows in one copy)
  struct Many {
    char *d = nullptr;
    size_t cap = 0;                              // bytes; growing it drops the cached graphs (their addresses move)
    // (B, flags of every update, buffer, engine path, buffer epoch, length drawn from): as in agent.cu
    using Key = std::tuple<int64_t, std::vector<int>, uintptr_t, int, uint64_t, int64_t>;
    ManyGraphs<Key> graphs;
  } many;
  // sync-BN (gcrl_sac_set_sync_bn): the update is cut into graph segments, each ending in the collective the caller
  // runs before the next one (gcrl_sac_update_segment)
  int sync_world = 0, sync_rank = 0;
  float *bn_gather = nullptr;                    // [world][2 ldh]: per-rank BatchNorm partial statistics
  struct SegRec { GraphRec graph; int collective; };
  std::map<std::tuple<int, int>, std::vector<SegRec>> seg_graphs;     // (B, flags)
  std::vector<SegRec> *seg_build = nullptr;      // the segment list being captured
  uint64_t seg_mark = 0;
  float *critic_grads = nullptr;                 // [n][critic_stride]: the ensemble's flat gradients, contiguous
  int critic_stride = 0;
  // activations
  std::vector<float *> xhat, ah;                 // actor: [L] x [maxB, ldh]
  float *invstd = nullptr;                       // [L][ldh]
  std::vector<std::vector<float *>> ch;          // critics: [n][L] x [maxB, ldh]
  std::vector<float *> th;                       // target critic scratch [L]
  float *dz[2] = {nullptr, nullptr};
  std::vector<float *> dzc;                      // [2 n] x [min(maxB, kEnsembleBatchMax), ldh]: per-critic gradient ping-pong
  int64_t pset = 0;                              // floats per partial-gradient set (one set per critic)
  float *sa = nullptr, *nsa = nullptr, *spi = nullptr, *br = nullptr, *bd = nullptr;
  float *bs = nullptr, *ba = nullptr, *bns = nullptr, *br0 = nullptr, *bd0 = nullptr;
  float *q = nullptr, *qt = nullptr, *y = nullptr, *dq = nullptr;     // [n][maxB], [n][maxB], [maxB], [n][maxB*4]
  float *logp = nullptr, *act4 = nullptr, *std4 = nullptr, *gate4 = nullptr, *dact = nullptr, *dzh = nullptr;
  float *eps_next = nullptr, *eps_cur = nullptr;
  float *per_w = nullptr, *per_td = nullptr;     // prioritised replay: importance weights in, TD errors out [maxB]
  bool per_on = false;                           // flags bit3 of the update being issued
  // quantile critics (gcrl_sac_create_quantile; nq == 0: scalar critics): M atoms per critic, d dropped per critic,
  // K = n (M - d) kept target atoms.  q / qt / dq then hold [n][maxB][ldm] (qstride floats per critic), y [maxB][ldy]
  int nq = 0, nq_drop = 0, nq_keep = 0, ldm = 0, ldy = 0;
  int64_t qstride = 0;
  float *qscratch = nullptr, *qrow = nullptr;   // quantile_critic_loss's scratch [2 n maxB], rows [maxB]
  float *partials = nullptr;
  int64_t slab = 0;
  float *sumsq = nullptr;
  float *mdev = nullptr;                         // [32] device metrics block
  float *alpha_state = nullptr;                  // [4] log_alpha, alpha, m, v: mdev + 32 (one copy takes both)
  StepScalars *d_scalars = nullptr;
  PinnedRing scal_stage, io_stage;
  float *d_io = nullptr;
  size_t io_cap = 0;
};

namespace {

enum : int { M_CLOSS = 0 /*[8]*/, M_TD = 8, M_Q = 9, M_CGN = 10 /*[8]*/, M_ALOSS = 18, M_AGN = 19, M_ALPHA_LOSS = 20 };

int blocks_for(int64_t work, int per_block) {
  return int(std::max<int64_t>(1, std::min<int64_t>((work + per_block - 1) / per_block, int64_t(sm_count()) * 8)));
}

// Collectives a graph segment ends in (gcrl_sac_update_segment): what the caller runs before the next segment.
enum : int { COLL_DONE = 0, COLL_GATHER_BN = 1, COLL_AVG_CRITIC = 2, COLL_AVG_ACTOR = 3 };

// Close the graph segment being captured and open the next one.  Only the segmented capture reaches this.
void seg_cut(gcrl_sac *ag, int collective, bool last = false) {
  ag->seg_build->push_back(gcrl_sac::SegRec{end_capture(ag->cap_stream, launch_counter() - ag->seg_mark), collective});
  ag->seg_mark = launch_counter();
  if (!last) begin_capture(ag->cap_stream);
}

// ---- tensor-core engine (tcgen05, 3xTF32; precision >= 1) --------------------------------------------
// Hidden-layer forward, input-gradient and weight-gradient GEMMs of an update.  precision 2: every batch >= 128 rows;
// precision 1: once B * H^2 reaches the break-even measured against the fp32 tiles for SAC / TQC on a B200 (DESIGN.md
// 4, profiles/r03_sac_precision.json): between 1024 and 2048 rows at H = 256, at or below 512 rows at H = 512 (the
// ensemble's launches fill the SMs at fewer rows per member when the layers are wider).
constexpr int64_t kSacTcMinWork = int64_t(2048) * 256 * 256;
bool use_tc(const gcrl_sac *ag, int B, int N, int K) {
  if (!tc_dense_supported(B, N, K)) return false;
  return ag->cfg.precision == 2 ? B >= 128
                                : (ag->cfg.precision == 1 && int64_t(B) * ag->H * ag->H >= kSacTcMinWork);
}
// every hidden-layer shape of an update passes the same test (K = padded input widths, all multiples of 4)
bool engine_tc(const gcrl_sac *ag, int B) { return use_tc(ag, B, ag->H, ag->ldh); }

// eager, outside capture: the halves of every network whose weights changed since they were last split
void ensure_split(gcrl_sac *ag, cudaStream_t st) {
  ag->actor.copies.split_if_stale(ag->actor.p, st);
  for (int i = 0; i < ag->n; ++i) {
    ag->critic[i].copies.split_if_stale(ag->critic[i].p, st);
    ag->target[i].copies.split_if_stale(ag->target[i].p, st);
  }
}
void mark_split_stale(gcrl_sac *ag) {
  ag->actor.copies.stale = true;
  for (int i = 0; i < ag->n; ++i) ag->critic[i].copies.stale = ag->target[i].copies.stale = true;
}

// partial weight / bias gradients of one hidden Linear [H][ldw] on input X[B][K] (K: padded for layer 0)
int linear_wgrad(gcrl_sac *ag, const float *dZ, const float *X, int ldx, int K, bool tc_ok, float *pW, int ldw,
                 float *pB, int B, cudaStream_t st) {
  const int Kp = pad4(K);     // operand rows and weight rows are zero-padded to ld
  if (ag->tc_update && tc_ok && tc_wgrad_supported(B, ag->H, Kp))
    return launch_tc_wgrad(dZ, ag->ldh, X, ldx, pW, ldw, ag->slab, pB, ag->slab, B, ag->H, Kp, kSplits, st);
  return launch_linear_wgrad(dZ, ag->ldh, X, ldx, pW, ldw, ag->slab, pB, ag->slab, B, ag->H, K, kSplits, st);
}

// Tensor cores: dX = dZ W (.) leaky'(act) of hidden layer l >= 1 for the critics first .. first + m - 1 in one launch
// (gradients dz_in[j] -> dz_out[j]), with the transposed weight copies as the K-major operand
void critics_dgrad_tc(gcrl_sac *ag, int first, int m, int l, float *const *dz_in, float *const *dz_out, int B,
                      cudaStream_t st) {
  TcDenseProblem pr[kMaxBatchedLinear];
  for (int j = 0; j < m; ++j) {
    const WeightCopies &tc = ag->critic[first + j].copies;
    pr[j] = TcDenseProblem{dz_in[j], ag->ldh, tc.pT_hi + tc.t_off[l], tc.pT_lo + tc.t_off[l], tc.ldt[l], nullptr,
                           ag->ch[first + j][l - 1], dz_out[j]};
  }
  launch_tc_dense_ensemble(pr, m, ag->ldh, ag->ldh, B, ag->H, ag->H, 1, st);
}

// The whole ensemble on the same input rows: one launch per layer (blockIdx.z = critic, or the members of the
// tensor-core ensemble launch) instead of n.
// Activations land in ag->ch[i][l] (the caches of the backward pass, or plain scratch for the targets).
void critics_fwd(gcrl_sac *ag, const MlpParams *nets, const float *X, float *q_out, int B, cudaStream_t st) {
  const int n = ag->n, L = ag->L;
  LinearFwdProblem pr[kMaxBatchedLinear];
  TcDenseProblem tp[kMaxBatchedLinear];
  for (int l = 0; l < L; ++l) {
    if (ag->tc_update) {      // layer 0: K = ldc, the operand rows [s | a | 0] and the weight rows are zero-padded
      for (int i = 0; i < n; ++i)
        tp[i] = TcDenseProblem{l == 0 ? X : ag->ch[i][l - 1], l == 0 ? ag->ldc : ag->ldh, nets[i].copies.p_hi + nets[i].w_off[l],
                               nets[i].copies.p_lo + nets[i].w_off[l], nets[i].ldw[l], nets[i].b(l), nullptr, ag->ch[i][l]};
      launch_tc_dense_ensemble(tp, n, 0, ag->ldh, B, ag->H, l == 0 ? ag->ldc : ag->H, 0, st);
      continue;
    }
    for (int i = 0; i < n; ++i)
      pr[i] = LinearFwdProblem{l == 0 ? X : ag->ch[i][l - 1], l == 0 ? ag->ldc : ag->ldh, nets[i].W(l), nets[i].ldw[l],
                               nets[i].b(l), ag->ch[i][l], ag->ldh};
    launch_linear_fwd_batched(pr, n, B, ag->H, l == 0 ? ag->D + ag->A : ag->H, ACT_LEAKY, st);
  }
  if (ag->nq > 0) {           // quantile critics: the H -> M head on the fp32 tiles, atoms [B][ldm] per critic
    for (int i = 0; i < n; ++i)
      pr[i] = LinearFwdProblem{ag->ch[i][L - 1], ag->ldh, nets[i].W(L), nets[i].ldw[L], nets[i].b(L),
                               q_out + int64_t(i) * ag->qstride, ag->ldm};
    launch_linear_fwd_batched(pr, n, B, ag->nq, ag->H, ACT_NONE, st);
    return;
  }
  HeadFwdProblem hp[kMaxBatchedLinear];
  for (int i = 0; i < n; ++i)
    hp[i] = HeadFwdProblem{ag->ch[i][L - 1], nets[i].W(L), nets[i].b(L), q_out + int64_t(i) * ag->maxB};
  launch_head_fwd_batched(hp, n, ag->ldh, nets[0].ldw[L], B, ag->H, st);
}

// actor forward on rows[:, :D]; action -> rows[:, D:D+A]
void actor_fwd(gcrl_sac *ag, float *rows, const float *eps, int B, bool train, bool cache, float *act_out,
               cudaStream_t st) {
  ActorNet &a = ag->actor;
  const float *in = rows;
  int ldin = ag->ldc, K = ag->D;
  for (int l = 0; l < ag->L; ++l) {
    if (train && ag->tc_update)       // (select_action, train == false, stays on the fp32 path)
      launch_tc_dense(in, ldin, a.copies.p_hi + a.w_off[l], a.ldw[l], a.p + a.b_off[l], nullptr, 0, ag->xhat[l], ag->ldh, B,
                      ag->H, pad4(K), 2, st, a.copies.p_lo + a.w_off[l]);
    else
      launch_linear_fwd(in, ldin, a.p + a.w_off[l], a.ldw[l], a.p + a.b_off[l], ag->xhat[l], ag->ldh, B, ag->H, K,
                        ACT_NONE, st);
    if (train && ag->sync_world > 0) {
      GCRL_REQUIRE(ag->seg_build != nullptr, "a sync-BN agent trains through gcrl_sac_update_segment only");
      bn_stats_kernel<<<(ag->H + 31) / 32, dim3(32, 32), 0, st>>>(
          ag->xhat[l], ag->ldh, B, ag->H, ag->bn_gather + size_t(ag->sync_rank) * 2 * ag->ldh, ag->ldh);
      GCRL_LAUNCHED();
      seg_cut(ag, COLL_GATHER_BN);
      bn_fwd_sync_kernel<<<(ag->H + 31) / 32, dim3(32, 32), 0, st>>>(
          ag->xhat[l], ag->ldh, B, ag->H, a.p + a.gam_off[l], a.p + a.bet_off[l], a.rmean + size_t(l) * ag->ldh,
          a.rvar + size_t(l) * ag->ldh, ag->invstd + size_t(l) * ag->ldh, ag->ah[l], ag->bn_gather, ag->sync_world,
          ag->ldh);
      GCRL_LAUNCHED();
    } else {
      bn_fwd_kernel<<<(ag->H + 31) / 32, dim3(32, 32), 0, st>>>(ag->xhat[l], ag->ldh, B, ag->H, a.p + a.gam_off[l],
                                                                a.p + a.bet_off[l], a.rmean + size_t(l) * ag->ldh,
                                                                a.rvar + size_t(l) * ag->ldh,
                                                                ag->invstd + size_t(l) * ag->ldh, ag->ah[l], train ? 1 : 0);
      GCRL_LAUNCHED();
    }
    in = ag->ah[l]; ldin = ag->ldh; K = ag->H;
  }
  PolicyFwdArgs p{};
  p.feat = ag->ah[ag->L - 1]; p.ldh = ag->ldh;
  p.Wm = a.p + a.wm_off; p.bm = a.p + a.bm_off; p.Ws = a.p + a.ws_off; p.bs = a.p + a.bs_off; p.ldw = ag->ldh;
  p.eps = eps;
  p.rows = rows; p.ldr = ag->ldc; p.col0 = ag->D;
  p.act_out = act_out; p.ld_act = ag->A;
  p.logp = ag->logp;
  if (cache) { p.act4 = ag->act4; p.std4 = ag->std4; p.gate4 = ag->gate4; }
  p.M = B; p.K = ag->H; p.A = ag->A;
  policy_fwd_kernel<<<blocks_for(B, 8), 256, 0, st>>>(p);
  GCRL_LAUNCHED();
}

void reduce_critic(gcrl_sac *ag, MlpParams &c, const int *splits, int head_splits, cudaStream_t st,
                   const float *partials = nullptr) {
  if (partials == nullptr) partials = ag->partials;
  ReduceArgs r{};
  for (int l = 0; l < c.layers; ++l) {
    const int sp = l == c.layers - 1 ? head_splits : splits[l];
    r.seg[r.nseg++] = SegDesc{c.w_off[l], c.out_d[l] * c.ldw[l], partials, sp, ag->slab, c.w_off[l]};
    r.seg[r.nseg++] = SegDesc{c.b_off[l], c.out_d[l], partials, sp, ag->slab, c.b_off[l]};
  }
  r.total = c.total; r.grad = c.g; r.sumsq_partials = ag->sumsq;
  r.metric_partials = nullptr; r.metric_splits = 0; r.metric_scale = 0.f; r.metrics = ag->mdev;
  r.slot_loss = r.slot_td = r.slot_q = -1;
  launch_reduce_grads(r, st);
}

// tc / ttc: the tensor-core copies of the network and of its target (no W^T: targetT stays nullptr)
void adam(gcrl_sac *ag, float *p, float *m, float *v, const float *g, int total, int which, float *target,
          bool polyak, int slot_norm, cudaStream_t st, WeightCopies &tc, WeightCopies *ttc) {
  AdamArgs a{};
  a.p = p; a.m = m; a.v = v; a.g = g; a.n = total;
  a.sumsq_partials = ag->sumsq; a.nsumsq = reduce_grid(total);
  a.max_norm = ag->cfg.grad_clip;
  a.weight_decay = ag->cfg.weight_decay;
  a.sc = ag->d_scalars; a.which = which;
  a.target = target; a.tau = ag->cfg.tau; a.one_minus_tau = float(1.0 - double(ag->cfg.tau));
  a.polyak = (polyak && target) ? 1 : 0;
  a.metrics = ag->mdev; a.slot_norm = slot_norm;
  a.tmap = tc.tmap; a.pT = tc.pT; a.targetT = nullptr;
  launch_adam(a, st);
  if (ag->tc_update) {          // this update's later GEMMs read the stepped weights through the tensor cores
    tc.split(p, st);
    if (a.polyak && ttc != nullptr) ttc->split(target, st);
  }
}

void adam_critic(gcrl_sac *ag, int i, int flags, cudaStream_t st) {
  MlpParams &c = ag->critic[i];
  adam(ag, c.p, c.m, c.v, c.g, c.total, 0, ag->target[i].p, (flags & 2) != 0, M_CGN + i, st, c.copies,
       &ag->target[i].copies);
}

// sums of squares of an (averaged) flat gradient that is already in place
void rereduce(gcrl_sac *ag, float *g, int total, cudaStream_t st) {
  ReduceArgs r{};
  r.nseg = 1;
  r.seg[0] = SegDesc{0, total, nullptr, 0, 0, 0};
  r.total = total; r.grad = g; r.sumsq_partials = ag->sumsq;
  r.metrics = ag->mdev; r.slot_loss = r.slot_td = r.slot_q = -1;
  launch_reduce_grads(r, st);
}

// ---- quantile critics: the launches around the loss kernels and the head's backward ----------------------------
// The loss of n critics of M atoms with K kept targets, on any buffers (the agent's and gcrl_quantile_critic_loss):
// target atoms zt -> y [B][ldy]; critic atoms z -> dZ in dz (same layout as z), the per-critic losses into
// out[slot_loss + i], the batch-mean TD into out[slot_td] and the per-row TD into td_rows (or nullptr).
// scratch: n * (B + ceil(B / rows)) floats, the TD parts [n][B] then the loss partials [n][nblk].
void quantile_critic_loss(const float *zt, const float *z, int64_t zstride, int ldm, int n, int M, int K,
                          const float *logp, const float *r, const float *d, const float *w, float gamma, float coef,
                          const float *alpha_dev, float *y, int ldy, float *dz, float *out, int slot_loss, int slot_td,
                          float *td_rows, float *scratch, int B, cudaStream_t st) {
  const int total = n * M;
  auto target = total <= 32 ? quantile_target_kernel<1>
              : total <= 64 ? quantile_target_kernel<2> : total <= 128 ? quantile_target_kernel<4> : quantile_target_kernel<8>;
  target<<<blocks_for(B, 8), 256, 0, st>>>(zt, zstride, ldm, n, M, K, logp, r, d, gamma, coef, alpha_dev, y, ldy, B);
  GCRL_LAUNCHED();
  const int rows = std::max(1, kQhThreads / M);
  const int nblk = (B + rows - 1) / rows;
  float *td_part = scratch, *loss_part = scratch + int64_t(n) * B;
  quantile_huber_kernel<<<dim3(nblk, n), kQhThreads, 0, st>>>(z, zstride, ldm, M, y, ldy, K, w, dz, loss_part, td_part,
                                                              B, rows);
  GCRL_LAUNCHED();
  quantile_metrics_kernel<<<1, 1024, 0, st>>>(loss_part, nblk, td_part, n, B, float(B) * float(M) * float(K), out,
                                              slot_loss, slot_td, td_rows);
  GCRL_LAUNCHED();
}

// target atoms in qt -> y; critic atoms in q -> dZ in dq, per-critic losses, td (and the prioritised TD rows)
void quantile_critic_loss(gcrl_sac *ag, int B, cudaStream_t st) {
  quantile_critic_loss(ag->qt, ag->q, ag->qstride, ag->ldm, ag->n, ag->nq, ag->nq_keep, ag->logp, ag->br, ag->bd,
                       ag->per_on ? ag->per_w : nullptr, ag->cfg.gamma, ag->cfg.entropy_coef, ag->alpha_state + 1,
                       ag->y, ag->ldy, ag->dq, ag->mdev, M_CLOSS, M_TD, ag->per_on ? ag->per_td : nullptr,
                       ag->qscratch, B, st);
}

// *out = mean over the batch of quantile_row_mean_kernel's row values of the atoms z (see there for logp / dz)
void quantile_row_mean(gcrl_sac *ag, const float *z, const float *logp, float *dz, float *out, int B, cudaStream_t st) {
  quantile_row_mean_kernel<<<blocks_for(B, 8), 256, 0, st>>>(z, ag->qstride, ag->ldm, ag->n, ag->nq, logp,
                                                             ag->cfg.entropy_coef, ag->alpha_state + 1, ag->qrow, dz,
                                                             -1.0f / (float(B) * float(ag->n * ag->nq)), B);
  GCRL_LAUNCHED();
  alpha_mean_kernel<<<1, 1024, 0, st>>>(ag->qrow, B, 0.f, out);
  GCRL_LAUNCHED();
}

// The H -> M head of critics first .. first + m - 1, from dZ [B][ldm] in dq: with wgrad, the weight-gradient partial
// slabs into each critic's partial set (pset_stride floats apart); always dX = dZ W (.) leaky'(h) into
// dz_out[j * dz_step].  Returns the weight gradient's number of batch slabs.
int quantile_head_bwd(gcrl_sac *ag, int first, int m, float *const *dz_out, bool wgrad, int64_t pset_stride, int B,
                      cudaStream_t st, int dz_step = 1) {
  const int L = ag->L;
  int splits = 0;
  if (wgrad) {
    WgradProblem wp[kMaxWgradProblems];
    for (int j = 0; j < m; ++j) {
      const MlpParams &c = ag->critic[first + j];
      float *part = ag->partials + j * pset_stride;
      wp[j] = WgradProblem{ag->dq + (first + j) * ag->qstride, ag->ldm, ag->ch[first + j][L - 1], ag->ldh,
                           part + c.w_off[L], c.ldw[L], part + c.b_off[L], ag->nq, ag->H};
    }
    splits = launch_multi_wgrad(wp, m, B, ag->slab, kSplits, st);
  }
  LinearDgradProblem dg[kMaxBatchedLinear];
  for (int j = 0; j < m; ++j) {
    const MlpParams &c = ag->critic[first + j];
    dg[j] = LinearDgradProblem{ag->dq + (first + j) * ag->qstride, ag->ldm, c.W(L), c.ldw[L], ag->ch[first + j][L - 1],
                               ag->ldh, dz_out[j * dz_step], ag->ldh};
  }
  launch_linear_dgrad_batched(dg, m, B, ag->nq, ag->H, st);
  return splits;
}

enum : int { PH_CGRAD = 1, PH_CSTEP = 2, PH_AGRAD = 4, PH_ASTEP = 8, PH_ALL = 15 };

// critic_update (SAC :548-639, TQC :951-1042).  mask PH_ALL: every critic is stepped right after its own
// backward; data-parallel: PH_CGRAD leaves the n flat gradients in critic_grads (all-reduced by the
// caller), PH_CSTEP clips and steps on the averaged gradients.
void critic_update(gcrl_sac *ag, int B, int flags, int mask, cudaStream_t st) {
  const int n = ag->n, L = ag->L, K0 = ag->D + ag->A;
  const bool tqc = ag->cfg.algo == GCRL_ALGO_TQC;
  const bool dp = mask != PH_ALL;
  if (mask & PH_CGRAD) {
  // next action and log-probability = actor.sample(next_state) in train mode (batch statistics; running statistics move)
  actor_fwd(ag, ag->nsa, ag->eps_next, B, true, false, nullptr, st);
  critics_fwd(ag, ag->target, ag->nsa, ag->qt, B, st);         // ch[i] as scratch: overwritten by the critic forward
  if (ag->nq > 0) {
    critics_fwd(ag, ag->critic, ag->sa, ag->q, B, st);
    quantile_critic_loss(ag, B, st);
  } else {
  sac_target_kernel<<<blocks_for(B, 256), 256, 0, st>>>(ag->qt, ag->maxB, n, ag->keep, ag->logp, ag->br, ag->bd,
                                                       ag->cfg.gamma, ag->cfg.entropy_coef, ag->alpha_state + 1,
                                                       ag->y, B);
  GCRL_LAUNCHED();
  critics_fwd(ag, ag->critic, ag->sa, ag->q, B, st);
  critic_metrics_kernel<<<1, 1024, 0, st>>>(ag->q, ag->maxB, n, ag->y, B, ag->mdev + M_CLOSS, 0,
                                            ag->per_on ? ag->per_w : nullptr, ag->per_on ? ag->per_td : nullptr);
  GCRL_LAUNCHED();
  }
  if (B <= kEnsembleBatchMax) {
    // the ensemble's backward passes share their launches: one head launch, one weight-gradient and one
    // input-gradient launch per layer (per-critic gradient buffers and partial sets), then reduce + AdamW per critic
    HeadBwdArgs hs[kMaxBatchedLinear];
    for (int i = 0; i < n; ++i) {
      const MlpParams &c = ag->critic[i];
      float *part = ag->partials + int64_t(i) * ag->pset;
      HeadBwdArgs h{};
      h.mode = 0; h.loss_kind = 0; h.clamp_y = 0; h.nout = 1;
      h.q = ag->q + int64_t(i) * ag->maxB; h.y_in = ag->y;
      if (ag->per_on) h.is_w = ag->per_w;
      h.Hact = ag->ch[i][L - 1]; h.ldh = ag->ldh;
      h.W = c.W(L); h.ldw = c.ldw[L];
      h.dZprev = ag->dzc[2 * i]; h.lddz = ag->ldh;
      h.pW = part + c.w_off[L]; h.w_split_stride = ag->slab;
      h.pB = part + c.b_off[L]; h.b_split_stride = ag->slab;
      h.metric_partials = part + ag->slab * kSplits;            // scratch tail, unused
      h.M = B; h.K = ag->H;
      hs[i] = h;
    }
    const int head_splits = ag->nq > 0 ? quantile_head_bwd(ag, 0, n, ag->dzc.data(), true, ag->pset, B, st, 2)
                                       : launch_head_bwd_batched(hs, n, kSplits, st);
    int splits[8] = {};
    int cur = 0;
    for (int l = L - 1; l >= 0; --l) {
      WgradProblem wp[kMaxWgradProblems];
      for (int i = 0; i < n; ++i) {
        const MlpParams &c = ag->critic[i];
        float *part = ag->partials + int64_t(i) * ag->pset;
        wp[i] = WgradProblem{ag->dzc[2 * i + cur], ag->ldh, l == 0 ? ag->sa : ag->ch[i][l - 1], l == 0 ? ag->ldc : ag->ldh,
                             part + c.w_off[l], c.ldw[l], part + c.b_off[l], ag->H, l == 0 ? K0 : ag->H};
      }
      if (ag->tc_update) {       // per critic: the slabs of one weight-gradient launch already fill the SMs
        for (int i = 0; i < n; ++i)
          splits[l] = linear_wgrad(ag, wp[i].dZ, wp[i].X, wp[i].ldx, wp[i].K, true, wp[i].pW, wp[i].ldw, wp[i].pB, B, st);
      } else {
        splits[l] = launch_multi_wgrad(wp, n, B, ag->slab, kSplits, st);
      }
      if (l > 0 && ag->tc_update) {
        float *din[kMaxBatchedLinear], *dout[kMaxBatchedLinear];
        for (int i = 0; i < n; ++i) { din[i] = ag->dzc[2 * i + cur]; dout[i] = ag->dzc[2 * i + (cur ^ 1)]; }
        critics_dgrad_tc(ag, 0, n, l, din, dout, B, st);
        cur ^= 1;
      } else if (l > 0) {
        LinearDgradProblem dg[kMaxBatchedLinear];
        for (int i = 0; i < n; ++i) {
          const MlpParams &c = ag->critic[i];
          dg[i] = LinearDgradProblem{ag->dzc[2 * i + cur], ag->ldh, c.W(l), c.ldw[l], ag->ch[i][l - 1], ag->ldh,
                                     ag->dzc[2 * i + (cur ^ 1)], ag->ldh};
        }
        launch_linear_dgrad_batched(dg, n, B, ag->H, ag->H, st);
        cur ^= 1;
      }
    }
    for (int i = 0; i < n; ++i) {
      MlpParams &c = ag->critic[i];
      reduce_critic(ag, c, splits, head_splits, st, ag->partials + int64_t(i) * ag->pset);
      if (!dp) adam_critic(ag, i, flags, st);
    }
  } else
  for (int i = 0; i < n; ++i) {
    MlpParams &c = ag->critic[i];
    HeadBwdArgs h{};
    h.mode = 0; h.loss_kind = 0; h.clamp_y = 0; h.nout = 1;
    h.q = ag->q + int64_t(i) * ag->maxB; h.y_in = ag->y;
    if (ag->per_on) h.is_w = ag->per_w;
    h.Hact = ag->ch[i][L - 1]; h.ldh = ag->ldh;
    h.W = c.W(L); h.ldw = c.ldw[L];
    h.dZprev = ag->dz[0]; h.lddz = ag->ldh;
    h.pW = ag->partials + c.w_off[L]; h.w_split_stride = ag->slab;
    h.pB = ag->partials + c.b_off[L]; h.b_split_stride = ag->slab;
    h.metric_partials = ag->partials + ag->slab * kSplits;      // scratch tail, unused
    h.M = B; h.K = ag->H;
    const int head_splits = ag->nq > 0 ? quantile_head_bwd(ag, i, 1, ag->dz, true, 0, B, st) : launch_head_bwd(h, kSplits, st);
    int splits[8] = {};
    int cur = 0;
    for (int l = L - 1; l >= 0; --l) {
      const float *xin = l == 0 ? ag->sa : ag->ch[i][l - 1];
      const int ldin = l == 0 ? ag->ldc : ag->ldh;
      const int K = l == 0 ? K0 : ag->H;
      splits[l] = linear_wgrad(ag, ag->dz[cur], xin, ldin, K, true, ag->partials + c.w_off[l], c.ldw[l],
                               ag->partials + c.b_off[l], B, st);
      if (l > 0) {
        if (ag->tc_update)
          critics_dgrad_tc(ag, i, 1, l, &ag->dz[cur], &ag->dz[cur ^ 1], B, st);
        else
          launch_linear_dgrad(ag->dz[cur], ag->ldh, c.W(l), c.ldw[l], ag->ch[i][l - 1], ag->ldh, ag->dz[cur ^ 1],
                              ag->ldh, B, ag->H, ag->H, st);
        cur ^= 1;
      }
    }
    reduce_critic(ag, c, splits, head_splits, st);
    if (!dp) adam_critic(ag, i, flags, st);
  }
  }
  if (ag->seg_build != nullptr) seg_cut(ag, COLL_AVG_CRITIC);
  if (dp && (mask & PH_CSTEP)) {
    for (int i = 0; i < n; ++i) {
      MlpParams &c = ag->critic[i];
      rereduce(ag, c.g, c.total, st);
      adam_critic(ag, i, flags, st);
    }
  }
  if (tqc && (mask & PH_CSTEP)) {   // logged Q = mean over the STEPPED critics (:1016-1019)
    critics_fwd(ag, ag->critic, ag->sa, ag->qt, B, st);        // the backward pass is done with ch[i]
    if (ag->nq > 0) {
      quantile_row_mean(ag, ag->qt, nullptr, nullptr, ag->mdev + M_Q, B, st);
      return;
    }
    critic_metrics_kernel<<<1, 1024, 0, st>>>(ag->qt, ag->maxB, n, nullptr, B, ag->mdev + M_CLOSS, 1, nullptr, nullptr);
    GCRL_LAUNCHED();
  }
}

// actor_update (SAC :513-530, TQC :912-934) + alpha_update (:532-546 / :936-949)
void actor_update(gcrl_sac *ag, int B, int flags, int mask, cudaStream_t st) {
  const int n = ag->n, L = ag->L, D = ag->D, A = ag->A;
  ActorNet &a = ag->actor;
  const bool dp = mask != PH_ALL;
  if (mask & PH_AGRAD) {
  actor_fwd(ag, ag->spi, ag->eps_cur, B, true, true, nullptr, st);
  critics_fwd(ag, ag->critic, ag->spi, ag->q, B, st);
  if (ag->nq > 0) {     // no truncation: loss mean_b(coef log pi - mean_ik Z_ik), every atom's gradient -1 / (B n M)
    quantile_row_mean(ag, ag->q, ag->logp, ag->dq, ag->mdev + M_ALOSS, B, st);
  } else {
  actor_trunc_kernel<<<1, 1024, 0, st>>>(ag->q, ag->maxB, n, ag->keep, ag->logp, ag->cfg.entropy_coef,
                                        ag->alpha_state + 1, ag->dq, ag->mdev + M_ALOSS, B);
  GCRL_LAUNCHED();
  }
  if (B <= kEnsembleBatchMax) {        // the ensemble's input-gradient chains share their launches
    HeadBwdArgs hs[kMaxBatchedLinear];
    for (int i = 0; i < n; ++i) {
      const MlpParams &c = ag->critic[i];
      HeadBwdArgs h{};
      h.mode = 2; h.nout = 1; h.dz_in = ag->dq + int64_t(i) * ag->maxB * 4;
      h.Hact = ag->ch[i][L - 1]; h.ldh = ag->ldh;
      h.W = c.W(L); h.ldw = c.ldw[L];
      h.dZprev = ag->dzc[2 * i]; h.lddz = ag->ldh;
      h.pW = nullptr; h.pB = nullptr;            // critic weight gradients are discarded
      h.M = B; h.K = ag->H;
      hs[i] = h;
    }
    if (ag->nq > 0) quantile_head_bwd(ag, 0, n, ag->dzc.data(), false, 0, B, st, 2);
    else launch_head_bwd_batched(hs, n, kSplits, st);
    int cur = 0;
    for (int l = L - 1; l >= 1; --l) {
      if (ag->tc_update) {
        float *din[kMaxBatchedLinear], *dout[kMaxBatchedLinear];
        for (int i = 0; i < n; ++i) { din[i] = ag->dzc[2 * i + cur]; dout[i] = ag->dzc[2 * i + (cur ^ 1)]; }
        critics_dgrad_tc(ag, 0, n, l, din, dout, B, st);
        cur ^= 1;
        continue;
      }
      LinearDgradProblem dg[kMaxBatchedLinear];
      for (int i = 0; i < n; ++i) {
        const MlpParams &c = ag->critic[i];
        dg[i] = LinearDgradProblem{ag->dzc[2 * i + cur], ag->ldh, c.W(l), c.ldw[l], ag->ch[i][l - 1], ag->ldh,
                                   ag->dzc[2 * i + (cur ^ 1)], ag->ldh};
      }
      launch_linear_dgrad_batched(dg, n, B, ag->H, ag->H, st);
      cur ^= 1;
    }
    for (int i = 0; i < n; ++i) {                // summed over the critics in index order
      const MlpParams &c = ag->critic[i];
      action_grad_acc_kernel<<<blocks_for(B, 8), 256, 0, st>>>(ag->dzc[2 * i + cur], ag->ldh, c.W(0), c.ldw[0], D,
                                                              ag->dact, B, ag->H, A, i > 0 ? 1 : 0);
      GCRL_LAUNCHED();
    }
  } else
  for (int i = 0; i < n; ++i) {
    const MlpParams &c = ag->critic[i];
    HeadBwdArgs h{};
    h.mode = 2; h.nout = 1; h.dz_in = ag->dq + int64_t(i) * ag->maxB * 4;
    h.Hact = ag->ch[i][L - 1]; h.ldh = ag->ldh;
    h.W = c.W(L); h.ldw = c.ldw[L];
    h.dZprev = ag->dz[0]; h.lddz = ag->ldh;
    h.pW = nullptr; h.pB = nullptr;              // critic weight gradients are discarded
    h.M = B; h.K = ag->H;
    if (ag->nq > 0) quantile_head_bwd(ag, i, 1, ag->dz, false, 0, B, st);
    else launch_head_bwd(h, kSplits, st);
    int cur = 0;
    for (int l = L - 1; l >= 1; --l) {
      if (ag->tc_update)
        critics_dgrad_tc(ag, i, 1, l, &ag->dz[cur], &ag->dz[cur ^ 1], B, st);
      else
        launch_linear_dgrad(ag->dz[cur], ag->ldh, c.W(l), c.ldw[l], ag->ch[i][l - 1], ag->ldh, ag->dz[cur ^ 1], ag->ldh,
                            B, ag->H, ag->H, st);
      cur ^= 1;
    }
    action_grad_acc_kernel<<<blocks_for(B, 8), 256, 0, st>>>(ag->dz[cur], ag->ldh, c.W(0), c.ldw[0], D, ag->dact, B,
                                                            ag->H, A, i > 0 ? 1 : 0);
    GCRL_LAUNCHED();
  }
  policy_bwd_kernel<<<blocks_for(int64_t(B) * 4, 256), 256, 0, st>>>(ag->dact, ag->act4, ag->std4, ag->gate4,
                                                                    ag->eps_cur, A, ag->cfg.entropy_coef,
                                                                    ag->alpha_state + 1, ag->dzh, B);
  GCRL_LAUNCHED();
  int rows = (B + kSplits - 1) / kSplits;
  rows = std::min(kHeadRows, std::max(rows, 16));
  const int head_slabs = (B + rows - 1) / rows;
  GCRL_REQUIRE(head_slabs <= kSplits, "batch too large for the policy-head partial buffers");
  policy_head_bwd_kernel<<<head_slabs, 256, 0, st>>>(ag->dzh, ag->ah[L - 1], ag->ldh, a.p + a.wm_off, a.p + a.ws_off,
                                                    ag->ldh, A, ag->dz[0], ag->ldh, ag->partials + a.wm_off,
                                                    ag->partials + a.bm_off, ag->partials + a.ws_off,
                                                    ag->partials + a.bs_off, ag->slab, B, ag->H, rows);
  GCRL_LAUNCHED();
  int splits[8] = {};
  int cur = 0;
  for (int l = L - 1; l >= 0; --l) {
    if (ag->sync_world > 0) {
      GCRL_REQUIRE(ag->seg_build != nullptr, "a sync-BN agent trains through gcrl_sac_update_segment only");
      bn_bwd_stats_kernel<<<(ag->H + 31) / 32, dim3(32, 32), 0, st>>>(
          ag->dz[cur], ag->ah[l], ag->xhat[l], ag->ldh, B, ag->H, ag->bn_gather + size_t(ag->sync_rank) * 2 * ag->ldh,
          ag->ldh);
      GCRL_LAUNCHED();
      seg_cut(ag, COLL_GATHER_BN);
      bn_bwd_sync_kernel<<<(ag->H + 31) / 32, dim3(32, 32), 0, st>>>(
          ag->dz[cur], ag->ah[l], ag->xhat[l], ag->ldh, B, ag->H, a.p + a.gam_off[l], ag->invstd + size_t(l) * ag->ldh,
          a.g + a.gam_off[l], a.g + a.bet_off[l], ag->bn_gather, ag->sync_world, ag->sync_rank, ag->ldh);
      GCRL_LAUNCHED();
    } else {
      bn_bwd_kernel<<<(ag->H + 31) / 32, dim3(32, 32), 0, st>>>(ag->dz[cur], ag->ah[l], ag->xhat[l], ag->ldh, B, ag->H,
                                                                a.p + a.gam_off[l], ag->invstd + size_t(l) * ag->ldh,
                                                                a.g + a.gam_off[l], a.g + a.bet_off[l]);
      GCRL_LAUNCHED();
    }
    const float *xin = l == 0 ? ag->spi : ag->ah[l - 1];
    const int ldin = l == 0 ? ag->ldc : ag->ldh;
    const int K = l == 0 ? D : ag->H;
    // layer 0 on the tensor cores only when K needs no padding: the columns D.. of spi hold the sampled action now
    splits[l] = linear_wgrad(ag, ag->dz[cur], xin, ldin, K, l > 0 || D % 4 == 0, ag->partials + a.w_off[l], a.ldw[l],
                             ag->partials + a.b_off[l], B, st);
    if (l > 0) {
      if (ag->tc_update)      // bare product: bn_bwd applies ReLU' itself
        launch_tc_dense(ag->dz[cur], ag->ldh, a.copies.pT_hi + a.copies.t_off[l], a.copies.ldt[l], nullptr, nullptr, 0,
                        ag->dz[cur ^ 1], ag->ldh, B, ag->H, ag->H, 3, st, a.copies.pT_lo + a.copies.t_off[l]);
      else
        launch_linear_dgrad(ag->dz[cur], ag->ldh, a.p + a.w_off[l], a.ldw[l], nullptr, 0, ag->dz[cur ^ 1], ag->ldh, B,
                            ag->H, ag->H, st);
      cur ^= 1;
    }
  }
  ReduceArgs r{};
  for (int l = 0; l < L; ++l) {
    r.seg[r.nseg++] = SegDesc{a.w_off[l], ag->H * a.ldw[l], ag->partials, splits[l], ag->slab, a.w_off[l]};
    r.seg[r.nseg++] = SegDesc{a.b_off[l], ag->H, ag->partials, splits[l], ag->slab, a.b_off[l]};
    r.seg[r.nseg++] = SegDesc{a.gam_off[l], ag->H, nullptr, 0, 0, 0};     // written by bn_bwd, already reduced
    r.seg[r.nseg++] = SegDesc{a.bet_off[l], ag->H, nullptr, 0, 0, 0};
  }
  r.seg[r.nseg++] = SegDesc{a.wm_off, A * ag->ldh, ag->partials, head_slabs, ag->slab, a.wm_off};
  r.seg[r.nseg++] = SegDesc{a.bm_off, A, ag->partials, head_slabs, ag->slab, a.bm_off};
  r.seg[r.nseg++] = SegDesc{a.ws_off, A * ag->ldh, ag->partials, head_slabs, ag->slab, a.ws_off};
  r.seg[r.nseg++] = SegDesc{a.bs_off, A, ag->partials, head_slabs, ag->slab, a.bs_off};
  r.total = a.total; r.grad = a.g; r.sumsq_partials = ag->sumsq;
  r.metrics = ag->mdev; r.slot_loss = r.slot_td = r.slot_q = -1;
  launch_reduce_grads(r, st);
  if (flags & 4) {
    alpha_mean_kernel<<<1, 1024, 0, st>>>(ag->logp, B, ag->cfg.target_entropy, a.g + a.total);
    GCRL_LAUNCHED();
  }
  }
  if (ag->seg_build != nullptr) seg_cut(ag, COLL_AVG_ACTOR);
  if (mask & PH_ASTEP) {
    if (dp) rereduce(ag, a.g, a.total, st);
    adam(ag, a.p, a.m, a.v, a.g, a.total, 1, nullptr, false, M_AGN, st, a.copies, nullptr);
    if (flags & 4) {
      alpha_step_kernel<<<1, 1, 0, st>>>(a.g + a.total, reinterpret_cast<const float *>(ag->d_scalars + 1),
                                        ag->alpha_state, ag->mdev + M_ALPHA_LOSS);
      GCRL_LAUNCHED();
    } else {
      GCRL_CUDA(cudaMemsetAsync(ag->mdev + M_ALPHA_LOSS, 0, 4, st));
    }
  }
}

void read_metrics(gcrl_sac *ag, int flags, float *metrics_host, cudaStream_t st);

void run_body(gcrl_sac *ag, int B, int flags, int mask, cudaStream_t st) {
  if (mask & (PH_CGRAD | PH_CSTEP)) critic_update(ag, B, flags, mask == PH_ALL ? PH_ALL : (mask & (PH_CGRAD | PH_CSTEP)), st);
  if ((mask & (PH_AGRAD | PH_ASTEP)) && (flags & 1))
    actor_update(ag, B, flags, mask == PH_ALL ? PH_ALL : (mask & (PH_AGRAD | PH_ASTEP)), st);
}

// the engine an update at this batch runs on; the tensor-core one needs the split weight copies current
void select_engine(gcrl_sac *ag, int B, cudaStream_t st) {
  ag->tc_update = engine_tc(ag, B);
  if (ag->tc_update) ensure_split(ag, st);          // (the update itself re-splits what it steps)
  else mark_split_stale(ag);                        // weights move without their split copies following
}

// Replay (or capture on first use) the CUDA graph of (B, flags, phase mask): ~170 launches per TQC update
// become one graph launch; everything that varies per step travels through device scalars.
void run_phases(gcrl_sac *ag, int B, int flags, int mask, cudaStream_t st) {
  // (a graph captured before gcrl_sac_set_sync_bn would otherwise replay with local statistics)
  GCRL_REQUIRE(ag->sync_world == 0, "a sync-BN agent trains through gcrl_sac_update_segment only");
  ag->per_on = (flags & 8) != 0;
  if (!ag->use_graphs) {
    run_body(ag, B, flags, mask, st);
    return;
  }
  const auto key = std::make_tuple(B, flags, mask);
  auto it = ag->graphs.find(key);
  if (it == ag->graphs.end())
    it = ag->graphs.emplace(key, capture_graph(ag->cap_stream, [&](cudaStream_t cs) { run_body(ag, B, flags, mask, cs); })).first;
  launch_graph(it->second, st);
}

// ---- n updates in one graph (gcrl_sac_update_many) -------------------------------------------------------------
size_t many_bytes(const gcrl_sac *ag, int n, int64_t B) {
  return size_t(n) * (kManyScalBytes + size_t(B) * (sizeof(int64_t) + 2 * ag->A * sizeof(float) + sizeof(float)) +
                      kMetricFloats * sizeof(float));
}
char *many_scalars(const gcrl_sac *ag, int i) { return ag->many.d + size_t(i) * kManyScalBytes; }
int64_t *many_positions(const gcrl_sac *ag, int n, int64_t B, int i) {
  return reinterpret_cast<int64_t *>(ag->many.d + size_t(n) * kManyScalBytes) + size_t(i) * B;
}
float *many_eps(const gcrl_sac *ag, int n, int64_t B, int which /*0 next, 1 cur*/) {
  return reinterpret_cast<float *>(many_positions(ag, n, B, n)) + size_t(which) * n * B * ag->A;
}
float *many_metrics(const gcrl_sac *ag, int n, int64_t B, int i) {
  return many_eps(ag, n, B, 2) + size_t(i) * kMetricFloats;
}
float *many_td(const gcrl_sac *ag, int n, int64_t B, int i) { return many_metrics(ag, n, B, n) + size_t(i) * B; }

// While update i of an n-update call is recorded (or issued eagerly), the agent's per-update inputs -- AdamW and
// alpha scalars, rsample noise -- point at slot i, so every argument builder of critic_update / actor_update picks
// the slot up; the sampler reads the slot's totals and positions.
struct ManySlot {
  gcrl_sac *ag;
  StepScalars *sc; float *en, *ec;
  const SampleScalars *ssc; const int64_t *idx; float *metrics;
  float *td;
  ManySlot(gcrl_sac *a, int i, int n, int B)
      : ag(a), sc(a->d_scalars), en(a->eps_next), ec(a->eps_cur),
        ssc(reinterpret_cast<const SampleScalars *>(many_scalars(a, i) + 2 * sizeof(StepScalars))),
        idx(many_positions(a, n, B, i)), metrics(many_metrics(a, n, B, i)), td(many_td(a, n, B, i)) {
    a->d_scalars = reinterpret_cast<StepScalars *>(many_scalars(a, i));
    a->eps_next = many_eps(a, n, B, 0) + size_t(i) * B * a->A;
    a->eps_cur = many_eps(a, n, B, 1) + size_t(i) * B * a->A;
  }
  ~ManySlot() { ag->d_scalars = sc; ag->eps_next = en; ag->eps_cur = ec; }
  ManySlot(const ManySlot &) = delete;
  ManySlot &operator=(const ManySlot &) = delete;
};

// n updates back to back from the HER buffer `her` or the uniform / prioritised buffer `rb` (the other is NULL): the
// slot's draw, operand rows, the update, then -- prioritised -- the priority write-back and the TD errors into the
// slot's row, and the metrics and alpha state into the slot's row (copy nodes, not launches)
void run_many_body(gcrl_sac *ag, gcrl_her *her, gcrl_replay *rb, int B, int n, const int *flags, cudaStream_t st) {
  for (int i = 0; i < n; ++i) {
    ManySlot slot(ag, i, n, B);
    if (rb != nullptr)
      replay_many_sample(rb, B, n, i, ag->bs, ag->ba, ag->br0, ag->bns, ag->bd0, ag->per_w, st);
    else
      her_sample_graphed(her, B, slot.ssc, slot.idx, ag->bs, ag->ba, ag->br0, ag->bns, ag->bd0, st);
    launch_ingest_batch(ag->bs, ag->ba, ag->br0, ag->bns, ag->bd0, ag->D, ag->A, B, ag->sa, ag->nsa, ag->spi, ag->ldc,
                        ag->br, ag->bd, st);
    run_body(ag, B, flags[i], PH_ALL, st);
    if (ag->per_on) {
      replay_many_write_back(rb, B, ag->per_td, st);
      GCRL_CUDA(cudaMemcpyAsync(slot.td, ag->per_td, size_t(B) * sizeof(float), cudaMemcpyDeviceToDevice, st));
    }
    GCRL_CUDA(cudaMemcpyAsync(slot.metrics, ag->mdev, kMetricFloats * sizeof(float), cudaMemcpyDeviceToDevice, st));
  }
}

// A prioritised call is captured when its key repeats only (see ManyGraphs::launch); a HER buffer has 0 for the
// key's epoch and length.
void run_many(gcrl_sac *ag, gcrl_her *her, gcrl_replay *rb, int B, int n, const int *flags, cudaStream_t st) {
  select_engine(ag, B, st);
  ag->per_on = rb != nullptr && replay_prioritized(rb);
  const uintptr_t buf = rb != nullptr ? reinterpret_cast<uintptr_t>(rb) : reinterpret_cast<uintptr_t>(her);
  ag->many.graphs.launch({int64_t(B), std::vector<int>(flags, flags + n), buf, ag->tc_update ? 1 : 0,
                          rb != nullptr ? replay_epoch(rb) : 0, ag->per_on ? replay_many_n(rb) : 0},
                         !ag->per_on, [&](cudaStream_t cs) { run_many_body(ag, her, rb, B, n, flags, cs); }, st,
                         ag->use_graphs, ag->cap_stream);
}

// Segmented update (sync-BN): the body is captured ONCE per (B, flags) as a chain of graphs, cut wherever a
// collective has to run (BatchNorm statistics, the two gradient averages); segment `seg` replays graph `seg` and
// reports the collective the caller owes before the next one.
constexpr int PH_SEGMENTED = PH_ALL | 16;          // all four phases, data-parallel form (mask != PH_ALL)

int run_segment(gcrl_sac *ag, int B, int flags, int seg, cudaStream_t st) {
  GCRL_REQUIRE(ag->use_graphs, "sync-BN needs CUDA graphs (unset GCRL_B200_NO_GRAPH)");
  ag->per_on = (flags & 8) != 0;
  const auto key = std::make_tuple(B, flags);
  auto it = ag->seg_graphs.find(key);
  if (it == ag->seg_graphs.end()) {
    std::vector<gcrl_sac::SegRec> segs;
    ag->seg_build = &segs;
    ag->seg_mark = launch_counter();
    begin_capture(ag->cap_stream);
    try {
      run_body(ag, B, flags, PH_SEGMENTED, ag->cap_stream);
      seg_cut(ag, COLL_DONE, true);
    } catch (...) {
      abort_capture(ag->cap_stream);
      for (auto &r : segs) cudaGraphExecDestroy(r.graph.exec);
      ag->seg_build = nullptr;
      count_launch(ag->seg_mark - launch_counter());     // what the open segment recorded (each cut took its own)
      throw;
    }
    ag->seg_build = nullptr;
    it = ag->seg_graphs.emplace(key, std::move(segs)).first;
  }
  GCRL_REQUIRE(seg >= 0 && seg < int(it->second.size()), "segment index past the end of the update");
  const auto &r = it->second[size_t(seg)];
  launch_graph(r.graph, st);
  return r.collective;
}

// The next update's AdamW step counters -> sc[0] (critic / actor scalars) and the first 4 floats of sc[1] (alpha's)
void fill_scalars(gcrl_sac *ag, double lr_c, double lr_a, int flags, StepScalars *sc) {
  auto fill = [&](int t, double lr, float *out) {
    out[0] = float(lr / (1.0 - std::pow(0.9, double(t))));
    out[1] = float(std::sqrt(1.0 - std::pow(0.999, double(t))));
    out[2] = float(1.0 - lr * double(ag->cfg.weight_decay));
    out[3] = 0.f;
  };
  ag->adam_t_c += 1;
  fill(ag->adam_t_c, lr_c, &sc->step_size_c);
  if (flags & 1) ag->adam_t_a += 1;
  fill(std::max(1, ag->adam_t_a), lr_a, &sc->step_size_a);
  float *al = reinterpret_cast<float *>(sc + 1);
  al[0] = 0.f; al[1] = 1.f; al[2] = 1.f; al[3] = 0.f;
  if ((flags & 1) && (flags & 4)) {
    ag->adam_t_alpha += 1;
    fill(ag->adam_t_alpha, double(ag->cfg.alpha_lr), al);
  }
}

// The step counters advance in fill_scalars, before the update is enqueued; unless commit() is reached they are
// put back (and, after keep_draws, the device index-stream epoch of the sampled buffer with them).
struct StepCounterGuard {
  gcrl_sac *ag;
  int t_c, t_a, t_al;
  gcrl_her *buf = nullptr;
  unsigned long long draw_epoch = 0;
  bool done = false;
  explicit StepCounterGuard(gcrl_sac *a) : ag(a), t_c(a->adam_t_c), t_a(a->adam_t_a), t_al(a->adam_t_alpha) {}
  void keep_draws(gcrl_her *b) { buf = b; draw_epoch = her_draw_epoch(b); }
  void commit() { done = true; }
  ~StepCounterGuard() {
    if (done) return;
    ag->adam_t_c = t_c; ag->adam_t_a = t_a; ag->adam_t_alpha = t_al;
    if (buf != nullptr) her_draw_epoch(buf) = draw_epoch;
  }
  StepCounterGuard(const StepCounterGuard &) = delete;
  StepCounterGuard &operator=(const StepCounterGuard &) = delete;
};

// phase < 0: the whole update.  phase 0..3: the data-parallel cut (critic grads | critic steps | actor grads |
// actor step), the caller averaging critic_grads / the actor gradient across ranks in between.
void sac_update(gcrl_sac *ag, int phase, gcrl_her *buf, int64_t B64, const int64_t *idx_host, const float *s,
                const float *a, const float *r, const float *ns, const float *d, const float *eps_next,
                const float *eps_cur, double lr_c, double lr_a, int flags, float *metrics_host, cudaStream_t st,
                int seg = -1, int *collective = nullptr) {
  GCRL_REQUIRE(ag != nullptr, "agent handle is NULL");
  GCRL_REQUIRE(B64 >= 2 && B64 <= ag->maxB, "batch size outside [2, max_batch] (BatchNorm needs > 1 row)");
  const int B = int(B64);
  select_engine(ag, B, st);
  if (seg > 0) {
    GCRL_REQUIRE(ag->dp_B == B && ag->dp_flags == flags, "segment > 0 must follow segment 0 of the same update");
    *collective = run_segment(ag, B, flags, seg, st);
    return;
  }
  if (phase > 0) {
    GCRL_REQUIRE(ag->dp_B == B && ag->dp_flags == flags, "phase 1..3 must follow phase 0 of the same update");
    run_phases(ag, B, flags, phase == 1 ? PH_CSTEP : (phase == 2 ? PH_AGRAD : PH_ASTEP), st);
    if (phase == 3) ag->dp_open = false;
    return;
  }
  GCRL_REQUIRE(eps_next != nullptr && (eps_cur != nullptr || !(flags & 1)), "NULL rsample noise tensor");
  if (buf != nullptr) {
    GCRL_REQUIRE(her_state_dim(buf) == ag->D && her_act_dim(buf) == ag->A, "buffer / agent shape mismatch");
    GCRL_REQUIRE(her_device(buf) == ag->device, "buffer and agent live on different devices");
    her_sample_into(buf, B, idx_host, ag->bs, ag->ba, ag->br0, ag->bns, ag->bd0, nullptr, st);
    s = ag->bs; a = ag->ba; r = ag->br0; ns = ag->bns; d = ag->bd0;
  } else {
    GCRL_REQUIRE(s && a && r && ns && d, "NULL batch pointer");
  }
  launch_ingest_batch(s, a, r, ns, d, ag->D, ag->A, B, ag->sa, ag->nsa, ag->spi, ag->ldc, ag->br, ag->bd, st);
  GCRL_CUDA(cudaMemcpyAsync(ag->eps_next, eps_next, size_t(B) * ag->A * 4, cudaMemcpyDeviceToDevice, st));
  if (flags & 1)
    GCRL_CUDA(cudaMemcpyAsync(ag->eps_cur, eps_cur, size_t(B) * ag->A * 4, cudaMemcpyDeviceToDevice, st));
  // the step counters move only if the update is issued: a throw below (capture, CUDA error, a misuse check)
  // must not leave the bias corrections one step ahead of the Python schedulers
  StepCounterGuard guard(ag);
  int slot;
  auto *sc = reinterpret_cast<StepScalars *>(ag->scal_stage.acquire(2 * sizeof(StepScalars), &slot));
  fill_scalars(ag, lr_c, lr_a, flags, sc);
  GCRL_CUDA(cudaMemcpyAsync(ag->d_scalars, sc, sizeof(StepScalars) + 16, cudaMemcpyHostToDevice, st));
  ag->scal_stage.release(slot, st);
  if (seg == 0) {
    ag->dp_B = B; ag->dp_flags = flags;
    *collective = run_segment(ag, B, flags, 0, st);
    guard.commit();
    return;
  }
  if (phase == 0) {
    ag->dp_B = B; ag->dp_flags = flags;
    run_phases(ag, B, flags, PH_CGRAD, st);
    ag->dp_open = true;
    guard.commit();
    return;
  }
  run_phases(ag, B, flags, PH_ALL, st);
  read_metrics(ag, flags, metrics_host, st);
  guard.commit();
}

// the 12 floats an update returns (include/gcrl_b200.h), from its device metrics block hm[32] and alpha state hs[4]
void metrics_tuple(const gcrl_sac *ag, int flags, const float *hm, const float *hs, float *metrics_host) {
  const int n = ag->n;
  if (ag->cfg.algo == GCRL_ALGO_SAC) {
    metrics_host[0] = hm[M_CLOSS]; metrics_host[1] = hm[M_CLOSS + 1];
    metrics_host[5] = hm[M_CGN]; metrics_host[6] = hm[M_CGN + 1];
  } else {                                   // np.mean over the per-critic Python floats (:1013-1014)
    double sl = 0.0, sg = 0.0;
    for (int i = 0; i < n; ++i) { sl += double(hm[M_CLOSS + i]); sg += double(hm[M_CGN + i]); }
    metrics_host[0] = metrics_host[1] = float(sl / n);
    metrics_host[5] = metrics_host[6] = float(sg / n);
  }
  metrics_host[2] = (flags & 1) ? hm[M_ALOSS] : 0.f;
  metrics_host[3] = hm[M_TD];
  metrics_host[4] = hm[M_Q];
  metrics_host[7] = (flags & 1) ? hm[M_AGN] : 0.f;
  metrics_host[8] = (flags & 1) ? hm[M_ALPHA_LOSS] : 0.f;
  metrics_host[9] = hs[1];
  metrics_host[10] = hs[0];
  metrics_host[11] = 0.f;
}

void read_metrics(gcrl_sac *ag, int flags, float *metrics_host, cudaStream_t st) {
  if (metrics_host != nullptr) {
    float hm[32], hs[4];
    GCRL_CUDA(cudaMemcpyAsync(hm, ag->mdev, sizeof(hm), cudaMemcpyDeviceToHost, st));
    GCRL_CUDA(cudaMemcpyAsync(hs, ag->alpha_state, sizeof(hs), cudaMemcpyDeviceToHost, st));
    GCRL_CUDA(cudaStreamSynchronize(st));
    metrics_tuple(ag, flags, hm, hs, metrics_host);
  }
}

// the per-update slots of an n-update call laid out for (n, B)
void ensure_many(gcrl_sac *ag, int n, int64_t B) {
  auto &mn = ag->many;
  const size_t need = many_bytes(ag, n, B);
  if (need <= mn.cap) return;
  mn.graphs.clear();   // cudaFree waits for replays still reading them
  if (mn.d) GCRL_CUDA(cudaFree(mn.d));
  mn.d = nullptr;
  mn.cap = 0;
  mn.d = dev_alloc<char>(need);
  mn.cap = need;
}

// The metric rows [n][36] and, when td_host is given, the TD rows [n][B] that follow them: ONE read-back per call;
// to pageable memory the copy returns once it (and the updates before it) completed
void read_many_rows(gcrl_sac *ag, int n, int64_t B, const int *flags, float *metrics_host, float *td_host,
                    cudaStream_t st) {
  if (metrics_host == nullptr && td_host == nullptr) return;
  const size_t m = size_t(n) * kMetricFloats;
  std::vector<float> rows(m + (td_host != nullptr ? size_t(n) * B : 0));
  GCRL_CUDA(cudaMemcpyAsync(rows.data(), many_metrics(ag, n, B, 0), rows.size() * sizeof(float), cudaMemcpyDeviceToHost,
                            st));
  if (metrics_host != nullptr)
    for (int i = 0; i < n; ++i) {
      const float *r = rows.data() + size_t(i) * kMetricFloats;
      metrics_tuple(ag, flags[i], r, r + 32, metrics_host + size_t(i) * 12);
    }
  if (td_host != nullptr) std::memcpy(td_host, rows.data() + m, size_t(n) * B * sizeof(float));
}


// (rows, cols, ld, weight offset, bias offset) of actor Linear `layer`
void actor_linear_geom(const gcrl_sac *ag, int layer, int *rows, int *cols, int *ld, int *woff, int *boff) {
  const ActorNet &a = ag->actor;
  GCRL_REQUIRE(layer >= 0 && layer <= ag->L + 1, "bad actor layer index");
  if (layer < ag->L) {
    *rows = ag->H; *cols = layer == 0 ? ag->D : ag->H; *ld = a.ldw[layer]; *woff = a.w_off[layer]; *boff = a.b_off[layer];
  } else {
    *rows = ag->A; *cols = ag->H; *ld = ag->ldh;
    *woff = layer == ag->L ? a.wm_off : a.ws_off;
    *boff = layer == ag->L ? a.bm_off : a.bs_off;
  }
}

}  // namespace

// Every entry point checks the handle's type tag: a gcrl_sac handle passed to the other family's functions would be
// reinterpreted as a different struct (garbage shapes and pointers).
static inline void require_handle(const gcrl_sac *h) {
  if (h == nullptr) throw ::gcrl::Error(GCRL_ERR_INVALID, "handle is NULL");
  if (h->magic != 0x54434153u) throw ::gcrl::Error(GCRL_ERR_INVALID, "handle is not a SAC / TQC agent (gcrl_sac_create)");
}

// gcrl_sac_update_many (HER buffer `her`) and gcrl_sac_update_many_replay (uniform / prioritised buffer `rb`): one of
// the two is NULL.  Nothing moves before the last refusal: the buffer's own checks (replay_many_stage) come first.
static void update_many(gcrl_sac *ag, gcrl_her *her, gcrl_replay *rb, int64_t B, int n, const int *flags,
                        const int64_t *idx_host, const int64_t *pos_host, const double *u_host, const double *beta,
                        const float *eps_next_dev, const float *eps_cur_dev, const double *lr_critic,
                        const double *lr_actor, float *metrics_host, float *td_host, void *stream) {
  require_handle(ag);
  GCRL_REQUIRE(her != nullptr || rb != nullptr, "buffer handle is NULL");
  GCRL_REQUIRE(B >= 2 && B <= ag->maxB, "batch size outside [2, max_batch] (BatchNorm needs > 1 row)");
  GCRL_REQUIRE(n >= 1 && n <= GCRL_MAX_MANY_STEPS, "n must be in [1, GCRL_MAX_MANY_STEPS]");
  GCRL_REQUIRE(flags != nullptr && lr_critic != nullptr && lr_actor != nullptr, "NULL flags / learning rates");
  const bool per = rb != nullptr && replay_prioritized(rb);
  bool any_actor = false;
  for (int i = 0; i < n; ++i) {
    if (her != nullptr) {
      GCRL_REQUIRE((flags[i] & ~7) == 0, "flags of an n-update call may hold bits 0-2 only");
    } else {
      GCRL_REQUIRE((flags[i] & ~15) == 0, "flags of an n-update call from a replay buffer may hold bits 0-3 only");
      GCRL_REQUIRE(((flags[i] & 8) != 0) == per, "flags bit3 must be set exactly when the buffer is prioritised");
    }
    any_actor = any_actor || (flags[i] & 1) != 0;
  }
  GCRL_REQUIRE(eps_next_dev != nullptr && (eps_cur_dev != nullptr || !any_actor), "NULL rsample noise tensor");
  GCRL_REQUIRE(ag->sync_world == 0, "a sync-BN agent trains through gcrl_sac_update_segment only");
  GCRL_REQUIRE(!ag->dp_open, "a phase-wise data-parallel update is open (phase 3 not issued)");
  if (her != nullptr) {
    GCRL_REQUIRE(her_state_dim(her) == ag->D && her_act_dim(her) == ag->A, "buffer / agent shape mismatch");
    GCRL_REQUIRE(her_device(her) == ag->device, "buffer and agent live on different devices");
    const int64_t len = her_len(her);
    if (len < B) throw Error(GCRL_ERR_UNDERFILLED, "[ERROR] Not enough in buffer to sample");
    if (idx_host != nullptr)
      for (int64_t i = 0; i < int64_t(n) * B; ++i)
        if (idx_host[i] < 0 || idx_host[i] >= len) throw Error(GCRL_ERR_INVALID, "sample index out of range [0, len)");
  } else {
    GCRL_REQUIRE(replay_state_dim(rb) == ag->D && replay_act_dim(rb) == ag->A, "buffer / agent shape mismatch");
    GCRL_REQUIRE(replay_device(rb) == ag->device, "buffer and agent live on different devices");
  }
  GCRL_CUDA(cudaSetDevice(ag->device));
  cudaStream_t st = as_stream(stream);
  if (rb != nullptr) replay_many_stage(rb, B, n, pos_host, u_host, beta, st);
  ensure_many(ag, n, B);
  StepCounterGuard guard(ag);
  if (her != nullptr) guard.keep_draws(her);
  // every update's scalars (HER: the device stream's draw epochs in order), then every update's positions: ONE copy
  const size_t scal = size_t(n) * kManyScalBytes, pos = idx_host != nullptr ? size_t(n) * B * sizeof(int64_t) : 0;
  int slot;
  char *p = ag->io_stage.acquire(scal + pos, &slot);
  for (int i = 0; i < n; ++i) {
    char *s = p + size_t(i) * kManyScalBytes;
    fill_scalars(ag, lr_critic[i], lr_actor[i], flags[i], reinterpret_cast<StepScalars *>(s));
    const SampleScalars ss = her != nullptr ? her_next_scalars(her, idx_host != nullptr) : SampleScalars{};
    std::memcpy(s + 2 * sizeof(StepScalars), &ss, sizeof(SampleScalars));
  }
  if (pos) std::memcpy(p + scal, idx_host, pos);
  GCRL_CUDA(cudaMemcpyAsync(ag->many.d, p, scal + pos, cudaMemcpyHostToDevice, st));
  ag->io_stage.release(slot, st);
  // stable addresses for the captured graph
  const size_t noise = size_t(n) * B * ag->A * sizeof(float);
  GCRL_CUDA(cudaMemcpyAsync(many_eps(ag, n, B, 0), eps_next_dev, noise, cudaMemcpyDeviceToDevice, st));
  if (any_actor) GCRL_CUDA(cudaMemcpyAsync(many_eps(ag, n, B, 1), eps_cur_dev, noise, cudaMemcpyDeviceToDevice, st));
  run_many(ag, her, rb, int(B), n, flags, st);
  guard.commit();
  read_many_rows(ag, n, B, flags, metrics_host, per ? td_host : nullptr, st);
}

// gcrl_sac_create (nq == 0: scalar critics) and gcrl_sac_create_quantile (nq atoms per critic, nq_drop dropped)
static void sac_create(gcrl_sac **out, int device, const gcrl_sac_config *cfg, int nq, int nq_drop) {
  GCRL_REQUIRE(out != nullptr && cfg != nullptr, "NULL argument");
  GCRL_REQUIRE(cfg->algo == GCRL_ALGO_SAC || cfg->algo == GCRL_ALGO_TQC, "unknown algo");
  GCRL_REQUIRE(cfg->state_dim >= 1 && cfg->act_dim >= 1 && cfg->act_dim <= 4, "need state_dim >= 1 and 1 <= act_dim <= 4");
  GCRL_REQUIRE(cfg->hidden_dim >= 1 && cfg->hidden_dim <= 4096, "hidden_dim outside [1, 4096]");
  GCRL_REQUIRE(cfg->layer_count >= 1 && cfg->layer_count <= 6, "layer_count outside [1, 6]");
  GCRL_REQUIRE(cfg->n_critics >= 1 && cfg->n_critics <= kMaxCritics, "n_critics outside [1, 8]");
  if (nq == 0) {
    GCRL_REQUIRE(cfg->drop_top >= 0 && cfg->drop_top < cfg->n_critics, "drop_top outside [0, n_critics)");
  } else {
    GCRL_REQUIRE(cfg->algo == GCRL_ALGO_TQC, "quantile critics need algo GCRL_ALGO_TQC");
    GCRL_REQUIRE(nq >= 1 && nq_drop >= 0 && nq_drop < nq,
                 "quantile critics need n_quantiles >= 1 and 0 <= drop_per_net < n_quantiles");
    GCRL_REQUIRE(cfg->n_critics * nq <= 256, "quantile critics need n_critics * n_quantiles <= 256");
  }
  GCRL_REQUIRE(cfg->max_batch >= 2 && cfg->max_batch <= kSplits * 256, "max_batch outside [2, 32768]");
  GCRL_REQUIRE(cfg->precision >= 0 && cfg->precision <= 2, "precision must be 0 (fp32 FFMA), 1 (tensor cores for large batches) or 2 (tensor cores whenever supported)");
  GCRL_CUDA(cudaSetDevice(device));
  auto *ag = new gcrl_sac();
  try {
    ag->device = device; ag->cfg = *cfg;
    ag->D = cfg->state_dim; ag->A = cfg->act_dim; ag->H = cfg->hidden_dim; ag->L = cfg->layer_count;
    ag->n = cfg->n_critics; ag->keep = cfg->n_critics - cfg->drop_top;
    ag->ldh = pad4(ag->H); ag->ldc = pad4(ag->D + ag->A); ag->maxB = cfg->max_batch;
    ag->nq = nq; ag->nq_drop = nq_drop; ag->nq_keep = cfg->n_critics * (nq - nq_drop);
    ag->ldm = pad4(nq); ag->ldy = pad4(ag->nq_keep);
    ag->qstride = nq > 0 ? ag->maxB * ag->ldm : ag->maxB;
    GCRL_REQUIRE(4 * ag->L + 4 <= kMaxSegs, "layer_count too large for the reduction descriptor");
    const int D = ag->D, A = ag->A, H = ag->H, L = ag->L, n = ag->n;
    const size_t mb = size_t(ag->maxB), act = mb * ag->ldh;
    ag->actor.init(D, H, A, L);
    const int nout = nq > 0 ? nq : 1;
    for (int i = 0; i < n; ++i) { ag->critic[i].layout(D + A, H, nout, L); ag->target[i].layout(D + A, H, nout, L); }
    ag->critic_stride = ag->critic[0].total;
    ag->critic_grads = dev_alloc<float>(size_t(n) * ag->critic_stride);
    GCRL_CUDA(cudaMemset(ag->critic_grads, 0, size_t(n) * ag->critic_stride * 4));
    for (int i = 0; i < n; ++i) {     // the critics' gradients: one buffer, so one all-reduce covers the ensemble
      ag->critic[i].alloc(true, ag->critic_grads + size_t(i) * ag->critic_stride);
      ag->target[i].alloc(false);
    }
    for (int l = 0; l < L; ++l) { ag->xhat.push_back(dev_alloc<float>(act)); ag->ah.push_back(dev_alloc<float>(act)); }
    ag->invstd = dev_alloc<float>(size_t(L) * ag->ldh);
    ag->ch.resize(n);
    for (int i = 0; i < n; ++i)
      for (int l = 0; l < L; ++l) ag->ch[i].push_back(dev_alloc<float>(act));
    for (int l = 0; l < L; ++l) ag->th.push_back(dev_alloc<float>(act));
    for (auto &p : ag->dz) p = dev_alloc<float>(act);
    for (int i = 0; i < 2 * n; ++i) ag->dzc.push_back(dev_alloc<float>(size_t(std::min<int64_t>(mb, kEnsembleBatchMax)) * ag->ldh));
    for (float **p : {&ag->sa, &ag->nsa, &ag->spi}) *p = dev_alloc<float>(mb * ag->ldc);
    for (float **p : {&ag->br, &ag->bd, &ag->br0, &ag->bd0, &ag->logp, &ag->per_w, &ag->per_td}) *p = dev_alloc<float>(mb);
    ag->y = dev_alloc<float>(mb * (nq > 0 ? ag->ldy : 1));
    ag->bs = dev_alloc<float>(mb * D); ag->bns = dev_alloc<float>(mb * D); ag->ba = dev_alloc<float>(mb * A);
    ag->q = dev_alloc<float>(n * ag->qstride); ag->qt = dev_alloc<float>(n * ag->qstride);
    ag->dq = dev_alloc<float>(n * std::max<int64_t>(ag->qstride, mb * 4));
    if (nq > 0) {
      ag->qscratch = dev_alloc<float>(mb * (2 * n + 1));
      ag->qrow = ag->qscratch + 2 * mb * n;
    }
    for (float **p : {&ag->act4, &ag->std4, &ag->gate4, &ag->dact, &ag->eps_next, &ag->eps_cur}) *p = dev_alloc<float>(mb * 4);
    ag->dzh = dev_alloc<float>(mb * 8);
    ag->slab = std::max(ag->actor.total, ag->critic[0].total);
    ag->pset = int64_t(kSplits) * ag->slab + int64_t(kSplits) * 4;
    ag->partials = dev_alloc<float>(size_t(ag->pset) * n);
    ag->sumsq = dev_alloc<float>(size_t(reduce_grid(int(ag->slab))) + 8);
    ag->mdev = dev_alloc<float>(kMetricFloats);
    GCRL_CUDA(cudaMemset(ag->mdev, 0, kMetricFloats * 4));
    ag->alpha_state = ag->mdev + 32;
    const float init_alpha[4] = {0.f, 1.f, 0.f, 0.f};       // log_alpha = 0 (:424)
    GCRL_CUDA(cudaMemcpy(ag->alpha_state, init_alpha, sizeof(init_alpha), cudaMemcpyHostToDevice));
    ag->d_scalars = dev_alloc<StepScalars>(2);
    if (cfg->precision >= 1) {
      // tensor-core engine: halves of every network; W^T of the hidden layers 1..L-1 of a trainable one (the input
      // gradient of a critic's layer 0 is only needed at the action columns, action_grad_acc_kernel)
      tc_dense_init();
      ag->actor.init_copies();
      for (int i = 0; i < n; ++i) {
        ag->critic[i].init_copies(1, L, true);
        ag->target[i].init_copies(0, 0, true);
      }
    }
    GCRL_CUDA(cudaStreamCreateWithFlags(&ag->cap_stream, cudaStreamNonBlocking));
    ag->use_graphs = graphs_enabled();
    ag->scal_stage.init(256);
    ag->io_stage.init(size_t(1) << 16);
  } catch (...) {
    delete ag;
    throw;
  }
  *out = ag;
}

extern "C" {

int gcrl_sac_create(gcrl_sac **out, int device, const gcrl_sac_config *cfg) {
  GCRL_API_BEGIN
  sac_create(out, device, cfg, 0, 0);
  GCRL_API_END
}

int gcrl_sac_create_quantile(gcrl_sac **out, int device, const gcrl_sac_config *cfg, int n_quantiles,
                             int drop_per_net) {
  GCRL_API_BEGIN
  GCRL_REQUIRE(n_quantiles >= 1, "quantile critics need n_quantiles >= 1");
  sac_create(out, device, cfg, n_quantiles, drop_per_net);
  GCRL_API_END
}

int gcrl_sac_destroy(gcrl_sac *ag) {
  GCRL_API_BEGIN
  if (ag == nullptr) return GCRL_OK;
  cudaSetDevice(ag->device);
  cudaDeviceSynchronize();
  ag->actor.destroy();
  for (int i = 0; i < ag->n; ++i) { ag->critic[i].destroy(); ag->target[i].destroy(); }
  for (auto &v : {ag->xhat, ag->ah, ag->th}) for (float *p : v) cudaFree(p);
  for (auto &v : ag->ch) for (float *p : v) cudaFree(p);
  for (float *p : ag->dzc) cudaFree(p);
  for (float *p : {ag->invstd, ag->dz[0], ag->dz[1], ag->sa, ag->nsa, ag->spi, ag->br, ag->bd, ag->bs, ag->ba, ag->bns,
                   ag->br0, ag->bd0, ag->q, ag->qt, ag->y, ag->dq, ag->logp, ag->act4, ag->std4, ag->gate4, ag->dact,
                   ag->dzh, ag->eps_next, ag->eps_cur, ag->partials, ag->sumsq, ag->mdev, ag->d_io,
                   ag->critic_grads, ag->per_w, ag->per_td, ag->qscratch})
    if (p) cudaFree(p);
  for (auto &kv : ag->graphs) cudaGraphExecDestroy(kv.second.exec);
  ag->many.graphs.clear();
  if (ag->many.d) cudaFree(ag->many.d);
  for (auto &kv : ag->seg_graphs) for (auto &r : kv.second) cudaGraphExecDestroy(r.graph.exec);
  if (ag->bn_gather) cudaFree(ag->bn_gather);
  if (ag->cap_stream) cudaStreamDestroy(ag->cap_stream);
  cudaFree(ag->d_scalars);
  ag->scal_stage.destroy();
  ag->io_stage.destroy();
  delete ag;
  GCRL_API_END
}

int gcrl_sac_set_actor_linear(gcrl_sac *ag, int layer, const float *w, const float *b, void *stream) {
  GCRL_API_BEGIN
  require_handle(ag);
  GCRL_REQUIRE(ag && w && b, "NULL argument");
  GCRL_CUDA(cudaSetDevice(ag->device));
  int rows, cols, ld, woff, boff;
  actor_linear_geom(ag, layer, &rows, &cols, &ld, &woff, &boff);
  upload_rows(ag->actor.p + woff, w, rows, cols, ld, as_stream(stream));
  upload_rows(ag->actor.p + boff, b, 1, rows, rows, as_stream(stream));
  ag->actor.copies.weights_changed(ag->actor.p, as_stream(stream));
  GCRL_API_END
}

int gcrl_sac_get_actor_linear(gcrl_sac *ag, int layer, float *w, float *b, void *stream) {
  GCRL_API_BEGIN
  require_handle(ag);
  GCRL_REQUIRE(ag != nullptr, "NULL argument");
  GCRL_CUDA(cudaSetDevice(ag->device));
  int rows, cols, ld, woff, boff;
  actor_linear_geom(ag, layer, &rows, &cols, &ld, &woff, &boff);
  if (w) download_rows(w, ag->actor.p + woff, rows, cols, ld, as_stream(stream));
  if (b) download_rows(b, ag->actor.p + boff, 1, rows, rows, as_stream(stream));
  GCRL_API_END
}

int gcrl_sac_set_actor_bn(gcrl_sac *ag, int layer, const float *weight, const float *bias, const float *rm,
                          const float *rv, void *stream) {
  GCRL_API_BEGIN
  require_handle(ag);
  GCRL_REQUIRE(ag && layer >= 0 && layer < ag->L, "bad BatchNorm layer index");
  GCRL_CUDA(cudaSetDevice(ag->device));
  cudaStream_t st = as_stream(stream);
  ActorNet &a = ag->actor;
  if (weight) upload_rows(a.p + a.gam_off[layer], weight, 1, ag->H, ag->H, st);
  if (bias) upload_rows(a.p + a.bet_off[layer], bias, 1, ag->H, ag->H, st);
  if (rm) upload_rows(a.rmean + size_t(layer) * ag->ldh, rm, 1, ag->H, ag->H, st);
  if (rv) upload_rows(a.rvar + size_t(layer) * ag->ldh, rv, 1, ag->H, ag->H, st);
  GCRL_API_END
}

int gcrl_sac_get_actor_bn(gcrl_sac *ag, int layer, float *weight, float *bias, float *rm, float *rv, void *stream) {
  GCRL_API_BEGIN
  require_handle(ag);
  GCRL_REQUIRE(ag && layer >= 0 && layer < ag->L, "bad BatchNorm layer index");
  GCRL_CUDA(cudaSetDevice(ag->device));
  cudaStream_t st = as_stream(stream);
  ActorNet &a = ag->actor;
  if (weight) download_rows(weight, a.p + a.gam_off[layer], 1, ag->H, ag->H, st);
  if (bias) download_rows(bias, a.p + a.bet_off[layer], 1, ag->H, ag->H, st);
  if (rm) download_rows(rm, a.rmean + size_t(layer) * ag->ldh, 1, ag->H, ag->H, st);
  if (rv) download_rows(rv, a.rvar + size_t(layer) * ag->ldh, 1, ag->H, ag->H, st);
  GCRL_API_END
}

int gcrl_sac_set_critic_layer(gcrl_sac *ag, int critic, int target, int layer, const float *w, const float *b,
                              void *stream) {
  GCRL_API_BEGIN
  require_handle(ag);
  GCRL_REQUIRE(ag && w && b && critic >= 0 && critic < ag->n, "bad critic index / NULL data");
  MlpParams &c = target ? ag->target[critic] : ag->critic[critic];
  GCRL_REQUIRE(layer >= 0 && layer < c.layers, "bad layer index");
  GCRL_CUDA(cudaSetDevice(ag->device));
  upload_rows(c.p + c.w_off[layer], w, c.out_d[layer], c.in_d[layer], c.ldw[layer], as_stream(stream));
  upload_rows(c.p + c.b_off[layer], b, 1, c.out_d[layer], c.out_d[layer], as_stream(stream));
  c.copies.weights_changed(c.p, as_stream(stream));
  GCRL_API_END
}

int gcrl_sac_get_critic_layer(gcrl_sac *ag, int critic, int target, int layer, float *w, float *b, void *stream) {
  GCRL_API_BEGIN
  require_handle(ag);
  GCRL_REQUIRE(ag && critic >= 0 && critic < ag->n, "bad critic index");
  MlpParams &c = target ? ag->target[critic] : ag->critic[critic];
  GCRL_REQUIRE(layer >= 0 && layer < c.layers, "bad layer index");
  GCRL_CUDA(cudaSetDevice(ag->device));
  if (w) download_rows(w, c.p + c.w_off[layer], c.out_d[layer], c.in_d[layer], c.ldw[layer], as_stream(stream));
  if (b) download_rows(b, c.p + c.b_off[layer], 1, c.out_d[layer], c.out_d[layer], as_stream(stream));
  GCRL_API_END
}

int gcrl_sac_hard_update(gcrl_sac *ag, void *stream) {
  GCRL_API_BEGIN
  require_handle(ag);
  GCRL_REQUIRE(ag != nullptr, "agent handle is NULL");
  GCRL_CUDA(cudaSetDevice(ag->device));
  for (int i = 0; i < ag->n; ++i) {
    GCRL_CUDA(cudaMemcpyAsync(ag->target[i].p, ag->critic[i].p, size_t(ag->critic[i].total) * 4,
                              cudaMemcpyDeviceToDevice, as_stream(stream)));
    ag->target[i].copies.weights_changed(ag->target[i].p, as_stream(stream));
  }
  GCRL_API_END
}

int gcrl_sac_set_log_alpha(gcrl_sac *ag, float log_alpha, void *stream) {
  GCRL_API_BEGIN
  require_handle(ag);
  GCRL_REQUIRE(ag != nullptr, "agent handle is NULL");
  GCRL_CUDA(cudaSetDevice(ag->device));
  const float v[4] = {log_alpha, std::exp(log_alpha), 0.f, 0.f};   // fresh AdamW state (reset(), :763-765)
  GCRL_CUDA(cudaMemcpyAsync(ag->alpha_state, v, sizeof(v), cudaMemcpyHostToDevice, as_stream(stream)));
  GCRL_CUDA(cudaStreamSynchronize(as_stream(stream)));
  ag->adam_t_alpha = 0;
  GCRL_API_END
}

int gcrl_sac_get_log_alpha(gcrl_sac *ag, float *log_alpha, void *stream) {
  GCRL_API_BEGIN
  require_handle(ag);
  GCRL_REQUIRE(ag != nullptr && log_alpha != nullptr, "NULL argument");
  GCRL_CUDA(cudaSetDevice(ag->device));
  GCRL_CUDA(cudaMemcpyAsync(log_alpha, ag->alpha_state, 4, cudaMemcpyDeviceToHost, as_stream(stream)));
  GCRL_CUDA(cudaStreamSynchronize(as_stream(stream)));
  GCRL_API_END
}

int gcrl_sac_update_batch(gcrl_sac *ag, int64_t B, const float *s, const float *a, const float *r, const float *ns,
                          const float *d, const float *eps_next, const float *eps_cur, double lr_c, double lr_a,
                          int flags, float *metrics_host, void *stream) {
  GCRL_API_BEGIN
  GCRL_NVTX("gcrl_sac_update_batch");
  require_handle(ag);
  GCRL_REQUIRE(ag != nullptr, "agent handle is NULL");
  GCRL_CUDA(cudaSetDevice(ag->device));
  sac_update(ag, -1, nullptr, B, nullptr, s, a, r, ns, d, eps_next, eps_cur, lr_c, lr_a, flags, metrics_host,
             as_stream(stream));
  GCRL_API_END
}

int gcrl_sac_update_from_buffer(gcrl_sac *ag, gcrl_her *buf, int64_t B, const int64_t *idx_host,
                                const float *eps_next, const float *eps_cur, double lr_c, double lr_a, int flags,
                                float *metrics_host, void *stream) {
  GCRL_API_BEGIN
  GCRL_NVTX("gcrl_sac_update_from_buffer");
  require_handle(ag);
  GCRL_REQUIRE(ag != nullptr && buf != nullptr, "NULL handle");
  GCRL_CUDA(cudaSetDevice(ag->device));
  sac_update(ag, -1, buf, B, idx_host, nullptr, nullptr, nullptr, nullptr, nullptr, eps_next, eps_cur, lr_c, lr_a,
             flags, metrics_host, as_stream(stream));
  GCRL_API_END
}

int gcrl_sac_update_many(gcrl_sac *ag, gcrl_her *buf, int64_t B, int n, const int *flags, const int64_t *idx_host,
                         const float *eps_next_dev, const float *eps_cur_dev, const double *lr_critic,
                         const double *lr_actor, float *metrics_host, void *stream) {
  GCRL_API_BEGIN
  GCRL_NVTX("gcrl_sac_update_many");
  update_many(ag, buf, nullptr, B, n, flags, idx_host, nullptr, nullptr, nullptr, eps_next_dev, eps_cur_dev, lr_critic,
              lr_actor, metrics_host, nullptr, stream);
  GCRL_API_END
}

int gcrl_sac_update_many_replay(gcrl_sac *ag, gcrl_replay *buf, int64_t B, int n, const int *flags,
                                const int64_t *pos_host, const double *u_host, const double *beta,
                                const float *eps_next_dev, const float *eps_cur_dev, const double *lr_critic,
                                const double *lr_actor, float *metrics_host, float *td_host, void *stream) {
  GCRL_API_BEGIN
  GCRL_NVTX("gcrl_sac_update_many_replay");
  update_many(ag, nullptr, buf, B, n, flags, nullptr, pos_host, u_host, beta, eps_next_dev, eps_cur_dev, lr_critic,
              lr_actor, metrics_host, td_host, stream);
  GCRL_API_END
}

int gcrl_sac_update_phase(gcrl_sac *ag, int phase, gcrl_her *buf, int64_t B, const int64_t *idx_host, const float *s,
                          const float *a, const float *r, const float *ns, const float *d, const float *eps_next,
                          const float *eps_cur, double lr_c, double lr_a, int flags, void *stream) {
  GCRL_API_BEGIN
  GCRL_NVTX("gcrl_sac_update_phase");
  require_handle(ag);
  GCRL_REQUIRE(ag != nullptr && phase >= 0 && phase <= 3, "NULL handle / phase outside 0..3");
  GCRL_REQUIRE(ag->nq == 0, "data parallelism is not available for quantile critics (gcrl_sac_create_quantile)");
  GCRL_CUDA(cudaSetDevice(ag->device));
  sac_update(ag, phase, buf, B, idx_host, s, a, r, ns, d, eps_next, eps_cur, lr_c, lr_a, flags, nullptr,
             as_stream(stream));
  GCRL_API_END
}

int gcrl_sac_set_sync_bn(gcrl_sac *ag, int world, int rank) {
  GCRL_API_BEGIN
  require_handle(ag);
  GCRL_REQUIRE(ag->nq == 0, "data parallelism is not available for quantile critics (gcrl_sac_create_quantile)");
  GCRL_REQUIRE(world >= 0 && world <= 1024 && (world == 0 || (rank >= 0 && rank < world)),
               "need 0 <= world <= 1024 and 0 <= rank < world (world 0 switches sync-BN off)");
  GCRL_CUDA(cudaSetDevice(ag->device));
  GCRL_CUDA(cudaDeviceSynchronize());
  for (auto &kv : ag->seg_graphs) for (auto &r : kv.second) cudaGraphExecDestroy(r.graph.exec);
  ag->seg_graphs.clear();
  if (ag->bn_gather) { cudaFree(ag->bn_gather); ag->bn_gather = nullptr; }
  ag->sync_world = world; ag->sync_rank = world > 0 ? rank : 0;
  if (world > 0) {
    ag->bn_gather = dev_alloc<float>(size_t(world) * 2 * ag->ldh);
    GCRL_CUDA(cudaMemset(ag->bn_gather, 0, size_t(world) * 2 * ag->ldh * 4));
  }
  GCRL_API_END
}

int gcrl_sac_update_segment(gcrl_sac *ag, int segment, gcrl_her *buf, int64_t B, const int64_t *idx_host,
                            const float *s, const float *a, const float *r, const float *ns, const float *d,
                            const float *eps_next, const float *eps_cur, double lr_c, double lr_a, int flags,
                            int *collective, void *stream) {
  GCRL_API_BEGIN
  GCRL_NVTX("gcrl_sac_update_segment");
  require_handle(ag);
  GCRL_REQUIRE(segment >= 0 && collective != nullptr, "segment < 0 / NULL collective");
  GCRL_REQUIRE(ag->nq == 0, "data parallelism is not available for quantile critics (gcrl_sac_create_quantile)");
  GCRL_REQUIRE(ag->sync_world > 0, "gcrl_sac_set_sync_bn first");
  GCRL_CUDA(cudaSetDevice(ag->device));
  sac_update(ag, -1, buf, B, idx_host, s, a, r, ns, d, eps_next, eps_cur, lr_c, lr_a, flags, nullptr,
             as_stream(stream), segment, collective);
  GCRL_API_END
}

int gcrl_sac_per_buffers(gcrl_sac *ag, float **weights_dev, float **td_dev) {
  GCRL_API_BEGIN
  require_handle(ag);
  GCRL_REQUIRE(ag != nullptr && weights_dev != nullptr && td_dev != nullptr, "NULL argument");
  *weights_dev = ag->per_w;
  *td_dev = ag->per_td;
  GCRL_API_END
}

int gcrl_sac_dp_buffer(gcrl_sac *ag, int which, float **dev, int64_t *count) {
  GCRL_API_BEGIN
  require_handle(ag);
  GCRL_REQUIRE(ag != nullptr && dev != nullptr && count != nullptr, "NULL argument");
  switch (which) {
    case 0: *dev = ag->actor.g; *count = ag->actor.total + 4; break;                       // + alpha's batch mean
    case 1: *dev = ag->critic_grads; *count = int64_t(ag->n) * ag->critic_stride; break;
    case 2: *dev = ag->actor.rmean; *count = int64_t(2) * ag->L * ag->ldh; break;          // BatchNorm running stats
    case 3: *dev = ag->mdev; *count = 32; break;
    case 4:
      GCRL_REQUIRE(ag->bn_gather != nullptr, "gcrl_sac_set_sync_bn first");
      *dev = ag->bn_gather; *count = int64_t(ag->sync_world) * 2 * ag->ldh; break;          // [world][2 ldh]
    default:
      throw Error(GCRL_ERR_INVALID,
                  "which must be 0 (actor grad), 1 (critic grads), 2 (BN running stats), 3 (metrics), 4 (sync-BN slots)");
  }
  GCRL_API_END
}

int gcrl_sac_read_metrics(gcrl_sac *ag, int flags, float *metrics_host, void *stream) {
  GCRL_API_BEGIN
  require_handle(ag);
  GCRL_REQUIRE(ag != nullptr && metrics_host != nullptr, "NULL argument");
  GCRL_CUDA(cudaSetDevice(ag->device));
  read_metrics(ag, flags, metrics_host, as_stream(stream));
  GCRL_API_END
}

int gcrl_sac_act(gcrl_sac *ag, int64_t n, const float *obs_host, const float *eps_host, float *act_host,
                 void *stream) {
  GCRL_API_BEGIN
  require_handle(ag);
  GCRL_REQUIRE(ag && obs_host && act_host, "NULL argument");
  GCRL_REQUIRE(n >= 1 && n <= ag->maxB, "row count outside [1, max_batch]");
  GCRL_CUDA(cudaSetDevice(ag->device));
  cudaStream_t st = as_stream(stream);
  const int D = ag->D, A = ag->A;
  const size_t need = size_t(n) * (D + 2 * A);
  if (need > ag->io_cap) {
    GCRL_CUDA(cudaStreamSynchronize(st));
    if (ag->d_io) GCRL_CUDA(cudaFree(ag->d_io));
    ag->io_cap = need * 2;
    ag->d_io = dev_alloc<float>(ag->io_cap);
  }
  auto stage = [&](const float *host, size_t count, size_t off) {
    int slot;
    char *p = ag->io_stage.acquire(count * 4, &slot);
    std::memcpy(p, host, count * 4);
    GCRL_CUDA(cudaMemcpyAsync(ag->d_io + off, p, count * 4, cudaMemcpyHostToDevice, st));
    ag->io_stage.release(slot, st);
    return ag->d_io + off;
  };
  float *obs = stage(obs_host, size_t(n) * D, 0);
  float *eps = eps_host ? stage(eps_host, size_t(n) * A, size_t(n) * D) : nullptr;
  float *out = ag->d_io + size_t(n) * (D + A);
  launch_pack_rows(obs, D, nullptr, A, ag->spi, ag->ldc, int(n), st);
  actor_fwd(ag, ag->spi, eps, int(n), false, false, out, st);     // set_eval(): running statistics
  GCRL_CUDA(cudaMemcpyAsync(act_host, out, size_t(n) * A * 4, cudaMemcpyDeviceToHost, st));
  GCRL_CUDA(cudaStreamSynchronize(st));
  GCRL_API_END
}

int gcrl_quantile_critic_loss(int device, int n, int M, int drop, int64_t B, const float *zt_dev, const float *z_dev,
                              int ldm, int64_t zstride, const float *logp_dev, const float *r_dev, const float *d_dev,
                              const float *w_dev, float gamma, float coef, const float *alpha_dev, float *y_dev, int ldy,
                              float *dz_dev, float *out_dev, float *td_rows_dev, float *scratch_dev, void *stream) {
  GCRL_API_BEGIN
  GCRL_REQUIRE(n >= 1 && n <= kMaxCritics, "n_critics outside [1, 8]");
  GCRL_REQUIRE(M >= 1 && n * M <= 256, "need n_quantiles >= 1 and n_critics * n_quantiles <= 256");
  GCRL_REQUIRE(drop >= 0 && drop < M, "drop_per_net outside [0, n_quantiles)");
  GCRL_REQUIRE(B >= 1 && B < (int64_t(1) << 31), "batch size outside [1, 2^31)");
  const int K = n * (M - drop);
  GCRL_REQUIRE(ldm >= M && ldm % 4 == 0, "ldm must be >= n_quantiles and a multiple of 4");
  GCRL_REQUIRE(zstride >= B * ldm, "zstride must be >= B * ldm");
  GCRL_REQUIRE(ldy >= K && ldy % 4 == 0, "ldy must be >= n_critics * (n_quantiles - drop_per_net) and a multiple of 4");
  GCRL_REQUIRE(coef >= 0.f || alpha_dev != nullptr, "coef < 0 reads the coefficient from alpha_dev: NULL");
  GCRL_REQUIRE(zt_dev && z_dev && logp_dev && r_dev && d_dev && y_dev && dz_dev && out_dev && scratch_dev,
               "NULL argument");
  GCRL_CUDA(cudaSetDevice(device));
  quantile_critic_loss(zt_dev, z_dev, zstride, ldm, n, M, K, logp_dev, r_dev, d_dev, w_dev, gamma, coef, alpha_dev,
                       y_dev, ldy, dz_dev, out_dev, 0, n, td_rows_dev, scratch_dev, int(B), as_stream(stream));
  GCRL_API_END
}

}  // extern "C"
