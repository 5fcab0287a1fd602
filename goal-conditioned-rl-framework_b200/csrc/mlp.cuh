// Launch helpers for the MLP forward/backward/optimiser kernels (mlp.cu, optim.cu).
// All 2-D operands are (pointer, leading dimension) with the leading dimension a multiple
// of 4 floats and the base 16-byte aligned; logical sizes are arbitrary.
#pragma once
#include "common.cuh"
#include "her_device.cuh"

namespace gcrl {

constexpr float kLeakySlope = 0.01f;  // nn.LeakyReLU() default, reference src/model.py:20

enum ActMode : int { ACT_NONE = 0, ACT_LEAKY = 1 };

// Y[M,N] = act(X[M,K] * W[N,K]^T + bias[N])
void launch_linear_fwd(const float *X, int ldx, const float *W, int ldw, const float *bias, float *Y,
                       int ldy, int M, int N, int K, int act, cudaStream_t st);

// dX[M,K] = (dZ[M,N] * W[N,K]) (.) leaky'(Xact[M,K])     (Xact == nullptr: no activation factor)
void launch_linear_dgrad(const float *dZ, int lddz, const float *W, int ldw, const float *Xact,
                         int ldxa, float *dX, int lddx, int M, int N, int K, cudaStream_t st);

// Split-batch partial weight gradients:
//   pW[s][N][ldw] = sum_{m in slab s} dZ[m,n] * X[m,k],   pB[s][N] = sum_{m in slab s} dZ[m,n]
// Returns the number of slabs S written (<= max_splits).
int launch_linear_wgrad(const float *dZ, int lddz, const float *X, int ldx, float *pW, int ldw,
                        int64_t w_split_stride, float *pB, int64_t b_split_stride, int M, int N, int K,
                        int max_splits, cudaStream_t st);

// Skinny output layer, NOUT <= 4:  out[m, col0 + n] = f(H[m,:] . W[n,:] + bias[n]),  f = tanh | id
// ---- same-shape problems of an ensemble (the n critics) in one launch per layer ----
constexpr int kMaxBatchedLinear = 8;
struct LinearFwdProblem { const float *X; int ldx; const float *W; int ldw; const float *bias; float *Y; int ldy; };
struct LinearDgradProblem { const float *dZ; int lddz; const float *W; int ldw; const float *Xact; int ldxa; float *dX; int lddx; };
struct HeadFwdProblem { const float *Hact; const float *W; const float *bias; float *out; };   // out[m] = h[m] . W + bias
void launch_linear_fwd_batched(const LinearFwdProblem *pr, int n, int M, int N, int K, int act, cudaStream_t st);
void launch_linear_dgrad_batched(const LinearDgradProblem *pr, int n, int M, int N, int K, cudaStream_t st);
void launch_head_fwd_batched(const HeadFwdProblem *pr, int n, int ldh, int ldw, int M, int K, cudaStream_t st);

void launch_head_fwd(const float *Hact, int ldh, const float *W, int ldw, const float *bias, float *out,
                     int ldo, int col0, int M, int K, int nout, int tanh_out, cudaStream_t st);

struct HeadBwdArgs {
  // mode 0 (critic TD loss): dz = w_is * 2 (q - y) / M with
  //        y = r + gamma (1 - d) min(qt1, qt2)   [clamped to [y_lo, 0] when clamp_y]
  //        loss_kind 0: mse, 1: smooth-l1 (beta 1)   (TD3, reference src/agent.py:189-197)
  // mode 1 (actor loss through the critic): dz = -1 / M
  // mode 2 (actor head): dz[m,n] given in dz_in[m*4+n]
  int mode, loss_kind, clamp_y, nout;
  const float *q, *qt1, *qt2, *r, *d, *dz_in;
  const float *y_in;      // mode 0: Bellman target given per row (SAC / TQC) instead of built from qt1/qt2
  const float *q_other;   // TD3 critic 2: metrics use max(|q-y|, |q_other-y|) and (q+q_other)/2
  const float *is_w;      // mode 0, prioritised replay: per-sample importance weight of the loss (nullptr: 1)
  float *td_out;          // mode 0, prioritised replay: per-sample TD error (max with q_other's), or nullptr
  float gamma, y_lo;
  const float *Hact; int ldh;      // last hidden activation [M, K]
  const float *W; int ldw;         // head weight [nout, K]
  float *dZprev; int lddz;         // out: grad wrt last hidden pre-activation [M, K]
  float *pW; int64_t w_split_stride;  // out: partial head weight grads [S][nout][ldw] (nullptr: skip)
  float *pB; int64_t b_split_stride;  // out: partial head bias grads   [S][nout]
  float *metric_partials;          // out: [S][4] = sum loss, sum |y-q|, sum q, unused
  float *y_out;                    // optional [M]
  int M, K;
};
// Returns the number of row slabs S.
int launch_head_bwd(const HeadBwdArgs &a, int max_splits, cudaStream_t st);
int launch_head_bwd_batched(const HeadBwdArgs *a, int n, int max_splits, cudaStream_t st);   // nout == 1, same M / K

// Critic layer-1 input gradient restricted to the action columns, fused with tanh':
//   dz_out[m*4 + j] = (sum_n dZ1[m,n] W1[n, col0 + j]) * (1 - act[m, col0 + j]^2)
void launch_action_grad(const float *dZ1, int lddz, const float *W1, int ldw, const float *sa, int ldsa,
                        int col0, float *dz_out, int M, int N, int nact, cudaStream_t st);

// pack dense s[M,D], a[M,A] (optional) into rows [s | a | 0-pad] with leading dimension ldo
void launch_pack_rows(const float *s, int D, const float *a, int A, float *out, int ldo, int M,
                      cudaStream_t st);

// All weight gradients of one network in ONE launch (multi-problem split-batch GEMM):
//   problem i: pW_i[s][N_i][ldw_i] = sum_{m in slab s} dZ_i[m,n] * X_i[m,k]  (+ bias partials)
struct WgradProblem {
  const float *dZ; int lddz;
  const float *X; int ldx;
  float *pW; int ldw;
  float *pB;
  int N, K;          // layer output / input widths
  float *gW, *gB;    // WgradFinal: where this layer's weight / bias gradient lives in the flat gradient buffer
};
constexpr int kMaxWgradProblems = 8;   // == kMaxBatchedLinear: one problem per critic of an ensemble
// What wgrad_tile_kernel finalises next to the gradient: per-tile sums of squares for the clip and the
// batch-mean metrics of the phase.
struct WgradFinal {
  float *sumsq_partials;    // [tiles]
  const float *metric_partials; int metric_splits; float metric_scale;
  float *metrics; int slot_loss, slot_td, slot_q;
  // peer-memory data parallelism: the LAST CTA to finish tells every peer "this rank's gradient is complete"
  // (and publishes the metrics) -- the flag travels over NVLink while the averaging kernel is being launched
  unsigned int *const *peer_flags; unsigned int *epoch; unsigned int *ticket;
  float *outbox; int rank, world;
};
// Split-batch partial slabs (summed later by reduce_grads); returns the number of batch slabs S.
int launch_multi_wgrad(const WgradProblem *probs, int nprob, int M, int64_t split_stride, int max_splits,
                       cudaStream_t st);
// Complete gradients straight into probs[i].gW / gB + sums of squares + metrics in ONE launch (M <= 1024);
// returns the number of output tiles (= sums of squares written).
int launch_wgrad_complete(const WgradProblem *probs, int nprob, int M, const WgradFinal &fin, cudaStream_t st);
// Per-tile sums of squares of a complete gradient (probs[i].gW / gB, N, K, ldw), bit-identical to the ones
// launch_wgrad_complete leaves; returns the number of tiles.
int launch_wgrad_sumsq(const WgradProblem *probs, int nprob, float *sumsq_partials, cudaStream_t st);

// ---- row-slab fused update kernels (fused.cu) -----------------------------------------------
constexpr int kFusedMaxL = 6;
struct FusedNet {               // hidden layers 0..L-1 and the output head of one MLP
  const float *Wt[kFusedMaxL];  // transposed weights [in][ldt]   (forward)
  const float *W[kFusedMaxL];   // weights as stored  [out][ldw]  (input gradient)
  const float *b[kFusedMaxL];
  int ldt[kFusedMaxL], ldw[kFusedMaxL];
  const float *Wh, *bh;         // head [nout][ldwh]
  int ldwh;
  const float *flat, *flatT;    // the whole parameter buffer and its transposed copy (L2 prefetch at kernel start)
  int nflat, nflatT;
};
struct FusedCriticArgs {
  FusedNet ta, tc, c;           // target actor, target critic, critic
  FusedNet tc2; int has_tc2;    // TD3: second target critic (y uses the minimum)
  const float *noise;           // TD3: [B, A] standard-normal draws of the target-policy smoothing, or nullptr
  float policy_noise, noise_clamp;
  int loss_kind;                // 0 mse, 1 smooth-l1 (beta 1)
  const float *y_in;            // non-null: the Bellman target is given (TD3 critic 2); the target nets are skipped
  const float *q_other;         // non-null: metrics use max(|q-y|, |q_other-y|) and (q + q_other) / 2
  const float *is_w;            // prioritised replay: per-sample importance weight of the loss (nullptr: 1)
  float *td_out;                // prioritised replay: per-sample TD error [B] (max with q_other's), or nullptr
  const float *s, *a, *r, *ns, *d;   // dense batch
  // sample != 0: the kernel draws the batch itself from the HER episode store (her_device.cuh: position ->
  // episode -> packed row + future goal -> relabel + reward, per slab) and leaves the dense batch in bs .. bd
  // for the actor phase; one launch and one pass over the batch less than a separate sampler
  int sample;
  HerGeom geom;
  const SampleScalars *sample_sc;    // totals / draw epoch of this update (device struct, written by the host)
  const int64_t *sample_idx;         // positions (host index stream), used when sample_sc->use_idx
  float *bs, *ba, *br, *bns, *bd;    // dense batch out
  int B, D, A, H, L, ldh, ldc;
  float gamma, y_lo; int clamp_y;
  float *sa_out;                // [B][ldc]  = [s | a | 0] rows (layer-1 wgrad operand)
  float *h_out[kFusedMaxL];     // critic hidden activations [B][ldh]
  float *dz_out[kFusedMaxL];    // critic pre-activation gradients [B][ldh]
  float *dzh_out, *y_out, *q_out;   // [B]
  float *metric_partials;       // [grid][4]
};
struct FusedActorArgs {
  FusedNet actor, c;
  const float *s;
  int B, D, A, H, L, ldh;
  float *h_out[kFusedMaxL];     // actor hidden activations
  float *dz_out[kFusedMaxL];    // actor pre-activation gradients
  float *da_out;                // [B][4] gradient at the actor head's pre-activation
  float *metric_partials;
};
bool fused_supported(int B, int D, int A, int H, int L);
bool fused_sample_supported(const HerGeom &g);
int launch_fused_critic(const FusedCriticArgs &a, cudaStream_t st);   // returns the grid (metric slabs)
int launch_fused_actor(const FusedActorArgs &a, cudaStream_t st);

// ---- tensor-core dense layers (tc_gemm.cu): tcgen05 / TMEM / TMA, 3xTF32 split for fp32 accuracy ----
bool tc_dense_supported(int M, int N, int K);
void tc_dense_init();
bool tc_wgrad_supported(int M, int N, int K);
// tensor-core version of launch_linear_wgrad (same partial-slab contract); returns the number of slabs
int launch_tc_wgrad(const float *dZ, int lddz, const float *X, int ldx, float *pW, int ldw, int64_t w_split_stride,
                    float *pB, int64_t b_split_stride, int M, int N, int K, int max_splits, cudaStream_t st);
// out[M, N] = epilogue(X[M, K] * W[N, K]^T); mode 0: leaky(. + bias), 1: . * leaky'(act), 2: . + bias, 3: . (bare)
// W_lo != nullptr: the weights come pre-split (W = TF32 hi halves, W_lo = lo halves, same layout; launch_split_tf32)
void launch_tc_dense(const float *X, int ldx, const float *W, int ldw, const float *bias, const float *act,
                     int ldact, float *out, int ldo, int M, int N, int K, int mode, cudaStream_t st,
                     const float *W_lo = nullptr);
// the same for n <= 8 independent problems of one (M, N, K, mode) in one launch (e.g. the critics of an ensemble);
// each member's output equals the single-CTA launch_tc_dense of that member bit for bit
struct TcDenseProblem { const float *X; int ldx; const float *W_hi, *W_lo; int ldw; const float *bias, *act; float *out; };
void launch_tc_dense_ensemble(const TcDenseProblem *pr, int n, int ldact, int ldo, int M, int N, int K, int mode,
                              cudaStream_t st);
void launch_split_tf32(const float *src, float *hi, float *lo, int n, cudaStream_t st);

// ---- optimiser (optim.cu) --------------------------------------------------------------
struct SegDesc {          // one parameter segment of a flat network buffer
  int begin, count;       // [begin, begin+count) in the flat buffer
  const float *partials;  // [splits][split_stride] partial sums (nullptr: already reduced)
  int splits;
  int64_t split_stride;
  int offset;             // offset of this segment inside a partial slab
};
constexpr int kMaxSegs = 32;
struct ReduceArgs {
  SegDesc seg[kMaxSegs];
  int nseg, total;
  float *grad;            // flat gradient out
  float *sumsq_partials;  // [gridDim.x]
  // metrics finalisation (block 0): out[slot] = sum(partials[.][j]) * scale
  const float *metric_partials; int metric_splits; float metric_scale;
  float *metrics; int slot_loss, slot_td, slot_q;
};
int reduce_grid(int total);
void launch_reduce_grads(const ReduceArgs &a, cudaStream_t st);

struct StepScalars {       // written by the host before every update (device copy)
  // per optimiser: lr / (1 - b1^t), sqrt(1 - b2^t), 1 - lr * weight_decay, unused
  float step_size_c, bc2_sqrt_c, decay_c;
  unsigned int seq;        // update counter: the last optimiser kernel publishes it with the metrics (AdamArgs::publish)
  float step_size_a, bc2_sqrt_a, decay_a, pad1;
};
struct AdamArgs {
  float *p, *m, *v; const float *g; int n;
  const float *sumsq_partials; int nsumsq;
  float max_norm;          // < 0: no clipping
  float weight_decay;      // decoupled (AdamW); 0 for Adam
  const StepScalars *sc; int which;   // 0: critic scalars, 1: actor scalars
  float *target; float tau, one_minus_tau; int polyak;   // fused Polyak of `target` with the NEW p
  float *metrics; int slot_norm;
  // transposed weight copies kept in step with p / target (fused.cu's forward operand)
  const int *tmap;         // [n] index into pT, or -1 (bias / padding)
  float *pT, *targetT;
  // last optimiser kernel of an update: copy the 8 metrics (+ the data-parallel watchdog word) into MAPPED host
  // memory and then the update's sequence number -- the host polls that word instead of paying a D2H copy and a
  // stream synchronisation per update()
  float *publish;          // mapped host: float[8] metrics, uint32 seq, int32 err  (nullptr: do not publish)
  const float *publish_src;
  const int *publish_err;
};
void launch_adam(const AdamArgs &a, cudaStream_t st);
// data-parallel averaging over NVLink peer memory (optim.cu)
void launch_p2p_barrier(unsigned int *const *peer_flags, unsigned int *epoch, int rank, int world, int *err,
                        cudaStream_t st);
// flag barrier + rank-order average of one network's gradient + metric exchange, ONE launch (optim.cu)
struct P2PReduceHost {
  const float *const *peers; unsigned int *const *peer_flags; const float *const *peer_outbox;
  unsigned int *epoch, *ticket, *go; int *err;
  int rank, world, n;
  float *out, *sumsq_partials;
  const float *local_metrics; float *outbox, *metrics_avg; unsigned int metric_mask;
  int signalled;      // the producer of the gradient has already raised this rank's flag (WgradFinal::peer_flags)
};
int p2p_reduce_grid(int n);              // CTAs (= sums of squares) of the launch below
void launch_p2p_reduce(const P2PReduceHost &h, cudaStream_t st);
long long p2p_timeout_cycles();
void launch_polyak(float *target, const float *src, int n, float tau, float one_minus_tau,
                   const int *tmap, float *targetT, cudaStream_t st);
// pT[tmap[e]] = p[e] for every weight element
void launch_sync_transposed(const float *p, float *pT, const int *tmap, int n, cudaStream_t st);

// one launch: dense (s, a, r, ns, d) -> sa = [s|a|0], nsa = [ns|0], spi = [s|0], r, d copies
void launch_ingest_batch(const float *s, const float *a, const float *r, const float *ns, const float *d,
                         int D, int A, int M, float *sa, float *nsa, float *spi, int ldc, float *r_out,
                         float *d_out, cudaStream_t st);
// TD3 target-policy smoothing: x[m, col0+j] = clamp(x + clamp(noise[m*A+j] * sigma, +-c), -1, 1)
void launch_td3_smooth(float *x, int ldx, int col0, const float *noise, int A, int M, float sigma,
                       float clampv, cudaStream_t st);

}  // namespace gcrl
