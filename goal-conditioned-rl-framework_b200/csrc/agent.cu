// Off-policy learner: DDPG and TD3 update orchestration over the kernels in mlp.cu/optim.cu.
//
// Replaces (reference src/agent.py) DDPG.critic_update :1302-1343, actor_update :1288-1300,
// update_target_network :1255-1271 and update :1378-1404; TD3Agent.critic_update :164-251,
// actor_update :149-162, update_actor/update_critic :117-132, update :281-317.
//
// Device memory per agent: every network is one flat fp32 buffer (weights [out, ld(in)] then
// bias, per layer, 16 B aligned segments) with matching flat gradient / Adam m / Adam v
// buffers; activations are [max_batch, ld(hidden)] per layer; the [state | action] operand
// rows (sa, nsa, spi) fold torch.cat: the actor heads write their tanh output straight into
// the action columns.  An update is captured once per (batch, flags) into a CUDA graph and
// replayed; per-step scalars (lr / bias corrections) travel through a small device struct.
#include <algorithm>
#include <atomic>
#include <chrono>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <initializer_list>
#include <map>
#include <tuple>
#include <vector>

#include "buffer_api.cuh"
#include "graphs.cuh"
#include "mlp.cuh"
#include "params.cuh"

using namespace gcrl;

namespace {

struct Acts {  // post-activation outputs of the hidden layers, [max_batch, ldh] each
  std::vector<float *> h;
  void init(int hidden_layers, int64_t maxB, int ldh) {
    for (int l = 0; l < hidden_layers; ++l) h.push_back(dev_alloc<float>(size_t(maxB) * ldh));
  }
  void destroy() { for (auto p : h) cudaFree(p); }
};

enum NetId { ACTOR = 0, CRITIC1 = 1, T_ACTOR = 2, T_CRITIC1 = 3, CRITIC2 = 4, T_CRITIC2 = 5, NUM_NETS = 6 };
enum Slot { S_CLOSS = 0, S_ALOSS = 1, S_TD = 2, S_Q = 3, S_CGRAD = 4, S_AGRAD = 5, S_C2LOSS = 6, S_C2GRAD = 7 };

constexpr int kMaxSplits = 128;
constexpr size_t kScalBytes = sizeof(StepScalars) + sizeof(SampleScalars);   // the per-update device scalars

}  // namespace

struct gcrl_agent {
  uint32_t magic = 0x544E4741u;   // handle type tag: the two agent families share the Python base class
  int device = 0;
  gcrl_agent_config cfg{};
  int D = 0, A = 0, H = 0, L = 0, ldh = 0, ldc = 0;
  int64_t maxB = 0;
  bool td3 = false;
  MlpParams net[NUM_NETS];
  bool has[NUM_NETS] = {};
  int adam_t[NUM_NETS] = {};               // Adam step counters
  Acts acts_actor, acts_c1, acts_c2, acts_tgt;
  float *dz[2] = {nullptr, nullptr};       // ping-pong grad-wrt-preactivation buffers [maxB, ldh]
  float *sa = nullptr, *nsa = nullptr, *spi = nullptr;
  float *q1 = nullptr, *q2 = nullptr, *qt1 = nullptr, *qt2 = nullptr, *yv = nullptr, *dz_act = nullptr;
  float *br = nullptr, *bd = nullptr;      // reward / done copies
  float *bs = nullptr, *ba = nullptr, *bns = nullptr, *br0 = nullptr, *bd0 = nullptr;  // sampled batch
  float *partials = nullptr;               // [kMaxSplits][max net total]
  int64_t slab = 0;
  float *metric_partials = nullptr;        // [kMaxSplits][4]
  float *sumsq = nullptr;                  // [max(reduce grid, wgrad tiles)]
  int nsumsq = 0;                          // how many sums of squares the pending optimiser step reads
  float *metrics = nullptr;                // [8]
  StepScalars *d_scalars = nullptr;        // StepScalars, then the SampleScalars of the update (one H2D copy)
  SampleScalars *d_sample_sc = nullptr;
  int64_t *d_idx = nullptr;                // positions of the in-kernel sampler (host index stream) [maxB]
  float *h_pub = nullptr, *d_pub = nullptr; // mapped host memory the last optimiser kernel publishes the metrics to
  unsigned int pub_seq = 0;                // sequence number of the most recent update
  bool pub_valid = false;                  // ... and whether that update publishes (whole-update launches only)
  bool publish_now = false;                // capture-time: the optimiser step being recorded is the update's last
  gcrl_her *sample_buf = nullptr;          // the update being issued draws its batch inside the critic kernel
  SampleScalars sample_sc{};
  PinnedRing scal_stage;
  PinnedRing io_stage;
  float *d_io = nullptr;
  size_t io_cap = 0;
  float *noise = nullptr;                  // TD3 smoothing noise copy [maxB, A]
  std::vector<float *> dzl;                // fused path: per-layer pre-activation gradients [maxB, ldh]
  float *dzh = nullptr;                    // fused path: critic head dL/dq [maxB]
  float *per_w = nullptr, *per_td = nullptr;   // prioritised replay: importance weights in, TD errors out [maxB]
  bool per_on = false;                     // flags bit3 of the update being issued
  bool use_fused = true, fuse_sampler = true;
  bool tc_update = false;                  // the update being recorded / issued runs on the tensor-core engine
  int dp_B = -1, dp_flags = -1;            // the update the data-parallel phases belong to
  // data-parallel averaging over NVLink peer memory (gcrl_agent_dp_connect)
  struct P2P {
    bool on = false;
    int rank = 0, world = 1;
    unsigned int *flags = nullptr, *epoch = nullptr;     // [8] arrival counters written by the peers; my barrier count
    unsigned int *go = nullptr;                          // local release word: CTA 0 saw every peer's flag
    unsigned int *ticket = nullptr, *wticket = nullptr;  // CTA tickets of the barrier + average launch / the weight-gradient launch
    bool signalled = false;                              // capture-time: the gradient's producer raises the flag itself
    int *err = nullptr;
    float *outbox = nullptr, *metrics_avg = nullptr;     // [2][8] metrics published to / [8] averaged over the ranks
    float *gavg[NUM_NETS] = {};                          // averaged gradient of every trainable network
    unsigned int **d_peer_flags = nullptr;               // device arrays of `world` peer pointers
    float **d_peer_outbox = nullptr;
    float **d_peer_g[NUM_NETS] = {};
    std::vector<void *> opened;                          // cudaIpcOpenMemHandle results
  } p2p;
  bool dp_open = false;                    // a phase-wise data-parallel update: phase 0 issued, phase 3 not yet
  bool use_graphs = true;
  cudaStream_t cap_stream = nullptr;       // capture-only stream (the caller's may be the legacy one)
  std::map<std::tuple<int64_t, int, int, uintptr_t>, GraphRec> graphs;   // (B, flags, phase mask, sampled buffer)
  // n consecutive updates in one graph (gcrl_agent_update_many): everything a captured update reads that changes
  // from one update to the next has one slot per update; allocated on first use
  struct Many {
    char *d = nullptr;                     // [GCRL_MAX_MANY_STEPS] x kScalBytes scalars, then positions [n][B] int64
    float *noise = nullptr;                // TD3 smoothing noise [n][B][A]
    float *h_pub = nullptr, *d_pub = nullptr;   // mapped publish blocks [GCRL_MAX_MANY_STEPS][16] of updates 0 .. n-2
    float *td = nullptr;                   // prioritised replay: every update's per-sample TD errors [n][B]
    // (B, flags of every update, buffer, engine path, buffer epoch, length drawn from): a uniform or HER buffer has
    // 0 for the last one, a graph serves any length; a HER buffer also has 0 for the epoch
    using Key = std::tuple<int64_t, std::vector<int>, uintptr_t, int, uint64_t, int64_t>;
    ManyGraphs<Key> graphs;
  } many;
};

namespace {

// Tensor-core (tcgen05, 3xTF32) dense layers: large batches only -- below ~1k rows a 128-row tile
// grid cannot fill the 148 SMs and the fp32 tiles / row-slab kernels win.
constexpr int kTcMinBatch = 2048;     // measured break-even with the fp32 tiles (the column tile narrows to fill the SMs)
bool use_tc(const gcrl_agent *ag, int B, int N, int K) {
  if (!tc_dense_supported(B, N, K)) return false;
  return ag->cfg.precision == 2 ? B >= 128 : (ag->cfg.precision == 1 && B >= kTcMinBatch);
}

// does an update / forward at this batch run its hidden layers on the tensor cores (pre-split weights needed)?
bool engine_tc(const gcrl_agent *ag, int B) { return use_tc(ag, B, ag->H, (ag->H + 3) & ~3); }

// the TF32 hi / lo copies of every network whose parameters changed since they were last split (eager, outside capture)
void ensure_split(gcrl_agent *ag, cudaStream_t st) {
  for (int i = 0; i < NUM_NETS; ++i)
    if (ag->has[i]) ag->net[i].copies.split_if_stale(ag->net[i].p, st);
}
void mark_split_stale(gcrl_agent *ag) {
  for (int i = 0; i < NUM_NETS; ++i) ag->net[i].copies.stale = true;
}

// ---- forward / backward building blocks ----------------------------------------------------
// hidden stack: X[B, K0] -> acts.h[0..L-1]
void forward_hidden(const gcrl_agent *ag, const MlpParams &n, const float *X, int ldx, int K0, const Acts &acts,
                    int B, cudaStream_t st) {
  const float *in = X;
  int ldin = ldx, K = K0;
  for (int l = 0; l < ag->L; ++l) {
    // layer 0: the operand rows and the weight rows are zero-padded to ld, so the padded K is exact
    const int Kp = (K + 3) & ~3;
    if (use_tc(ag, B, ag->H, Kp))
      launch_tc_dense(in, ldin, n.copies.p_hi + n.w_off[l], n.ldw[l], n.b(l), nullptr, 0, acts.h[l], ag->ldh, B, ag->H, Kp,
                      0, st, n.copies.p_lo + n.w_off[l]);
    else
      launch_linear_fwd(in, ldin, n.W(l), n.ldw[l], n.b(l), acts.h[l], ag->ldh, B, ag->H, K, ACT_LEAKY, st);
    in = acts.h[l];
    ldin = ag->ldh;
    K = ag->H;
  }
}

// Backward through the hidden stack given dz[cur] = grad wrt the pre-activation of the last hidden
// layer.  Writes split partial weight/bias grads; returns per-layer split counts.  When
// `to_input` the chain continues to dZ of layer 0 (left in dz[*cur_out]).
// x_pad_zero: X's columns K0 .. K0 padded to a multiple of 4 are zero.  The actor's input rows [s | a | 0] hold the
// actions there, which the tensor-core weight gradient would sum into the padding columns of layer 0's gradient
// (inflating its norm, hence the clip, and stepping the padding weights).
void backward_hidden(gcrl_agent *ag, const MlpParams &n, const float *X, int ldx, int K0, bool x_pad_zero,
                     const Acts &acts, int B, int cur, bool want_wgrad, int *splits /*[layers]*/, int *cur_out,
                     cudaStream_t st) {
  for (int l = ag->L - 1; l >= 0; --l) {
    const float *xin = l == 0 ? X : acts.h[l - 1];
    const int ldin = l == 0 ? ldx : ag->ldh;
    const int K = l == 0 ? K0 : ag->H;
    if (want_wgrad) {
      const int Kp = (K + 3) & ~3;     // the tensor cores reduce over Kp columns of the operand rows
      if ((Kp == K || x_pad_zero) && use_tc(ag, B, ag->H, Kp) && tc_wgrad_supported(B, ag->H, Kp))
        splits[l] = launch_tc_wgrad(ag->dz[cur], ag->ldh, xin, ldin, ag->partials + n.w_off[l], n.ldw[l], ag->slab,
                                    ag->partials + n.b_off[l], ag->slab, B, ag->H, Kp, kMaxSplits, st);
      else
        splits[l] = launch_linear_wgrad(ag->dz[cur], ag->ldh, xin, ldin, ag->partials + n.w_off[l], n.ldw[l],
                                        ag->slab, ag->partials + n.b_off[l], ag->slab, B, ag->H, K,
                                        kMaxSplits, st);
    }
    if (l > 0) {
      if (use_tc(ag, B, ag->H, ag->H))   // dX = dZ Wt^T with the transposed weight copy as the K-major operand
        launch_tc_dense(ag->dz[cur], ag->ldh, n.copies.pT_hi + n.copies.t_off[l], n.copies.ldt[l], nullptr,
                        acts.h[l - 1], ag->ldh, ag->dz[cur ^ 1], ag->ldh, B, ag->H, ag->H, 1, st,
                        n.copies.pT_lo + n.copies.t_off[l]);
      else
        launch_linear_dgrad(ag->dz[cur], ag->ldh, n.W(l), n.ldw[l], acts.h[l - 1], ag->ldh, ag->dz[cur ^ 1],
                            ag->ldh, B, ag->H, ag->H, st);
      cur ^= 1;
    }
  }
  *cur_out = cur;
}

// partial slabs -> flat gradient of `n` (+ per-CTA sums of squares, + batch-mean metrics).
// rereduce: the gradient is already in n.g (it was averaged across ranks); only the sums of
// squares for the global-norm clip are recomputed.
void reduce_grads(gcrl_agent *ag, MlpParams &n, const int *splits, int head_splits, bool rereduce, int slot_loss,
                  int slot_td, int slot_q, int metric_splits, int B, cudaStream_t st) {
  ReduceArgs r{};
  r.nseg = 0;
  for (int l = 0; l < n.layers; ++l) {
    const int sp = rereduce ? 0 : (l == n.layers - 1 ? head_splits : splits[l]);
    const float *src = rereduce ? nullptr : ag->partials;
    SegDesc w{n.w_off[l], n.out_d[l] * n.ldw[l], src, sp, ag->slab, n.w_off[l]};
    SegDesc b{n.b_off[l], n.out_d[l], src, sp, ag->slab, n.b_off[l]};
    r.seg[r.nseg++] = w;
    r.seg[r.nseg++] = b;
  }
  r.total = n.total;
  r.grad = n.g;
  r.sumsq_partials = ag->sumsq;
  r.metric_partials = metric_splits > 0 ? ag->metric_partials : nullptr;
  r.metric_splits = metric_splits;
  r.metric_scale = 1.0f / float(B);
  r.metrics = ag->metrics;
  r.slot_loss = slot_loss; r.slot_td = slot_td; r.slot_q = slot_q;
  ag->nsumsq = reduce_grid(n.total);
  launch_reduce_grads(r, st);
}

// global-norm clip + Adam(W) (+ fused Polyak of `target` with the stepped parameters)
void adam_step(gcrl_agent *ag, MlpParams &n, int which, float max_norm, int slot_norm, MlpParams *target, bool polyak,
               cudaStream_t st, const float *grad = nullptr) {
  AdamArgs a{};
  a.p = n.p; a.m = n.m; a.v = n.v; a.g = grad ? grad : n.g; a.n = n.total;
  a.sumsq_partials = ag->sumsq; a.nsumsq = ag->nsumsq;
  a.max_norm = max_norm;
  a.weight_decay = ag->cfg.weight_decay;
  a.sc = ag->d_scalars; a.which = which;
  a.target = target ? target->p : nullptr; a.tau = ag->cfg.tau; a.one_minus_tau = float(1.0 - double(ag->cfg.tau));
  a.polyak = (polyak && target) ? 1 : 0;
  a.metrics = ag->p2p.on ? ag->p2p.metrics_avg : ag->metrics;   // the norm of the averaged gradient is global already
  a.slot_norm = slot_norm;
  a.tmap = n.copies.tmap; a.pT = n.copies.pT; a.targetT = target ? target->copies.pT : nullptr;
  if (ag->publish_now) {
    a.publish = ag->d_pub;
    a.publish_src = a.metrics;
    a.publish_err = ag->p2p.on ? ag->p2p.err : nullptr;
  }
  launch_adam(a, st);
  if (ag->tc_update) {          // this update's later layers read the stepped weights through the tensor cores
    n.copies.split(n.p, st);
    if (a.polyak) target->copies.split(target->p, st);
  }
}

// ---- phases ------------------------------------------------------------------------------------
// phase 0/1: critic(s).  Operands sa / nsa / br / bd must be resident.
void critic_forward_backward(gcrl_agent *ag, int which_critic, int B, int *splits, int *head_splits,
                             int *metric_splits, cudaStream_t st) {
  const MlpParams &c = ag->net[which_critic == 0 ? CRITIC1 : CRITIC2];
  const Acts &acts = which_critic == 0 ? ag->acts_c1 : ag->acts_c2;
  float *q = which_critic == 0 ? ag->q1 : ag->q2;
  const int K0 = ag->D + ag->A;
  HeadBwdArgs h{};
  h.mode = 0;
  h.loss_kind = ag->td3 ? 1 : 0;
  h.clamp_y = ag->td3 ? 0 : 1;                       // DDPG clamps y to [-1/(1-gamma), 0] (:1317)
  h.nout = 1;
  h.q = q; h.qt1 = ag->qt1; h.qt2 = ag->td3 ? ag->qt2 : nullptr;
  h.q_other = (ag->td3 && which_critic == 1) ? ag->q1 : nullptr;
  if (ag->per_on) { h.is_w = ag->per_w; h.td_out = ag->per_td; }
  h.r = ag->br; h.d = ag->bd;
  h.gamma = ag->cfg.gamma;
  h.y_lo = float(-1.0 / (1.0 - double(ag->cfg.gamma)));
  h.Hact = acts.h[ag->L - 1]; h.ldh = ag->ldh;
  h.W = c.W(ag->L); h.ldw = c.ldw[ag->L];
  h.dZprev = ag->dz[0]; h.lddz = ag->ldh;
  h.pW = ag->partials + c.w_off[ag->L]; h.w_split_stride = ag->slab;
  h.pB = ag->partials + c.b_off[ag->L]; h.b_split_stride = ag->slab;
  h.metric_partials = ag->metric_partials;
  h.y_out = ag->yv;
  h.M = B; h.K = ag->H;
  *head_splits = launch_head_bwd(h, kMaxSplits, st);
  *metric_splits = *head_splits;
  int cur;
  backward_hidden(ag, c, ag->sa, ag->ldc, K0, true, acts, B, 0, true, splits, &cur, st);
}

void targets_and_critic_forward(gcrl_agent *ag, int B, const float *noise, cudaStream_t st) {
  const int D = ag->D, A = ag->A, K0 = D + A;
  // a' = target_actor(s')  -> action columns of nsa                          (:1312 / :179)
  forward_hidden(ag, ag->net[T_ACTOR], ag->nsa, ag->ldc, D, ag->acts_tgt, B, st);
  launch_head_fwd(ag->acts_tgt.h[ag->L - 1], ag->ldh, ag->net[T_ACTOR].W(ag->L), ag->net[T_ACTOR].ldw[ag->L],
                  ag->net[T_ACTOR].b(ag->L), ag->nsa, ag->ldc, D, B, ag->H, A, 1, st);
  if (ag->td3) {
    GCRL_REQUIRE(noise != nullptr, "TD3 update needs the [B, A] standard-normal noise tensor");
    launch_td3_smooth(ag->nsa, ag->ldc, D, noise, A, B, ag->cfg.policy_noise, ag->cfg.noise_clamp, st);
  }
  // q' = target_critic([s', a'])                                               (:1313-1315)
  forward_hidden(ag, ag->net[T_CRITIC1], ag->nsa, ag->ldc, K0, ag->acts_tgt, B, st);
  launch_head_fwd(ag->acts_tgt.h[ag->L - 1], ag->ldh, ag->net[T_CRITIC1].W(ag->L),
                  ag->net[T_CRITIC1].ldw[ag->L], ag->net[T_CRITIC1].b(ag->L), ag->qt1, 1, 0, B, ag->H, 1, 0, st);
  if (ag->td3) {
    forward_hidden(ag, ag->net[T_CRITIC2], ag->nsa, ag->ldc, K0, ag->acts_tgt, B, st);
    launch_head_fwd(ag->acts_tgt.h[ag->L - 1], ag->ldh, ag->net[T_CRITIC2].W(ag->L),
                    ag->net[T_CRITIC2].ldw[ag->L], ag->net[T_CRITIC2].b(ag->L), ag->qt2, 1, 0, B, ag->H, 1, 0,
                    st);
  }
  // q = critic([s, a])                                                          (:1319)
  forward_hidden(ag, ag->net[CRITIC1], ag->sa, ag->ldc, K0, ag->acts_c1, B, st);
  launch_head_fwd(ag->acts_c1.h[ag->L - 1], ag->ldh, ag->net[CRITIC1].W(ag->L), ag->net[CRITIC1].ldw[ag->L],
                  ag->net[CRITIC1].b(ag->L), ag->q1, 1, 0, B, ag->H, 1, 0, st);
  if (ag->td3) {
    forward_hidden(ag, ag->net[CRITIC2], ag->sa, ag->ldc, K0, ag->acts_c2, B, st);
    launch_head_fwd(ag->acts_c2.h[ag->L - 1], ag->ldh, ag->net[CRITIC2].W(ag->L), ag->net[CRITIC2].ldw[ag->L],
                    ag->net[CRITIC2].b(ag->L), ag->q2, 1, 0, B, ag->H, 1, 0, st);
  }
}

struct PhaseState {
  int splits[8] = {};
  int head_splits = 0, metric_splits = 0;
};

// ---- row-slab fused path (fused.cu): DDPG, B <= 1024 ---------------------------------------------
bool fused_ok(const gcrl_agent *ag, int B) {
  return ag->use_fused && fused_supported(B, ag->D, ag->A, ag->H, ag->L);
}

FusedNet fused_net(const gcrl_agent *ag, const MlpParams &n) {
  FusedNet f{};
  const WeightCopies &c = n.copies;
  for (int l = 0; l < ag->L; ++l) {
    f.Wt[l] = c.pT + c.t_off[l]; f.ldt[l] = c.ldt[l];
    f.W[l] = n.p + n.w_off[l];   f.ldw[l] = n.ldw[l];
    f.b[l] = n.p + n.b_off[l];
  }
  f.Wh = n.p + n.w_off[ag->L]; f.ldwh = n.ldw[ag->L]; f.bh = n.p + n.b_off[ag->L];
  f.flat = n.p; f.nflat = n.total; f.flatT = c.pT; f.nflatT = c.total_t;
  return f;
}

// batch-mean metrics that are final when critic `which`'s gradient is: DDPG critic loss / td / q; TD3 critic 1: its
// loss; critic 2: loss, td, q (they ride on that gradient's barrier under peer-memory data parallelism)
unsigned int critic_metric_mask(const gcrl_agent *ag, int which) {
  return !ag->td3 ? ((1u << S_CLOSS) | (1u << S_TD) | (1u << S_Q))
                  : (which == 0 ? (1u << S_CLOSS) : ((1u << S_C2LOSS) | (1u << S_TD) | (1u << S_Q)));
}

// weight gradients of all layers of `n` in ONE launch that also completes the split-batch sums into the flat
// gradient n.g, the per-tile sums of squares and the batch-mean metrics (mlp.cu: multi_wgrad_kernel);
// hidden-layer operands: dzl[l] and (l == 0 ? sa : acts.h[l-1]); head operand: dz_head [B][ld_head] and acts.h[L-1]
void fused_wgrads(gcrl_agent *ag, MlpParams &n, const Acts &acts, int K0, const float *dz_head, int ld_head, int B,
                  int slot_loss, int slot_td, int slot_q, int metric_splits, cudaStream_t st) {
  WgradProblem pr[kMaxWgradProblems];
  const int L = ag->L;
  for (int l = 0; l < L; ++l) {
    pr[l] = WgradProblem{ag->dzl[l], ag->ldh, l == 0 ? ag->sa : acts.h[l - 1], l == 0 ? ag->ldc : ag->ldh,
                         ag->partials + n.w_off[l], n.ldw[l], ag->partials + n.b_off[l], ag->H,
                         l == 0 ? K0 : ag->H, n.g + n.w_off[l], n.g + n.b_off[l]};
  }
  pr[L] = WgradProblem{dz_head, ld_head, acts.h[L - 1], ag->ldh, ag->partials + n.w_off[L], n.ldw[L],
                       ag->partials + n.b_off[L], n.out_d[L], ag->H, n.g + n.w_off[L], n.g + n.b_off[L]};
  WgradFinal fin{};
  fin.sumsq_partials = ag->sumsq;
  fin.metric_partials = metric_splits > 0 ? ag->metric_partials : nullptr;
  fin.metric_splits = metric_splits;
  fin.metric_scale = 1.0f / float(B);
  fin.metrics = ag->metrics;
  fin.slot_loss = slot_loss; fin.slot_td = slot_td; fin.slot_q = slot_q;
  if (ag->p2p.on) {         // the last CTA raises this rank's flag at every peer (p2p_average then only waits)
    auto &pp = ag->p2p;
    fin.peer_flags = pp.d_peer_flags; fin.epoch = pp.epoch; fin.ticket = pp.wticket; fin.outbox = pp.outbox;
    fin.rank = pp.rank; fin.world = pp.world;
    pp.signalled = true;
  }
  ag->nsumsq = launch_wgrad_complete(pr, L + 1, B, fin, st);
}

// the same per-tile sums of squares for a gradient that is already complete in n.g (data-parallel phases: the
// cross-rank average replaced it) -- bit-identical to what fused_wgrads leaves for the same values
void fused_grad_sumsq(gcrl_agent *ag, MlpParams &n, cudaStream_t st) {
  WgradProblem pr[kMaxWgradProblems];
  for (int l = 0; l < n.layers; ++l) {
    pr[l] = WgradProblem{};
    pr[l].ldw = n.ldw[l]; pr[l].N = n.out_d[l]; pr[l].K = n.in_d[l];
    pr[l].gW = n.g + n.w_off[l]; pr[l].gB = n.g + n.b_off[l];
  }
  ag->nsumsq = launch_wgrad_sumsq(pr, n.layers, ag->sumsq, st);
}

FusedCriticArgs fused_critic_args(gcrl_agent *ag, int B, int which = 0) {
  FusedCriticArgs a{};
  a.ta = fused_net(ag, ag->net[T_ACTOR]);
  a.tc = fused_net(ag, ag->net[T_CRITIC1]);
  a.c = fused_net(ag, ag->net[which == 0 ? CRITIC1 : CRITIC2]);
  if (ag->td3) {
    a.tc2 = fused_net(ag, ag->net[T_CRITIC2]);
    a.has_tc2 = 1;
    a.noise = ag->noise;
    a.policy_noise = ag->cfg.policy_noise; a.noise_clamp = ag->cfg.noise_clamp;
    a.loss_kind = 1;
    if (which == 1) { a.y_in = ag->yv; a.q_other = ag->q1; }     // target and Q1 left by the critic-1 launch
  }
  if (ag->per_on) { a.is_w = ag->per_w; a.td_out = ag->per_td; }
  a.s = ag->bs; a.a = ag->ba; a.r = ag->br0; a.ns = ag->bns; a.d = ag->bd0;
  if (ag->sample_buf != nullptr && which == 0) {        // the kernel draws the batch itself (TD3 critic 2 reuses it)
    a.sample = 1;
    a.geom = her_geom(ag->sample_buf);
    a.sample_sc = ag->d_sample_sc;
    a.sample_idx = ag->d_idx;
    a.bs = ag->bs; a.ba = ag->ba; a.br = ag->br0; a.bns = ag->bns; a.bd = ag->bd0;
  }
  a.B = B; a.D = ag->D; a.A = ag->A; a.H = ag->H; a.L = ag->L; a.ldh = ag->ldh; a.ldc = ag->ldc;
  a.gamma = ag->cfg.gamma;
  a.y_lo = float(-1.0 / (1.0 - double(ag->cfg.gamma)));
  a.clamp_y = ag->td3 ? 0 : 1;                         // DDPG clamps y to [-1/(1-gamma), 0] (:1317); TD3 does not
  a.sa_out = which == 0 ? ag->sa : nullptr;
  const Acts &acts = which == 0 ? ag->acts_c1 : ag->acts_c2;
  for (int l = 0; l < ag->L; ++l) { a.h_out[l] = acts.h[l]; a.dz_out[l] = ag->dzl[l]; }
  a.dzh_out = ag->dzh; a.y_out = ag->yv; a.q_out = which == 0 ? ag->q1 : ag->q2;
  a.metric_partials = ag->metric_partials;
  return a;
}

void fused_critic_phase_grads(gcrl_agent *ag, int B, int which, cudaStream_t st) {
  const FusedCriticArgs a = fused_critic_args(ag, B, which);
  const int slabs = launch_fused_critic(a, st);
  MlpParams &c = ag->net[which == 0 ? CRITIC1 : CRITIC2];
  // TD3: td error / Q metrics come from the critic-2 launch (they need both critics' Q)
  const bool metrics_here = !ag->td3 || which == 1;
  fused_wgrads(ag, c, which == 0 ? ag->acts_c1 : ag->acts_c2, ag->D + ag->A, ag->dzh, 1, B,
               which == 0 ? S_CLOSS : S_C2LOSS, metrics_here ? S_TD : -1, metrics_here ? S_Q : -1, slabs, st);
}

void fused_actor_phase_grads(gcrl_agent *ag, int B, cudaStream_t st) {
  FusedActorArgs a{};
  a.actor = fused_net(ag, ag->net[ACTOR]);
  a.c = fused_net(ag, ag->net[CRITIC1]);
  a.s = ag->bs;
  a.B = B; a.D = ag->D; a.A = ag->A; a.H = ag->H; a.L = ag->L; a.ldh = ag->ldh;
  for (int l = 0; l < ag->L; ++l) { a.h_out[l] = ag->acts_actor.h[l]; a.dz_out[l] = ag->dzl[l]; }
  a.da_out = ag->dz_act;
  a.metric_partials = ag->metric_partials;
  const int slabs = launch_fused_actor(a, st);
  fused_wgrads(ag, ag->net[ACTOR], ag->acts_actor, ag->D, ag->dz_act, 4, B, S_ALOSS, -1, -1, slabs, st);
}

// critic(s): forward, loss, backward, partials -> flat local-mean gradient(s) + metrics
void critic_phase_grads(gcrl_agent *ag, int B, const float *noise, cudaStream_t st) {
  if (fused_ok(ag, B)) { fused_critic_phase_grads(ag, B, 0, st); return; }
  PhaseState ps;
  targets_and_critic_forward(ag, B, noise, st);
  critic_forward_backward(ag, 0, B, ps.splits, &ps.head_splits, &ps.metric_splits, st);
  reduce_grads(ag, ag->net[CRITIC1], ps.splits, ps.head_splits, false, S_CLOSS, ag->td3 ? -1 : S_TD,
               ag->td3 ? -1 : S_Q, ps.metric_splits, B, st);
}
void critic2_phase_grads(gcrl_agent *ag, int B, cudaStream_t st) {   // TD3 only; reuses dz / partials
  if (fused_ok(ag, B)) { fused_critic_phase_grads(ag, B, 1, st); return; }
  PhaseState ps;
  critic_forward_backward(ag, 1, B, ps.splits, &ps.head_splits, &ps.metric_splits, st);
  reduce_grads(ag, ag->net[CRITIC2], ps.splits, ps.head_splits, false, S_C2LOSS, S_TD, S_Q, ps.metric_splits,
               B, st);
}

// clip + Adam (+ Polyak) of critic `which`; rereduce: gradients were replaced by the cross-rank
// average, so the sums of squares are recomputed first.
// p2p mode: ONE launch per network -- flag barrier (every rank's local gradient of `net` is complete), average of
// the peers' buffers into p2p.gavg[net] (+ the sums of squares the clip needs), and the batch-mean metrics that
// are final at this point (`metric_mask`, slot bits) averaged over the ranks on the same barrier.
const float *p2p_average(gcrl_agent *ag, int net, unsigned int metric_mask, cudaStream_t st) {
  auto &pp = ag->p2p;
  P2PReduceHost h{};
  h.peers = pp.d_peer_g[net]; h.peer_flags = pp.d_peer_flags; h.peer_outbox = pp.d_peer_outbox;
  h.epoch = pp.epoch; h.ticket = pp.ticket; h.go = pp.go; h.err = pp.err;
  h.rank = pp.rank; h.world = pp.world; h.n = ag->net[net].total;
  h.out = pp.gavg[net]; h.sumsq_partials = ag->sumsq;
  h.local_metrics = ag->metrics; h.outbox = pp.outbox; h.metrics_avg = pp.metrics_avg; h.metric_mask = metric_mask;
  h.signalled = pp.signalled ? 1 : 0;
  pp.signalled = false;
  launch_p2p_reduce(h, st);
  ag->nsumsq = p2p_reduce_grid(ag->net[net].total);
  return pp.gavg[net];
}

void critic_phase_step(gcrl_agent *ag, int which, int flags, bool rereduce, cudaStream_t st) {
  const bool polyak = ag->td3 ? true : ((flags & 2) != 0);
  const int id = which == 0 ? CRITIC1 : CRITIC2;
  MlpParams &c = ag->net[id];
  const float *grad = nullptr;
  // metrics final before this barrier: DDPG critic loss / td / q; TD3 critic 1: its loss; critic 2: loss, td, q
  const unsigned int mm = critic_metric_mask(ag, which);
  if (ag->p2p.on) grad = p2p_average(ag, id, mm, st);
  else if (rereduce && fused_ok(ag, ag->dp_B)) fused_grad_sumsq(ag, c, st);
  else if (rereduce) reduce_grads(ag, c, nullptr, 0, true, -1, -1, -1, 0, 1, st);
  // TD3 critic 1 is NOT clipped (:201 is commented out), critic 2 is
  const float clip = (ag->td3 && which == 0) ? -1.0f : ag->cfg.grad_clip;
  adam_step(ag, c, 0, clip, which == 0 ? S_CGRAD : S_C2GRAD, &ag->net[which == 0 ? T_CRITIC1 : T_CRITIC2],
            polyak, st, grad);
}

// DDPG: the actor target blends the PRE-step actor, before the actor step (:1397-1401)
void ddpg_actor_target_polyak(gcrl_agent *ag, int flags, cudaStream_t st) {
  if (!ag->td3 && (flags & 2)) {
    MlpParams &t = ag->net[T_ACTOR];
    launch_polyak(t.p, ag->net[ACTOR].p, ag->net[ACTOR].total, ag->cfg.tau, float(1.0 - double(ag->cfg.tau)),
                  ag->net[ACTOR].copies.tmap, t.copies.pT, st);
    if (ag->tc_update) t.copies.split(t.p, st);
  }
}

void actor_phase_grads(gcrl_agent *ag, int B, cudaStream_t st) {
  if (fused_ok(ag, B)) { fused_actor_phase_grads(ag, B, st); return; }
  PhaseState pstate, *ps = &pstate;
  const int D = ag->D, A = ag->A, K0 = D + A, L = ag->L;
  const MlpParams &actor = ag->net[ACTOR];
  const MlpParams &c = ag->net[CRITIC1];
  // a = actor(s) -> action columns of spi; q = critic([s, a]) with the stepped critic (:1289-1290)
  forward_hidden(ag, actor, ag->spi, ag->ldc, D, ag->acts_actor, B, st);
  launch_head_fwd(ag->acts_actor.h[L - 1], ag->ldh, actor.W(L), actor.ldw[L], actor.b(L), ag->spi, ag->ldc, D,
                  B, ag->H, A, 1, st);
  forward_hidden(ag, c, ag->spi, ag->ldc, K0, ag->acts_c1, B, st);
  launch_head_fwd(ag->acts_c1.h[L - 1], ag->ldh, c.W(L), c.ldw[L], c.b(L), ag->q1, 1, 0, B, ag->H, 1, 0, st);
  // d(-mean q)/d(critic hidden) ... down to the action columns
  HeadBwdArgs h{};
  h.mode = 1; h.nout = 1; h.q = ag->q1;
  h.Hact = ag->acts_c1.h[L - 1]; h.ldh = ag->ldh;
  h.W = c.W(L); h.ldw = c.ldw[L];
  h.dZprev = ag->dz[0]; h.lddz = ag->ldh;
  h.pW = nullptr; h.pB = nullptr;                     // critic weight grads are discarded (:1293-1294)
  h.metric_partials = ag->metric_partials;
  h.M = B; h.K = ag->H;
  const int actor_metric_splits = launch_head_bwd(h, kMaxSplits, st);
  int cur;
  int dummy[8];
  backward_hidden(ag, c, ag->spi, ag->ldc, K0, true, ag->acts_c1, B, 0, false, dummy, &cur, st);
  launch_action_grad(ag->dz[cur], ag->ldh, c.W(0), c.ldw[0], ag->spi, ag->ldc, D, ag->dz_act, B, ag->H, A, st);
  // actor head + hidden stack backward
  HeadBwdArgs ha{};
  ha.mode = 2; ha.nout = A; ha.dz_in = ag->dz_act;
  ha.Hact = ag->acts_actor.h[L - 1]; ha.ldh = ag->ldh;
  ha.W = actor.W(L); ha.ldw = actor.ldw[L];
  ha.dZprev = ag->dz[0]; ha.lddz = ag->ldh;
  ha.pW = ag->partials + actor.w_off[L]; ha.w_split_stride = ag->slab;
  ha.pB = ag->partials + actor.b_off[L]; ha.b_split_stride = ag->slab;
  ha.M = B; ha.K = ag->H;
  ps->head_splits = launch_head_bwd(ha, kMaxSplits, st);
  backward_hidden(ag, actor, ag->spi, ag->ldc, D, false, ag->acts_actor, B, 0, true, ps->splits, &cur, st);
  // the actor-loss metric partials (critic head pass) are still intact: the actor head pass has mode 2
  reduce_grads(ag, ag->net[ACTOR], ps->splits, ps->head_splits, false, S_ALOSS, -1, -1, actor_metric_splits, B,
               st);
}

void actor_phase_step(gcrl_agent *ag, bool rereduce, cudaStream_t st) {
  MlpParams &a = ag->net[ACTOR];
  const float *grad = nullptr;
  if (ag->p2p.on) grad = p2p_average(ag, ACTOR, 1u << S_ALOSS, st);
  else if (rereduce && fused_ok(ag, ag->dp_B)) fused_grad_sumsq(ag, a, st);
  else if (rereduce) reduce_grads(ag, a, nullptr, 0, true, -1, -1, -1, 0, 1, st);
  adam_step(ag, a, 1, ag->cfg.grad_clip, S_AGRAD, &ag->net[T_ACTOR], ag->td3, st, grad);
}

// The next update's Adam step counters and sequence number -> its StepScalars, followed by `ss`, at `out` (host)
void fill_scalars(gcrl_agent *ag, double lr_c, double lr_a, bool actor_steps, const SampleScalars &ss, char *out) {
  auto fill = [&](int t, double lr, float *out) {
    const double bc1 = 1.0 - std::pow(0.9, double(t));
    const double bc2 = 1.0 - std::pow(0.999, double(t));
    out[0] = float(lr / bc1);
    out[1] = float(std::sqrt(bc2));
    out[2] = float(1.0 - lr * double(ag->cfg.weight_decay));
  };
  auto *sc = reinterpret_cast<StepScalars *>(out);
  std::memcpy(sc + 1, &ss, sizeof(SampleScalars));
  ag->adam_t[CRITIC1] += 1;
  if (ag->td3) ag->adam_t[CRITIC2] += 1;
  fill(ag->adam_t[CRITIC1], lr_c, &sc->step_size_c);
  if (actor_steps) ag->adam_t[ACTOR] += 1;
  fill(std::max(1, ag->adam_t[ACTOR]), lr_a, &sc->step_size_a);
  sc->pad1 = 0.f;
  sc->seq = ++ag->pub_seq;
}

void write_scalars(gcrl_agent *ag, double lr_c, double lr_a, bool actor_steps, cudaStream_t st) {
  int slot;
  char *sc = ag->scal_stage.acquire(kScalBytes, &slot);
  fill_scalars(ag, lr_c, lr_a, actor_steps, ag->sample_sc, sc);
  GCRL_CUDA(cudaMemcpyAsync(ag->d_scalars, sc, kScalBytes, cudaMemcpyHostToDevice, st));
  ag->scal_stage.release(slot, st);
}

// The Adam step counters and the update sequence number advance in write_scalars, before the update is enqueued.
// If anything after that throws (argument checks, a CUDA error, graph capture), the Python schedulers do not step
// either, so the counters are restored -- otherwise every later bias correction would be off by one step.
// keep_draws: the device index-stream epoch of `buf` is restored too (an n-update call draws all its epochs first).
struct AdamStepGuard {
  gcrl_agent *ag;
  int t[NUM_NETS];
  bool per_on; int dp_B, dp_flags;
  unsigned int pub_seq;
  gcrl_her *buf = nullptr;
  unsigned long long draw_epoch = 0;
  bool done = false;
  explicit AdamStepGuard(gcrl_agent *a)
      : ag(a), per_on(a->per_on), dp_B(a->dp_B), dp_flags(a->dp_flags), pub_seq(a->pub_seq) {
    std::copy(a->adam_t, a->adam_t + NUM_NETS, t);
  }
  void keep_draws(gcrl_her *b) { buf = b; draw_epoch = her_draw_epoch(b); }
  void commit() { done = true; }
  ~AdamStepGuard() {
    if (done) return;
    std::copy(t, t + NUM_NETS, ag->adam_t);
    ag->per_on = per_on; ag->dp_B = dp_B; ag->dp_flags = dp_flags;
    ag->pub_seq = pub_seq;
    if (buf != nullptr) her_draw_epoch(buf) = draw_epoch;
  }
};

// phase masks: bit0 critic grads, bit1 critic step, bit2 actor grads, bit3 actor step.
// A single-GPU update runs all four back to back (mask 15); the data-parallel path runs them one
// at a time with the caller's gradient all-reduce in between (steps then re-reduce).
enum : int { PH_CGRAD = 1, PH_CSTEP = 2, PH_AGRAD = 4, PH_ASTEP = 8, PH_ALL = 15 };

void run_update_body(gcrl_agent *ag, int B, const float *noise, int flags, int mask, cudaStream_t st) {
  const bool dp = mask != PH_ALL;
  if (mask & PH_CGRAD) {
    GCRL_NVTX("gcrl: critic phase (targets, loss, backward, weight gradients)");
    critic_phase_grads(ag, B, noise, st);
    if (ag->td3 && dp) critic2_phase_grads(ag, B, st);
  }
  const bool actor_steps = (flags & 1) != 0;
  if (mask & PH_CSTEP) {
    GCRL_NVTX("gcrl: critic step (average, clip, Adam, Polyak)");
    ddpg_actor_target_polyak(ag, flags, st);
    ag->publish_now = !dp && !actor_steps && !ag->td3;
    critic_phase_step(ag, 0, flags, dp, st);
    if (ag->td3) {
      if (!dp) critic2_phase_grads(ag, B, st);
      ag->publish_now = !dp && !actor_steps;
      critic_phase_step(ag, 1, flags, dp, st);
    }
    ag->publish_now = false;
  }
  if ((mask & PH_AGRAD) && (flags & 1)) {
    GCRL_NVTX("gcrl: actor phase (policy, Q, backward, weight gradients)");
    actor_phase_grads(ag, B, st);
  }
  if ((mask & PH_ASTEP) && (flags & 1)) {
    GCRL_NVTX("gcrl: actor step (average, clip, Adam, Polyak)");
    ag->publish_now = !dp;
    actor_phase_step(ag, dp, st);
    ag->publish_now = false;
  }
}

// the engine an update at this batch runs on; the tensor-core one needs the split weight copies current
void select_engine(gcrl_agent *ag, int B, cudaStream_t st) {
  ag->tc_update = !fused_ok(ag, B) && engine_tc(ag, B);
  if (ag->tc_update) ensure_split(ag, st);          // (the update itself re-splits what it steps)
  else mark_split_stale(ag);                        // weights move without their split copies following
}

// Replay (or capture on first use) the graph of (B, flags, phase mask).  TD3 noise pointers vary
// per call, so the noise is first copied into an internal buffer by the caller.
void run_update(gcrl_agent *ag, int B, const float *noise, int flags, int mask, cudaStream_t st) {
  select_engine(ag, B, st);
  if (!ag->use_graphs) {
    run_update_body(ag, B, noise, flags, mask, st);
    return;
  }
  const auto key = std::make_tuple(int64_t(B), flags, mask, reinterpret_cast<uintptr_t>(ag->sample_buf));
  auto it = ag->graphs.find(key);
  if (it == ag->graphs.end())
    it = ag->graphs.emplace(key, capture_graph(ag->cap_stream, [&](cudaStream_t cs) { run_update_body(ag, B, noise, flags, mask, cs); })).first;
  launch_graph(it->second, st);
}

// While update i of an n-update call is recorded (or issued eagerly), the agent's per-update inputs -- scalars,
// sampler positions, TD3 noise, publish block -- point at slot i, so every argument builder picks the slot up.
// The last update publishes through the single-update block: gcrl_agent_read_metrics then sees it as after
// gcrl_agent_update_from_buffer.
struct ManySlot {
  gcrl_agent *ag;
  StepScalars *sc; SampleScalars *ssc; int64_t *idx; float *noise, *pub;
  ManySlot(gcrl_agent *a, int i, int n, int B)
      : ag(a), sc(a->d_scalars), ssc(a->d_sample_sc), idx(a->d_idx), noise(a->noise), pub(a->d_pub) {
    a->d_scalars = reinterpret_cast<StepScalars *>(a->many.d + size_t(i) * kScalBytes);
    a->d_sample_sc = reinterpret_cast<SampleScalars *>(a->d_scalars + 1);
    a->d_idx = reinterpret_cast<int64_t *>(a->many.d + size_t(n) * kScalBytes) + size_t(i) * B;
    if (a->td3) a->noise = a->many.noise + size_t(i) * B * a->A;
    if (i < n - 1) a->d_pub = a->many.d_pub + size_t(i) * 16;
  }
  ~ManySlot() { ag->d_scalars = sc; ag->d_sample_sc = ssc; ag->d_idx = idx; ag->noise = noise; ag->d_pub = pub; }
  ManySlot(const ManySlot &) = delete;
  ManySlot &operator=(const ManySlot &) = delete;
};

// n updates back to back from the HER buffer `her` or the uniform / prioritised buffer `rb` (the other is NULL).
// Update i draws its batch from slot i -- HER: from the slot's totals and positions, unless the row-slab critic kernel
// draws it (ag->sample_buf set) -- and, prioritised, writes its priorities back and copies its TD errors into row i.
void run_many_body(gcrl_agent *ag, gcrl_her *her, gcrl_replay *rb, int B, int n, const int *flags, cudaStream_t st) {
  for (int i = 0; i < n; ++i) {
    ManySlot slot(ag, i, n, B);
    if (ag->sample_buf == nullptr) {
      if (rb != nullptr)
        replay_many_sample(rb, B, n, i, ag->bs, ag->ba, ag->br0, ag->bns, ag->bd0, ag->per_w, st);
      else
        her_sample_graphed(her, B, ag->d_sample_sc, ag->d_idx, ag->bs, ag->ba, ag->br0, ag->bns, ag->bd0, st);
      if (!fused_ok(ag, B))
        launch_ingest_batch(ag->bs, ag->ba, ag->br0, ag->bns, ag->bd0, ag->D, ag->A, B, ag->sa, ag->nsa, ag->spi, ag->ldc,
                            ag->br, ag->bd, st);
    }
    run_update_body(ag, B, ag->td3 ? ag->noise : nullptr, flags[i], PH_ALL, st);
    if (ag->per_on) {
      replay_many_write_back(rb, B, ag->per_td, st);
      GCRL_CUDA(cudaMemcpyAsync(ag->many.td + size_t(i) * B, ag->per_td, size_t(B) * 4, cudaMemcpyDeviceToDevice, st));
    }
  }
}

int many_path(const gcrl_agent *ag, int B) {
  return (ag->sample_buf != nullptr ? 1 : 0) | (fused_ok(ag, B) ? 2 : 0) | (ag->tc_update ? 4 : 0);
}

// A prioritised call is captured when its key repeats only (see ManyGraphs::launch); a HER buffer has 0 for the
// key's epoch and length.
void run_many(gcrl_agent *ag, gcrl_her *her, gcrl_replay *rb, int B, int n, const int *flags, cudaStream_t st) {
  select_engine(ag, B, st);
  const uintptr_t buf = rb != nullptr ? reinterpret_cast<uintptr_t>(rb) : reinterpret_cast<uintptr_t>(her);
  ag->many.graphs.launch({int64_t(B), std::vector<int>(flags, flags + n), buf, many_path(ag, B),
                          rb != nullptr ? replay_epoch(rb) : 0, ag->per_on ? replay_many_n(rb) : 0},
                         !ag->per_on, [&](cudaStream_t cs) { run_many_body(ag, her, rb, B, n, flags, cs); }, st,
                         ag->use_graphs, ag->cap_stream);
}

// The row-slab critic kernel draws the batch itself from `buf` (else the sampler is a launch of its own).  Its
// in-kernel sampler draws one-step rows only: an n-step buffer always takes the standalone sampler.
bool samples_in_kernel(const gcrl_agent *ag, const gcrl_her *buf, int64_t B) {
  return fused_ok(ag, int(B)) && ag->fuse_sampler && her_n_step(buf) == 1 && fused_sample_supported(her_geom(buf));
}

// Stage one batch (sampled from `buf`, or the caller's dense device batch) into the operand rows.
void ingest(gcrl_agent *ag, gcrl_her *buf, int64_t B, const int64_t *idx_host, const float *s, const float *a,
            const float *r, const float *ns, const float *d, const float *noise_dev, const float **noise_out,
            cudaStream_t st) {
  ag->sample_buf = nullptr;
  if (buf != nullptr) {
    GCRL_REQUIRE(her_state_dim(buf) == ag->D && her_act_dim(buf) == ag->A, "buffer / agent shape mismatch");
    GCRL_REQUIRE(her_device(buf) == ag->device, "buffer and agent live on different devices");
    if (samples_in_kernel(ag, buf, B)) {
      // row-slab path: the critic-phase kernel draws its own rows; here only the positions (host index stream)
      // and the buffer's totals travel to the device
      if (her_len(buf) < B) throw Error(GCRL_ERR_UNDERFILLED, "[ERROR] Not enough in buffer to sample");
      if (idx_host != nullptr) {
        const int64_t len = her_len(buf);
        for (int64_t i = 0; i < B; ++i)
          if (idx_host[i] < 0 || idx_host[i] >= len) throw Error(GCRL_ERR_INVALID, "sample index out of range [0, len)");
        int slot;
        char *p = ag->io_stage.acquire(size_t(B) * sizeof(int64_t), &slot);
        std::memcpy(p, idx_host, size_t(B) * sizeof(int64_t));
        GCRL_CUDA(cudaMemcpyAsync(ag->d_idx, p, size_t(B) * sizeof(int64_t), cudaMemcpyHostToDevice, st));
        ag->io_stage.release(slot, st);
      }
      ag->sample_sc = her_next_scalars(buf, idx_host != nullptr);
      ag->sample_buf = buf;
    } else {
      her_sample_into(buf, B, idx_host, ag->bs, ag->ba, ag->br0, ag->bns, ag->bd0, nullptr, st);
    }
    s = ag->bs; a = ag->ba; r = ag->br0; ns = ag->bns; d = ag->bd0;
  } else {
    GCRL_REQUIRE(s && a && r && ns && d, "NULL batch pointer");
  }
  GCRL_REQUIRE(!ag->td3 || noise_dev != nullptr, "TD3 update needs the [B, A] standard-normal noise tensor");
  if (fused_ok(ag, int(B))) {
    // the fused kernels read the dense batch in place (stable addresses for the captured graph)
    if (buf == nullptr) {
      const size_t n = size_t(B) * 4;
      GCRL_CUDA(cudaMemcpyAsync(ag->bs, s, n * ag->D, cudaMemcpyDeviceToDevice, st));
      GCRL_CUDA(cudaMemcpyAsync(ag->ba, a, n * ag->A, cudaMemcpyDeviceToDevice, st));
      GCRL_CUDA(cudaMemcpyAsync(ag->br0, r, n, cudaMemcpyDeviceToDevice, st));
      GCRL_CUDA(cudaMemcpyAsync(ag->bns, ns, n * ag->D, cudaMemcpyDeviceToDevice, st));
      GCRL_CUDA(cudaMemcpyAsync(ag->bd0, d, n, cudaMemcpyDeviceToDevice, st));
    }
  } else {
    launch_ingest_batch(s, a, r, ns, d, ag->D, ag->A, int(B), ag->sa, ag->nsa, ag->spi, ag->ldc, ag->br, ag->bd, st);
  }
  *noise_out = nullptr;
  if (ag->td3) {  // stable address for the captured graph
    GCRL_CUDA(cudaMemcpyAsync(ag->noise, noise_dev, size_t(B) * ag->A * 4, cudaMemcpyDeviceToDevice, st));
    *noise_out = ag->noise;
  }
}

// the per-update slots of n-update calls, on first use
void ensure_many(gcrl_agent *ag) {
  auto &mn = ag->many;
  if (mn.d != nullptr) return;
  mn.d = dev_alloc<char>(GCRL_MAX_MANY_STEPS * (kScalBytes + size_t(ag->maxB) * sizeof(int64_t)));
  if (ag->td3) mn.noise = dev_alloc<float>(size_t(GCRL_MAX_MANY_STEPS) * ag->maxB * ag->A);
  GCRL_CUDA(cudaHostAlloc(reinterpret_cast<void **>(&mn.h_pub), GCRL_MAX_MANY_STEPS * 64, cudaHostAllocMapped));
  std::memset(mn.h_pub, 0, GCRL_MAX_MANY_STEPS * 64);
  GCRL_CUDA(cudaHostGetDevicePointer(reinterpret_cast<void **>(&mn.d_pub), mn.h_pub, 0));
}

void check_batch(const gcrl_agent *ag, int64_t B) {
  GCRL_REQUIRE(ag != nullptr, "agent handle is NULL");
  GCRL_REQUIRE(B >= 1 && B <= ag->maxB, "batch size outside [1, max_batch]");
}

float *stage_to_device(gcrl_agent *ag, const float *host, size_t count, size_t offset_floats,
                       cudaStream_t st) {
  int slot;
  char *p = ag->io_stage.acquire(count * 4, &slot);
  std::memcpy(p, host, count * 4);
  GCRL_CUDA(cudaMemcpyAsync(ag->d_io + offset_floats, p, count * 4, cudaMemcpyHostToDevice, st));
  ag->io_stage.release(slot, st);
  return ag->d_io + offset_floats;
}

void ensure_io(gcrl_agent *ag, size_t floats, cudaStream_t st) {
  if (floats > ag->io_cap) {
    GCRL_CUDA(cudaStreamSynchronize(st));
    if (ag->d_io) GCRL_CUDA(cudaFree(ag->d_io));
    ag->io_cap = floats * 2;
    ag->d_io = dev_alloc<float>(ag->io_cap);
  }
}

// Wait until the publish block `pub` (mapped host: float[8] metrics, uint32 seq, int32 err) carries sequence number
// `seq`: the update's last optimiser kernel writes the metrics and then that word (no D2H copy, no stream
// synchronisation, no driver call on the critical path), then copy the metrics out.
void read_published(const float *pub, unsigned int want, float *metrics_host, cudaStream_t st) {
  const volatile unsigned int *seq = reinterpret_cast<const volatile unsigned int *>(pub) + 8;
  const auto t0 = std::chrono::steady_clock::now();
  unsigned long spins = 0;
  while (*seq != want) {
    if ((++spins & 0xFFFF) == 0) {
      if (cudaStreamQuery(st) != cudaErrorNotReady) {       // finished (or failed) without publishing this number
        GCRL_CUDA(cudaStreamSynchronize(st));
        if (*seq == want) break;
        throw Error(GCRL_ERR_CUDA, "the update finished without publishing its metrics");
      }
      if (std::chrono::steady_clock::now() - t0 > std::chrono::seconds(120))
        throw Error(GCRL_ERR_CUDA, "timed out waiting for the update's metrics");
    }
  }
  std::atomic_thread_fence(std::memory_order_acquire);
  std::memcpy(metrics_host, pub, 8 * sizeof(float));
}

void finish_metrics(gcrl_agent *ag, float *metrics_host, cudaStream_t st) {
  if (metrics_host == nullptr) return;
  auto dp_error = [](int err) {
    return Error(GCRL_ERR_CUDA, "data-parallel barrier timed out: rank " + std::to_string((err - 1) / 16) +
                                    " never saw the flag of rank " + std::to_string((err - 1) % 16));
  };
  if (ag->pub_valid) {
    read_published(ag->h_pub, ag->pub_seq, metrics_host, st);
    const int err = reinterpret_cast<const int *>(ag->h_pub)[9];
    if (err) throw dp_error(err);
    return;
  }
  GCRL_CUDA(cudaMemcpyAsync(metrics_host, ag->p2p.on ? ag->p2p.metrics_avg : ag->metrics, 8 * sizeof(float),
                            cudaMemcpyDeviceToHost, st));
  GCRL_CUDA(cudaStreamSynchronize(st));
  if (ag->p2p.on) {
    int err = 0;
    GCRL_CUDA(cudaMemcpy(&err, ag->p2p.err, sizeof(int), cudaMemcpyDeviceToHost));
    if (err) throw dp_error(err);
  }
}

// metrics_host[n][8] of an n-update call: the last update publishes as a single one does; stream order then has the
// earlier blocks complete
void read_many_metrics(gcrl_agent *ag, int n, float *metrics_host, cudaStream_t st) {
  if (metrics_host == nullptr) return;
  finish_metrics(ag, metrics_host + size_t(n - 1) * 8, st);
  for (int i = 0; i < n - 1; ++i)
    read_published(ag->many.h_pub + size_t(i) * 16, ag->pub_seq - unsigned(n - 1 - i), metrics_host + size_t(i) * 8, st);
}

}  // namespace

// Every entry point checks the handle's type tag: a gcrl_agent handle passed to the other family's functions would be
// reinterpreted as a different struct (garbage shapes and pointers).
static inline void require_handle(const gcrl_agent *h) {
  if (h == nullptr) throw ::gcrl::Error(GCRL_ERR_INVALID, "handle is NULL");
  if (h->magic != 0x544E4741u) throw ::gcrl::Error(GCRL_ERR_INVALID, "handle is not a DDPG / TD3 agent (gcrl_agent_create)");
}

// gcrl_agent_update_many (HER buffer `her`) and gcrl_agent_update_many_replay (uniform / prioritised buffer `rb`): one
// of the two is NULL.  Nothing moves before the last refusal: the buffer's own checks (replay_many_stage) come first.
static void update_many(gcrl_agent *ag, gcrl_her *her, gcrl_replay *rb, int64_t B, int n, const int *flags,
                        const int64_t *idx_host, const int64_t *pos_host, const double *u_host, const double *beta,
                        const float *noise_dev, const double *lr_critic, const double *lr_actor, float *metrics_host,
                        float *td_host, void *stream) {
  require_handle(ag);
  check_batch(ag, B);
  GCRL_REQUIRE(her != nullptr || rb != nullptr, "buffer handle is NULL");
  GCRL_REQUIRE(n >= 1 && n <= GCRL_MAX_MANY_STEPS, "n must be in [1, GCRL_MAX_MANY_STEPS]");
  GCRL_REQUIRE(flags != nullptr && lr_critic != nullptr && lr_actor != nullptr, "NULL flags / learning rates");
  const bool per = rb != nullptr && replay_prioritized(rb);
  for (int i = 0; i < n; ++i) {
    if (her != nullptr) {
      GCRL_REQUIRE((flags[i] & ~3) == 0, "flags of an n-update call may hold bit0 and bit1 only");
    } else {
      GCRL_REQUIRE((flags[i] & ~11) == 0, "flags of an n-update call from a replay buffer may hold bits 0, 1 and 3 only");
      GCRL_REQUIRE(((flags[i] & 8) != 0) == per, "flags bit3 must be set exactly when the buffer is prioritised");
    }
  }
  GCRL_REQUIRE(!ag->p2p.on, "n-update calls are not available under peer-memory data parallelism");
  GCRL_REQUIRE(!ag->dp_open, "a phase-wise data-parallel update is open (phase 3 not issued)");
  if (her != nullptr) {
    GCRL_REQUIRE(her_state_dim(her) == ag->D && her_act_dim(her) == ag->A, "buffer / agent shape mismatch");
    GCRL_REQUIRE(her_device(her) == ag->device, "buffer and agent live on different devices");
  } else {
    GCRL_REQUIRE(replay_state_dim(rb) == ag->D && replay_act_dim(rb) == ag->A, "buffer / agent shape mismatch");
    GCRL_REQUIRE(replay_device(rb) == ag->device, "buffer and agent live on different devices");
  }
  GCRL_REQUIRE(!ag->td3 || noise_dev != nullptr, "TD3 update needs the [n, B, A] standard-normal noise tensor");
  if (her != nullptr) {
    const int64_t len = her_len(her);
    if (len < B) throw Error(GCRL_ERR_UNDERFILLED, "[ERROR] Not enough in buffer to sample");
    if (idx_host != nullptr)
      for (int64_t i = 0; i < int64_t(n) * B; ++i)
        if (idx_host[i] < 0 || idx_host[i] >= len) throw Error(GCRL_ERR_INVALID, "sample index out of range [0, len)");
  }
  GCRL_CUDA(cudaSetDevice(ag->device));
  cudaStream_t st = as_stream(stream);
  if (rb != nullptr) replay_many_stage(rb, B, n, pos_host, u_host, beta, st);
  auto &mn = ag->many;
  ensure_many(ag);
  if (per && mn.td == nullptr) mn.td = dev_alloc<float>(size_t(GCRL_MAX_MANY_STEPS) * ag->maxB);
  AdamStepGuard guard(ag);
  if (her != nullptr) guard.keep_draws(her);
  ag->per_on = per;
  // every update's scalars (HER: the device stream's draw epochs in order), then every update's positions: ONE copy
  const size_t scal = size_t(n) * kScalBytes, pos = idx_host != nullptr ? size_t(n) * B * sizeof(int64_t) : 0;
  int slot;
  char *p = ag->io_stage.acquire(scal + pos, &slot);
  for (int i = 0; i < n; ++i) {
    if (her != nullptr) ag->sample_sc = her_next_scalars(her, idx_host != nullptr);
    fill_scalars(ag, lr_critic[i], lr_actor[i], (flags[i] & 1) != 0, her != nullptr ? ag->sample_sc : SampleScalars{},
                 p + size_t(i) * kScalBytes);
  }
  if (pos) std::memcpy(p + scal, idx_host, pos);
  GCRL_CUDA(cudaMemcpyAsync(mn.d, p, scal + pos, cudaMemcpyHostToDevice, st));
  ag->io_stage.release(slot, st);
  if (ag->td3)   // stable addresses for the captured graph
    GCRL_CUDA(cudaMemcpyAsync(mn.noise, noise_dev, size_t(n) * B * ag->A * 4, cudaMemcpyDeviceToDevice, st));
  ag->sample_buf = her != nullptr && samples_in_kernel(ag, her, B) ? her : nullptr;
  run_many(ag, her, rb, int(B), n, flags, st);
  ag->pub_valid = true;
  guard.commit();
  read_many_metrics(ag, n, metrics_host, st);
  if (per && td_host != nullptr) {
    // ONE read-back per call; to pageable memory the copy returns once it (and the updates before it) completed
    std::vector<float> rows(size_t(n) * B);
    GCRL_CUDA(cudaMemcpyAsync(rows.data(), mn.td, rows.size() * sizeof(float), cudaMemcpyDeviceToHost, st));
    std::memcpy(td_host, rows.data(), rows.size() * sizeof(float));
  }
}

extern "C" {

int gcrl_agent_create(gcrl_agent **out, int device, const gcrl_agent_config *cfg) {
  GCRL_API_BEGIN
  GCRL_REQUIRE(out != nullptr && cfg != nullptr, "NULL argument");
  GCRL_REQUIRE(cfg->algo == GCRL_ALGO_DDPG || cfg->algo == GCRL_ALGO_TD3, "unknown algo");
  GCRL_REQUIRE(cfg->state_dim >= 1 && cfg->act_dim >= 1 && cfg->act_dim <= 4,
               "need state_dim >= 1 and 1 <= act_dim <= 4");
  GCRL_REQUIRE(cfg->hidden_dim >= 1 && cfg->hidden_dim <= 4096, "hidden_dim outside [1, 4096]");
  GCRL_REQUIRE(cfg->layer_count >= 1 && cfg->layer_count <= 6, "layer_count outside [1, 6]");
  GCRL_REQUIRE(cfg->max_batch >= 1, "max_batch must be >= 1");
  GCRL_REQUIRE(cfg->precision >= 0 && cfg->precision <= 2, "precision must be 0 (fp32 FFMA), 1 (tensor cores for large batches) or 2 (tensor cores whenever supported)");
  GCRL_CUDA(cudaSetDevice(device));
  auto *ag = new gcrl_agent();
  try {
    ag->device = device;
    ag->cfg = *cfg;
    ag->D = cfg->state_dim; ag->A = cfg->act_dim; ag->H = cfg->hidden_dim; ag->L = cfg->layer_count;
    ag->ldh = pad4(ag->H);
    ag->ldc = pad4(ag->D + ag->A);
    ag->maxB = cfg->max_batch;
    ag->td3 = cfg->algo == GCRL_ALGO_TD3;
    GCRL_REQUIRE(ag->maxB <= int64_t(kMaxSplits) * 512, "max_batch too large for the partial buffers");
    const int D = ag->D, A = ag->A, H = ag->H, L = ag->L;
    auto init_net = [&](int id, int in, int out, bool trainable) {
      MlpParams &n = ag->net[id];
      n.layout(in, H, out, L);
      n.init_copies(0, n.layers, false);   // W^T of every layer: the row-slab kernels read Wt, prefetch all of flatT
      n.alloc(trainable);
      ag->has[id] = true;
    };
    init_net(ACTOR, D, A, true);
    init_net(CRITIC1, D + A, 1, true);
    init_net(T_ACTOR, D, A, false);
    init_net(T_CRITIC1, D + A, 1, false);
    if (ag->td3) {
      init_net(CRITIC2, D + A, 1, true);
      init_net(T_CRITIC2, D + A, 1, false);
    }
    const int64_t mb = ag->maxB;
    ag->acts_actor.init(L, mb, ag->ldh);
    ag->acts_c1.init(L, mb, ag->ldh);
    if (ag->td3) ag->acts_c2.init(L, mb, ag->ldh);
    ag->acts_tgt.init(L, mb, ag->ldh);
    for (auto &p : ag->dz) p = dev_alloc<float>(size_t(mb) * ag->ldh);
    ag->sa = dev_alloc<float>(size_t(mb) * ag->ldc);
    ag->nsa = dev_alloc<float>(size_t(mb) * ag->ldc);
    ag->spi = dev_alloc<float>(size_t(mb) * ag->ldc);
    for (float **p : {&ag->q1, &ag->q2, &ag->qt1, &ag->qt2, &ag->yv, &ag->br, &ag->bd, &ag->br0, &ag->bd0})
      *p = dev_alloc<float>(size_t(mb));
    ag->dz_act = dev_alloc<float>(size_t(mb) * 4);
    ag->noise = dev_alloc<float>(size_t(mb) * 4);
    for (int l = 0; l < L; ++l) ag->dzl.push_back(dev_alloc<float>(size_t(mb) * ag->ldh));
    ag->dzh = dev_alloc<float>(size_t(mb));
    ag->per_w = dev_alloc<float>(size_t(mb));
    ag->per_td = dev_alloc<float>(size_t(mb));
    const char *nf = getenv("GCRL_B200_NO_FUSED");
    ag->use_fused = !(nf && nf[0] == '1');
    ag->bs = dev_alloc<float>(size_t(mb) * D);
    ag->bns = dev_alloc<float>(size_t(mb) * D);
    ag->ba = dev_alloc<float>(size_t(mb) * A);
    ag->slab = std::max(ag->net[ACTOR].total, ag->net[CRITIC1].total);
    ag->partials = dev_alloc<float>(size_t(kMaxSplits) * ag->slab);
    ag->metric_partials = dev_alloc<float>(size_t(256) * 4);
    const int ht = (H + 31) / 32;              // 32 x 32 output tiles of the largest net (multi_wgrad_kernel)
    const int wtiles = ht * ((D + A + 31) / 32) + (L - 1) * ht * ht + ht + 8;
    ag->sumsq = dev_alloc<float>(size_t(std::max(reduce_grid(int(ag->slab)), wtiles)) + 8);
    ag->metrics = dev_alloc<float>(8);
    GCRL_CUDA(cudaMemset(ag->metrics, 0, 8 * sizeof(float)));
    ag->d_scalars = reinterpret_cast<StepScalars *>(dev_alloc<char>(sizeof(StepScalars) + sizeof(SampleScalars)));
    ag->d_sample_sc = reinterpret_cast<SampleScalars *>(ag->d_scalars + 1);
    ag->d_idx = dev_alloc<int64_t>(size_t(mb));
    GCRL_CUDA(cudaHostAlloc(reinterpret_cast<void **>(&ag->h_pub), 64, cudaHostAllocMapped));
    std::memset(ag->h_pub, 0, 64);
    GCRL_CUDA(cudaHostGetDevicePointer(reinterpret_cast<void **>(&ag->d_pub), ag->h_pub, 0));
    const char *nfs = getenv("GCRL_B200_NO_FUSED_SAMPLER");
    ag->fuse_sampler = !(nfs && nfs[0] == '1');
    ag->scal_stage.init(256);
    GCRL_CUDA(cudaStreamCreateWithFlags(&ag->cap_stream, cudaStreamNonBlocking));
    ag->use_graphs = graphs_enabled();
    ag->io_stage.init(size_t(1) << 16);
    if (ag->cfg.precision >= 1) {
      // the TF32 halves of tcgen05 come last: the row-slab kernels' buffers keep their places (next to each other,
      // in the order tmap, Wt, p, g, m, v), without which B = 256 steps ran 0.5 % slower on a B200
      tc_dense_init();
      for (int i = 0; i < NUM_NETS; ++i)
        if (ag->has[i]) ag->net[i].copies.alloc_halves();
    }
  } catch (...) {
    delete ag;
    throw;
  }
  *out = ag;
  GCRL_API_END
}

int gcrl_agent_destroy(gcrl_agent *ag) {
  GCRL_API_BEGIN
  if (ag == nullptr) return GCRL_OK;
  cudaSetDevice(ag->device);
  cudaDeviceSynchronize();
  for (auto &kv : ag->graphs) cudaGraphExecDestroy(kv.second.exec);
  ag->many.graphs.clear();
  if (ag->many.d) cudaFree(ag->many.d);
  if (ag->many.noise) cudaFree(ag->many.noise);
  if (ag->many.h_pub) cudaFreeHost(ag->many.h_pub);
  if (ag->many.td) cudaFree(ag->many.td);
  for (void *p : ag->p2p.opened) cudaIpcCloseMemHandle(p);
  for (void *p : {(void *)ag->p2p.flags, (void *)ag->p2p.epoch, (void *)ag->p2p.ticket, (void *)ag->p2p.wticket, (void *)ag->p2p.go,
                  (void *)ag->p2p.err, (void *)ag->p2p.outbox,
                  (void *)ag->p2p.metrics_avg, (void *)ag->p2p.d_peer_flags, (void *)ag->p2p.d_peer_outbox})
    if (p) cudaFree(p);
  for (int i = 0; i < NUM_NETS; ++i) {
    if (ag->p2p.gavg[i]) cudaFree(ag->p2p.gavg[i]);
    if (ag->p2p.d_peer_g[i]) cudaFree(ag->p2p.d_peer_g[i]);
  }
  for (int i = 0; i < NUM_NETS; ++i)
    if (ag->has[i]) ag->net[i].destroy();
  ag->acts_actor.destroy(); ag->acts_c1.destroy(); ag->acts_c2.destroy(); ag->acts_tgt.destroy();
  for (float *p : {ag->dz[0], ag->dz[1], ag->sa, ag->nsa, ag->spi, ag->q1, ag->q2, ag->qt1, ag->qt2, ag->yv,
                   ag->dz_act, ag->br, ag->bd, ag->bs, ag->ba, ag->bns, ag->br0, ag->bd0, ag->partials,
                   ag->metric_partials, ag->sumsq, ag->metrics, ag->d_io, ag->noise, ag->dzh, ag->per_w, ag->per_td})
    if (p) cudaFree(p);
  for (float *p : ag->dzl) cudaFree(p);
  cudaFree(ag->d_scalars);
  cudaFree(ag->d_idx);
  if (ag->h_pub) cudaFreeHost(ag->h_pub);
  if (ag->cap_stream) cudaStreamDestroy(ag->cap_stream);
  ag->scal_stage.destroy();
  ag->io_stage.destroy();
  delete ag;
  GCRL_API_END
}

int gcrl_agent_num_layers(const gcrl_agent *ag, int net) {
  if (ag == nullptr || ag->magic != 0x544E4741u || net < 0 || net >= NUM_NETS || !ag->has[net]) return -1;
  return ag->net[net].layers;
}

int gcrl_agent_layer_shape(const gcrl_agent *ag, int net, int layer, int *out_dim, int *in_dim) {
  GCRL_API_BEGIN
  require_handle(ag);
  GCRL_REQUIRE(ag && net >= 0 && net < NUM_NETS && ag->has[net], "bad network id");
  GCRL_REQUIRE(layer >= 0 && layer < ag->net[net].layers, "bad layer index");
  if (out_dim) *out_dim = ag->net[net].out_d[layer];
  if (in_dim) *in_dim = ag->net[net].in_d[layer];
  GCRL_API_END
}

int gcrl_agent_set_layer(gcrl_agent *ag, int net, int layer, const float *weight_host,
                         const float *bias_host, void *stream) {
  GCRL_API_BEGIN
  require_handle(ag);
  GCRL_REQUIRE(ag && net >= 0 && net < NUM_NETS && ag->has[net], "bad network id");
  MlpParams &n = ag->net[net];
  GCRL_REQUIRE(layer >= 0 && layer < n.layers && weight_host && bias_host, "bad layer / NULL data");
  GCRL_CUDA(cudaSetDevice(ag->device));
  cudaStream_t st = as_stream(stream);
  upload_rows(n.p + n.w_off[layer], weight_host, n.out_d[layer], n.in_d[layer], n.ldw[layer], st);
  upload_rows(n.p + n.b_off[layer], bias_host, 1, n.out_d[layer], n.out_d[layer], st);
  n.copies.weights_changed(n.p, st);
  GCRL_CUDA(cudaStreamSynchronize(st));
  GCRL_API_END
}

int gcrl_agent_get_layer(gcrl_agent *ag, int net, int layer, float *weight_host, float *bias_host,
                         void *stream) {
  GCRL_API_BEGIN
  require_handle(ag);
  GCRL_REQUIRE(ag && net >= 0 && net < NUM_NETS && ag->has[net], "bad network id");
  MlpParams &n = ag->net[net];
  GCRL_REQUIRE(layer >= 0 && layer < n.layers, "bad layer index");
  GCRL_CUDA(cudaSetDevice(ag->device));
  cudaStream_t st = as_stream(stream);
  if (weight_host) download_rows(weight_host, n.p + n.w_off[layer], n.out_d[layer], n.in_d[layer], n.ldw[layer], st);
  if (bias_host) download_rows(bias_host, n.p + n.b_off[layer], 1, n.out_d[layer], n.out_d[layer], st);
  GCRL_API_END
}

// Adam state of one layer of a trainable network, in the layout of set_layer / get_layer
// (exp_avg = m, exp_avg_sq = v of torch.optim.Adam); `set` != 0 uploads, else downloads.
static int adam_layer_io(gcrl_agent *ag, int net, int layer, float *m_w, float *m_b, float *v_w, float *v_b, int set,
                         void *stream) {
  GCRL_API_BEGIN
  require_handle(ag);
  GCRL_REQUIRE(ag && net >= 0 && net < NUM_NETS && ag->has[net] && ag->net[net].m, "bad (or non-trainable) network id");
  MlpParams &n = ag->net[net];
  GCRL_REQUIRE(layer >= 0 && layer < n.layers && m_w && m_b && v_w && v_b, "bad layer / NULL data");
  GCRL_CUDA(cudaSetDevice(ag->device));
  cudaStream_t st = as_stream(stream);
  const int o = n.out_d[layer], i = n.in_d[layer], ld = n.ldw[layer];
  float *dev[2] = {n.m, n.v};
  float *hw[2] = {m_w, v_w}, *hb[2] = {m_b, v_b};
  for (int k = 0; k < 2; ++k) {
    if (set) {
      upload_rows(dev[k] + n.w_off[layer], hw[k], o, i, ld, st);
      upload_rows(dev[k] + n.b_off[layer], hb[k], 1, o, o, st);
    } else {
      download_rows(hw[k], dev[k] + n.w_off[layer], o, i, ld, st);
      download_rows(hb[k], dev[k] + n.b_off[layer], 1, o, o, st);
    }
  }
  GCRL_API_END
}

int gcrl_agent_get_adam_layer(gcrl_agent *ag, int net, int layer, float *m_w, float *m_b, float *v_w, float *v_b,
                              void *stream) {
  return adam_layer_io(ag, net, layer, m_w, m_b, v_w, v_b, 0, stream);
}
int gcrl_agent_set_adam_layer(gcrl_agent *ag, int net, int layer, const float *m_w, const float *m_b, const float *v_w,
                              const float *v_b, void *stream) {
  return adam_layer_io(ag, net, layer, const_cast<float *>(m_w), const_cast<float *>(m_b), const_cast<float *>(v_w),
                       const_cast<float *>(v_b), 1, stream);
}
int gcrl_agent_get_adam_step(gcrl_agent *ag, int net, int *step) {
  GCRL_API_BEGIN
  require_handle(ag);
  GCRL_REQUIRE(ag && step && net >= 0 && net < NUM_NETS && ag->has[net] && ag->net[net].m, "bad network id");
  *step = ag->adam_t[net];
  GCRL_API_END
}
int gcrl_agent_set_adam_step(gcrl_agent *ag, int net, int step) {
  GCRL_API_BEGIN
  require_handle(ag);
  GCRL_REQUIRE(ag && step >= 0 && net >= 0 && net < NUM_NETS && ag->has[net] && ag->net[net].m, "bad network id");
  ag->adam_t[net] = step;
  GCRL_API_END
}

int gcrl_agent_hard_update(gcrl_agent *ag, void *stream) {
  GCRL_API_BEGIN
  require_handle(ag);
  GCRL_REQUIRE(ag != nullptr, "agent handle is NULL");
  GCRL_CUDA(cudaSetDevice(ag->device));
  cudaStream_t st = as_stream(stream);
  const int pairs[3][2] = {{T_ACTOR, ACTOR}, {T_CRITIC1, CRITIC1}, {T_CRITIC2, CRITIC2}};
  for (auto &pr : pairs)
    if (ag->has[pr[0]]) {
      MlpParams &t = ag->net[pr[0]];
      const MlpParams &src = ag->net[pr[1]];
      GCRL_CUDA(cudaMemcpyAsync(t.p, src.p, size_t(src.total) * 4, cudaMemcpyDeviceToDevice, st));
      GCRL_CUDA(cudaMemcpyAsync(t.copies.pT, src.copies.pT, size_t(src.copies.total_t) * 4, cudaMemcpyDeviceToDevice,
                                st));
      t.copies.stale = true;
    }
  GCRL_API_END
}

// Polyak step theta_t <- tau theta + (1 - tau) theta_t of selected target networks, outside update()
// (DDPG.update_target_network(hard_update=False, tau), src/agent.py:1259-1271; TD3 update_actor / update_critic
// :117-132).  which: bit0 actor, bit1 critic(s).
int gcrl_agent_soft_update(gcrl_agent *ag, int which, double tau, void *stream) {
  GCRL_API_BEGIN
  require_handle(ag);
  GCRL_REQUIRE(which >= 1 && which <= 3 && tau >= 0.0 && tau <= 1.0, "which in 1..3, tau in [0, 1]");
  GCRL_CUDA(cudaSetDevice(ag->device));
  cudaStream_t st = as_stream(stream);
  const int pairs[3][3] = {{T_ACTOR, ACTOR, 1}, {T_CRITIC1, CRITIC1, 2}, {T_CRITIC2, CRITIC2, 2}};
  for (auto &pr : pairs)
    if ((which & pr[2]) && ag->has[pr[0]]) {
      MlpParams &t = ag->net[pr[0]];
      const MlpParams &srcn = ag->net[pr[1]];
      launch_polyak(t.p, srcn.p, srcn.total, float(tau), float(1.0 - tau), srcn.copies.tmap, t.copies.pT, st);
      t.copies.stale = true;
    }
  GCRL_API_END
}

int gcrl_agent_reset_optim(gcrl_agent *ag, void *stream) {
  GCRL_API_BEGIN
  require_handle(ag);
  GCRL_REQUIRE(ag != nullptr, "agent handle is NULL");
  GCRL_CUDA(cudaSetDevice(ag->device));
  cudaStream_t st = as_stream(stream);
  for (int i : {ACTOR, CRITIC1, CRITIC2})
    if (ag->has[i]) {
      GCRL_CUDA(cudaMemsetAsync(ag->net[i].m, 0, size_t(ag->net[i].total) * 4, st));
      GCRL_CUDA(cudaMemsetAsync(ag->net[i].v, 0, size_t(ag->net[i].total) * 4, st));
      ag->adam_t[i] = 0;
    }
  GCRL_API_END
}

int gcrl_agent_update_batch(gcrl_agent *ag, int64_t B, const float *s_dev, const float *a_dev,
                            const float *r_dev, const float *ns_dev, const float *d_dev,
                            const float *noise_dev, double lr_critic, double lr_actor, int flags,
                            float *metrics_host, void *stream) {
  GCRL_API_BEGIN
  GCRL_NVTX("gcrl_agent_update_batch");
  require_handle(ag);
  check_batch(ag, B);
  GCRL_CUDA(cudaSetDevice(ag->device));
  cudaStream_t st = as_stream(stream);
  const float *noise = nullptr;
  AdamStepGuard guard(ag);
  ag->per_on = (flags & 8) != 0;
  ingest(ag, nullptr, B, nullptr, s_dev, a_dev, r_dev, ns_dev, d_dev, noise_dev, &noise, st);
  write_scalars(ag, lr_critic, lr_actor, (flags & 1) != 0, st);
  run_update(ag, int(B), noise, flags, PH_ALL, st);
  ag->pub_valid = true;
  guard.commit();
  finish_metrics(ag, metrics_host, st);
  GCRL_API_END
}

int gcrl_agent_update_from_buffer(gcrl_agent *ag, gcrl_her *buf, int64_t B, const int64_t *idx_host,
                                  const float *noise_dev, double lr_critic, double lr_actor, int flags,
                                  float *metrics_host, void *stream) {
  GCRL_API_BEGIN
  GCRL_NVTX("gcrl_agent_update_from_buffer");
  require_handle(ag);
  check_batch(ag, B);
  GCRL_REQUIRE(buf != nullptr, "buffer handle is NULL");
  GCRL_CUDA(cudaSetDevice(ag->device));
  cudaStream_t st = as_stream(stream);
  const float *noise = nullptr;
  AdamStepGuard guard(ag);
  ag->per_on = (flags & 8) != 0;
  ingest(ag, buf, B, idx_host, nullptr, nullptr, nullptr, nullptr, nullptr, noise_dev, &noise, st);
  write_scalars(ag, lr_critic, lr_actor, (flags & 1) != 0, st);
  run_update(ag, int(B), noise, flags, PH_ALL, st);
  ag->pub_valid = true;
  guard.commit();
  finish_metrics(ag, metrics_host, st);
  GCRL_API_END
}

int gcrl_agent_update_many(gcrl_agent *ag, gcrl_her *buf, int64_t B, int n, const int *flags, const int64_t *idx_host,
                           const float *noise_dev, const double *lr_critic, const double *lr_actor, float *metrics_host,
                           void *stream) {
  GCRL_API_BEGIN
  GCRL_NVTX("gcrl_agent_update_many");
  update_many(ag, buf, nullptr, B, n, flags, idx_host, nullptr, nullptr, nullptr, noise_dev, lr_critic, lr_actor,
              metrics_host, nullptr, stream);
  GCRL_API_END
}

int gcrl_agent_update_many_replay(gcrl_agent *ag, gcrl_replay *buf, int64_t B, int n, const int *flags,
                                  const int64_t *pos_host, const double *u_host, const double *beta,
                                  const float *noise_dev, const double *lr_critic, const double *lr_actor,
                                  float *metrics_host, float *td_host, void *stream) {
  GCRL_API_BEGIN
  GCRL_NVTX("gcrl_agent_update_many_replay");
  update_many(ag, nullptr, buf, B, n, flags, nullptr, pos_host, u_host, beta, noise_dev, lr_critic, lr_actor,
              metrics_host, td_host, stream);
  GCRL_API_END
}

int gcrl_agent_read_metrics(gcrl_agent *ag, float *metrics_host, void *stream) {
  GCRL_API_BEGIN
  require_handle(ag);
  GCRL_REQUIRE(ag != nullptr && metrics_host != nullptr, "NULL argument");
  GCRL_CUDA(cudaSetDevice(ag->device));
  finish_metrics(ag, metrics_host, as_stream(stream));
  GCRL_API_END
}

int gcrl_agent_act(gcrl_agent *ag, int64_t n, const float *obs_host, float *act_host, void *stream) {
  GCRL_API_BEGIN
  GCRL_NVTX("gcrl_agent_act");
  require_handle(ag);
  check_batch(ag, n);
  GCRL_REQUIRE(obs_host && act_host, "NULL argument");
  GCRL_CUDA(cudaSetDevice(ag->device));
  cudaStream_t st = as_stream(stream);
  const int D = ag->D, A = ag->A, L = ag->L;
  ensure_io(ag, size_t(n) * (D + 4), st);
  float *obs = stage_to_device(ag, obs_host, size_t(n) * D, 0, st);
  // uses the actor-phase scratch (spi / acts_actor): select_action never overlaps an update
  launch_pack_rows(obs, D, nullptr, A, ag->spi, ag->ldc, int(n), st);
  if (engine_tc(ag, int(n))) ensure_split(ag, st);
  const MlpParams &actor = ag->net[ACTOR];
  forward_hidden(ag, actor, ag->spi, ag->ldc, D, ag->acts_actor, int(n), st);
  float *out = ag->d_io + size_t(n) * D;
  launch_head_fwd(ag->acts_actor.h[L - 1], ag->ldh, actor.W(L), actor.ldw[L], actor.b(L), out, A, 0, int(n),
                  ag->H, A, 1, st);
  GCRL_CUDA(cudaMemcpyAsync(act_host, out, size_t(n) * A * 4, cudaMemcpyDeviceToHost, st));
  GCRL_CUDA(cudaStreamSynchronize(st));
  GCRL_API_END
}

int gcrl_agent_q(gcrl_agent *ag, int64_t n, const float *obs_host, const float *act_host, float *q_host,
                 void *stream) {
  GCRL_API_BEGIN
  require_handle(ag);
  check_batch(ag, n);
  GCRL_REQUIRE(obs_host && act_host && q_host, "NULL argument");
  GCRL_CUDA(cudaSetDevice(ag->device));
  cudaStream_t st = as_stream(stream);
  const int D = ag->D, A = ag->A, L = ag->L;
  ensure_io(ag, size_t(n) * (D + A + 1), st);
  float *obs = stage_to_device(ag, obs_host, size_t(n) * D, 0, st);
  float *act = stage_to_device(ag, act_host, size_t(n) * A, size_t(n) * D, st);
  launch_pack_rows(obs, D, act, A, ag->spi, ag->ldc, int(n), st);
  if (engine_tc(ag, int(n))) ensure_split(ag, st);
  const MlpParams &c = ag->net[CRITIC1];
  forward_hidden(ag, c, ag->spi, ag->ldc, D + A, ag->acts_c1, int(n), st);
  float *out = ag->d_io + size_t(n) * (D + A);
  launch_head_fwd(ag->acts_c1.h[L - 1], ag->ldh, c.W(L), c.ldw[L], c.b(L), out, 1, 0, int(n), ag->H, 1, 0, st);
  GCRL_CUDA(cudaMemcpyAsync(q_host, out, size_t(n) * 4, cudaMemcpyDeviceToHost, st));
  GCRL_CUDA(cudaStreamSynchronize(st));
  GCRL_API_END
}

int gcrl_agent_per_buffers(gcrl_agent *ag, float **weights_dev, float **td_dev) {
  GCRL_API_BEGIN
  require_handle(ag);
  GCRL_REQUIRE(ag != nullptr && weights_dev != nullptr && td_dev != nullptr, "NULL argument");
  *weights_dev = ag->per_w;
  *td_dev = ag->per_td;
  GCRL_API_END
}

// ---- data-parallel phase hooks ---------------------------------------------------------------------
int gcrl_agent_update_phase(gcrl_agent *ag, int phase, gcrl_her *buf, int64_t B, const int64_t *idx_host,
                            const float *s_dev, const float *a_dev, const float *r_dev, const float *ns_dev,
                            const float *d_dev, const float *noise_dev, double lr_critic, double lr_actor,
                            int flags, void *stream) {
  GCRL_API_BEGIN
  GCRL_NVTX("gcrl_agent_update_phase");
  require_handle(ag);
  check_batch(ag, B);
  GCRL_REQUIRE(phase >= 0 && phase <= 3, "phase must be 0..3");
  GCRL_CUDA(cudaSetDevice(ag->device));
  cudaStream_t st = as_stream(stream);
  if (phase == 0) {
    const float *noise = nullptr;
    AdamStepGuard guard(ag);
    ag->per_on = (flags & 8) != 0;
    ingest(ag, buf, B, idx_host, s_dev, a_dev, r_dev, ns_dev, d_dev, noise_dev, &noise, st);
    write_scalars(ag, lr_critic, lr_actor, (flags & 1) != 0, st);
    ag->dp_B = int(B);
    ag->dp_flags = flags;
    run_update(ag, int(B), noise, flags, PH_CGRAD, st);
    ag->pub_valid = false;                 // phase-cut update: metrics through the D2H copy
    ag->dp_open = true;
    guard.commit();
  } else {
    GCRL_REQUIRE(ag->dp_B == int(B) && ag->dp_flags == flags, "phase 1..3 must follow phase 0 of the same update");
    run_update(ag, int(B), ag->td3 ? ag->noise : nullptr, flags, phase == 1 ? PH_CSTEP : (phase == 2 ? PH_AGRAD : PH_ASTEP), st);
    if (phase == 3) ag->dp_open = false;
  }
  GCRL_API_END
}

int gcrl_agent_time_critic_kernel(gcrl_agent *ag, int64_t B, int iters, float *ms_per_launch, void *stream) {
  GCRL_API_BEGIN
  require_handle(ag);
  check_batch(ag, B);
  GCRL_REQUIRE(iters >= 1 && ms_per_launch != nullptr, "bad argument");
  GCRL_REQUIRE(fused_ok(ag, int(B)), "the fused critic-phase kernel does not serve this batch / shape");
  GCRL_CUDA(cudaSetDevice(ag->device));
  cudaStream_t st = as_stream(stream);
  gcrl_her *const sampled = ag->sample_buf;        // time the kernel on the resident dense batch
  ag->sample_buf = nullptr;
  const FusedCriticArgs a = fused_critic_args(ag, int(B));
  ag->sample_buf = sampled;
  cudaEvent_t e0, e1;
  GCRL_CUDA(cudaEventCreate(&e0));
  GCRL_CUDA(cudaEventCreate(&e1));
  for (int i = 0; i < 3; ++i) launch_fused_critic(a, st);
  GCRL_CUDA(cudaEventRecord(e0, st));
  for (int i = 0; i < iters; ++i) launch_fused_critic(a, st);
  GCRL_CUDA(cudaEventRecord(e1, st));
  GCRL_CUDA(cudaEventSynchronize(e1));
  float ms = 0.f;
  GCRL_CUDA(cudaEventElapsedTime(&ms, e0, e1));
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  *ms_per_launch = ms / float(iters);
  GCRL_API_END
}

// ---- data-parallel averaging over NVLink peer memory ---------------------------------------------------
// Buffers a rank shares with its peers, in this order: flags, metrics outbox, then the flat gradient of every
// trainable network (actor, critic, critic_2 for TD3).
static int dp_items(gcrl_agent *ag, void **ptrs) {
  int n = 0;
  ptrs[n++] = ag->p2p.flags;
  ptrs[n++] = ag->p2p.outbox;
  for (int id : {int(ACTOR), int(CRITIC1), int(CRITIC2)})
    if (ag->has[id]) ptrs[n++] = ag->net[id].g;
  return n;
}

int gcrl_agent_dp_export(gcrl_agent *ag, unsigned char *handles /*[n_items][64]*/, int *n_items) {
  GCRL_API_BEGIN
  require_handle(ag);
  GCRL_REQUIRE(ag != nullptr && n_items != nullptr, "NULL argument");
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
  GCRL_CUDA(cudaSetDevice(ag->device));
  auto &pp = ag->p2p;
  if (pp.flags == nullptr) {
    pp.flags = dev_alloc<unsigned int>(8);
    pp.epoch = dev_alloc<unsigned int>(1);
    pp.ticket = dev_alloc<unsigned int>(1);
    pp.wticket = dev_alloc<unsigned int>(1);
    GCRL_CUDA(cudaMemset(pp.wticket, 0, sizeof(unsigned int)));
    pp.go = dev_alloc<unsigned int>(1);
    GCRL_CUDA(cudaMemset(pp.go, 0, sizeof(unsigned int)));
    pp.err = dev_alloc<int>(1);
    pp.outbox = dev_alloc<float>(16);
    pp.metrics_avg = dev_alloc<float>(8);
    GCRL_CUDA(cudaMemset(pp.flags, 0, 8 * sizeof(unsigned int)));
    GCRL_CUDA(cudaMemset(pp.epoch, 0, sizeof(unsigned int)));
    GCRL_CUDA(cudaMemset(pp.ticket, 0, sizeof(unsigned int)));
    GCRL_CUDA(cudaMemset(pp.err, 0, sizeof(int)));
    GCRL_CUDA(cudaMemset(pp.outbox, 0, 16 * sizeof(float)));
    GCRL_CUDA(cudaMemset(pp.metrics_avg, 0, 8 * sizeof(float)));
    GCRL_CUDA(cudaDeviceSynchronize());
  }
  void *ptrs[8];
  const int n = dp_items(ag, ptrs);
  *n_items = n;
  if (handles != nullptr)
    for (int i = 0; i < n; ++i)
      GCRL_CUDA(cudaIpcGetMemHandle(reinterpret_cast<cudaIpcMemHandle_t *>(handles + size_t(i) * 64), ptrs[i]));
  GCRL_API_END
}

int gcrl_agent_dp_connect(gcrl_agent *ag, int rank, int world, const unsigned char *all_handles /*[world][n_items][64]*/) {
  GCRL_API_BEGIN
  require_handle(ag);
  GCRL_REQUIRE(ag != nullptr && all_handles != nullptr, "NULL argument");
  GCRL_REQUIRE(world >= 1 && world <= 8 && rank >= 0 && rank < world, "need 1 <= world <= 8 and 0 <= rank < world");
  GCRL_REQUIRE(ag->p2p.flags != nullptr, "call gcrl_agent_dp_export first");
  GCRL_CUDA(cudaSetDevice(ag->device));
  auto &pp = ag->p2p;
  void *mine[8];
  const int n = dp_items(ag, mine);
  std::vector<std::vector<void *>> peer(static_cast<size_t>(world), std::vector<void *>(static_cast<size_t>(n), nullptr));
  for (int r = 0; r < world; ++r)
    for (int i = 0; i < n; ++i) {
      if (r == rank) { peer[r][i] = mine[i]; continue; }
      cudaIpcMemHandle_t h;
      std::memcpy(&h, all_handles + (size_t(r) * n + i) * 64, 64);
      void *p = nullptr;
      GCRL_CUDA(cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess));
      pp.opened.push_back(p);
      peer[r][i] = p;
    }
  auto upload = [&](int item) {
    std::vector<void *> v(static_cast<size_t>(world), nullptr);
    for (int r = 0; r < world; ++r) v[size_t(r)] = peer[size_t(r)][size_t(item)];
    void **d = dev_alloc<void *>(size_t(world));
    GCRL_CUDA(cudaMemcpy(d, v.data(), size_t(world) * sizeof(void *), cudaMemcpyHostToDevice));
    return d;
  };
  pp.d_peer_flags = reinterpret_cast<unsigned int **>(upload(0));
  pp.d_peer_outbox = reinterpret_cast<float **>(upload(1));
  int item = 2;
  for (int id : {int(ACTOR), int(CRITIC1), int(CRITIC2)})
    if (ag->has[id]) {
      pp.d_peer_g[id] = reinterpret_cast<float **>(upload(item++));
      pp.gavg[id] = dev_alloc<float>(size_t(ag->net[id].total));
      GCRL_CUDA(cudaMemset(pp.gavg[id], 0, size_t(ag->net[id].total) * 4));
    }
  pp.rank = rank; pp.world = world; pp.on = true;
  for (auto &kv : ag->graphs) cudaGraphExecDestroy(kv.second.exec);      // graphs captured without the averaging
  ag->graphs.clear();
  GCRL_CUDA(cudaDeviceSynchronize());
  GCRL_API_END
}

int gcrl_agent_dp_barrier(gcrl_agent *ag, void *stream) {
  GCRL_API_BEGIN
  require_handle(ag);
  GCRL_REQUIRE(ag != nullptr && ag->p2p.on, "peer-memory data parallelism is not connected");
  GCRL_CUDA(cudaSetDevice(ag->device));
  auto &pp = ag->p2p;
  launch_p2p_barrier(pp.d_peer_flags, pp.epoch, pp.rank, pp.world, pp.err, as_stream(stream));
  GCRL_API_END
}

int gcrl_agent_grad_buffer(gcrl_agent *ag, int net, float **grad_dev, int64_t *count) {
  GCRL_API_BEGIN
  require_handle(ag);
  GCRL_REQUIRE(ag && net >= 0 && net < NUM_NETS && ag->has[net] && ag->net[net].g, "bad network id");
  if (grad_dev) *grad_dev = ag->net[net].g;
  if (count) *count = ag->net[net].total;
  GCRL_API_END
}

int gcrl_agent_metrics_buffer(gcrl_agent *ag, float **metrics_dev) {
  GCRL_API_BEGIN
  require_handle(ag);
  GCRL_REQUIRE(ag != nullptr && metrics_dev != nullptr, "NULL argument");
  *metrics_dev = ag->metrics;
  GCRL_API_END
}

int gcrl_agent_param_buffers(gcrl_agent *ag, int net, const float **flat_dev, int64_t *count,
                             const float **flat_t_dev, int64_t *count_t) {
  GCRL_API_BEGIN
  require_handle(ag);
  GCRL_REQUIRE(ag && net >= 0 && net < NUM_NETS && ag->has[net] && ag->net[net].p, "bad network id");
  const MlpParams &n = ag->net[net];
  if (flat_dev) *flat_dev = n.p;
  if (count) *count = n.total;
  if (flat_t_dev) *flat_t_dev = n.copies.pT;
  if (count_t) *count_t = n.copies.pT ? n.copies.total_t : 0;
  GCRL_API_END
}

}  // extern "C"
