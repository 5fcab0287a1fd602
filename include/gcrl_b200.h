/*
 * gcrl_b200.h -- C ABI of the B200-native HER-sample + off-policy-update hot path.
 *
 * Drop-in boundary for CodeKnight314/Goal-Conditioned-RL-Framework.  The reference
 * has no FFI of its own (it is pure Python), so each entry point below replaces a
 * reference *method*; the citation next to it is the reference file:line it stands
 * in for.  INTEGRATION.md shows the ctypes binding and the two-line import change a
 * maintainer makes in src/env.py.
 *
 * Conventions
 *   - plain C types only; no torch / CUDA types in signatures.  `stream` is a
 *     cudaStream_t passed as void* (NULL = legacy default stream).
 *   - every function returns GCRL_OK (0) or an error code; gcrl_last_error() gives
 *     the message for the calling thread.
 *   - "dev" pointers are device pointers on the handle's GPU, "host" pointers are
 *     ordinary host memory borrowed for the duration of the call.
 *   - one host thread drives one handle; work is ordered on the stream passed in.
 *   - there is NO CPU fallback: without a CUDA device every compute entry point
 *     fails with GCRL_ERR_CUDA.
 */
#ifndef GCRL_B200_H
#define GCRL_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GCRL_ABI_VERSION 5

#define GCRL_OK 0
#define GCRL_ERR_INVALID 1      /* bad argument / shape                                  */
#define GCRL_ERR_UNDERFILLED 2  /* sample(B) with len < B: AssertionError, buffer.py:122 */
#define GCRL_ERR_CUDA 3         /* CUDA runtime error (or no device)                     */
#define GCRL_ERR_CAPACITY 4     /* transition / episode ring would overflow              */

int gcrl_abi_version(void);
const char *gcrl_last_error(void);
int gcrl_device_count(int *count);
/* Number of CUDA kernels this library has launched in the calling process so far (graph
 * replays count their kernel nodes).  Diagnostics / bench.py's "gpu_launches". */
uint64_t gcrl_kernel_launches(void);

/* ------------------------------------------------------------------------------------
 * HER replay buffer -- replaces HERBuffer, src/buffer.py:92-179
 * ------------------------------------------------------------------------------------
 * Device-resident episode store.  An episode of T transitions stands for
 * E = (T-1)(k+1)+1 *entries* in the reference's deque order (src/buffer.py:145-179):
 * for t = 0..T-1 the original, then -- if t < T-1 -- k future-relabelled copies.
 * Entries are never materialised: gcrl_her_sample() maps a deque position to
 * (episode, t, j) and relabels on the fly.  `max_entries` is the deque's maxlen
 * (per-ENTRY FIFO eviction, src/buffer.py:101); `cap_transitions` sizes the ring of
 * stored transitions (<= 0: max_entries + 254, always sufficient).
 */
typedef struct gcrl_her gcrl_her;

int gcrl_her_create(gcrl_her **out, int device, int64_t max_entries, int64_t cap_transitions,
                    int state_dim /* D = obs + goal */, int goal_dim, int act_dim, int k_future,
                    uint64_t seed);
int gcrl_her_destroy(gcrl_her *h);

/* Commit one finished episode (what HERBuffer.push does when `done or len >= 50`,
 * src/buffer.py:117-119 -> apply_her :143-179).  Row t is the tuple pushed at
 * src/env.py:215-224: s[t] = state, ns[t] = next_state (both [D], goal in the last
 * goal_dim columns), a[t], r[t], d[t] (0/1), ag[t] = achieved goal of the NEXT
 * observation.  fut[t*k + j] (t < T-1) is the absolute future index f in [t+1, T-1]
 * drawn by `random.randint(t+1, T-1)` at src/buffer.py:153 (other goal-selection strategies: their
 * range, gcrl_her_set_goal_selection); NULL = draw them from the handle's own counter-based generator.
 * All pointers are host memory.  1 <= T <= 255. */
int gcrl_her_push_episode(gcrl_her *h, int T, const float *s, const float *a, const float *ns,
                          const float *r, const float *d, const float *ag, const uint8_t *fut,
                          void *stream);

/* Distance threshold of the sparse relabel reward -(||achieved - goal||_2 > threshold) (HERBuffer's `threshold`
 * constructor argument, src/buffer.py:93; panda-gym's tasks use 0.05, the default).  Takes effect for the
 * following samples. */
int gcrl_her_set_threshold(gcrl_her *h, float threshold);

/* Goal selection (Andrychowicz et al. 2017).  A relabelled transition at step t of an episode of T steps takes the
 * achieved goal of step f as its goal:
 *   GCRL_HER_FUTURE  (default) f in [t+1, T-1] -- random.randint(t+1, T-1), the reference's only strategy
 *   GCRL_HER_FINAL   f = T-1
 *   GCRL_HER_EPISODE f in [0, T-1]
 * online_k == 0 (eager, the default): the k_future relabelled copies of the store's entry mapping; fut[] of
 * gcrl_her_push_episode must lie in the strategy's range (f == T-1 for FINAL), and fut == NULL draws it there.
 * online_k > 0 (online relabelling): the store holds each transition once (it must be created with k_future = 0,
 * so len() counts transitions), and each sampled row is relabelled at sample time with probability
 * online_k / (online_k + 1) to a goal step drawn uniformly from the strategy's range (FUTURE / FINAL: none at
 * t = T-1); coin and goal step come from a hash of (seed, draw epoch, batch row), and every sample call of an
 * online store advances the draw epoch.  gcrl_her_push_episode then takes no fut (fut != NULL: GCRL_ERR_INVALID).
 * Refused (GCRL_ERR_INVALID) once an episode has been committed. */
#define GCRL_HER_FUTURE 0
#define GCRL_HER_FINAL 1
#define GCRL_HER_EPISODE 2
int gcrl_her_set_goal_selection(gcrl_her *h, int strategy, int online_k);
/* n-step returns, as Stable-Baselines3's `n_steps` for its off-policy algorithms (1: one-step rows, the default).
 * A sampled row at step t of an episode of T stored steps, with goal g (original or relabelled), covers the window
 * t .. t+k-1, k = min(n, T - t): reward R = r_t + gamma (r_{t+1} + ... + gamma r_{t+k-1}) (unfused fp32, from the
 * back; relabelled rows recompute every r_{t+i} for g), next state = ns of row t+k-1 (goal columns <- g), done =
 * 1 - gamma^(k-1) (1 - done_{t+k-1}) (relabelled rows: done_{t+k-1} = 0).  A learner's gamma (1 - done) is then the
 * n-step bootstrap weight gamma^k (1 - done_{t+k-1}), exactly while gamma^(k-1) >= 1/2 and within 2^-25 beyond.
 * 1 <= n <= 255; 0 < gamma <= 1 when n > 1.  Refused (GCRL_ERR_INVALID) once an episode has been committed. */
int gcrl_her_set_n_step(gcrl_her *h, int n, float gamma);
/* The draw epoch of the device index stream and of online relabelling (one per sample call that draws on the
 * device; in online mode one per sample call).  A checkpoint saves it so that a resumed run draws the same rows. */
uint64_t gcrl_her_get_draw_epoch(const gcrl_her *h);
int gcrl_her_set_draw_epoch(gcrl_her *h, uint64_t epoch);
/* Diagnostics (cache experiments, profiles/cold_start.py): the device episode and bucket index tables that map a
 * deque position to its row, with their sizes in bytes. */
int gcrl_her_index_tables(gcrl_her *h, const void **eps_dev, int64_t *eps_bytes, const void **buckets_dev,
                          int64_t *bucket_bytes);
int64_t gcrl_her_len(const gcrl_her *h);            /* __len__, src/buffer.py:137-138   */
int64_t gcrl_her_total_entries(const gcrl_her *h);  /* entries ever appended            */
int64_t gcrl_her_live_transitions(const gcrl_her *h);
int gcrl_her_clear(gcrl_her *h);
/* Export of the live window for a true resume (the reference never checkpoints its replay buffer,
 * src/env.py:430-440): the episodes that still hold a live entry, oldest first, exactly as committed
 * (rows as pushed, the future indices that were drawn).  Re-pushing them in order into a fresh buffer
 * with the same max_entries reproduces every deque position.  s == NULL: query T only. */
int64_t gcrl_her_live_episodes(const gcrl_her *h);
int gcrl_her_get_episode(gcrl_her *h, int64_t i, int *T, float *s, float *a, float *ns, float *r, float *d,
                         float *ag, uint8_t *fut, void *stream);

/* sample(batch_size), src/buffer.py:121-135.  Outputs are DEVICE pointers:
 * states [B,D], actions [B,A], rewards [B,1], next_states [B,D], dones [B,1] float32.
 * idx_host: B deque positions in [0, len) (the stream `random.sample(range(len), B)`
 * yields -- identical to random.sample(deque, B) at src/buffer.py:124), or NULL to draw
 * B distinct positions on the device (keyed Feistel permutation of [0, len), i.e.
 * uniform without replacement like random.sample).  idx_out_dev (optional, int64[B])
 * receives the positions used.  Returns GCRL_ERR_UNDERFILLED when len < B. */
int gcrl_her_sample(gcrl_her *h, int64_t B, const int64_t *idx_host, float *states_dev,
                    float *actions_dev, float *rewards_dev, float *next_states_dev,
                    float *dones_dev, int64_t *idx_out_dev, void *stream);
/* Same, positions already on the device. */
int gcrl_her_sample_dev_idx(gcrl_her *h, int64_t B, const int64_t *idx_dev, float *states_dev,
                            float *actions_dev, float *rewards_dev, float *next_states_dev,
                            float *dones_dev, void *stream);
/* Same as gcrl_her_sample but the five outputs are HOST buffers (device->host copies
 * and a stream synchronise inside the call). */
int gcrl_her_sample_host(gcrl_her *h, int64_t B, const int64_t *idx_host, float *states,
                         float *actions, float *rewards, float *next_states, float *dones,
                         int64_t *idx_out, void *stream);

/* Host-side mirror of CPython's `random` draws on this path (no GPU involved): advance a copy of the
 * interpreter's MT19937 state (the 624 words and position of random.getstate()) exactly as
 * random.randint(lo[i], hi[i]) (src/buffer.py:153) / random.sample(range(n), k) (== random.sample(deque, k),
 * src/buffer.py:124) would, CPython 3.12 algorithms.  The caller writes the state back with
 * random.setstate(), so every other consumer of the global stream sees the reference's interleaving. */
int gcrl_pyrandom_randint(uint32_t *mt624, int *pos, int64_t count, const int32_t *lo, const int32_t *hi,
                          int32_t *out);
int gcrl_pyrandom_sample_range(uint32_t *mt624, int *pos, int64_t n, int64_t k, int64_t *out);

/* ------------------------------------------------------------------------------------
 * Running normaliser -- replaces RunningNormalizer, src/utils.py:68-117
 * ------------------------------------------------------------------------------------ */
typedef struct gcrl_norm gcrl_norm;

int gcrl_norm_create(gcrl_norm **out, int device, int dim, double clip_range, double eps_count);
int gcrl_norm_destroy(gcrl_norm *h);
/* update(x), src/utils.py:75-94.  x: host [n, dim], float64 (is_f64 != 0) or float32. */
int gcrl_norm_update(gcrl_norm *h, const void *x_host, int64_t n, int is_f64, void *stream);
/* Data-parallel update (one process per GPU, every rank sees its own envs' observations): the local batch's
 * moments per column, moments_host [dim][3] = (n, mean, M2 = sum (x - mean)^2), no state change; the caller
 * all-gathers them and every rank folds ALL ranks' moments, in rank order, into its running state with
 * gcrl_norm_update_moments (moments_host [parts][dim][3]) -- Chan's merge, then _update_from_moments
 * (src/utils.py:82-94) once.  N ranks on per-rank batches == one rank on the concatenated batch to float64
 * rounding, and the replicas stay bit-identical. */
int gcrl_norm_batch_moments(gcrl_norm *h, const void *x_host, int64_t n, int is_f64, double *moments_host,
                            void *stream);
int gcrl_norm_update_moments(gcrl_norm *h, const double *moments_host, int parts, void *stream);
/* Same with x already on the device. */
int gcrl_norm_update_dev(gcrl_norm *h, const void *x_dev, int64_t n, int is_f64, void *stream);
/* normalize(x), src/utils.py:96-98: clip((x-mean)/(sqrt(var)+1e-8), +-clip) in float64.
 * host in -> host out (float64 [n, dim]); synchronises the stream. */
int gcrl_norm_apply(gcrl_norm *h, const void *x_host, int64_t n, int is_f64, double *out_host,
                    void *stream);
/* Device variant: float32 output written at out_dev[row*out_stride + out_col0 + c]
 * (lets the caller build obs||goal rows, src/agent.py:1434-1445, without a concat). */
int gcrl_norm_apply_dev_f32(gcrl_norm *h, const void *x_dev, int64_t n, int is_f64,
                            float *out_dev, int64_t out_stride, int64_t out_col0, void *stream);
int gcrl_norm_get_state(gcrl_norm *h, double *mean, double *var, double *count,
                        double *clip_range, void *stream);
int gcrl_norm_set_state(gcrl_norm *h, const double *mean, const double *var, double count,
                        double clip_range, void *stream);

/* ------------------------------------------------------------------------------------
 * Off-policy agents -- replace DDPG (src/agent.py:1173-1465) and TD3Agent (:12-386)
 * ------------------------------------------------------------------------------------ */
typedef struct gcrl_agent gcrl_agent;

#define GCRL_ALGO_DDPG 0
#define GCRL_ALGO_TD3 1

typedef struct gcrl_agent_config {
  int32_t algo;          /* GCRL_ALGO_*                                                */
  int32_t state_dim;     /* D = obs + goal (env.py:120 passes obs_dim + dg_dim)        */
  int32_t act_dim;
  int32_t hidden_dim;    /* BaseAgentConfig.hidden_dim, src/utils.py:11                */
  int32_t layer_count;   /* number of hidden layers, src/utils.py:12                   */
  int32_t max_batch;     /* largest B an update will see                               */
  float gamma;           /* src/utils.py:23                                            */
  float tau;             /* src/utils.py:33                                            */
  float grad_clip;       /* < 0: no clipping (grad_clip None)                          */
  float policy_noise;    /* TD3 target smoothing sigma, src/agent.py:175               */
  float noise_clamp;     /* TD3, src/agent.py:176                                      */
  float weight_decay;    /* 0 = Adam (DDPG); 0.01 = AdamW default (TD3)                */
  int32_t precision;     /* 0 = fp32 FFMA everywhere; 1 = hidden-layer forward / input-gradient
                            GEMMs on tcgen05 tensor cores (3xTF32 split, fp32-level accuracy)
                            once the batch reaches 2048 rows; 2 = the same for every batch
                            >= 128 rows (tests)                                           */
  int32_t reserved;
} gcrl_agent_config;

int gcrl_agent_create(gcrl_agent **out, int device, const gcrl_agent_config *cfg);
int gcrl_agent_destroy(gcrl_agent *h);

/* Networks: 0 actor, 1 critic(_1), 2 target_actor, 3 target_critic(_1), 4 critic_2,
 * 5 target_critic_2.  Parameters are exchanged per layer in the reference checkpoint
 * layout: weight [out, in] row-major fp32, bias [out] (state_dict keys
 * base_net.{0,2,..} / net.{0,2,..}, src/model.py:24-26,64-65; save/load :32-37). */
int gcrl_agent_num_layers(const gcrl_agent *h, int net);
int gcrl_agent_layer_shape(const gcrl_agent *h, int net, int layer, int *out_dim, int *in_dim);
int gcrl_agent_set_layer(gcrl_agent *h, int net, int layer, const float *weight_host,
                         const float *bias_host, void *stream);
int gcrl_agent_get_layer(gcrl_agent *h, int net, int layer, float *weight_host,
                         float *bias_host, void *stream);
/* Optimiser state for a true resume (the reference checkpoints weights only, src/env.py:430-440,
 * so its "resume" restarts Adam from zero): exp_avg / exp_avg_sq of torch.optim.Adam for one layer of
 * a trainable network (0 actor, 1 critic, 4 critic_2), same layout as get_layer, and the step count. */
int gcrl_agent_get_adam_layer(gcrl_agent *h, int net, int layer, float *m_weight, float *m_bias,
                              float *v_weight, float *v_bias, void *stream);
int gcrl_agent_set_adam_layer(gcrl_agent *h, int net, int layer, const float *m_weight, const float *m_bias,
                              const float *v_weight, const float *v_bias, void *stream);
int gcrl_agent_get_adam_step(gcrl_agent *h, int net, int *step);
int gcrl_agent_set_adam_step(gcrl_agent *h, int net, int step);
/* update_target_network(hard_update=True), src/agent.py:1255-1258 */
int gcrl_agent_hard_update(gcrl_agent *h, void *stream);
/* Polyak step theta_t <- tau theta + (1 - tau) theta_t of the target actor (which bit0) and / or the target critic(s)
 * (bit1), outside update(): DDPG.update_target_network(hard_update=False, tau) src/agent.py:1259-1271, TD3Agent.update_actor
 * / update_critic :117-132.  (Inside update() the Polyak steps are fused into the optimiser kernels.) */
int gcrl_agent_soft_update(gcrl_agent *h, int which, double tau, void *stream);
/* Optimiser state is zeroed (Adam step counters too): a fresh torch.optim.Adam. */
int gcrl_agent_reset_optim(gcrl_agent *h, void *stream);

/* One update on an explicit device batch (critic_update :1302-1343, Polyak :1259-1271,
 * actor_update :1288-1300, in the order of update() :1378-1404).
 *   flags bit0: run the actor step; bit1: Polyak soft update (before the actor step).
 *   noise_dev: TD3 only, [B, A] standard-normal draws (the randn_like at agent.py:175),
 *   NULL for DDPG.
 *   metrics_host (optional, float[8]): critic_loss, actor_loss, td_error, q_value,
 *   critic_grad_norm, actor_grad_norm, critic2_loss, critic2_grad_norm -- copied back
 *   and the stream synchronised when non-NULL; NULL leaves the update fully async. */
int gcrl_agent_update_batch(gcrl_agent *h, int64_t B, const float *s_dev, const float *a_dev,
                            const float *r_dev, const float *ns_dev, const float *d_dev,
                            const float *noise_dev, double lr_critic, double lr_actor,
                            int flags, float *metrics_host, void *stream);
/* Fused hot path: sample B transitions from `buf` (positions idx_host or on-device
 * draw) and run the update, one call (update(), src/agent.py:1378-1404). */
int gcrl_agent_update_from_buffer(gcrl_agent *h, gcrl_her *buf, int64_t B,
                                  const int64_t *idx_host, const float *noise_dev,
                                  double lr_critic, double lr_actor, int flags,
                                  float *metrics_host, void *stream);
/* n consecutive updates from `buf`, issued as ONE graph launch.  Equivalent, bit for bit, to n calls of
 * gcrl_agent_update_from_buffer with flags[i], lr_critic[i], lr_actor[i], the positions idx_host + i*B (or the
 * device index stream's next n draws when idx_host is NULL) and the TD3 noise noise_dev + i*B*A.
 * flags[i] may hold bit0 and bit1 only (no prioritised weights: a HER buffer has no priorities).
 * metrics_host: float[n][8], row i = what update i would have returned; NULL leaves the call async, and
 * gcrl_agent_read_metrics then returns the last row.  1 <= n <= GCRL_MAX_MANY_STEPS.
 * Refused (GCRL_ERR_INVALID) on a handle connected for peer data parallelism and while a phase-wise
 * data-parallel update is open (phase 0 issued, phase 3 not yet).  On any error no Adam step counter, update
 * sequence number or device index-stream draw has advanced. */
#define GCRL_MAX_MANY_STEPS 64
int gcrl_agent_update_many(gcrl_agent *h, gcrl_her *buf, int64_t B, int n, const int *flags,
                           const int64_t *idx_host, const float *noise_dev, const double *lr_critic,
                           const double *lr_actor, float *metrics_host, void *stream);
/* Device metrics of the most recent update (float[8], same order). */
int gcrl_agent_read_metrics(gcrl_agent *h, float *metrics_host, void *stream);

/* actor(obs) for select_action, src/agent.py:1345-1366: obs host [n, D] -> act host
 * [n, A] = tanh-squashed network output (the caller applies the reference's second
 * tanh, noise and clipping). */
int gcrl_agent_act(gcrl_agent *h, int64_t n, const float *obs_host, float *act_host,
                   void *stream);
/* Q(s, a) with the online critic; host in / host out [n, 1] (tests, diagnostics). */
int gcrl_agent_q(gcrl_agent *h, int64_t n, const float *obs_host, const float *act_host,
                 float *q_host, void *stream);

/* Data-parallel hooks (one process per GPU, buffer sharded by episode, weights replicated).
 * The update above is cut at the two points where gradients are averaged across ranks:
 *   phase 0: ingest the local batch (sampled from `buf` at idx_host / on-device draw when buf is
 *            non-NULL, else the dense device batch) -> target + critic forward, loss, backward ->
 *            flat critic gradient(s) = mean over the LOCAL batch, local metrics;
 *   [caller: all-reduce AVG of gcrl_agent_grad_buffer(critic) (and critic_2 for TD3)]
 *   phase 1: global-norm clip on the averaged gradient + Adam (+ Polyak per flags);
 *   phase 2: actor forward through the stepped critic, backward -> flat actor gradient;
 *   [caller: all-reduce AVG of gcrl_agent_grad_buffer(actor)]
 *   phase 3: clip + Adam (actor).
 * Phases 2/3 are no-ops when flags bit0 is clear.  With world size 1 and no all-reduce the four
 * phases reproduce gcrl_agent_update_* bit for bit. */
int gcrl_agent_update_phase(gcrl_agent *h, int phase, gcrl_her *buf, int64_t B,
                            const int64_t *idx_host, const float *s_dev, const float *a_dev,
                            const float *r_dev, const float *ns_dev, const float *d_dev,
                            const float *noise_dev, double lr_critic, double lr_actor, int flags,
                            void *stream);
/* Data-parallel averaging over NVLink peer memory instead of a collective library: every rank exports
 * CUDA-IPC handles of its flag array, metrics outbox and flat gradient buffers (gcrl_agent_dp_export:
 * handles may be NULL to query n_items; 64 bytes each), the caller all-gathers them (any transport), and
 * gcrl_agent_dp_connect maps the peers' buffers.  From then on gcrl_agent_update_batch / _from_buffer
 * average the critic and actor gradients (and the batch-mean metrics) across the ranks inside the one
 * captured graph: flag barrier over peer memory, every rank sums all ranks' buffers in rank order
 * (bit-identical replicas), clip + Adam on the average.  All ranks must issue the same sequence of updates
 * (same batch size and flags).  world <= 8 (one NVSwitch domain). */
int gcrl_agent_dp_export(gcrl_agent *h, unsigned char *handles, int *n_items);
int gcrl_agent_dp_connect(gcrl_agent *h, int rank, int world, const unsigned char *all_handles);
/* One flag barrier over the connected ranks on `stream` (a single-warp kernel), outside any update: aligns
 * the ranks, e.g. before a timed region.  Every rank must call it the same number of times. */
int gcrl_agent_dp_barrier(gcrl_agent *h, void *stream);
/* flat fp32 gradient of a trainable network: device pointer + element count (for NCCL) */
int gcrl_agent_grad_buffer(gcrl_agent *h, int net, float **grad_dev, int64_t *count);
/* device float[8] holding the metrics of the most recent update (averaged across ranks by the
 * caller when a data-parallel run wants global losses) */
int gcrl_agent_metrics_buffer(gcrl_agent *h, float **metrics_dev);
/* Diagnostics (cache experiments, profiles/cold_start.py): a network's flat parameter buffer and its transposed
 * copy, device pointers and element counts (NULL and 0 when the network keeps no transposed copy). */
int gcrl_agent_param_buffers(gcrl_agent *h, int net, const float **flat_dev, int64_t *count,
                             const float **flat_t_dev, int64_t *count_t);

/* ------------------------------------------------------------------------------------
 * Stochastic-actor agents -- replace SACAgent (src/agent.py:388-770) and TQCAgent (:773-1171)
 * ------------------------------------------------------------------------------------
 * Actor = SACActorModel (src/model.py:86-141): L x (Linear -> BatchNorm1d -> ReLU), mean_head,
 * log_std_head.  Critics = an ensemble of n scalar Critic MLPs with n target copies; the value
 * used in the Bellman target and in the actor loss is the mean of the (n - drop_top) smallest
 * critic outputs per sample: SAC n = 2, drop_top = 1 (torch.min, :566,:519); "TQC" n = 5,
 * drop_top = 2 (sort / slice / mean, :971-976, :919-921).  BatchNorm runs in train mode (batch
 * statistics, running statistics updated) for both policy samples of an update, exactly as the
 * reference does under set_train() (:701-706), including inside torch.no_grad (:556-557). */
typedef struct gcrl_sac gcrl_sac;

#define GCRL_ALGO_SAC 2
#define GCRL_ALGO_TQC 3

typedef struct gcrl_sac_config {
  int32_t algo;            /* GCRL_ALGO_SAC | GCRL_ALGO_TQC                                   */
  int32_t state_dim;       /* D = obs + goal                                                   */
  int32_t act_dim;         /* 1..4                                                             */
  int32_t hidden_dim;
  int32_t layer_count;
  int32_t max_batch;
  int32_t n_critics;       /* SAC 2; TQC 5 (getattr default, src/agent.py:789)                 */
  int32_t drop_top;        /* SAC 1 (= min); TQC 2 (src/agent.py:790)                          */
  float gamma, tau, grad_clip;
  float weight_decay;      /* AdamW default 0.01 (:420-425)                                    */
  float entropy_coef;      /* >= 0: literal coefficient (SAC: 0.2, :521,:569); < 0: use the
                              learned alpha = exp(log_alpha) (TQC, :928,:978)                  */
  float target_entropy;    /* SAC -A/2 (:423); TQC -A (:815)                                   */
  float alpha_lr;          /* SACAgentConfig.alpha_lr, src/utils.py:37                         */
  int32_t precision;       /* 0 = fp32 FFMA everywhere; 1 = the critics' and the actor's hidden-layer forward,
                              input-gradient and weight-gradient GEMMs on tcgen05 tensor cores (3xTF32 split,
                              fp32-level accuracy; the critic ensemble in one launch per layer) once
                              B * H^2 >= 2048 * 256^2 (B = batch, H = hidden_dim: 2048 rows at H = 256, 512 at
                              H = 512, 8192 at H = 128); 2 = the same for every batch >= 128 rows (tests).
                              select_action stays on the fp32 path.  Other values: GCRL_ERR_INVALID          */
} gcrl_sac_config;

int gcrl_sac_create(gcrl_sac **out, int device, const gcrl_sac_config *cfg);
/* TQC with quantile critics: as gcrl_sac_create, but every critic ends in an H -> n_quantiles Linear, the target
 * keeps the n_critics * (n_quantiles - drop_per_net) smallest pooled atoms and the critics minimise the quantile
 * Huber loss.  cfg->algo must be GCRL_ALGO_TQC; cfg->drop_top is not used.  1 <= n_quantiles,
 * 0 <= drop_per_net < n_quantiles, n_critics * n_quantiles <= 256; otherwise GCRL_ERR_INVALID.
 * Every other gcrl_sac_* call works on such a handle (gcrl_sac_get / set_critic_layer move an [n_quantiles, H]
 * head) except data parallelism: gcrl_sac_set_sync_bn, gcrl_sac_update_phase and gcrl_sac_update_segment refuse
 * it with GCRL_ERR_INVALID. */
int gcrl_sac_create_quantile(gcrl_sac **out, int device, const gcrl_sac_config *cfg, int n_quantiles,
                             int drop_per_net);
int gcrl_sac_destroy(gcrl_sac *h);

/* Parameter exchange in the reference's state_dict layout (fp32, weight [out, in] row-major).
 * Actor Linear layers: 0..L-1 = base_net.{3l}; L = mean_head; L+1 = log_std_head.
 * Actor BatchNorm l = base_net.{3l+1}: weight, bias, running_mean, running_var [H].
 * Critics: critic 0..n-1 (critic_1/critic_2 or critics.{i}), target != 0 for the target copy;
 * layer = net.{2 layer}. */
int gcrl_sac_set_actor_linear(gcrl_sac *h, int layer, const float *weight_host, const float *bias_host,
                              void *stream);
int gcrl_sac_get_actor_linear(gcrl_sac *h, int layer, float *weight_host, float *bias_host, void *stream);
int gcrl_sac_set_actor_bn(gcrl_sac *h, int layer, const float *weight, const float *bias,
                          const float *running_mean, const float *running_var, void *stream);
int gcrl_sac_get_actor_bn(gcrl_sac *h, int layer, float *weight, float *bias, float *running_mean,
                          float *running_var, void *stream);
int gcrl_sac_set_critic_layer(gcrl_sac *h, int critic, int target, int layer, const float *weight_host,
                              const float *bias_host, void *stream);
int gcrl_sac_get_critic_layer(gcrl_sac *h, int critic, int target, int layer, float *weight_host,
                              float *bias_host, void *stream);
int gcrl_sac_hard_update(gcrl_sac *h, void *stream);          /* update_target_network, :483-485 */
int gcrl_sac_set_log_alpha(gcrl_sac *h, float log_alpha, void *stream);
int gcrl_sac_get_log_alpha(gcrl_sac *h, float *log_alpha, void *stream);

/* One update (update(), src/agent.py:659-699 / :1062-1100) on an explicit device batch.
 *   eps_next_dev / eps_cur_dev: [B, A] standard-normal draws behind Normal.rsample
 *   (src/model.py:134) for the next-state sample (critic_update) and the state sample
 *   (actor_update; may be NULL when flags bit0 is clear).
 *   flags bit0: actor step (+ alpha bookkeeping); bit1: Polyak of the target critics
 *   (SAC: step % gradient_step == 0, :681; TQC: always, :1086); bit2: alpha update
 *   (step > alpha_min_steps, :533).
 *   metrics_host (optional, float[12]): q1_loss, q2_loss, actor_loss, td_error, q_value,
 *   critic_1_grad, critic_2_grad, actor_grad, alpha_loss, alpha, log_alpha, unused -- the
 *   reference's return tuple (:684-698); for TQC slots 0/1 and 5/6 carry the ensemble means
 *   (:1013-1014). */
int gcrl_sac_update_batch(gcrl_sac *h, int64_t B, const float *s_dev, const float *a_dev,
                          const float *r_dev, const float *ns_dev, const float *d_dev,
                          const float *eps_next_dev, const float *eps_cur_dev, double lr_critic,
                          double lr_actor, int flags, float *metrics_host, void *stream);
int gcrl_sac_update_from_buffer(gcrl_sac *h, gcrl_her *buf, int64_t B, const int64_t *idx_host,
                                const float *eps_next_dev, const float *eps_cur_dev, double lr_critic,
                                double lr_actor, int flags, float *metrics_host, void *stream);
/* n consecutive SAC / TQC updates from `buf` as ONE graph launch.  Bit for bit equal to n calls of
 * gcrl_sac_update_from_buffer with flags[i], lr_critic[i], lr_actor[i], the positions idx_host + i*B (or the device
 * index stream's next n draws when idx_host is NULL), eps_next_dev + i*B*A and eps_cur_dev + i*B*A (row i of
 * eps_cur read only when flags[i] bit0 is set; eps_cur_dev may be NULL when no flags[i] has it).
 * flags[i]: bits 0-2 only (a HER buffer has no priorities).
 * metrics_host: float[n][12], row i = what update i returns, read back once per call; NULL leaves the call async,
 * and gcrl_sac_read_metrics then returns the last update's tuple.  1 <= n <= GCRL_MAX_MANY_STEPS.
 * Refused (GCRL_ERR_INVALID) on a sync-BN agent (gcrl_sac_set_sync_bn world != 0) and while a phase-wise
 * data-parallel update is open.  On any error, no AdamW step counter (critics, actor, alpha) and no device
 * index-stream epoch has moved. */
int gcrl_sac_update_many(gcrl_sac *h, gcrl_her *buf, int64_t B, int n, const int *flags, const int64_t *idx_host,
                         const float *eps_next_dev, const float *eps_cur_dev, const double *lr_critic,
                         const double *lr_actor, float *metrics_host, void *stream);
/* Data-parallel hooks (one process per GPU, episode-sharded buffer, replicated weights): the update cut
 * at the points where gradients are averaged across ranks --
 *   phase 0: ingest the local batch, policy sample, targets, all critic forwards / backwards
 *            -> the ensemble's flat gradients (gcrl_sac_dp_buffer which = 1), local metrics;
 *   phase 1: clip + AdamW (+ Polyak per flags) of every critic on the averaged gradients;
 *   phase 2: actor forward / backward through the stepped critics -> actor gradient, followed in the same
 *            buffer by alpha's batch mean (which = 0);
 *   phase 3: clip + AdamW of the actor, alpha step.
 * BatchNorm uses the LOCAL batch statistics on every rank (torch DistributedDataParallel's default
 * without SyncBatchNorm); the caller averages the running statistics (which = 2) after phase 3 so that
 * the replicas' eval-mode policies stay identical.  With world size 1 the four phases reproduce
 * gcrl_sac_update_* bit for bit. */
int gcrl_sac_update_phase(gcrl_sac *h, int phase, gcrl_her *buf, int64_t B, const int64_t *idx_host,
                          const float *s_dev, const float *a_dev, const float *r_dev, const float *ns_dev,
                          const float *d_dev, const float *eps_next_dev, const float *eps_cur_dev,
                          double lr_critic, double lr_actor, int flags, void *stream);
/* which: 0 actor gradient (+ 4 trailing floats: alpha's batch mean), 1 all critic gradients (contiguous),
 * 2 BatchNorm running mean | var of every layer, 3 the 32-float device metrics block, 4 the sync-BN slots
 * [world][2 * pad4(hidden)] (after gcrl_sac_set_sync_bn; this rank's slot is row `rank`). */
int gcrl_sac_dp_buffer(gcrl_sac *h, int which, float **dev, int64_t *count);
/* Sync-BN: BatchNorm1d of SACActorModel (src/model.py:103-111) normalises with the statistics of the WHOLE
 * global batch, so that `world` ranks on B rows each equal one rank on the concatenated world * B rows (the 1-GPU
 * semantics; all ranks must use the same B).  gcrl_sac_set_sync_bn(world, rank) switches it on (world = 0: off;
 * world = 1 reproduces gcrl_sac_update_* bit for bit).  The update is then issued as a chain of graph segments:
 *     for (seg = 0;; ++seg) {
 *       gcrl_sac_update_segment(h, seg, ..., &collective, stream);
 *       if (collective == 0) break;                       update complete
 *       1: all-gather the sync-BN slots (which = 4: every rank contributes row `rank`, in place)
 *       2: average the critic gradients (which = 1)      3: average the actor gradient + alpha mean (which = 0)
 *     }
 * on `stream`, every rank issuing the same sequence.  Segment 0 takes the batch (arguments as
 * gcrl_sac_update_phase phase 0); later segments only need (B, flags) to match.  2 * layer_count gathers for the
 * forward passes of a critic+actor update, layer_count for the backward pass; the running statistics come out
 * identical on every rank (no average of which = 2 needed). */
int gcrl_sac_set_sync_bn(gcrl_sac *h, int world, int rank);
int gcrl_sac_update_segment(gcrl_sac *h, int segment, gcrl_her *buf, int64_t B, const int64_t *idx_host,
                            const float *s_dev, const float *a_dev, const float *r_dev, const float *ns_dev,
                            const float *d_dev, const float *eps_next_dev, const float *eps_cur_dev,
                            double lr_critic, double lr_actor, int flags, int *collective, void *stream);
/* The metrics tuple of the most recent update (float[12], same order as gcrl_sac_update_batch). */
int gcrl_sac_read_metrics(gcrl_sac *h, int flags, float *metrics_host, void *stream);

/* select_action, :641-647: eval-mode actor (running statistics).  eps_host NULL = deterministic
 * tanh(mean); otherwise tanh(mean + std * eps).  obs host [n, D] -> act host [n, A]. */
int gcrl_sac_act(gcrl_sac *h, int64_t n, const float *obs_host, const float *eps_host, float *act_host,
                 void *stream);

/* ------------------------------------------------------------------------------------
 * Uniform and prioritised replay -- replace ReplayBuffer (src/buffer.py:8-35) and PERBuffer
 * (src/buffer.py:38-89), the buffers behind agent.update() when buffer_type is not "HER"
 * ------------------------------------------------------------------------------------
 * A bounded FIFO of transitions on the device (deque(maxlen=capacity) semantics: position 0 is the
 * oldest live entry).  Packed host row: s[D] | a[A] | r | ns[D] | d  (2D + A + 2 floats). */
typedef struct gcrl_replay gcrl_replay;

/* PERBuffer(max_len, alpha) when prioritized != 0 (:39-44), else ReplayBuffer(max_len) (:9-11). */
int gcrl_replay_create(gcrl_replay **out, int device, int64_t capacity, int state_dim, int act_dim,
                       int prioritized, double alpha);
int gcrl_replay_destroy(gcrl_replay *h);
/* push() x n (:13-14, :46-48): rows host [n, 2D + A + 2]; new entries get priority 1.0. */
int gcrl_replay_push(gcrl_replay *h, int64_t n, const float *rows_host, void *stream);
int64_t gcrl_replay_len(gcrl_replay *h);          /* __len__, :34-35 / :83-84 */
int64_t gcrl_replay_total(gcrl_replay *h);        /* entries ever appended    */
/* ReplayBuffer.sample (:16-32) at the positions the caller drew (random.sample(range(len), B) --
 * the same Mersenne-Twister stream as random.sample(deque, B)); device outputs s [B, D], a [B, A],
 * r [B], ns [B, D], d [B].  GCRL_ERR_INVALID "Not enough in buffer to sample" mirrors the assert. */
int gcrl_replay_sample(gcrl_replay *h, int64_t B, const int64_t *idx_host, float *s_dev, float *a_dev,
                       float *r_dev, float *ns_dev, float *d_dev, void *stream);
/* PERBuffer.sample(batch_size, beta) (:50-81).  u_host[B] = the uniforms np.random.choice consumes
 * (RandomState.random_sample(B)); positions = searchsorted(cumsum(P) / cumsum(P)[-1], u, "right") with
 * P = priorities / priorities.sum() in float32, bit-exact (see per.cu); weights_dev[B] =
 * (N P[i])^-beta / max.  idx_host_out (optional): the drawn deque positions, copied back with a stream
 * synchronise; NULL keeps the call asynchronous. */
int gcrl_replay_sample_prioritized(gcrl_replay *h, int64_t B, const double *u_host, double beta,
                                   float *s_dev, float *a_dev, float *r_dev, float *ns_dev, float *d_dev,
                                   float *weights_dev, int64_t *idx_host_out, void *stream);
/* update_priorities(indices, td) (:86-89): priority = (|td| + 1e-6)^alpha in float32, applied in list
 * order (the last duplicate wins).  idx_host[B] = deque positions, or NULL = the positions drawn by the
 * preceding sample_prioritized (kept on the device; no host round trip). */
int gcrl_replay_update_priorities(gcrl_replay *h, int64_t B, const int64_t *idx_host, const float *td_dev,
                                  void *stream);
/* priorities in deque order, host float[len] (tests, checkpoints) */
int gcrl_replay_get_priorities(gcrl_replay *h, float *prio_host, void *stream);
int gcrl_replay_set_priorities(gcrl_replay *h, const float *prio_host, int64_t n, void *stream);
/* stored rows [first, first + n) in deque order, packed host rows (tests, checkpoints) */
int gcrl_replay_get_rows(gcrl_replay *h, int64_t first, int64_t n, float *rows_host, void *stream);
/* Of the last sample_prioritized: the float32 priority sum, and whether the float64 cumsum had additions that
 * round (1: every rounding tracked, per.cu) or none (0: order-independent fixed-point scan). */
int gcrl_replay_last_sample_info(gcrl_replay *h, float *priority_sum, int *sequential_cumsum, void *stream);
/* The deque positions drawn by the last sample_prioritized (what the reference returns as `indices`). */
int gcrl_replay_last_positions(gcrl_replay *h, int64_t B, int64_t *idx_host, void *stream);
/* Of the last sample_prioritized: P (float32 [len]) and the searched table (float64 [len]). */
int gcrl_replay_last_tables(gcrl_replay *h, float *p_host, double *cdf_host, void *stream);

/* The prioritised branch of critic_update (src/agent.py:1322-1324,1338-1340; TD3 :193-197,:232-233;
 * SAC :577-596,:620-621; TQC :993-997,:1021-1024): with flags bit3 set, gcrl_agent_update_* /
 * gcrl_sac_update_* weight every sample's critic loss with weights_dev[b] (mean(w * loss)) and write the
 * per-sample TD error |y - q| (max over the critics) to td_dev[b].  The two device arrays (max_batch
 * floats each) belong to the agent. */
int gcrl_agent_per_buffers(gcrl_agent *h, float **weights_dev, float **td_dev);
int gcrl_sac_per_buffers(gcrl_sac *h, float **weights_dev, float **td_dev);

/* n consecutive updates sampling from a uniform or prioritised buffer, issued as ONE graph launch (prioritised:
 * once the same (B, flags, length) repeats; while the ring is still filling every call issues its updates directly).
 * Equivalent, bit for bit, to n rounds of
 *   uniform:     gcrl_replay_sample(pos_host + i*B) -> gcrl_agent_update_batch / gcrl_sac_update_batch;
 *   prioritised: gcrl_replay_sample_prioritized(u_host + i*B, beta[i]) -> the update with flags[i] bit3 ->
 *                gcrl_replay_update_priorities(NULL, td) -> TD errors into td_host + i*B,
 * with flags[i], lr_critic[i], lr_actor[i] and the noise rows of update i as in gcrl_agent_update_many /
 * gcrl_sac_update_many.  flags[i] bit3 must be set exactly when the buffer is prioritised; beyond it, the flag bits of
 * those calls.  pos_host [n][B] (uniform) or u_host [n][B] and beta [n] (prioritised); the other pointers may be NULL.
 * metrics_host: float[n][8] / float[n][12] as in those calls; td_host (prioritised, may be NULL): float[n][B], read
 * back with one copy at the end of the call.  Afterwards the buffer's last positions and sample info are those of
 * update n - 1.  Refused as gcrl_agent_update_many / gcrl_sac_update_many are, and GCRL_ERR_UNDERFILLED when len < B;
 * on any error no step counter, sequence number or priority has moved. */
int gcrl_agent_update_many_replay(gcrl_agent *h, gcrl_replay *buf, int64_t B, int n, const int *flags,
                                  const int64_t *pos_host, const double *u_host, const double *beta,
                                  const float *noise_dev, const double *lr_critic, const double *lr_actor,
                                  float *metrics_host, float *td_host, void *stream);
int gcrl_sac_update_many_replay(gcrl_sac *h, gcrl_replay *buf, int64_t B, int n, const int *flags,
                                const int64_t *pos_host, const double *u_host, const double *beta,
                                const float *eps_next_dev, const float *eps_cur_dev, const double *lr_critic,
                                const double *lr_actor, float *metrics_host, float *td_host, void *stream);

/* ------------------------------------------------------------------------------------
 * Diagnostics / micro-benchmarks
 * ------------------------------------------------------------------------------------
 * One dense layer on device buffers (what nn.Linear + LeakyReLU, src/model.py:17-30, and its
 * autograd input-gradient compute), with a selectable engine:
 *   engine 0: fp32 FFMA tiles (mlp.cu);  engine 1: tcgen05 tensor cores, 3xTF32 split (tc_gemm.cu).
 *   mode 0: y = leaky(x w^T + bias);  mode 1: y = (x w^T) * leaky'(act) (engine 1 only);
 *   mode 2: y = x w^T + bias.
 * x [M, K] (ldx), w [N, K] (ldw), y [M, N] (ldy); leading dimensions multiples of 4 floats. */
/* Average duration (CUDA events on `stream`, back to back, warm) of the critic-phase kernel of the
 * small-batch path (fused.cu / cluster.cu: target actor + target critic + critic forward, Bellman
 * target, loss, critic input gradients) on the batch left resident by the last update of size B.
 * Feeds bench.py's roofline object; it recomputes the same activations, no state changes. */
int gcrl_agent_time_critic_kernel(gcrl_agent *h, int64_t B, int iters, float *ms_per_launch, void *stream);

int gcrl_dense_layer(int device, int engine, int mode, int64_t M, int N, int K, const float *x_dev,
                     int ldx, const float *w_dev, int ldw, const float *bias_dev, const float *act_dev,
                     int ldact, float *y_dev, int ldy, void *stream);

/* Split-batch weight gradient of one dense layer (autograd of nn.Linear over the batch):
 *   pw[s][n][k] = sum_{m in slab s} dz[m, n] x[m, k],  pb[s][n] = sum_{m in slab s} dz[m, n]
 * for s < *splits_out <= max_splits slabs of batch rows (the caller sums the slabs in order).
 * engine 0: fp32 FFMA tiles; engine 1: tcgen05, MN-major operands, 3xTF32 split. */
/* The tensor-core dense layer as the agents call it: the weight operand pre-split into its TF32 hi / lo halves
 * (gcrl_split_tf32: hi = rna_tf32(w), lo = rna_tf32(w - hi); same layout as w), so that the kernel only splits the
 * activation tile.  Same modes as gcrl_dense_layer, and mode 3: y = x w^T (bare product; bias and act unused). */
int gcrl_split_tf32(int device, const float *src_dev, float *hi_dev, float *lo_dev, int64_t n, void *stream);
int gcrl_dense_layer_presplit(int device, int mode, int64_t M, int N, int K, const float *x_dev, int ldx,
                              const float *w_hi_dev, const float *w_lo_dev, int ldw, const float *bias_dev,
                              const float *act_dev, int ldact, float *y_dev, int ldy, void *stream);
/* n <= 8 independent pre-split dense layers of one shape and mode in ONE tcgen05 launch (the critic ensemble of the
 * SAC / TQC tensor-core engine): member i reads x_dev[i], w_hi_dev[i], w_lo_dev[i], bias_dev[i] / act_dev[i] and
 * writes y_dev[i] (host arrays of device pointers; bias_dev / act_dev may be NULL where the mode does not read them).
 * Each member's y equals gcrl_dense_layer_presplit of that member on the single-CTA kernel, bit for bit. */
int gcrl_dense_layer_ensemble(int device, int n, int mode, int64_t M, int N, int K, const float *const *x_dev,
                              int ldx, const float *const *w_hi_dev, const float *const *w_lo_dev, int ldw,
                              const float *const *bias_dev, const float *const *act_dev, int ldact,
                              float *const *y_dev, int ldy, void *stream);

int gcrl_dense_wgrad(int device, int engine, int64_t M, int N, int K, const float *dz_dev, int lddz,
                     const float *x_dev, int ldx, float *pw_dev, int ldw, int64_t w_split_stride,
                     float *pb_dev, int64_t b_split_stride, int max_splits, int *splits_out, void *stream);

/* The quantile-critic loss of a TQC update on caller buffers: the same three launches
 * (quantile_target_kernel<KPL> -> quantile_huber_kernel -> quantile_metrics_kernel) an update issues.
 *   1 <= n <= 8 critics of M >= 1 atoms, n * M <= 256, 0 <= drop < M dropped per critic, K = n (M - drop) kept
 *   zt, z : [n][B][ldm] target / current atoms, critic i at + i * zstride (ldm >= M, multiple of 4; the agent's is
 *           pad4(M); zstride >= B * ldm)
 *   logp, r, d : [B];  w : [B] importance weights or NULL;  coef >= 0: entropy coefficient, < 0: *alpha_dev
 *   y  : [B][ldy] sorted, truncated targets, ldy >= K, multiple of 4
 *   dz : [n][B][ldm] (same layout as z);  out : float[n + 1], per-critic losses then the batch-mean TD;
 *   td_rows : [B] or NULL;  scratch : n * (B + ceil(B / max(1, 256 / M))) floats
 * Only columns < M of z / zt and < K of y, and rows < B, are read or written. */
int gcrl_quantile_critic_loss(int device, int n, int M, int drop, int64_t B, const float *zt_dev, const float *z_dev,
                              int ldm, int64_t zstride, const float *logp_dev, const float *r_dev, const float *d_dev,
                              const float *w_dev, float gamma, float coef, const float *alpha_dev, float *y_dev, int ldy,
                              float *dz_dev, float *out_dev, float *td_rows_dev, float *scratch_dev, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* GCRL_B200_H */
