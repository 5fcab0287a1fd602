// The library-internal side of the HER buffer (her.cu) and the uniform / prioritised replay buffer (per.cu) that the
// agents (agent.cu, sac.cu) sample from.
#pragma once
#include "her_device.cuh"

struct gcrl_her;
namespace gcrl {
SampleScalars her_next_scalars(gcrl_her *h, bool positions_given);
const HerGeom &her_geom(const gcrl_her *h);
int64_t her_len(const gcrl_her *h);
void her_sample_into(gcrl_her *h, int64_t B, const int64_t *idx_host, float *s, float *a, float *r,
                     float *ns, float *d, int64_t *idx_out, cudaStream_t st);
int her_state_dim(const gcrl_her *h);
int her_act_dim(const gcrl_her *h);
int her_device(const gcrl_her *h);
int her_n_step(const gcrl_her *h);
void her_sample_graphed(gcrl_her *h, int64_t B, const SampleScalars *sc_dev, const int64_t *idx_dev, float *s,
                        float *a, float *r, float *ns, float *d, cudaStream_t st);
unsigned long long &her_draw_epoch(gcrl_her *h);
bool replay_prioritized(const gcrl_replay *h);
int replay_state_dim(const gcrl_replay *h);
int replay_act_dim(const gcrl_replay *h);
int replay_device(const gcrl_replay *h);
uint64_t replay_epoch(const gcrl_replay *h);
int64_t replay_many_n(const gcrl_replay *h);
void replay_many_stage(gcrl_replay *h, int64_t B, int n, const int64_t *pos_host, const double *u_host,
                       const double *beta, cudaStream_t st);
void replay_many_sample(gcrl_replay *h, int64_t B, int n, int i, float *s, float *a, float *r, float *ns, float *d,
                        float *weights_dev, cudaStream_t st);
void replay_many_write_back(gcrl_replay *h, int64_t B, const float *td_dev, cudaStream_t st);
}  // namespace gcrl
