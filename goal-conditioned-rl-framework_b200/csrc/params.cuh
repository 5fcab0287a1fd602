// Parameter containers of the agents (agent.cu: DDPG / TD3, sac.cu: SAC / TQC): how a network sits in one flat fp32
// buffer, and the copies of its weights that follow that buffer.
#pragma once
#include <vector>

#include "mlp.cuh"

namespace gcrl {

inline int pad4(int x) { return (x + 3) & ~3; }

// host rows [rows][cols] <-> device rows [rows][ld]; the upload writes the zero padding of each row too.  Both
// synchronise `st` before they return.
void upload_rows(float *dst, const float *src, int rows, int cols, int ld, cudaStream_t st);
void download_rows(float *dst, const float *src, int rows, int cols, int ld, cudaStream_t st);

// Weight copies of a flat parameter buffer p[total]: for the listed Linear layers a transposed copy W^T[in][ldt]
// (the operand of the row-slab kernels and of the tensor-core input gradient dX = dZ W), and with `halves` the TF32
// hi / lo halves of p and of W^T (the tensor-core engine's pre-split weight operand, tc_gemm.cu).  The optimiser and
// the Polyak kernel write W^T through tmap with every step; the halves are refreshed after every optimiser / Polyak
// step of an update that runs on the tensor cores, and before such an update once p changed in any other way (stale).
struct WeightCopies {
  struct Linear { int layer, w_off, rows, cols, ldw; };   // W[rows][ldw] at p + w_off
  std::vector<int> t_off, ldt;   // per Linear layer (t_off -1: no transposed copy)
  int total = 0, total_t = 0;
  int *tmap = nullptr;           // [total] -> index into pT, -1 elsewhere; nullptr when nothing is transposed
  float *pT = nullptr, *p_hi = nullptr, *p_lo = nullptr, *pT_hi = nullptr, *pT_lo = nullptr;
  bool stale = true;

  void init(int total, int nlinear, const std::vector<Linear> &transposed, bool halves);
  void alloc_halves();                                    // (those that do not exist yet)
  void split(const float *p, cudaStream_t st) {            // the halves of p, then of W^T
    launch_split_tf32(p, p_hi, p_lo, total, st);
    if (pT != nullptr) launch_split_tf32(pT, pT_hi, pT_lo, total_t, st);
  }
  void split_if_stale(const float *p, cudaStream_t st) {   // eager, outside capture
    if (p_hi == nullptr || !stale) return;
    split(p, st);
    stale = false;
  }
  // weights written from outside an update: W^T follows now, the halves before the next tensor-core update
  void weights_changed(const float *p, cudaStream_t st) {
    if (tmap != nullptr) launch_sync_transposed(p, pT, tmap, total, st);
    stale = true;
  }
  void destroy();
};

// A stack of Linear layers in one flat buffer: layer l is W[out_d][ldw] at w_off, then its bias at b_off (16 B-aligned
// segments), with flat gradient / Adam m / Adam v buffers of the same layout.
struct MlpParams {
  int layers = 0;
  std::vector<int> in_d, out_d, ldw, w_off, b_off;
  int total = 0;
  float *p = nullptr, *g = nullptr, *m = nullptr, *v = nullptr;
  bool owns_g = false;
  WeightCopies copies;

  void layout(int in, int hid, int out, int hidden_layers);   // no allocation
  // p; trainable: m, v and g, or g = grad_store (a slice of the caller's storage)
  void alloc(bool trainable, float *grad_store = nullptr);
  void init_copies(int t_first, int t_last, bool halves);     // W^T of the Linear layers [t_first, t_last)
  void destroy();
  const float *W(int l) const { return p + w_off[l]; }
  const float *b(int l) const { return p + b_off[l]; }
};

}  // namespace gcrl
