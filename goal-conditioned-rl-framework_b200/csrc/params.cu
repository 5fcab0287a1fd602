// Host side of the parameter containers (params.cuh).
#include <cstring>
#include <initializer_list>

#include "params.cuh"

namespace gcrl {

void upload_rows(float *dst, const float *src, int rows, int cols, int ld, cudaStream_t st) {
  std::vector<float> padded(size_t(rows) * ld, 0.f);
  for (int r = 0; r < rows; ++r) std::memcpy(&padded[size_t(r) * ld], src + size_t(r) * cols, size_t(cols) * 4);
  GCRL_CUDA(cudaMemcpyAsync(dst, padded.data(), padded.size() * 4, cudaMemcpyHostToDevice, st));
  GCRL_CUDA(cudaStreamSynchronize(st));
}

void download_rows(float *dst, const float *src, int rows, int cols, int ld, cudaStream_t st) {
  std::vector<float> padded(size_t(rows) * ld);
  GCRL_CUDA(cudaMemcpyAsync(padded.data(), src, padded.size() * 4, cudaMemcpyDeviceToHost, st));
  GCRL_CUDA(cudaStreamSynchronize(st));
  for (int r = 0; r < rows; ++r) std::memcpy(dst + size_t(r) * cols, &padded[size_t(r) * ld], size_t(cols) * 4);
}

void WeightCopies::init(int total_, int nlinear, const std::vector<Linear> &transposed, bool halves) {
  total = total_;
  t_off.assign(size_t(nlinear), -1);
  ldt.assign(size_t(nlinear), 0);
  if (halves) alloc_halves();
  if (transposed.empty()) return;
  std::vector<int> map(size_t(total), -1);
  for (const Linear &t : transposed) {
    ldt[t.layer] = pad4(t.rows);
    t_off[t.layer] = total_t;
    for (int o = 0; o < t.rows; ++o)
      for (int i = 0; i < t.cols; ++i) map[size_t(t.w_off) + size_t(o) * t.ldw + i] = total_t + i * ldt[t.layer] + o;
    total_t += t.cols * ldt[t.layer];
  }
  tmap = dev_alloc<int>(total);
  GCRL_CUDA(cudaMemcpy(tmap, map.data(), size_t(total) * sizeof(int), cudaMemcpyHostToDevice));
  pT = dev_alloc<float>(total_t);
  GCRL_CUDA(cudaMemset(pT, 0, size_t(total_t) * 4));
  if (halves) alloc_halves();
}

void WeightCopies::alloc_halves() {
  if (p_hi == nullptr) { p_hi = dev_alloc<float>(total); p_lo = dev_alloc<float>(total); }
  if (pT != nullptr && pT_hi == nullptr) { pT_hi = dev_alloc<float>(total_t); pT_lo = dev_alloc<float>(total_t); }
}

void WeightCopies::destroy() {
  for (void *q : {(void *)tmap, (void *)pT, (void *)p_hi, (void *)p_lo, (void *)pT_hi, (void *)pT_lo})
    if (q) cudaFree(q);
}

void MlpParams::layout(int in, int hid, int out, int hidden_layers) {
  layers = hidden_layers + 1;
  int off = 0;
  for (int l = 0; l < layers; ++l) {
    in_d.push_back(l == 0 ? in : hid);
    out_d.push_back(l == layers - 1 ? out : hid);
    ldw.push_back(pad4(in_d[l]));
    w_off.push_back(off); off += out_d[l] * ldw[l];
    b_off.push_back(off); off += pad4(out_d[l]);
  }
  total = off;
}

void MlpParams::alloc(bool trainable, float *grad_store) {
  auto zeros = [&] {
    float *q = dev_alloc<float>(total);
    GCRL_CUDA(cudaMemset(q, 0, size_t(total) * 4));
    return q;
  };
  p = zeros();
  if (!trainable) return;
  owns_g = grad_store == nullptr;
  g = owns_g ? zeros() : grad_store;
  m = zeros();
  v = zeros();
}

void MlpParams::init_copies(int t_first, int t_last, bool halves) {
  std::vector<WeightCopies::Linear> tr;
  for (int l = t_first; l < t_last; ++l) tr.push_back({l, w_off[l], out_d[l], in_d[l], ldw[l]});
  copies.init(total, layers, tr, halves);
}

void MlpParams::destroy() {
  for (float *q : {p, m, v, owns_g ? g : nullptr})
    if (q) cudaFree(q);
  copies.destroy();
}

}  // namespace gcrl
