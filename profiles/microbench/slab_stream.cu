// Micro-benchmark behind the round-2 redesign of the row-slab kernels (fused.cu): how fast can ONE CTA per SM
// stream a network's weights (every CTA needs all of them) and do the slab FMAs?
//   mode 0: per-thread __ldg of 16-byte column slices (the round-1 scheme)
//   mode 1: producer warp + cp.async.bulk ring in shared memory, consumers LDS.128 + FFMA
//   mode 2: mode 1 with 2-CTA clusters, each CTA fetching half of every chunk and multicasting it to both
//   mode 5: 2D split over a cluster of C CTAs sharing S rows: CTA c computes columns [c H/C, (c+1) H/C) of every
//           layer for all S rows (the K chunks of fused.cu's slab_matmul at H = 256), then stores its slice into
//           every peer's activation buffer (16-byte st.shared::cluster) and meets them at a split cluster barrier
// Output: us per launch for a chain of `steps` 256x256 layer steps on R rows per CTA.
// Build: nvcc -gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -o slab_stream slab_stream.cu
#include <cooperative_groups.h>
#include <cuda_runtime.h>
#include <cstdio>
#include <cstdlib>
#include <cstdint>
#include <vector>
namespace cg = cooperative_groups;
template <typename F> float time_it(F f, int iters = 20);

#define CK(x) do { cudaError_t e = (x); if (e != cudaSuccess) { printf("%s: %s\n", #x, cudaGetErrorString(e)); exit(1); } } while (0)

constexpr int H = 256;
constexpr int kConsumerWarps = 16, kConsumers = kConsumerWarps * 32;

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t bar, uint32_t cta) {
  uint32_t remote;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(remote) : "r"(bar), "r"(cta));
  asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(remote) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tWAIT_%=:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
      "@p bra DONE_%=;\n\tbra WAIT_%=;\n\tDONE_%=:\n\t}" ::"r"(bar), "r"(parity) : "memory");
}
__device__ __forceinline__ void mbar_wait_cluster(uint32_t bar, uint32_t parity) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tWAIT_%=:\n\t"
      "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%0], %1;\n\t"
      "@p bra DONE_%=;\n\tbra WAIT_%=;\n\tDONE_%=:\n\t}" ::"r"(bar), "r"(parity) : "memory");
}
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void *src, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}
__device__ __forceinline__ void bulk_g2s_mc(uint32_t dst, const void *src, uint32_t bytes, uint32_t bar, uint16_t mask) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster [%0], [%1], %2, [%3], %4;"
               ::"r"(dst), "l"(src), "r"(bytes), "r"(bar), "h"(mask) : "memory");
}
__device__ __forceinline__ void bar_consumers() { asm volatile("bar.sync 1, %0;" ::"n"(kConsumers) : "memory"); }

template <int R> __device__ __forceinline__ void load_rows(const float *p, float (&x)[R]) {
  if constexpr (R == 2) { const float2 t = *reinterpret_cast<const float2 *>(p); x[0] = t.x; x[1] = t.y; }
  else { const float4 t = *reinterpret_cast<const float4 *>(p); x[0] = t.x; x[1] = t.y; x[2] = t.z; x[3] = t.w; }
}

// combine of the K-split partials + bias/leaky epilogue, as in fused.cu
template <int R>
__device__ __forceinline__ void combine(float (&acc)[4][R], float *red, float *yT, int warp, int lane, int tid) {
  const int cw = warp & 1, ks = warp >> 1, j0 = (cw * 32 + lane) * 4;
#pragma unroll
  for (int c = 0; c < 4; ++c)
#pragma unroll
    for (int r = 0; r < R; ++r) red[(ks * H + j0 + c) * R + r] = acc[c][r];
  bar_consumers();
  for (int e = tid; e < H * R; e += kConsumers) {
    float s = 0.f;
#pragma unroll
    for (int k2 = 0; k2 < 8; ++k2) s += red[k2 * H * R + e];
    yT[e] = s > 0.f ? s : 0.01f * s;
  }
  bar_consumers();
}

template <int MODE> __device__ __forceinline__ float4 ldw(const float4 *p) {
  float4 v;
  if constexpr (MODE == 0) return __ldg(p);
  else if constexpr (MODE == 1) asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p));
  else if constexpr (MODE == 2) asm volatile("ld.global.cg.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p));
  else asm volatile("ld.global.nc.L1::evict_first.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p));
  return v;
}
template <int R, int MODE>
__global__ void __launch_bounds__(kConsumers, 1) ldg_kernel(const float *W, int nlayers, int steps, float *out) {
  __shared__ float xT[2][H * R];
  extern __shared__ float4 dyn[];
  float *red = reinterpret_cast<float *>(dyn);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  for (int e = tid; e < H * R; e += kConsumers) xT[0][e] = 0.001f * (e % 7);
  __syncthreads();
  const int cw = warp & 1, ks = warp >> 1, j0 = (cw * 32 + lane) * 4;
  for (int s = 0; s < steps; ++s) {
    const float *M = W + size_t(s % nlayers) * H * H + size_t(ks * 32) * H + j0;
    const float *x = xT[s & 1] + ks * 32 * R;
    float acc[4][R] = {};
#pragma unroll 8
    for (int i = 0; i < 32; ++i) {
      const float4 w = ldw<MODE>(reinterpret_cast<const float4 *>(M + size_t(i) * H));
      float xv[R];
      load_rows<R>(x + i * R, xv);
#pragma unroll
      for (int r = 0; r < R; ++r) {
        acc[0][r] = fmaf(w.x, xv[r], acc[0][r]); acc[1][r] = fmaf(w.y, xv[r], acc[1][r]);
        acc[2][r] = fmaf(w.z, xv[r], acc[2][r]); acc[3][r] = fmaf(w.w, xv[r], acc[3][r]);
      }
    }
    combine<R>(acc, red, xT[(s + 1) & 1], warp, lane, tid);
  }
  if (tid < R) out[blockIdx.x * R + tid] = xT[steps & 1][tid];
}

// ring of STAGES chunks of CR K-rows (CR * 1 KB each); warp 16 is the producer
template <int R, int CR, int STAGES, int CL>
__global__ void __launch_bounds__(kConsumers + 32, 1) ring_kernel(const float *W, int nlayers, int steps, float *out) {
  extern __shared__ float4 dyn[];
  float *ring = reinterpret_cast<float *>(dyn);                 // STAGES * CR * H floats
  float *red = ring + STAGES * CR * H;                          // 8 * H * R
  float *xT = red + 8 * H * R;                                  // 2 * H * R
  __shared__ __align__(8) uint64_t full[STAGES], empty[STAGES];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  uint32_t cta_rank = 0;
  if (CL > 1) cta_rank = cg::this_cluster().block_rank();
  if (tid == 0) {
    for (int s = 0; s < STAGES; ++s) { mbar_init(smem_u32(&full[s]), 1); mbar_init(smem_u32(&empty[s]), kConsumerWarps * CL); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  for (int e = tid; e < H * R; e += blockDim.x) xT[e] = 0.001f * (e % 7);
  __syncthreads();
  if (CL > 1) cg::this_cluster().sync();
  constexpr int chunks_per_layer = H / CR;
  constexpr uint32_t chunk_bytes = CR * H * 4;
  const int total_chunks = steps * chunks_per_layer;
  if (warp == kConsumerWarps) {
    if (lane == 0) {
      for (int c = 0; c < total_chunks; ++c) {
        const int st = c % STAGES, it = c / STAGES;
        if (it > 0) { if (CL > 1) mbar_wait_cluster(smem_u32(&empty[st]), (it - 1) & 1); else mbar_wait(smem_u32(&empty[st]), (it - 1) & 1); }
        const int layer = (c / chunks_per_layer) % nlayers, cc = c % chunks_per_layer;
        const float *src = W + size_t(layer) * H * H + size_t(cc) * CR * H;
        mbar_expect_tx(smem_u32(&full[st]), chunk_bytes);
        if (CL == 1) {
          bulk_g2s(smem_u32(ring + st * CR * H), src, chunk_bytes, smem_u32(&full[st]));
        } else {
          const uint32_t part = chunk_bytes / CL;
          bulk_g2s_mc(smem_u32(ring + st * CR * H) + cta_rank * part, reinterpret_cast<const char *>(src) + cta_rank * part,
                      part, smem_u32(&full[st]), uint16_t((1u << CL) - 1));
        }
      }
    }
  } else {
    const int cw = warp & 1, ks = warp >> 1, j0 = (cw * 32 + lane) * 4;
    constexpr int RW = CR / 8;       // K-rows of a chunk per K-group
    int c = 0;
    for (int s = 0; s < steps; ++s) {
      const float *x = xT + (s & 1) * H * R;
      float acc[4][R] = {};
      for (int cc = 0; cc < chunks_per_layer; ++cc, ++c) {
        const int st = c % STAGES, it = c / STAGES;
        mbar_wait(smem_u32(&full[st]), it & 1);
        const float *wc = ring + st * CR * H + (ks * RW) * H + j0;
        const float *xc = x + (cc * CR + ks * RW) * R;
#pragma unroll
        for (int i = 0; i < RW; ++i) {
          const float4 w = *reinterpret_cast<const float4 *>(wc + i * H);
          float xv[R];
          load_rows<R>(xc + i * R, xv);
#pragma unroll
          for (int r = 0; r < R; ++r) {
            acc[0][r] = fmaf(w.x, xv[r], acc[0][r]); acc[1][r] = fmaf(w.y, xv[r], acc[1][r]);
            acc[2][r] = fmaf(w.z, xv[r], acc[2][r]); acc[3][r] = fmaf(w.w, xv[r], acc[3][r]);
          }
        }
        __syncwarp();
        if (lane == 0) {
          if (CL == 1) mbar_arrive(smem_u32(&empty[st]));
          else for (uint32_t p = 0; p < CL; ++p) mbar_arrive_cluster(smem_u32(&empty[st]), p);
        }
      }
      combine<R>(acc, red, xT + ((s + 1) & 1) * H * R, warp, lane, tid);
    }
    if (tid < R) out[blockIdx.x * R + tid] = xT[(steps & 1) * H * R + tid];
  }
  if (CL > 1) cg::this_cluster().sync();
}

// mode 3: N-split over a 2-CTA cluster: the pair carries R rows, each CTA streams HALF of every layer's columns
// (per-thread __ldg), the half results are exchanged through distributed shared memory, one cluster barrier per layer
template <int R>
__global__ void __launch_bounds__(kConsumers, 1) nsplit_kernel(const float *W, int nlayers, int steps, float *out) {
  __shared__ __align__(16) float xT[2][H * R];
  extern __shared__ float4 dyn[];
  float *red = reinterpret_cast<float *>(dyn);       // [16][128][R]
  cg::cluster_group cluster = cg::this_cluster();
  const unsigned rank = cluster.block_rank();
  float *peer_x0 = cluster.map_shared_rank(&xT[0][0], rank ^ 1);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  for (int e = tid; e < H * R; e += kConsumers) xT[0][e] = 0.001f * (e % 7);
  __syncthreads();
  cluster.sync();
  const int ks = warp, j0 = rank * 128 + lane * 4;          // 16 K-groups of 16 rows, 128 columns per CTA
  for (int s = 0; s < steps; ++s) {
    const float *M = W + size_t(s % nlayers) * H * H + size_t(ks * 16) * H + j0;
    const float *x = xT[s & 1] + ks * 16 * R;
    float acc[4][R] = {};
#pragma unroll 16
    for (int i = 0; i < 16; ++i) {
      const float4 w = __ldg(reinterpret_cast<const float4 *>(M + size_t(i) * H));
      float xv[R];
      load_rows<R>(x + i * R, xv);
#pragma unroll
      for (int r = 0; r < R; ++r) {
        acc[0][r] = fmaf(w.x, xv[r], acc[0][r]); acc[1][r] = fmaf(w.y, xv[r], acc[1][r]);
        acc[2][r] = fmaf(w.z, xv[r], acc[2][r]); acc[3][r] = fmaf(w.w, xv[r], acc[3][r]);
      }
    }
#pragma unroll
    for (int c = 0; c < 4; ++c)
#pragma unroll
      for (int r = 0; r < R; ++r) red[(ks * 128 + lane * 4 + c) * R + r] = acc[c][r];
    __syncthreads();
    float *ynext = xT[(s + 1) & 1];
    float *ypeer = peer_x0 + ((s + 1) & 1) * H * R;
    for (int e = tid; e < 128 * R; e += kConsumers) {
      float v = 0.f;
#pragma unroll
      for (int k2 = 0; k2 < 16; ++k2) v += red[k2 * 128 * R + e];
      v = v > 0.f ? v : 0.01f * v;
      ynext[rank * 128 * R + e] = v;
      ypeer[rank * 128 * R + e] = v;
    }
    cluster.sync();
  }
  if (tid < R) out[blockIdx.x * R + tid] = xT[steps & 1][tid];
}
template <int R> void run_nsplit(const float *W, int nl, int steps, float *out, int grid) {
  const size_t smem = size_t(16) * 128 * R * 4;
  auto k = nsplit_kernel<R>;
  CK(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem)));
  cudaLaunchConfig_t cfg{}; cfg.gridDim = dim3(grid); cfg.blockDim = dim3(kConsumers); cfg.dynamicSmemBytes = smem;
  cudaLaunchAttribute attr[1]; attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr; cfg.numAttrs = 1;
  const float us = time_it([&] { CK(cudaLaunchKernelEx(&cfg, k, W, nl, steps, out)); });
  printf("nsplit R=%d (rows per 2-CTA pair) grid=%3d steps=%d: %7.2f us  (%.2f us/step)\n", R, grid, steps, us, us / steps);
}

// mode 4: as mode 0, but software-pipelined: the 8 weight loads of K-batch b+1 are issued BEFORE the 64 FMAs of
// batch b (register double buffer), so a warp's load latency overlaps its own arithmetic
template <int R, int DEPTH>
__global__ void __launch_bounds__(kConsumers, 1) ldg_pipe_kernel(const float *W, int nlayers, int steps, float *out) {
  __shared__ float xT[2][H * R];
  extern __shared__ float4 dyn[];
  float *red = reinterpret_cast<float *>(dyn);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  for (int e = tid; e < H * R; e += kConsumers) xT[0][e] = 0.001f * (e % 7);
  __syncthreads();
  const int cw = warp & 1, ks = warp >> 1, j0 = (cw * 32 + lane) * 4;
  constexpr int NB = 32 / DEPTH;     // batches of DEPTH rows per K-group
  for (int s = 0; s < steps; ++s) {
    const float *M = W + size_t(s % nlayers) * H * H + size_t(ks * 32) * H + j0;
    const float *x = xT[s & 1] + ks * 32 * R;
    float acc[4][R] = {};
    float4 wb[2][DEPTH];
#pragma unroll
    for (int i = 0; i < DEPTH; ++i) wb[0][i] = __ldg(reinterpret_cast<const float4 *>(M + size_t(i) * H));
#pragma unroll
    for (int b = 0; b < NB; ++b) {
      if (b + 1 < NB) {
#pragma unroll
        for (int i = 0; i < DEPTH; ++i) wb[(b + 1) & 1][i] = __ldg(reinterpret_cast<const float4 *>(M + size_t((b + 1) * DEPTH + i) * H));
      }
#pragma unroll
      for (int i = 0; i < DEPTH; ++i) {
        const float4 w = wb[b & 1][i];
        float xv[R];
        load_rows<R>(x + (b * DEPTH + i) * R, xv);
#pragma unroll
        for (int r = 0; r < R; ++r) {
          acc[0][r] = fmaf(w.x, xv[r], acc[0][r]); acc[1][r] = fmaf(w.y, xv[r], acc[1][r]);
          acc[2][r] = fmaf(w.z, xv[r], acc[2][r]); acc[3][r] = fmaf(w.w, xv[r], acc[3][r]);
        }
      }
    }
    combine<R>(acc, red, xT[(s + 1) & 1], warp, lane, tid);
  }
  if (tid < R) out[blockIdx.x * R + tid] = xT[steps & 1][tid];
}
template <int R, int DEPTH> void run_ldg_pipe(const float *W, int nl, int steps, float *out, int grid) {
  const size_t smem = size_t(8) * H * R * 4;
  const float us = time_it([&] { ldg_pipe_kernel<R, DEPTH><<<grid, kConsumers, smem>>>(W, nl, steps, out); });
  printf("ldg-pipelined R=%d depth=%2d grid=%3d steps=%d: %7.2f us  (%.2f us/step)\n", R, DEPTH, grid, steps, us, us / steps);
}

// mode 5: 2D split.  Thread = (4-column group, R = S / C row group, K chunk): 8 K chunks of 32 rows as in fused.cu at
// H = 256, so a thread does the same R-row, 4-column, 32-deep FMA chain as the R-row kernel, but the 4 lanes of a
// warp that share a column group load the same weight float4 (one L1 wavefront for 8 float4 per warp).
// PF = 1: between the barrier's arrive and wait, the first 8 weight float4 of the next step go into registers.
__device__ __forceinline__ void st_cluster4(uint32_t local, uint32_t cta, float4 v) {
  uint32_t remote;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(remote) : "r"(local), "r"(cta));
  asm volatile("st.shared::cluster.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(remote), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w)
               : "memory");
}
template <int C, int S, int PF>
__global__ void __launch_bounds__(kConsumers, 1) csplit_kernel(const float *W, int nlayers, int steps, float *out) {
  constexpr int R = S / C, Nc = H / C, G = Nc / 4, KC = 32;
  static_assert(G * C * (H / KC) == kConsumers, "one thread per (column group, row group, K chunk)");
  extern __shared__ float4 dyn[];
  float *xT = reinterpret_cast<float *>(dyn);            // [2][H][S]
  float *red = xT + 2 * H * S;                           // [8][Nc][S]
  const unsigned rank = cg::this_cluster().block_rank();
  const int tid = threadIdx.x, cgp = tid % G, rg = (tid / G) % C, ks = tid / (G * C);
  const int j0 = rank * Nc + cgp * 4;
  for (int e = tid; e < H * S; e += kConsumers) xT[e] = 0.001f * (e % 7);
  cg::this_cluster().sync();
  float4 wpre[8];
  auto preload = [&](int s) {
    const float *M = W + size_t(s % nlayers) * H * H + size_t(ks * KC) * H + j0;
#pragma unroll
    for (int i = 0; i < 8; ++i) wpre[i] = __ldg(reinterpret_cast<const float4 *>(M + size_t(i) * H));
  };
  if (PF) preload(0);
  for (int s = 0; s < steps; ++s) {
    const float *M = W + size_t(s % nlayers) * H * H + size_t(ks * KC) * H + j0;
    const float *x = xT + (s & 1) * H * S + ks * KC * S + rg * R;
    float acc[4][R] = {};
#pragma unroll
    for (int i = 0; i < KC; ++i) {
      const float4 w = (PF && i < 8) ? wpre[i & 7] : __ldg(reinterpret_cast<const float4 *>(M + size_t(i) * H));
      float xv[R];
      if constexpr (R == 1) xv[0] = x[i * S];
      else if constexpr (R == 2) { const float2 t = *reinterpret_cast<const float2 *>(x + i * S); xv[0] = t.x; xv[1] = t.y; }
      else {
#pragma unroll
        for (int q = 0; q < R / 4; ++q) {
          const float4 t = *reinterpret_cast<const float4 *>(x + i * S + 4 * q);
          xv[4 * q] = t.x; xv[4 * q + 1] = t.y; xv[4 * q + 2] = t.z; xv[4 * q + 3] = t.w;
        }
      }
#pragma unroll
      for (int r = 0; r < R; ++r) {
        acc[0][r] = fmaf(w.x, xv[r], acc[0][r]); acc[1][r] = fmaf(w.y, xv[r], acc[1][r]);
        acc[2][r] = fmaf(w.z, xv[r], acc[2][r]); acc[3][r] = fmaf(w.w, xv[r], acc[3][r]);
      }
    }
#pragma unroll
    for (int c = 0; c < 4; ++c)
#pragma unroll
      for (int r = 0; r < R; ++r) red[(ks * Nc + cgp * 4 + c) * S + rg * R + r] = acc[c][r];
    __syncthreads();
    const uint32_t ynext = smem_u32(xT + ((s + 1) & 1) * H * S + rank * Nc * S);
    for (int e4 = tid; e4 < Nc * S / 4; e4 += kConsumers) {
      float v[4];
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        float t = red[e4 * 4 + q];
#pragma unroll
        for (int k2 = 1; k2 < H / KC; ++k2) t += red[k2 * Nc * S + e4 * 4 + q];
        v[q] = t > 0.f ? t : 0.01f * t;
      }
      const float4 v4 = make_float4(v[0], v[1], v[2], v[3]);
#pragma unroll
      for (int p = 0; p < C; ++p) st_cluster4(ynext + e4 * 16, (rank + p) % C, v4);
    }
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    if (PF && s + 1 < steps) preload(s + 1);
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
  }
  if (tid < S) out[(blockIdx.x / C) * S + tid] = xT[(steps & 1) * H * S + tid];
}
template <int C, int S, int PF> void run_csplit(const float *W, int nl, int steps, float *out, int grid) {
  const size_t smem = (size_t(2) * H * S + size_t(8) * (H / C) * S) * 4;
  auto k = csplit_kernel<C, S, PF>;
  CK(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem)));
  CK(cudaFuncSetAttribute(k, cudaFuncAttributeNonPortableClusterSizeAllowed, 1));
  cudaLaunchConfig_t cfg{}; cfg.gridDim = dim3(grid); cfg.blockDim = dim3(kConsumers); cfg.dynamicSmemBytes = smem;
  cudaLaunchAttribute attr[1]; attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = C; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr; cfg.numAttrs = 1;
  int nclusters = 0;
  CK(cudaOccupancyMaxActiveClusters(&nclusters, k, &cfg));
  const float us = time_it([&] { CK(cudaLaunchKernelEx(&cfg, k, W, nl, steps, out)); });
  printf("csplit C=%d S=%2d R=%d prefetch=%d grid=%3d (%3d rows) steps=%d: %7.2f us  (%.2f us/step, smem %zu KB, "
         "max active clusters %d, need %d)\n", C, S, S / C, PF, grid, grid / C * S, steps, us, us / steps, smem >> 10,
         nclusters, grid / C);
}

template <typename F> float time_it(F f, int iters) {
  cudaEvent_t e0, e1; CK(cudaEventCreate(&e0)); CK(cudaEventCreate(&e1));
  for (int i = 0; i < 3; ++i) f();
  CK(cudaDeviceSynchronize());
  CK(cudaEventRecord(e0));
  for (int i = 0; i < iters; ++i) f();
  CK(cudaEventRecord(e1)); CK(cudaEventSynchronize(e1));
  float ms; CK(cudaEventElapsedTime(&ms, e0, e1));
  CK(cudaGetLastError());
  return ms * 1000.f / iters;
}

template <int R, int CR, int STAGES, int CL> void run_ring(const float *W, int nl, int steps, float *out, int grid) {
  const size_t smem = (size_t(STAGES) * CR * H + 8 * H * R + 2 * H * R) * 4;
  auto k = ring_kernel<R, CR, STAGES, CL>;
  CK(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem)));
  cudaLaunchConfig_t cfg{}; cfg.gridDim = dim3(grid); cfg.blockDim = dim3(kConsumers + 32); cfg.dynamicSmemBytes = smem;
  cudaLaunchAttribute attr[1]; attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = CL; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr; cfg.numAttrs = 1;
  const float us = time_it([&] { CK(cudaLaunchKernelEx(&cfg, k, W, nl, steps, out)); });
  printf("ring  R=%d chunk=%2dKB stages=%d cluster=%d grid=%3d steps=%d: %7.2f us  (%.2f us/step, smem %zu KB)\n", R, CR, STAGES, CL,
         grid, steps, us, us / steps, smem >> 10);
}
template <int R, int MODE = 0> void run_ldg(const float *W, int nl, int steps, float *out, int grid) {
  const size_t smem = size_t(8) * H * R * 4;
  const float us = time_it([&] { ldg_kernel<R, MODE><<<grid, kConsumers, smem>>>(W, nl, steps, out); });
  printf("ldg   R=%d mode=%d grid=%3d steps=%d: %7.2f us  (%.2f us/step)\n", R, MODE, grid, steps, us, us / steps);
}

int main(int argc, char **argv) {
  const int nl = 9, steps = 14;
  const bool cluster_only = argc > 1 && argv[1][0] == 'c';   // `slab_stream c`: the mode-5 table + its baseline
  float *W, *out;
  CK(cudaMalloc(&W, size_t(nl) * H * H * 4));
  CK(cudaMalloc(&out, 4096 * 4));
  std::vector<float> h(size_t(nl) * H * H);
  for (size_t i = 0; i < h.size(); ++i) h[i] = float((i * 2654435761u) % 1000) * 1e-5f - 0.005f;
  CK(cudaMemcpy(W, h.data(), h.size() * 4, cudaMemcpyHostToDevice));
  if (cluster_only) {
    for (int rep = 0; rep < 2; ++rep) {
      run_ldg<2, 0>(W, nl, steps, out, 128);
      run_csplit<4, 8, 0>(W, nl, steps, out, 128);
      run_csplit<4, 16, 0>(W, nl, steps, out, 128);
      run_csplit<4, 32, 0>(W, nl, steps, out, 128);
      run_csplit<8, 8, 0>(W, nl, steps, out, 128);
      run_csplit<8, 16, 0>(W, nl, steps, out, 128);
      run_csplit<8, 32, 0>(W, nl, steps, out, 128);
      run_csplit<4, 8, 1>(W, nl, steps, out, 128);
      run_csplit<8, 16, 1>(W, nl, steps, out, 128);
      run_csplit<8, 16, 0>(W, nl, steps, out, 8);
      run_csplit<8, 16, 0>(W, nl, steps, out, 64);
      run_csplit<8, 16, 0>(W, nl, steps, out, 144);
    }
    printf("done\n");
    return 0;
  }
  for (int grid : {1, 16, 64, 128, 148}) {
    run_ldg<2, 0>(W, nl, steps, out, grid);
    run_ldg<2, 1>(W, nl, steps, out, grid);
    run_ldg<2, 2>(W, nl, steps, out, grid);
    run_ldg<2, 3>(W, nl, steps, out, grid);
    run_ldg<4, 0>(W, nl, steps, out, grid);
    run_ldg<4, 1>(W, nl, steps, out, grid);
    run_ring<2, 32, 4, 1>(W, nl, steps, out, grid);
    run_ring<4, 32, 4, 1>(W, nl, steps, out, grid);
  }
  for (int grid : {64, 128, 148}) {
    run_ring<2, 32, 4, 2>(W, nl, steps, out, grid);
    run_ring<2, 32, 6, 2>(W, nl, steps, out, grid);
    run_ring<4, 32, 4, 2>(W, nl, steps, out, grid);
    run_ring<2, 32, 4, 4>(W, nl, steps, out, grid == 148 ? 144 : grid);
  }
  for (int grid : {1, 128}) {
    run_ldg_pipe<2, 4>(W, nl, steps, out, grid);
    run_ldg_pipe<2, 8>(W, nl, steps, out, grid);
    run_ldg_pipe<2, 16>(W, nl, steps, out, grid);
    run_ldg_pipe<4, 8>(W, nl, steps, out, grid);
  }
  for (int grid : {2, 64, 128, 148}) {
    run_nsplit<4>(W, nl, steps, out, grid);
    run_nsplit<8>(W, nl, steps, out, grid);
  }
  printf("done\n");
  return 0;
}
