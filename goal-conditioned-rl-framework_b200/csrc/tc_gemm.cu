// Dense hidden layers on the 5th-generation tensor cores (tcgen05 / TMEM / TMA), large-batch regime.
//
//   FWD  : Y[M,N]  = leaky(X[M,K] W[N,K]^T + b)          (nn.Linear + LeakyReLU, src/model.py:17-30)
//   DGRAD: dX[M,N] = (dZ[M,K] Wt[N,K]^T) (.) leaky'(act)  (autograd of the same; Wt = transposed copy)
//
// fp32 accuracy on TF32 tensor cores ("3xTF32"): every operand is split in shared memory into
//   hi = rna_tf32(x),  lo = rna_tf32(x - hi)   (x - hi is exact in fp32)
// and the product is accumulated in fp32 TMEM as  hi*hi + hi*lo + lo*hi  (the lo*lo term is
// 2^-22 relative).  Both halves are already valid TF32 bit patterns, so the result does not depend on
// how the tensor core would round raw fp32 inputs.
//
// One persistent CTA per SM, 10 warps:
//   warp 0      TMA producer    (cp.async.bulk.tensor, 64-byte swizzle, 4-stage ring of 16-wide K tiles)
//   warp 1      MMA issuer      (one elected thread: 6 x tcgen05.mma.kind::tf32 per K tile)
//   warps 2-5   epilogue        (tcgen05.ld 32 lanes x 32 columns, bias / activation, 16-byte stores)
//   warps 6-13  hi / lo splitter (generic-proxy pass over the landed stage, fence.proxy.async)
// Pipelines: full (TMA -> splitter), ready (splitter -> MMA), empty (MMA commit -> TMA),
// tmem_full / tmem_empty (MMA <-> epilogue; two accumulator stages of N columns, so the epilogue of
// tile i overlaps the MMAs of tile i+1).
#include <cuda.h>

#include <map>
#include <tuple>

#include "mlp.cuh"

namespace gcrl {
namespace {

constexpr int BM = 128;            // rows per tile = TMEM lanes = UMMA M
constexpr int BKF = 16;            // fp32 elements per K tile = one 64-byte swizzle row
constexpr int ROWB = BKF * 4;      // bytes per operand row in a stage
constexpr int STAGES = 4;
constexpr int kSplitWarps = 8;
constexpr int kSplitThreads = kSplitWarps * 32;
constexpr int kTcThreads = (6 + kSplitWarps) * 32;
constexpr int kPairThreads = kTcThreads + 4 * 32;   // pair kernel: a second set of 4 epilogue warps (14-17)
constexpr int kStgLd = 36;         // epilogue staging row stride in floats (16-byte aligned, conflict-free)

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return uint32_t(__cvta_generic_to_shared(p)); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  do {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(bar), "r"(parity)
        : "memory");
  } while (!ok);
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap *tm, uint32_t bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(dst), "l"(reinterpret_cast<uint64_t>(tm)), "r"(bar), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void umma_tf32(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                          uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
        "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]),
        "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]),
        "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr)
      : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// K-major, 64-byte-swizzled operand tile: rows of 64 bytes, 8-row groups 512 bytes apart.
// Descriptor (cute::UMMA::SmemDescriptor): start >> 4 [0,14), LBO >> 4 [16,30) (unused for swizzled
// K-major), SBO >> 4 [32,46), version 1 [46,48), layout [61,64): SWIZZLE_64B = 4 (SWIZZLE_128B = 2).
__device__ __forceinline__ uint64_t umma_desc_sw(uint32_t saddr) {
  constexpr uint64_t layout = ROWB == 128 ? 2 : 4;
  return uint64_t((saddr >> 4) & 0x3FFF) | (uint64_t(1) << 16) | (uint64_t((8 * ROWB) >> 4) << 32) |
         (uint64_t(1) << 46) | (layout << 61);
}

// MN-major operand (weight gradient): boxes of [16 batch rows][32 features] = 2048 bytes.  For 32-bit
// MN-major operands the only layout the tensor core accepts is the 128-byte swizzle with 32-byte atoms
// (cute::UMMA::Layout_MN_SW128_32B_Atom = Swizzle<2,5,2>, layout type 1; TMA: SWIZZLE_128B_ATOM_32B): the
// swizzle atom is 4 batch rows x 128 bytes, so the K groups inside a box are 512 bytes apart (SBO) and
// consecutive 32-feature MN blocks are one box apart (LBO).
__device__ __forceinline__ uint64_t umma_desc_mn(uint32_t saddr) {
  return uint64_t((saddr >> 4) & 0x3FFF) | (uint64_t(2048 >> 4) << 16) | (uint64_t(512 >> 4) << 32) |
         (uint64_t(1) << 46) | (uint64_t(1) << 61);
}

// One lane of a converged warp.  The producer and MMA warps run their loops with ALL lanes (uniform control flow) and
// elect the issuing lane only around the asynchronous instructions: the operands (descriptors, coordinates, barrier
// addresses) are then provably warp-uniform and live in uniform registers.  Inside an `if (lane == 0)` region the
// compiler wraps every UTCHMMA / UTMALDG in a broadcast loop (ELECT, 5 x R2UR.BROADCAST, BRA.U.ANY: ~200 clk per MMA
// for 128 clk of tensor work) -- that loop, not shared memory or L2, bounded the first versions of these kernels.
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "elect.sync _|p, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(pred));
  return pred != 0;
}

__device__ __forceinline__ uint32_t rna_tf32(float x) {
  uint32_t r;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
  return r;
}

// Epilogue of one 32-row x 32-column accumulator chunk that a warp has staged in shared memory (row stride kStgLd):
// lane = 4 columns of one of 4 rows, 8 row groups, so that every global access is a full 128-byte row segment.
// All 8 shared loads (and, for the input gradient, all 8 loads of the saved activation) are issued before the first
// store: with the loads, the arithmetic and the store of one row group chained through the same four registers the
// eight groups ran back to back at ~300 clk each, and the epilogue (10 us per 128 x 256 tile), not the MMAs (8 us),
// set the pace of the whole kernel (profiles/README.md, timeline of the CTA-pair kernel).
//   mode 0: leaky(acc + bias)   1: acc * leaky'(act)   2: acc + bias   3: acc   4: out + acc (the same lane of the
//   same CTA stored `out` for an earlier slab of this weight-gradient tile)
__device__ __forceinline__ void epilogue_store32(uint32_t stg, int lane, int row0, int col0, int rows_valid,
                                                 int cols_valid, int mode, const float *__restrict__ bias,
                                                 const float *__restrict__ act, int ldact, float *__restrict__ out,
                                                 int ldo) {
  const int sub_r = lane >> 3, sub_c = (lane & 7) * 4;
  const int col = col0 + sub_c;
  if (col >= cols_valid) return;                       // widths are multiples of 4 (padded leading dimensions)
  float4 x[8];
#pragma unroll
  for (int r8 = 0; r8 < 8; ++r8)
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];"
                 : "=f"(x[r8].x), "=f"(x[r8].y), "=f"(x[r8].z), "=f"(x[r8].w)
                 : "r"(stg + uint32_t((r8 * 4 + sub_r) * kStgLd + sub_c) * 4));
  if (mode == 1) {
    float4 h[8];
#pragma unroll
    for (int r8 = 0; r8 < 8; ++r8) {
      const int row = row0 + r8 * 4 + sub_r;
      h[r8] = row < rows_valid ? *reinterpret_cast<const float4 *>(act + size_t(row) * ldact + col)
                               : make_float4(1.f, 1.f, 1.f, 1.f);
    }
#pragma unroll
    for (int r8 = 0; r8 < 8; ++r8) {
      x[r8].x = h[r8].x > 0.f ? x[r8].x : x[r8].x * kLeakySlope;
      x[r8].y = h[r8].y > 0.f ? x[r8].y : x[r8].y * kLeakySlope;
      x[r8].z = h[r8].z > 0.f ? x[r8].z : x[r8].z * kLeakySlope;
      x[r8].w = h[r8].w > 0.f ? x[r8].w : x[r8].w * kLeakySlope;
    }
  } else if (mode == 4) {
#pragma unroll
    for (int r8 = 0; r8 < 8; ++r8) {
      const int row = row0 + r8 * 4 + sub_r;
      if (row < rows_valid) {
        const float4 o = *reinterpret_cast<const float4 *>(out + size_t(row) * ldo + col);
        x[r8].x += o.x; x[r8].y += o.y; x[r8].z += o.z; x[r8].w += o.w;
      }
    }
  } else if (mode != 3) {
    const float4 bv = __ldg(reinterpret_cast<const float4 *>(bias + col));
#pragma unroll
    for (int r8 = 0; r8 < 8; ++r8) {
      x[r8].x += bv.x; x[r8].y += bv.y; x[r8].z += bv.z; x[r8].w += bv.w;
      if (mode == 0) {
        x[r8].x = x[r8].x > 0.f ? x[r8].x : x[r8].x * kLeakySlope;
        x[r8].y = x[r8].y > 0.f ? x[r8].y : x[r8].y * kLeakySlope;
        x[r8].z = x[r8].z > 0.f ? x[r8].z : x[r8].z * kLeakySlope;
        x[r8].w = x[r8].w > 0.f ? x[r8].w : x[r8].w * kLeakySlope;
      }
    }
  }
#pragma unroll
  for (int r8 = 0; r8 < 8; ++r8) {
    const int row = row0 + r8 * 4 + sub_r;
    if (row < rows_valid) *reinterpret_cast<float4 *>(out + size_t(row) * ldo + col) = x[r8];
  }
}

struct TcArgs {
  float *out; int ldo;
  const float *bias;             // mode 0
  const float *act; int ldact;   // mode 1
  int M, N, K;                   // N <= BN * n_tiles
  int mode;                      // 0: leaky(acc + bias); 1: acc * leaky'(act); 2: acc + bias
  int n_tiles, m_tiles;
  // kind 1 (weight gradient): out[slab][n][k] = sum_{m in slab} A[m][n] B[m][k]; both operands MN-major,
  // the batch is the reduction; n_tiles = ceil(N / 128), k_tiles = ceil(K / BN); M rows in nslabs slabs
  int kind, rows_per_slab, nslabs, k_tiles;
  long long split_stride;
  int acc_slabs;                 // kind 1: a CTA adds the later slabs of its (n, k) block onto the first one it wrote
  float *colsum;                 // kind 1: bias-gradient partials pB[slab][n] = column sums of the slab's dZ rows, taken
  long long colsum_stride;       // by the splitter warps from the tiles they split anyway (nullptr: no bias gradient)
  int members;                   // ensemble kernel (NMEM > 1): problems of this shape in the launch
  int full_items;                // pair kernel: tiles taken whole; the rest are split into two 256 x 128 halves
};

template <int BN>
struct TcSmem {
  static constexpr int kA = BM * ROWB, kB = BN * ROWB;
  static constexpr int kStage = 2 * kA + 2 * kB;            // A_hi | A_lo | B_hi | B_lo
  static constexpr int kColsum = 16 * BM * 4;               // kind 1: [16 row lanes][128 features] column-sum scratch
  static constexpr int kBytes = STAGES * kStage + 1024 /*alignment slack*/ + 256 /*barriers*/ + 4 * 32 * kStgLd * 4 + kColsum;
};

// Operands of the launch: tensor maps A (activations), B (weights, or their TF32 hi halves), B lo halves (PRESPLIT)
// per member.  NMEM = 1: one problem, epilogue pointers in TcArgs.  NMEM > 1 (ensemble, e.g. the critics of one
// layer): a.members independent problems of the same (M, N, K, mode), each with its own epilogue pointers.
template <int NMEM>
struct TcOperands {
  CUtensorMap map[NMEM][3];
  float *out[NMEM];
  const float *bias[NMEM];
  const float *act[NMEM];
};
constexpr int kTcMaxMembers = 8;

// PRESPLIT: the B operand (the layer's weights) arrives already split into TF32 hi / lo halves (two tensors, kept
// next to the parameters and refreshed after every optimiser step): the producer loads both, the splitter warps only
// handle the activation tile -- a third of the shared-memory passes they made over a stage, off the TMA -> MMA
// critical path for 2/3 of the bytes.
template <int BN, bool PRESPLIT, int NMEM>
__global__ void __launch_bounds__(kTcThreads, 1)
tc_dense_kernel(const __grid_constant__ TcOperands<NMEM> ops, TcArgs a) {
  extern __shared__ uint8_t smem_raw[];
  using S = TcSmem<BN>;
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t bars = base + STAGES * S::kStage;
  // barrier layout (8 bytes each): full[S], ready[S], empty[S], tmem_full[2], tmem_empty[2], then tmem ptr
  auto full = [&](int s) { return bars + 8u * s; };
  auto ready = [&](int s) { return bars + 8u * (STAGES + s); };
  auto empty = [&](int s) { return bars + 8u * (2 * STAGES + s); };
  auto tfull = [&](int s) { return bars + 8u * (3 * STAGES + s); };
  auto tempty = [&](int s) { return bars + 8u * (3 * STAGES + 2 + s); };
  const uint32_t tmem_slot = bars + 8u * (3 * STAGES + 4);
  const uint32_t stage_base = bars + 256;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  if (warp == 1 && lane == 0) {
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(full(s), 1);
      mbar_init(ready(s), kSplitThreads);
      mbar_init(empty(s), 1);
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init(tfull(s), 1);
      mbar_init(tempty(s), 4);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  } else if (warp == 2) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "r"(2 * BN)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  uint32_t tmem_base;
  asm volatile("ld.shared.u32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_slot));

  const bool wg = a.kind == 1;
  const int per_member = a.m_tiles * a.n_tiles;
  const int total_tiles = wg ? a.nslabs * a.n_tiles * a.k_tiles : (NMEM > 1 ? a.members : 1) * per_member;
  // tile decode.  dense: (member, m block, n block), K tiles of BKF columns.  wgrad: (slab, n block, k block),
  // "K tiles" = 16 batch rows each.
  struct Tile { int m0, n0, nk, slab, out_slab, acc, mem; };
  auto decode = [&](int t) {
    Tile ti;
    ti.mem = 0;
    if (!wg) {
      if (NMEM > 1) {
        ti.mem = t / per_member;
        t -= ti.mem * per_member;
      }
      ti.m0 = (t / a.n_tiles) * BM; ti.n0 = (t % a.n_tiles) * BN; ti.nk = (a.K + BKF - 1) / BKF; ti.slab = 0;
      ti.out_slab = 0; ti.acc = 0;
    } else {
      const int per = a.n_tiles * a.k_tiles;
      ti.slab = t / per;
      // the grid is a multiple of `per`: the tiles a CTA visits are the same (n, k) block of different slabs, and it
      // adds the later ones onto the first (fewer partial slabs for reduce_grads to read)
      ti.out_slab = a.acc_slabs ? int(t % gridDim.x) / per : ti.slab;
      ti.acc = (a.acc_slabs && t >= int(gridDim.x)) ? 1 : 0;
      const int rem = t - ti.slab * per;
      ti.m0 = (rem / a.k_tiles) * BM;            // first output row (n index) of the tile
      ti.n0 = (rem % a.k_tiles) * BN;            // first output column (k index)
      const int r0 = ti.slab * a.rows_per_slab;
      ti.nk = (min(a.rows_per_slab, a.M - r0) + 15) / 16;
    }
    return ti;
  };

  if (warp == 0) {
    // ===== TMA producer (whole warp in the loop, one elected lane issues) =====
    uint32_t it = 0;
    for (int t = blockIdx.x; t < total_tiles; t += gridDim.x) {
      const Tile ti = decode(t);
      for (int kb = 0; kb < ti.nk; ++kb, ++it) {
        const int s = it % STAGES;
        mbar_wait(empty(s), ((it / STAGES) & 1) ^ 1);
        const uint32_t st = base + s * S::kStage;
        if (elect_one()) {
          const CUtensorMap *tm = ops.map[ti.mem];
          mbar_expect_tx(full(s), S::kA + (PRESPLIT ? 2 : 1) * S::kB);
          if (!wg) {
            tma_load_2d(st, &tm[0], full(s), kb * BKF, ti.m0);
            tma_load_2d(st + 2 * S::kA, &tm[1], full(s), kb * BKF, ti.n0);
            if (PRESPLIT) tma_load_2d(st + 2 * S::kA + S::kB, &tm[2], full(s), kb * BKF, ti.n0);
          } else {
            // boxes of 16 batch rows x 32 features (128-byte swizzle, 32-byte atoms), one per 32-feature MN block
            const int r = ti.slab * a.rows_per_slab + kb * 16;
#pragma unroll 1
            for (int b = 0; b < BM / 32; ++b) tma_load_2d(st + b * 2048, &tm[0], full(s), ti.m0 + 32 * b, r);
#pragma unroll 1
            for (int b = 0; b < BN / 32; ++b) tma_load_2d(st + 2 * S::kA + b * 2048, &tm[1], full(s), ti.n0 + 32 * b, r);
          }
        }
        __syncwarp();
      }
    }
  } else if (warp == 1) {
    // ===== MMA issuer (whole warp in the loop, one elected lane issues) =====
    {
      // instruction descriptor (cute::UMMA::InstrDescriptor): D = F32 [4,6) = 1, A/B = TF32 [7,10),[10,13) = 2,
      // K-major both, N >> 3 at [17,23), M >> 4 at [24,29)
      // kind 1: A and B MN-major (bits 15, 16)
      const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | (uint32_t(BN >> 3) << 17) | (uint32_t(BM >> 4) << 24) |
                             (wg ? (3u << 15) : 0u);
      uint32_t it = 0, tile_it = 0;
      for (int t = blockIdx.x; t < total_tiles; t += gridDim.x, ++tile_it) {
        const int nk = decode(t).nk;
        const int as = tile_it & 1;
        mbar_wait(tempty(as), ((tile_it >> 1) & 1) ^ 1);
        tc_fence_after();
        const uint32_t d = tmem_base + uint32_t(as * BN);
        for (int kb = 0; kb < nk; ++kb, ++it) {
          const int s = it % STAGES;
          mbar_wait(ready(s), (it / STAGES) & 1);
          tc_fence_after();
          const uint32_t st = base + s * S::kStage;
          const uint64_t a_hi = wg ? umma_desc_mn(st) : umma_desc_sw(st);
          const uint64_t a_lo = wg ? umma_desc_mn(st + S::kA) : umma_desc_sw(st + S::kA);
          const uint64_t b_hi = wg ? umma_desc_mn(st + 2 * S::kA) : umma_desc_sw(st + 2 * S::kA);
          const uint64_t b_lo = wg ? umma_desc_mn(st + 2 * S::kA + S::kB) : umma_desc_sw(st + 2 * S::kA + S::kB);
          if (elect_one()) {
#pragma unroll
            for (int k = 0; k < BKF / 8; ++k) {
              // UMMA K = 8 for tf32.  K-major: 32 bytes along the swizzled row (+2 in the >>4 address);
              // MN-major: the next 8-row group of every box (+1024 bytes)
              const uint64_t ko = wg ? uint64_t(k * (1024 >> 4)) : uint64_t(k * 2);
              umma_tf32(d, a_lo + ko, b_hi + ko, idesc, (kb | k) != 0 ? 1u : 0u);
              umma_tf32(d, a_hi + ko, b_lo + ko, idesc, 1u);
              umma_tf32(d, a_hi + ko, b_hi + ko, idesc, 1u);
            }
            umma_commit(empty(s));                      // smem stage reusable once these MMAs retire
          }
          __syncwarp();
        }
        if (elect_one()) umma_commit(tfull(as));        // accumulator complete
        __syncwarp();
      }
    }
  } else if (warp < 6) {
    // ===== epilogue: TMEM lanes (warp % 4) * 32 .. + 31 =====
    const int q = warp & 3;
    uint32_t tile_it = 0;
    for (int t = blockIdx.x; t < total_tiles; t += gridDim.x, ++tile_it) {
      const Tile ti = decode(t);
      const int m0 = ti.m0, n0 = ti.n0;
      const int rows_valid = wg ? a.N : a.M, cols_valid = wg ? a.ldo : a.N;
      float *const out = NMEM > 1 ? ops.out[ti.mem] : a.out;
      const float *const bias = NMEM > 1 ? ops.bias[ti.mem] : a.bias;
      const float *const act = NMEM > 1 ? ops.act[ti.mem] : a.act;
      float *const obase = out + (wg ? size_t(ti.out_slab) * size_t(a.split_stride) : size_t(0));
      const int emode = (wg && ti.acc) ? 4 : a.mode;
      const int as = tile_it & 1;
      mbar_wait(tfull(as), (tile_it >> 1) & 1);
      tc_fence_after();
      const uint32_t taddr = tmem_base + (uint32_t(q * 32) << 16) + uint32_t(as * BN);
      // 32 accumulator columns at a time: TMEM -> registers (lane = row) -> padded smem tile ->
      // (lane = 4 columns of one of 4 rows) so that every global access is a full 128-byte row segment
      const uint32_t stg = stage_base + uint32_t(q) * (32 * kStgLd * 4);
#pragma unroll 1
      for (int c = 0; c < BN; c += 32) {
        uint32_t v[32];
        tmem_ld32(taddr + uint32_t(c), v);
        __syncwarp();
#pragma unroll
        for (int j = 0; j < 32; j += 4)
          asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(stg + uint32_t(lane * kStgLd + j) * 4), "r"(v[j]),
                       "r"(v[j + 1]), "r"(v[j + 2]), "r"(v[j + 3])
                       : "memory");
        __syncwarp();
        epilogue_store32(stg, lane, m0 + q * 32, n0 + c, rows_valid, cols_valid, emode, bias, act, a.ldact, obase, a.ldo);
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(tempty(as));
    }
  } else {
    // ===== hi / lo splitter =====
    const int tid = threadIdx.x - 6 * 32;
    uint32_t it = 0;
    // kind 1: the dZ operand passes through these threads' registers, so the bias gradient (column sums of dZ over
    // the slab's rows) is taken here instead of by a second pass over dZ (6 x 20 us per B = 65 536 update).  A thread's
    // two dZ chunks sit at the same place of every stage: box = 32 features, 16 batch rows of 128 bytes, the 32-byte
    // units of a row XOR-swizzled with (row & 3) (SWIZZLE_128B_ATOM_32B).  Only the tile of the first k block writes.
    const bool colsum_on = wg && a.colsum != nullptr;
    const uint32_t cs_scratch = stage_base + 4 * 32 * kStgLd * 4;
    float cs[2][4] = {{0.f, 0.f, 0.f, 0.f}, {0.f, 0.f, 0.f, 0.f}};
    for (int t = blockIdx.x; t < total_tiles; t += gridDim.x) {
      const Tile tile = decode(t);
      const int nk = tile.nk;
      const bool cs_tile = colsum_on && tile.n0 == 0;
      for (int kb = 0; kb < nk; ++kb, ++it) {
        const int s = it % STAGES;
        mbar_wait(full(s), (it / STAGES) & 1);
        const uint32_t st = base + s * S::kStage;
        // chunk c (16 bytes) of the stage: A chunks first (hi at st, lo at st + kA), then B chunks
        // (hi at st + 2 kA, lo at + kB).  All loads of a thread are issued before the first store.
        constexpr int kChunksA = S::kA / 16, kChunks = PRESPLIT ? kChunksA : (S::kA + S::kB) / 16;
        constexpr int kPer = (kChunks + kSplitThreads - 1) / kSplitThreads;
        float x[kPer][4];
        uint32_t hi_addr[kPer], lo_addr[kPer];
#pragma unroll
        for (int u = 0; u < kPer; ++u) {
          const int c = tid + u * kSplitThreads;
          const bool isA = c < kChunksA;
          hi_addr[u] = isA ? st + 16u * c : st + 2 * S::kA + 16u * (c - kChunksA);
          lo_addr[u] = hi_addr[u] + (isA ? S::kA : S::kB);
          if (c < kChunks)
            asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];"
                         : "=f"(x[u][0]), "=f"(x[u][1]), "=f"(x[u][2]), "=f"(x[u][3])
                         : "r"(hi_addr[u]));
        }
        if (cs_tile) {
#pragma unroll
          for (int u = 0; u < 2; ++u)
#pragma unroll
            for (int e = 0; e < 4; ++e) cs[u][e] += x[u][e];
        }
#pragma unroll
        for (int u = 0; u < kPer; ++u) {
          const int c = tid + u * kSplitThreads;
          if (c < kChunks) {
            uint32_t h[4], l[4];
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              h[e] = rna_tf32(x[u][e]);
              l[e] = rna_tf32(x[u][e] - __uint_as_float(h[e]));
            }
            asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(hi_addr[u]), "r"(h[0]), "r"(h[1]), "r"(h[2]),
                         "r"(h[3])
                         : "memory");
            asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(lo_addr[u]), "r"(l[0]), "r"(l[1]), "r"(l[2]),
                         "r"(l[3])
                         : "memory");
          }
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic writes -> visible to the MMA (async proxy)
        mbar_arrive(ready(s));
      }
      if (cs_tile) {                                   // uniform over the splitter warps
#pragma unroll
        for (int u = 0; u < 2; ++u) {
          const int c = tid + u * kSplitThreads, cc = c & 127, row = cc >> 3;
          const int f = (c >> 7) * 32 + ((((cc >> 1) & 3) ^ (row & 3)) << 3) + (cc & 1) * 4;
          asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(cs_scratch + uint32_t(row * BM + f) * 4),
                       "f"(cs[u][0]), "f"(cs[u][1]), "f"(cs[u][2]), "f"(cs[u][3])
                       : "memory");
          cs[u][0] = cs[u][1] = cs[u][2] = cs[u][3] = 0.f;
        }
        asm volatile("bar.sync 1, %0;" ::"n"(kSplitThreads) : "memory");
        if (tid < BM && tile.m0 + tid < a.N) {
          float sum = 0.f;
#pragma unroll
          for (int r = 0; r < 16; ++r) {
            float v;
            asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(cs_scratch + uint32_t(r * BM + tid) * 4));
            sum += v;
          }
          float *const dst = a.colsum + (long long)tile.out_slab * a.colsum_stride + tile.m0 + tid;
          *dst = tile.acc ? *dst + sum : sum;            // same thread wrote it for the earlier slab
        }
        asm volatile("bar.sync 1, %0;" ::"n"(kSplitThreads) : "memory");
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(2 * BN) : "memory");
  }
}

// ---- CTA-pair variant (cta_group::2): dense forward / input gradient with pre-split weights, N % 256 == 0 -------
// Two CTAs on the two SMs of a TPC compute one 256-row x 256-column tile: each CTA stages ITS 128 activation rows
// (TMA -> in-smem hi / lo split, as above) and only ITS HALF (128 of the 256 rows) of the pre-split weight tile; the
// tensor cores of the pair read both halves.  Per 16-wide K tile and SM that is 24 KB of TMA writes instead of 40 and
// 48 KB of operand reads instead of 72 through the shared-memory port (128 B/clk; DESIGN.md 4).  The leader (cluster
// rank 0) issues every MMA; accumulators: rows 0-127 in the leader's TMEM, 128-255 in the peer's, two stages of 256
// columns each.  18 warps: 0 TMA producer, 1 MMA issuer (leader) / relay (peer), 2-5 and 14-17 epilogue (two warps
// per TMEM lane quarter, half of the columns each), 6-13 hi / lo splitter.
//   full[s]        TMA -> splitter                (per CTA)
//   split_done[s]  splitter -> MMA / relay        (per CTA, one arrival per splitter warp)
//   peer_ready[s]  the peer's relay thread (its otherwise idle MMA warp) -> leader: "my stage s is split"
//   empty[s]       MMA commit, multicast to both CTAs -> TMA
//   tfull[a]       MMA commit, multicast -> epilogue of both CTAs;  tempty[a]  both epilogues -> leader MMA
template <int STAGES2>
struct TcSmem2 {
  static constexpr int kA = BM * ROWB;                       // 128 activation rows
  static constexpr int kBh = 128 * ROWB;                     // this CTA's half of the 256 weight rows
  static constexpr int kStage = 2 * kA + 2 * kBh;            // A_hi | A_lo | B_hi | B_lo
  static constexpr int kBytes = STAGES2 * kStage + 1024 + 512 + 8 * 32 * kStgLd * 4;       // 8 epilogue warps
};

__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ uint32_t map_to_cta(uint32_t saddr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(saddr), "r"(rank));
  return r;
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
  // default semantics (release at CTA scope), as CUTLASS's ClusterBarrier::arrive: the .release.cluster form compiles
  // to MEMBAR + ERRBAR in front of the arrive, ~800 clk per call -- with one call per stage in the relay thread that
  // alone bounded the pair kernel at 27 us (profiles/README.md)
  asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
__device__ __forceinline__ void umma_tf32_pair(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                               uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma_commit_pair(uint32_t bar) {      // arrives on `bar` in BOTH CTAs of the pair
  const uint16_t mask = 3;
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
               ::"r"(bar), "h"(mask)
               : "memory");
}

template <int STAGES2>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kPairThreads, 1)
tc_dense_pair_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmBhi,
                     const __grid_constant__ CUtensorMap tmBlo, TcArgs a) {
  extern __shared__ uint8_t smem_raw[];
  using S = TcSmem2<STAGES2>;
  constexpr int BN = 256;
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t bars = base + STAGES2 * S::kStage;
  auto full = [&](int s) { return bars + 8u * s; };
  auto split_done = [&](int s) { return bars + 8u * (STAGES2 + s); };
  auto peer_ready = [&](int s) { return bars + 8u * (2 * STAGES2 + s); };
  auto empty = [&](int s) { return bars + 8u * (3 * STAGES2 + s); };
  auto tfull = [&](int s) { return bars + 8u * (4 * STAGES2 + s); };
  auto tempty = [&](int s) { return bars + 8u * (4 * STAGES2 + 2 + s); };
  const uint32_t tmem_slot = bars + 8u * (4 * STAGES2 + 4);
  const uint32_t stage_base = bars + 512;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const bool leader = rank == 0;

  if (warp == 1 && lane == 0) {
    for (int s = 0; s < STAGES2; ++s) {
      mbar_init(full(s), 1);
      mbar_init(split_done(s), kSplitWarps);
      mbar_init(peer_ready(s), 1);
      mbar_init(empty(s), 1);
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init(tfull(s), 1);
      mbar_init(tempty(s), 16);                        // 8 epilogue warps in each CTA of the pair
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  } else if (warp == 2) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "r"(2 * BN)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  cluster_sync_all();                                  // barriers of both CTAs initialised before any remote arrive
  tc_fence_after();
  uint32_t tmem_base;
  asm volatile("ld.shared.u32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_slot));

  const int pair = blockIdx.x >> 1, npairs = gridDim.x >> 1;
  const int nk = (a.K + BKF - 1) / BKF;
  // Work items: 256 x 256 tiles (m_tiles counts 256-row tiles); when the last round would leave at least half of the
  // pairs idle, its tiles are cut into two 256 x 128 halves taken by different pairs (MMA N = 128, 64 weight rows per
  // CTA), so the round costs about half a tile time: 256 tiles on 74 pairs take 3.5 rounds instead of 4.
  const int total_items = a.full_items + 2 * (a.m_tiles * a.n_tiles - a.full_items);
  struct Item { int m0, n0, ncols; };
  auto decode = [&](int w) {
    int t = w, half = 0, nc = BN;
    if (w >= a.full_items) {
      const int h = w - a.full_items;
      t = a.full_items + (h >> 1); half = h & 1; nc = BN / 2;
    }
    Item it;
    it.m0 = (t / a.n_tiles) * 256 + int(rank) * BM;
    it.n0 = (t % a.n_tiles) * BN + half * (BN / 2);
    it.ncols = nc;
    return it;
  };

  if (warp == 0) {
    // ===== TMA producer (both CTAs: own activation rows, own half of the weight rows) =====
    uint32_t it = 0;
    for (int w = pair; w < total_items; w += npairs) {
      const Item wi = decode(w);
      const int rows_b = wi.ncols / 2;                       // this CTA's share of the weight rows: 128 or 64
      const int nb = wi.n0 + int(rank) * rows_b;
      for (int kb = 0; kb < nk; ++kb, ++it) {
        const int s = it % STAGES2;
        mbar_wait(empty(s), ((it / STAGES2) & 1) ^ 1);
        const uint32_t st = base + s * S::kStage;
        if (elect_one()) {
          mbar_expect_tx(full(s), S::kA + 2 * rows_b * ROWB);
          tma_load_2d(st, &tmA, full(s), kb * BKF, wi.m0);
          for (int r = 0; r < rows_b; r += 64) {             // weight maps: boxes of 64 rows
            tma_load_2d(st + 2 * S::kA + r * ROWB, &tmBhi, full(s), kb * BKF, nb + r);
            tma_load_2d(st + 2 * S::kA + S::kBh + r * ROWB, &tmBlo, full(s), kb * BKF, nb + r);
          }
        }
        __syncwarp();
      }
    }
  } else if (warp == 1) {
    if (leader) {
      // ===== MMA issuer (leader only): M = 256 over the pair, N = 256 =====
      const uint32_t idesc_m = (1u << 4) | (2u << 7) | (2u << 10) | (uint32_t(256 >> 4) << 24);
      uint32_t it = 0, tile_it = 0;
      for (int w = pair; w < total_items; w += npairs, ++tile_it) {
        const uint32_t idesc = idesc_m | (uint32_t(decode(w).ncols >> 3) << 17);
        const int as = tile_it & 1;
        mbar_wait(tempty(as), ((tile_it >> 1) & 1) ^ 1);
        tc_fence_after();
        const uint32_t d = tmem_base + uint32_t(as * BN);
        for (int kb = 0; kb < nk; ++kb, ++it) {
          const int s = it % STAGES2;
          mbar_wait(split_done(s), (it / STAGES2) & 1);
          mbar_wait(peer_ready(s), (it / STAGES2) & 1);
          tc_fence_after();
          const uint32_t st = base + s * S::kStage;
          const uint64_t a_hi = umma_desc_sw(st), a_lo = umma_desc_sw(st + S::kA);
          const uint64_t b_hi = umma_desc_sw(st + 2 * S::kA), b_lo = umma_desc_sw(st + 2 * S::kA + S::kBh);
          if (elect_one()) {
#pragma unroll
            for (int k = 0; k < BKF / 8; ++k) {
              const uint64_t ko = uint64_t(k * 2);
              umma_tf32_pair(d, a_lo + ko, b_hi + ko, idesc, (kb | k) != 0 ? 1u : 0u);
              umma_tf32_pair(d, a_hi + ko, b_lo + ko, idesc, 1u);
              umma_tf32_pair(d, a_hi + ko, b_hi + ko, idesc, 1u);
            }
            umma_commit_pair(empty(s));
          }
          __syncwarp();
        }
        if (elect_one()) umma_commit_pair(tfull(as));
        __syncwarp();
      }
    } else {
      // ===== relay (peer only): "my stage is split" -> the leader's peer_ready =====
      uint32_t it = 0;
      for (int w = pair; w < total_items; w += npairs)
        for (int kb = 0; kb < nk; ++kb, ++it) {
          const int s = it % STAGES2;
          mbar_wait(split_done(s), (it / STAGES2) & 1);
          if (elect_one()) mbar_arrive_cluster(map_to_cta(peer_ready(s), 0));
          __syncwarp();
        }
    }
  } else if (warp < 6 || warp >= 14) {
    // ===== epilogue (both CTAs): own 128 rows; warps 2-5 take the first half of the columns, warps 14-17 the second
    // (a warp can only read the TMEM lane quarter warp % 4).  With 4 warps the epilogue of a tile (10 us with the
    // mainloop running beside it) was slower than its MMAs (8 us) and set the pace =====
    const int q = warp & 3, part = warp >= 14 ? 1 : 0;
    uint32_t tile_it = 0;
    for (int w = pair; w < total_items; w += npairs, ++tile_it) {
      const Item wi = decode(w);
      const int m0 = wi.m0, n0 = wi.n0;
      const int as = tile_it & 1;
      if (lane == 0) mbar_wait(tfull(as), (tile_it >> 1) & 1);
      __syncwarp();
      tc_fence_after();
      const uint32_t taddr = tmem_base + (uint32_t(q * 32) << 16) + uint32_t(as * BN);
      const uint32_t stg = stage_base + uint32_t(q + 4 * part) * (32 * kStgLd * 4);
      const int c_lo = part * (wi.ncols / 2), c_hi = c_lo + wi.ncols / 2;
#pragma unroll 1
      for (int c = c_lo; c < c_hi; c += 32) {
        uint32_t v[32];
        tmem_ld32(taddr + uint32_t(c), v);
        __syncwarp();
#pragma unroll
        for (int j = 0; j < 32; j += 4)
          asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(stg + uint32_t(lane * kStgLd + j) * 4), "r"(v[j]),
                       "r"(v[j + 1]), "r"(v[j + 2]), "r"(v[j + 3])
                       : "memory");
        __syncwarp();
        epilogue_store32(stg, lane, m0 + q * 32, n0 + c, a.M, a.N, a.mode, a.bias, a.act, a.ldact, a.out, a.ldo);
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive_cluster(map_to_cta(tempty(as), 0));
    }
  } else {
    // ===== hi / lo splitter (both CTAs): the activation tile only =====
    const int tid = threadIdx.x - 6 * 32;
    uint32_t it = 0;
    for (int w = pair; w < total_items; w += npairs) {
      for (int kb = 0; kb < nk; ++kb, ++it) {
        const int s = it % STAGES2;
        if (lane == 0) mbar_wait(full(s), (it / STAGES2) & 1);
        __syncwarp();
        const uint32_t st = base + s * S::kStage;
        constexpr int kChunks = S::kA / 16, kPer = kChunks / kSplitThreads;
        static_assert(kChunks % kSplitThreads == 0, "splitter threads must tile the activation stage");
        float x[kPer][4];
#pragma unroll
        for (int u = 0; u < kPer; ++u)
          asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];"
                       : "=f"(x[u][0]), "=f"(x[u][1]), "=f"(x[u][2]), "=f"(x[u][3])
                       : "r"(st + 16u * (tid + u * kSplitThreads)));
#pragma unroll
        for (int u = 0; u < kPer; ++u) {
          const uint32_t hi_addr = st + 16u * (tid + u * kSplitThreads);
          uint32_t h[4], l[4];
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            h[e] = rna_tf32(x[u][e]);
            l[e] = rna_tf32(x[u][e] - __uint_as_float(h[e]));
          }
          asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(hi_addr), "r"(h[0]), "r"(h[1]), "r"(h[2]), "r"(h[3])
                       : "memory");
          asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(hi_addr + S::kA), "r"(l[0]), "r"(l[1]), "r"(l[2]),
                       "r"(l[3])
                       : "memory");
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        __syncwarp();
        if (lane == 0) mbar_arrive(split_done(s));
      }
    }
  }

  tc_fence_before();
  cluster_sync_all();                                  // no CTA of the pair leaves while the other may still use it
  if (warp == 2) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(2 * BN) : "memory");
  }
}

// ---- host side ------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *,
                                  const cuuint64_t *, const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void *p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    GCRL_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres));
    if (p == nullptr || qres != cudaDriverEntryPointSuccess)
      throw Error(GCRL_ERR_CUDA, "cuTensorMapEncodeTiled is not available from the driver");
    fn = reinterpret_cast<EncodeTiledFn>(p);
  }
  return fn;
}

// fp32 row-major [rows, cols] with leading dimension ld -> box of (box_rows x box_cols floats), swizzle span =
// the box row (64 or 128 bytes); out-of-bounds elements read as zero (ragged M / N / K tails).
CUtensorMap make_map(const float *ptr, int64_t rows, int cols, int ld, int box_rows, int box_cols = BKF,
                     bool atom32 = false) {
  CUtensorMap m;
  const cuuint64_t dims[2] = {cuuint64_t(cols), cuuint64_t(rows)};
  const cuuint64_t strides[1] = {cuuint64_t(ld) * 4};
  const cuuint32_t box[2] = {cuuint32_t(box_cols), cuuint32_t(box_rows)};
  const cuuint32_t estr[2] = {1, 1};
  const CUresult r = encode_fn()(&m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float *>(ptr), dims, strides, box,
                                 estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                                 atom32 ? CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B
                                        : (box_cols * 4 == 128 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B),
                                 CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) throw Error(GCRL_ERR_CUDA, "cuTensorMapEncodeTiled failed (" + std::to_string(int(r)) + ")");
  return m;
}

template <int BN>
void set_attr() {
  static bool attr_set = false;
  if (!attr_set) {
    GCRL_CUDA(cudaFuncSetAttribute(tc_dense_kernel<BN, false, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                   TcSmem<BN>::kBytes));
    GCRL_CUDA(cudaFuncSetAttribute(tc_dense_kernel<BN, true, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                   TcSmem<BN>::kBytes));
    GCRL_CUDA(cudaFuncSetAttribute(tc_dense_kernel<BN, true, kTcMaxMembers>,
                                   cudaFuncAttributeMaxDynamicSharedMemorySize, TcSmem<BN>::kBytes));
    attr_set = true;
  }
}

template <int BN>
void launch_bn(const CUtensorMap &tmA, const CUtensorMap &tmB, const CUtensorMap *tmB2, const TcArgs &a,
               cudaStream_t st, int grid_wg = 0) {
  set_attr<BN>();
  const int tiles = a.kind == 1 ? a.nslabs * a.n_tiles * a.k_tiles : a.m_tiles * a.n_tiles;
  const int grid = grid_wg > 0 ? grid_wg : std::min(tiles, sm_count());
  TcOperands<1> ops{};
  ops.map[0][0] = tmA;
  ops.map[0][1] = tmB;
  ops.map[0][2] = tmB2 != nullptr ? *tmB2 : tmB;
  if (tmB2 != nullptr)
    tc_dense_kernel<BN, true, 1><<<grid, kTcThreads, TcSmem<BN>::kBytes, st>>>(ops, a);
  else
    tc_dense_kernel<BN, false, 1><<<grid, kTcThreads, TcSmem<BN>::kBytes, st>>>(ops, a);
  GCRL_LAUNCHED();
}

template <int BN>
void launch_bn_ensemble(const TcOperands<kTcMaxMembers> &ops, const TcArgs &a, cudaStream_t st) {
  set_attr<BN>();
  const int grid = std::min(a.members * a.m_tiles * a.n_tiles, sm_count());
  tc_dense_kernel<BN, true, kTcMaxMembers><<<grid, kTcThreads, TcSmem<BN>::kBytes, st>>>(ops, a);
  GCRL_LAUNCHED();
}

// CTA pairs that can be co-resident (one per TPC); 0 = the device cannot host the pair kernel.  Queried once,
// outside stream capture (tc_dense_init).
int pair_capacity() {
  static int pairs = -1;
  if (pairs < 0) {
    pairs = 0;
    GCRL_CUDA(cudaFuncSetAttribute(tc_dense_pair_kernel<5>, cudaFuncAttributeMaxDynamicSharedMemorySize, TcSmem2<5>::kBytes));
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3(unsigned(sm_count() & ~1));
    cfg.blockDim = dim3(kPairThreads);
    cfg.dynamicSmemBytes = TcSmem2<5>::kBytes;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = 2; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    cfg.attrs = at; cfg.numAttrs = 1;
    int n = 0;
    if (cudaOccupancyMaxActiveClusters(&n, tc_dense_pair_kernel<5>, &cfg) == cudaSuccess && n > 0)
      pairs = std::min(n, sm_count() / 2);
    else
      cudaGetLastError();
  }
  return pairs;
}

}  // namespace

// one-time host setup (driver entry point, shared-memory opt-in): call outside stream capture
void tc_dense_init() {
  encode_fn();
  set_attr<64>();
  set_attr<128>();
  set_attr<256>();
  pair_capacity();
}

bool tc_dense_supported(int M, int N, int K) {
  return M >= 1 && N >= 16 && (N % 16) == 0 && K >= 4 && (K % 4) == 0 && (N <= 256 || N % 256 == 0);
}

// Column tile of a dense launch of `members` problems: as wide as the layer when the row tiles of all members alone
// fill the SMs (the activation tile is then loaded and split once), narrower when the batch is small so that more
// CTAs share the work.
static int dense_column_tile(int M, int N, int members) {
  int BN = N <= 64 ? 64 : (N <= 128 ? 128 : 256);
  const int m_tiles_ = (M + BM - 1) / BM;
  while (BN > 64 && members * m_tiles_ * ((N + BN - 1) / BN) < (sm_count() * 3) / 4) BN >>= 1;
  return BN;
}

// out[M, N] = epilogue( X[M, K] * W[N, K]^T )
//   mode 0: leaky(. + bias)   mode 1: . * leaky'(act)   mode 2: . + bias   mode 3: . (bare product)
void launch_tc_dense(const float *X, int ldx, const float *W, int ldw, const float *bias, const float *act,
                     int ldact, float *out, int ldo, int M, int N, int K, int mode, cudaStream_t st,
                     const float *W_lo) {
  GCRL_REQUIRE(tc_dense_supported(M, N, K), "shape not supported by the tensor-core dense kernel");
  GCRL_REQUIRE((ldx % 4) == 0 && (ldw % 4) == 0 && (ldo % 4) == 0, "leading dimensions must be multiples of 4");
  const int BN = dense_column_tile(M, N, 1);
  TcArgs a{};
  a.out = out; a.ldo = ldo; a.bias = bias; a.act = act; a.ldact = ldact;
  a.M = M; a.N = N; a.K = K; a.mode = mode;
  a.m_tiles = (M + BM - 1) / BM;
  a.n_tiles = (N + BN - 1) / BN;
  // CTA pairs (256 x 256 tiles, each SM stages half of the weight tile) once they alone fill 3/4 of the TPCs
  const int pairs = (W_lo != nullptr && N % 256 == 0) ? pair_capacity() : 0;
  const int pair_tiles = ((M + 255) / 256) * (N / 256);
  // (M = 8192 as 64 half tiles on 64 pairs was tried: 20.5 us against 18.5 us for 128 single-CTA 128 x 128 tiles)
  if (pairs > 0 && 4 * pair_tiles >= 3 * pairs) {
    a.m_tiles = (M + 255) / 256;
    a.n_tiles = N / 256;
    const CUtensorMap tmA = make_map(X, M, K, ldx, BM);
    const CUtensorMap tmBhi = make_map(W, N, K, ldw, 64);
    const CUtensorMap tmBlo = make_map(W_lo, N, K, ldw, 64);
    const int used = std::min(pair_tiles, pairs);
    const int grid = 2 * used;
    const int rest = pair_tiles % used;                      // tiles of the last, partly filled round
    a.full_items = (rest > 0 && 2 * rest <= used) ? pair_tiles - rest : pair_tiles;
    tc_dense_pair_kernel<5><<<grid, kPairThreads, TcSmem2<5>::kBytes, st>>>(tmA, tmBhi, tmBlo, a);
    GCRL_LAUNCHED();
    return;
  }
  const CUtensorMap tmA = make_map(X, M, K, ldx, BM);
  const CUtensorMap tmB = make_map(W, N, K, ldw, BN);          // W_lo given: W holds the TF32 hi halves
  CUtensorMap tmB2;
  if (W_lo != nullptr) tmB2 = make_map(W_lo, N, K, ldw, BN);
  const CUtensorMap *p2 = W_lo != nullptr ? &tmB2 : nullptr;
  if (BN == 64) launch_bn<64>(tmA, tmB, p2, a, st);
  else if (BN == 128) launch_bn<128>(tmA, tmB, p2, a, st);
  else launch_bn<256>(tmA, tmB, p2, a, st);
}

// n independent problems of one shape in one launch (pre-split weights); every member's output is what
// launch_tc_dense computes for it alone.  One member goes through launch_tc_dense itself (CTA pairs included).
void launch_tc_dense_ensemble(const TcDenseProblem *pr, int n, int ldact, int ldo, int M, int N, int K, int mode,
                              cudaStream_t st) {
  GCRL_REQUIRE(n >= 1 && n <= kTcMaxMembers, "ensemble of 1..8 problems");
  if (n == 1) {
    launch_tc_dense(pr[0].X, pr[0].ldx, pr[0].W_hi, pr[0].ldw, pr[0].bias, pr[0].act, ldact, pr[0].out, ldo, M, N, K,
                    mode, st, pr[0].W_lo);
    return;
  }
  GCRL_REQUIRE(tc_dense_supported(M, N, K), "shape not supported by the tensor-core dense kernel");
  GCRL_REQUIRE((ldo % 4) == 0, "leading dimensions must be multiples of 4");
  const int BN = dense_column_tile(M, N, n);
  TcArgs a{};
  a.ldo = ldo; a.ldact = ldact;
  a.M = M; a.N = N; a.K = K; a.mode = mode;
  a.m_tiles = (M + BM - 1) / BM;
  a.n_tiles = (N + BN - 1) / BN;
  a.members = n;
  TcOperands<kTcMaxMembers> ops{};
  for (int i = 0; i < n; ++i) {
    GCRL_REQUIRE(pr[i].W_lo != nullptr && (pr[i].ldx % 4) == 0 && (pr[i].ldw % 4) == 0,
                 "ensemble members need pre-split weights and leading dimensions that are multiples of 4");
    ops.map[i][0] = make_map(pr[i].X, M, K, pr[i].ldx, BM);
    ops.map[i][1] = make_map(pr[i].W_hi, N, K, pr[i].ldw, BN);
    ops.map[i][2] = make_map(pr[i].W_lo, N, K, pr[i].ldw, BN);
    ops.out[i] = pr[i].out; ops.bias[i] = pr[i].bias; ops.act[i] = pr[i].act;
  }
  if (BN == 64) launch_bn_ensemble<64>(ops, a, st);
  else if (BN == 128) launch_bn_ensemble<128>(ops, a, st);
  else launch_bn_ensemble<256>(ops, a, st);
}

// hi = rna_tf32(x), lo = rna_tf32(x - hi): the halves the 3xTF32 product is built from
__global__ void __launch_bounds__(256) split_tf32_kernel(const float *__restrict__ src, float *__restrict__ hi,
                                                         float *__restrict__ lo, int n) {
  for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < n; e += gridDim.x * blockDim.x) {
    const float x = src[e];
    const uint32_t h = rna_tf32(x);
    hi[e] = __uint_as_float(h);
    lo[e] = __uint_as_float(rna_tf32(x - __uint_as_float(h)));
  }
}

void launch_split_tf32(const float *src, float *hi, float *lo, int n, cudaStream_t st) {
  const int grid = std::max(1, std::min((n + 255) / 256, sm_count() * 4));
  split_tf32_kernel<<<grid, 256, 0, st>>>(src, hi, lo, n);
  GCRL_LAUNCHED();
}

bool tc_wgrad_supported(int M, int N, int K) {
  return M >= 16 && N >= 4 && (N % 4) == 0 && K >= 4 && (K % 4) == 0;
}

// Split-batch partial weight gradients on the tensor cores (same contract as launch_linear_wgrad):
//   pW[s][N][ldw] = sum_{m in slab s} dZ[m,n] X[m,k],   pB[s][N] = sum_{m in slab s} dZ[m,n]
int launch_tc_wgrad(const float *dZ, int lddz, const float *X, int ldx, float *pW, int ldw, int64_t w_split_stride,
                    float *pB, int64_t b_split_stride, int M, int N, int K, int max_splits, cudaStream_t st) {
  GCRL_REQUIRE(tc_wgrad_supported(M, N, K), "shape not supported by the tensor-core weight-gradient kernel");
  GCRL_REQUIRE((lddz % 4) == 0 && (ldx % 4) == 0 && (ldw % 4) == 0, "leading dimensions must be multiples of 4");
  const int BN = K <= 64 ? 64 : (K <= 128 ? 128 : 256);
  TcArgs a{};
  a.kind = 1; a.mode = 3;
  a.out = pW; a.ldo = ldw;
  a.M = M; a.N = N; a.K = K;
  a.n_tiles = (N + BM - 1) / BM;
  a.k_tiles = (std::max(K, ldw) + BN - 1) / BN;      // every column of the padded slab rows is written
  a.m_tiles = 0;
  const int per = a.n_tiles * a.k_tiles;
  // slabs: fill the SMs, and keep the rows accumulated per TMEM tile <= 512 (the tensor core's fp32
  // accumulation error grows linearly with the number of MMAs chained into one accumulator; the slab
  // partials are summed in plain fp32 afterwards)
  int slabs = std::max(1, std::min(max_splits, std::max(sm_count() / per, (M + 511) / 512)));
  int rows = ((M + slabs - 1) / slabs + 15) & ~15;
  slabs = (M + rows - 1) / rows;
  a.rows_per_slab = rows; a.nslabs = slabs; a.split_stride = w_split_stride;
  // the bias-gradient partials ride on the splitter warps
  a.colsum = pB; a.colsum_stride = b_split_stride;
  const CUtensorMap tmA = make_map(dZ, M, N, lddz, 16, 32, true);
  const CUtensorMap tmB = make_map(X, M, K, ldx, 16, 32, true);
  // more tiles than SMs: a grid that is a multiple of the tiles per slab makes every CTA revisit the SAME (n, k) block
  // in later slabs, and it accumulates them in place (bias sums included) -- grid / per partial slabs for
  // reduce_grads instead of `slabs` (74 instead of 128 at M = 65 536: 102 -> 59 MB per network)
  const int tiles = slabs * per;
  int grid = std::min(tiles, sm_count()), written = slabs;
  if (tiles > grid && per <= sm_count()) {
    grid = (sm_count() / per) * per;
    a.acc_slabs = 1;
    written = grid / per;
  }
  if (BN == 64) launch_bn<64>(tmA, tmB, nullptr, a, st, grid);
  else if (BN == 128) launch_bn<128>(tmA, tmB, nullptr, a, st, grid);
  else launch_bn<256>(tmA, tmB, nullptr, a, st, grid);
  return written;
}

}  // namespace gcrl

extern "C" int gcrl_dense_layer(int device, int engine, int mode, int64_t M, int N, int K, const float *x_dev,
                                int ldx, const float *w_dev, int ldw, const float *bias_dev, const float *act_dev,
                                int ldact, float *y_dev, int ldy, void *stream) {
  GCRL_API_BEGIN
  using namespace gcrl;
  GCRL_REQUIRE(x_dev && w_dev && y_dev && M >= 1 && M < (int64_t(1) << 31), "bad argument");
  GCRL_REQUIRE(mode >= 0 && mode <= 2 && (mode == 1 ? act_dev != nullptr : bias_dev != nullptr), "bad mode / operands");
  GCRL_CUDA(cudaSetDevice(device));
  cudaStream_t st = as_stream(stream);
  if (engine == 1) {
    launch_tc_dense(x_dev, ldx, w_dev, ldw, bias_dev, act_dev, ldact, y_dev, ldy, int(M), N, K, mode, st);
  } else {
    GCRL_REQUIRE(engine == 0 && mode != 1, "engine 0 (fp32 FFMA) implements modes 0 and 2");
    GCRL_REQUIRE((ldx % 4) == 0 && (ldw % 4) == 0 && (ldy % 4) == 0, "leading dimensions must be multiples of 4");
    launch_linear_fwd(x_dev, ldx, w_dev, ldw, bias_dev, y_dev, ldy, int(M), N, K, mode == 0 ? ACT_LEAKY : ACT_NONE, st);
  }
  GCRL_API_END
}

extern "C" int gcrl_split_tf32(int device, const float *src_dev, float *hi_dev, float *lo_dev, int64_t n, void *stream) {
  GCRL_API_BEGIN
  using namespace gcrl;
  GCRL_REQUIRE(src_dev && hi_dev && lo_dev && n >= 0 && n < (int64_t(1) << 31), "bad argument");
  GCRL_CUDA(cudaSetDevice(device));
  if (n > 0) launch_split_tf32(src_dev, hi_dev, lo_dev, int(n), as_stream(stream));
  GCRL_API_END
}

extern "C" int gcrl_dense_layer_presplit(int device, int mode, int64_t M, int N, int K, const float *x_dev, int ldx,
                                         const float *w_hi_dev, const float *w_lo_dev, int ldw, const float *bias_dev,
                                         const float *act_dev, int ldact, float *y_dev, int ldy, void *stream) {
  GCRL_API_BEGIN
  using namespace gcrl;
  GCRL_REQUIRE(x_dev && w_hi_dev && w_lo_dev && y_dev && M >= 1 && M < (int64_t(1) << 31), "bad argument");
  GCRL_REQUIRE(mode >= 0 && mode <= 3 && (mode == 1 ? act_dev != nullptr : (mode == 3 || bias_dev != nullptr)),
               "bad mode / operands");
  GCRL_CUDA(cudaSetDevice(device));
  launch_tc_dense(x_dev, ldx, w_hi_dev, ldw, bias_dev, act_dev, ldact, y_dev, ldy, int(M), N, K, mode, as_stream(stream),
                  w_lo_dev);
  GCRL_API_END
}

extern "C" int gcrl_dense_layer_ensemble(int device, int n, int mode, int64_t M, int N, int K,
                                         const float *const *x_dev, int ldx, const float *const *w_hi_dev,
                                         const float *const *w_lo_dev, int ldw, const float *const *bias_dev,
                                         const float *const *act_dev, int ldact, float *const *y_dev, int ldy,
                                         void *stream) {
  GCRL_API_BEGIN
  using namespace gcrl;
  GCRL_REQUIRE(n >= 1 && n <= 8 && x_dev && w_hi_dev && w_lo_dev && y_dev && M >= 1 && M < (int64_t(1) << 31),
               "bad argument");
  GCRL_REQUIRE(mode >= 0 && mode <= 3 && (mode == 1 ? act_dev != nullptr : (mode == 3 || bias_dev != nullptr)),
               "bad mode / operands");
  TcDenseProblem pr[8];
  for (int i = 0; i < n; ++i) {
    GCRL_REQUIRE(x_dev[i] && w_hi_dev[i] && w_lo_dev[i] && y_dev[i], "NULL member operand");
    GCRL_REQUIRE(mode == 3 || (mode == 1 ? act_dev[i] != nullptr : bias_dev[i] != nullptr), "NULL member operand");
    pr[i] = TcDenseProblem{x_dev[i], ldx, w_hi_dev[i], w_lo_dev[i], ldw, (mode == 0 || mode == 2) ? bias_dev[i] : nullptr,
                           mode == 1 ? act_dev[i] : nullptr, y_dev[i]};
  }
  GCRL_CUDA(cudaSetDevice(device));
  launch_tc_dense_ensemble(pr, n, ldact, ldy, int(M), N, K, mode, as_stream(stream));
  GCRL_API_END
}

extern "C" int gcrl_dense_wgrad(int device, int engine, int64_t M, int N, int K, const float *dz_dev, int lddz,
                                const float *x_dev, int ldx, float *pw_dev, int ldw, int64_t w_split_stride,
                                float *pb_dev, int64_t b_split_stride, int max_splits, int *splits_out, void *stream) {
  GCRL_API_BEGIN
  using namespace gcrl;
  GCRL_REQUIRE(dz_dev && x_dev && pw_dev && splits_out && M >= 1 && M < (int64_t(1) << 31), "bad argument");
  GCRL_REQUIRE(engine == 0 || engine == 1, "engine must be 0 (fp32 FFMA) or 1 (tensor cores)");
  GCRL_CUDA(cudaSetDevice(device));
  cudaStream_t st = as_stream(stream);
  if (engine == 1) {
    *splits_out = launch_tc_wgrad(dz_dev, lddz, x_dev, ldx, pw_dev, ldw, w_split_stride, pb_dev, b_split_stride, int(M),
                                  N, K, max_splits, st);
  } else {
    GCRL_REQUIRE((lddz % 4) == 0 && (ldx % 4) == 0 && (ldw % 4) == 0, "leading dimensions must be multiples of 4");
    *splits_out = launch_linear_wgrad(dz_dev, lddz, x_dev, ldx, pw_dev, ldw, w_split_stride, pb_dev, b_split_stride,
                                      int(M), N, K, max_splits, st);
  }
  GCRL_API_END
}
