// az_net.cu -- policy/value network forward on the leaf batch (replaces Network.forward / forward_normalized /
// evaluate_batch: src/networks/flux.jl:127-132, src/networks/network.jl:264-271,308-315, and the Flux layers of
// src/networks/architectures/resnet.jl:53-92 and simplenet.jl:37-64).
//
// Activation layouts in HBM (fp16 rows of F = 128 channels, chosen once per network in ResNetImpl::init):
//   * DENSE, for the Connect-Four tower (7 x 6 boards, num_blocks > 0): row(board b, col x, row y) = b*W*H + y*W + x.
//     The tower kernels see it as a 4-D tensor (channel, x, y, board); the "same" padding of the 3x3 convolution is the
//     zero fill of TMA boxes that start at x = -1 (see az_k_conv_yrow).
//   * PADDED NHWC, for every other geometry: row(b, x, y) = b*BS + y*(W+1) + x, BS = (W+1)*(H+1), with column x = W and
//     row y = H kept at ZERO, so that the 3x3 "same" convolution becomes nine row-shifted GEMMs
//         out[p, co] = sum_{tap} sum_{ci} act[p + off(tap), ci] * Wt[co, tap*F + ci],   off = dy*(W+1) + dx
//     and each tap's A operand is ONE TMA box of consecutive rows (out-of-range rows are zero-filled by TMA).
//
// Kernels in this file (tcgen05 MMAs fed by TMA, fp16 operands, fp32 accumulators in TMEM):
//   az_k_stem<G>          leaf states -> first conv: the im2col tile is built in shared memory, one launch (both layouts)
//   az_k_tower_yrow       Connect-Four tower, ALL conv layers in one persistent launch: 2-CTA clusters (cta_group::2),
//                         resident weights, skip connection added on the tensor core from an fp16 + e4m3 residual stream
//   az_k_conv_yrow<EPI>   the same tower one conv layer per launch (AZ_TOWER=layer): the reference the persistent kernel
//                         is tested against bit for bit (with AZ_LO=16)
//   az_k_gemm_tc<BN,EPI>  generic warp-specialised implicit GEMM over the padded layout: the tower of every other
//                         geometry (tic-tac-toe, mancala, grid world), fp32 residual stream
//   az_k_head_conv        both heads' 1x1 convs as one N = 64 GEMM
//   az_k_heads_dense<G>   value dense + tanh and policy dense + softmax + legal-action mask, one launch
//   az_k_simplenet<G,NB>  fused fp32 MLP (SimpleNet)
//   az_k_fold_conv / az_k_fold_dense   parameter blob -> the kernels' weight layouts
// BatchNorm (test mode, eps = 1e-5) is folded into the conv / dense weights and biases when the blob is loaded.
#include <cuda.h>
#include <cuda_fp16.h>

#include <cmath>
#include <cstdlib>
#include <vector>

#include "az_internal.h"

#define AZ_TRY2(expr) do { int s__ = (expr); if (s__ != AZ_OK) return s__; } while (0)

// ------------------------------------------------------------------------------------------------
// PTX wrappers (sm_100a)
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ uint32_t mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t"
      "}" : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
  return ok;
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  while (!mbar_try_wait(bar, parity)) {}
}
__device__ __forceinline__ void tma_load_2d(void* dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1) {
  asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
               ::"r"(smem_u32(dst)), "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1) : "memory");
}
// One elected lane of a CONVERGED warp.  The producer / MMA warps run their loops warp-uniformly and predicate only the
// async instruction with this: inside a divergent `if (lane == 0)` region the compiler has to wrap every UTCHMMA /
// UTMALDG in an ELECT + R2UR.BROADCAST waterfall (~130 cycles per MMA, measured), because their operands are uniform registers.
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "elect.sync _|p, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t"
      "}" : "=r"(pred));
  return pred != 0;
}
// TMA bulk-tensor STORE smem -> global (tile written by the threads first, then fence.proxy.async + one issuing lane)
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* map, const void* src, int c0, int c1) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];"
               ::"l"(map), "r"(smem_u32(src)), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N> __device__ __forceinline__ void tma_store_wait_read() { asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory"); }
__device__ __forceinline__ void tma_store_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tcgen05_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tcgen05_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void umma_f16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}" ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t* r) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
        "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]),
        "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]),
        "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t* r) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
        "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}
// K-major, SWIZZLE_128B shared-memory matrix descriptor (cute::UMMA::SmemDescriptor): 8-row groups 1024 B apart
__device__ __forceinline__ uint64_t umma_desc_sw128(uint32_t saddr) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr & 0x3FFFF) >> 4);  // start address, bits [0,14)
  d |= (uint64_t)1 << 16;                   // leading byte offset (unused for swizzled K-major), bits [16,30)
  d |= (uint64_t)(1024 >> 4) << 32;         // stride byte offset, bits [32,46)
  d |= (uint64_t)1 << 46;                   // descriptor version (Blackwell), bits [46,48)
  d |= (uint64_t)2 << 61;                   // layout type SWIZZLE_128B, bits [61,64)
  return d;
}

// K-major, SWIZZLE_NONE descriptor for one 8-row x 16-element fp16 slice (two 8x8 core matrices of 128 B each, the second
// K half `lbo` bytes after the first): cute canonical layout ((8,n),2):((1,SBO),LBO) in 16-byte units
__device__ __forceinline__ uint64_t umma_desc_interleave(uint32_t saddr, uint32_t lbo, uint32_t sbo) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr & 0x3FFFF) >> 4);
  d |= (uint64_t)(lbo >> 4) << 16;
  d |= (uint64_t)(sbo >> 4) << 32;
  d |= (uint64_t)1 << 46;
  return d;  // layout type 0 = SWIZZLE_NONE
}

// ------------------------------------------------------------------------------------------------
// generic tcgen05 implicit-GEMM kernel (TMA producer warp -> 6-stage SWIZZLE_128B smem ring -> one elected lane issues
// tcgen05.mma M=128,N=BN,K=16 into double-buffered TMEM -> 4 epilogue warps): the tower convs of the padded layout
// ------------------------------------------------------------------------------------------------
namespace tc {
constexpr int BM = 128, BK = 64, STAGES = 6, F = 128;
constexpr int A_BYTES = BM * BK * 2;
constexpr int NUM_THREADS = 192;
enum { EPI_CONV1 = 0, EPI_CONV2 = 1 };
template <int BN>
struct Smem {
  uint8_t a[STAGES][A_BYTES];
  uint8_t b[STAGES][BN * BK * 2];
  uint64_t full[STAGES], empty[STAGES], tfull[2], tempty[2];
  uint32_t tmem_base;
  float bias[BN];
};
template <int BN>
constexpr uint32_t idesc() {  // f16 x f16 -> f32, K-major A and B, M = 128, N = BN
  return (1u << 4) | ((uint32_t)(BN >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);
}
}  // namespace tc

struct ConvGeom {
  int row_stride;  // W + 1
  int board_rows;  // (W+1)*(H+1)
  int valid_rows;  // (W+1)*H
  int wcols;       // W
  int off[9];
};
struct GemmArgs {
  const int32_t* n_boards;
  ConvGeom g;
  int kblocks;       // number of 64-wide K blocks: A coords = ((kb&1)*64, row + off[kb>>1]) (shifted-row conv)
  int rows_per_board;  // rows of the M dimension per board (board_rows)
  int alloc_rows;
  const float* bias;
  const float* resid32;  // EPI_CONV2
  int lo8;               // persistent tower: 1 = low-order residual part stored as e4m3 bytes (XL8), 0 = fp16 (XL16)
  int res_lo;            // per-layer Connect-Four kernel, EPI_CONV2: 1 = the residual has a low-order part (blocks >= 1), 0 = fp16 only (block 0)
  float* out32;          // EPI_CONV2 and the stem of the padded layout: fp32 residual stream
  __half* out16a;        // CONV1: T, CONV2: X16, head conv: policy features
  __half* out16b;        // head conv: value features
};

// (`ga` is __grid_constant__: the producer indexes ga.g.off[] with a run-time tap, which is then read from the parameter
// space in place instead of from a local-memory copy of the whole struct)
template <int BN, int EPI>
__global__ void __launch_bounds__(tc::NUM_THREADS, 1)
az_k_gemm_tc(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmW, const __grid_constant__ GemmArgs ga) {
  using namespace tc;
  using SmemT = Smem<BN>;
  constexpr int B_BYTES = BN * BK * 2;
  extern __shared__ uint8_t smem_raw[];
  SmemT& s = *reinterpret_cast<SmemT*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int rows_used = (*ga.n_boards) * ga.rows_per_board;
  const int num_tiles = (rows_used + BM - 1) / BM;
  const int kblocks = ga.kblocks;

  if (threadIdx.x == 0) {
    for (int i = 0; i < STAGES; i++) { mbar_init(&s.full[i], 1); mbar_init(&s.empty[i], 1); }
    for (int i = 0; i < 2; i++) { mbar_init(&s.tfull[i], 1); mbar_init(&s.tempty[i], 4); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (threadIdx.x >= 64 && threadIdx.x - 64 < BN) s.bias[threadIdx.x - 64] = ga.bias[threadIdx.x - 64];
  if (warp == 1) {  // TMEM: 2 accumulators x BN fp32 columns
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&s.tmem_base)), "r"((uint32_t)(2 * BN)) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem_base = s.tmem_base;
  // programmatic dependent launch: the prologue above overlapped the previous kernel's tail; all global data produced by
  // earlier kernels (activations, and the leaf count read below) is only touched after griddepcontrol.wait
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  asm volatile("griddepcontrol.wait;" ::: "memory");

  if (warp == 0) {
    {  // ===== TMA producer (warp-uniform; one elected lane issues) =====
      int stage = 0;
      uint32_t phase = 0;
      for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
        for (int kb = 0; kb < kblocks; kb++) {
          mbar_wait(&s.empty[stage], phase ^ 1);
          if (elect_one()) {
            mbar_expect_tx(&s.full[stage], A_BYTES + B_BYTES);
            tma_load_2d(s.a[stage], &tmA, &s.full[stage], (kb & 1) * BK, tile * BM + ga.g.off[kb >> 1]);
            tma_load_2d(s.b[stage], &tmW, &s.full[stage], kb * BK, 0);
          }
          __syncwarp();
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    {  // ===== MMA issuer (warp-uniform; one elected lane issues) =====
      int stage = 0;
      uint32_t phase = 0;
      int it = 0;
      for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x, it++) {
        const int acc = it & 1;
        const uint32_t aphase = (it >> 1) & 1;
        mbar_wait(&s.tempty[acc], aphase ^ 1);
        tcgen05_fence_after();
        const uint32_t tmem_d = tmem_base + acc * BN;
        for (int kb = 0; kb < kblocks; kb++) {
          mbar_wait(&s.full[stage], phase);
          tcgen05_fence_after();
          const uint64_t adesc = umma_desc_sw128(smem_u32(s.a[stage]));
          const uint64_t bdesc = umma_desc_sw128(smem_u32(s.b[stage]));
          if (elect_one()) {
#pragma unroll
            for (int k = 0; k < BK / 16; k++)  // advance 32 B (= 16 fp16) inside the 128-B swizzle row
              umma_f16(tmem_d, adesc + (uint64_t)(k * 2), bdesc + (uint64_t)(k * 2), idesc<BN>(), (kb | k) ? 1u : 0u);
            umma_commit(&s.empty[stage]);  // frees the smem stage when these MMAs retire
            if (kb == kblocks - 1) umma_commit(&s.tfull[acc]);
          }
          __syncwarp();
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else {  // ===== epilogue warps 2..5: TMEM lane quarter = warp % 4 =====
    const int quarter = warp & 3;
    int it = 0;
    for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x, it++) {
      const int acc = it & 1;
      const uint32_t aphase = (it >> 1) & 1;
      mbar_wait(&s.tfull[acc], aphase);
      tcgen05_fence_after();
      const int p = tile * BM + quarter * 32 + lane;
      const int r = p % ga.g.board_rows;
      const bool valid = (p < rows_used) && (r < ga.g.valid_rows) && ((r % ga.g.row_stride) != ga.g.wcols);
      const bool in_alloc = p < ga.alloc_rows;
#pragma unroll 1
      for (int c = 0; c < BN / 32; c++) {
        uint32_t v[32];
        tmem_ld32(tmem_base + acc * BN + c * 32 + ((uint32_t)(quarter * 32) << 16), v);
        float x[32];
#pragma unroll
        for (int j = 0; j < 32; j++) x[j] = __uint_as_float(v[j]) + s.bias[c * 32 + j];
        if (EPI == EPI_CONV2) {
          if (valid) {
            const float4* rp = reinterpret_cast<const float4*>(ga.resid32 + (size_t)p * F + c * 32);
#pragma unroll
            for (int j = 0; j < 8; j++) {
              float4 r4 = rp[j];
              x[4 * j] += r4.x; x[4 * j + 1] += r4.y; x[4 * j + 2] += r4.z; x[4 * j + 3] += r4.w;
            }
          }
        }
#pragma unroll
        for (int j = 0; j < 32; j++) x[j] = valid ? fmaxf(x[j], 0.0f) : 0.0f;
        if (!in_alloc) continue;
        if (EPI == EPI_CONV2) {
          float4* op = reinterpret_cast<float4*>(ga.out32 + (size_t)p * F + c * 32);
#pragma unroll
          for (int j = 0; j < 8; j++) op[j] = make_float4(x[4 * j], x[4 * j + 1], x[4 * j + 2], x[4 * j + 3]);
        }
        uint4 o[4];
        __half2* oh = reinterpret_cast<__half2*>(o);
#pragma unroll
        for (int j = 0; j < 16; j++) oh[j] = __floats2half2_rn(x[2 * j], x[2 * j + 1]);
        uint4* op = reinterpret_cast<uint4*>(ga.out16a + (size_t)p * F + c * 32);
#pragma unroll
        for (int j = 0; j < 4; j++) op[j] = o[j];
      }
      tcgen05_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&s.tempty[acc]);
    }
  }
  tcgen05_fence_before();
  __syncthreads();
  if (warp == 1) {
    tcgen05_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)(2 * BN)) : "memory");
  }
}

// ------------------------------------------------------------------------------------------------
// Connect-Four tower kernels: 2-CTA clusters (cta_group::2).  A single CTA issuing SS-mode M=128,N=128,K=16 MMAs is
// starved by SHARED-MEMORY bandwidth, not by L2 (stall sampling, profiles/r01_*): each MMA reads 8 KB of operands per
// 64 math cycles, which is all of the 128 B/clk smem port, and the TMA fills share that port.  Pairing two CTAs
// (M = 256 rows per pair) lets each CTA feed its own 128 A rows plus only HALF of B: each CTA owns half of the output
// channels (64) and keeps that half of the layer's weights resident in shared memory (18 chunks of 64co x 64k, 144 KB).
// Barrier protocol: TMA loads of both CTAs complete on the LEADER's `full` barrier; the leader's single MMA thread
// issues tcgen05.mma.cta_group::2 and multicasts tcgen05.commit to both CTAs' `empty` / `tfull` barriers; the 8
// epilogue warps of the pair arrive on the leader's `tempty`.
// ------------------------------------------------------------------------------------------------
namespace tc2 {
constexpr int BM = 128, BNH = 64, BK = 64;
constexpr int B_CHUNK = BNH * 128, NCHUNK = 18;
}  // namespace tc2

__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// TMA load whose completion bytes are credited to the LEADER CTA's mbarrier (peer bit cleared), cute::SM100_TMA_2SM_LOAD_2D
__device__ __forceinline__ void tma_load_2d_2sm(void* dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1) {
  asm volatile("cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
               ::"r"(smem_u32(dst)), "l"(map), "r"(smem_u32(bar) & 0xFEFFFFFFu), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void umma_f16_2sm(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}" ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void umma_commit_2sm(uint64_t* bar) {  // arrive on `bar` in both CTAs of the pair
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
               ::"r"(smem_u32(bar)), "h"((uint16_t)3) : "memory");
}
__device__ __forceinline__ void mbar_arrive_cluster(uint64_t* bar, uint32_t cta) {
  asm volatile(
      "{\n\t"
      ".reg .b32 ra;\n\t"
      "mapa.shared::cluster.u32 ra, %0, %1;\n\t"
      "mbarrier.arrive.shared::cluster.b64 _, [ra];\n\t"
      "}" ::"r"(smem_u32(bar)), "r"(cta) : "memory");
}

// ------------------------------------------------------------------------------------------------
// Connect-Four tower conv, one layer per launch ("y-row" kernel, round 2; AZ_TOWER=layer).  The persistent kernel below
// runs the same MMAs in the same order for every output row, so with the same residual format (AZ_LO=16) its outputs must
// equal this kernel's bit for bit: this kernel is the reference test_persistent_tower_equals_per_layer_kernels checks
// the persistent one against.
// Why not the padded layout on Connect Four (round 1, profiles/r01_final2_*): 56 MMA rows per 42 valid cells (25 % of
// the issued MMAs are padding), tile-round quantisation (604 tiles over 74 CTA pairs = 8.2 -> 9 rounds), three shifted
// shared-memory copies of every activation row, and zeroing / storing of pad rows.
//
// Here the activations are stored DENSE in HBM -- row(b, y, x) = b*42 + y*7 + x, 128 fp16 channels -- and seen by TMA
// as a 4-D tensor (channel, x, y, board).  One A stage = one board ROW y of 16 consecutive boards, 64 channels:
// box (64 ch, 8 x-slots, 1 y, 16 boards) with its origin at x = -1, i.e. 128 smem rows x 128 B (SWIZZLE_128B, one
// 1024-byte atom per board) where slot s of a board holds cell x = s - 1 and slot 0 is ZERO-FILLED by TMA (out of
// bounds); that zero slot, shared with the previous board's right edge, is the "same" padding of the convolution, so
// no pad row or pad column exists anywhere in memory.  An MMA tile is M = 256 rows = one output board row of 32
// boards (16 per CTA of the pair), 7 of every 8 rows valid (output row m <-> board m / 8, x = m % 8; x = 7 is discarded).
//   * ONE copy serves the three horizontal taps: the SWIZZLE_128B XOR is a function of the absolute shared-memory
//     address (measured: scripts/probes/umma_rowshift.cu, profiles/r02_rowshift_probe.txt -- a descriptor whose start is
//     advanced by any whole number of 128-byte rows reads exactly the shifted rows with base_offset = 0), so tap kx is
//     the same stage with the A descriptor started 2 - kx rows in.  Rows 128 / 129 of a stage are rows 0 / 1 of the
//     next stage in the ring (row 0 is a zero slot at all times; row 129 only feeds the discarded x = 7 output).
//     Shared-memory fill per MMA: 0.44 KB (round 1: 1.5 KB).
//   * schedule: input-row stationary.  For input row y the stage (y, half) feeds up to three OUTPUT rows
//     j = y+1, y, y-1 (vertical tap ky = j + 1 - y), each with its own TMEM accumulator: 4 x 128 columns roll through
//     the rows (three live + one being drained by the epilogue).  Taps that would read y = -1 or y = 6 are not issued
//     at all: 16 instead of 18 (j, ky) pairs per board column.
//   * MMA count per 32 boards and layer: 16 x 3 x 8 = 384 (round 1: 32 x 56 / 256 x 72 = 504, -24 %).
//   * balance: the unit of work is one output row of one 32-board group; the U = 6 x groups units are split into
//     gridDim/2 contiguous ranges of floor/ceil(U / pairs) units, so every CTA pair gets the same work to within one
//     unit whatever the leaf count of the tick (the halo row at each end of a range is loaded twice).
//   * boards are independent in this layout: rows of boards >= n_boards hold stale values that never reach a valid
//     board, so the epilogue needs no validity masking; x-slot 7 and boards past the allocation are clipped by the TMA
//     store (out-of-bounds elements of a store box are not written).
// Weights (this CTA's 64 output channels, 144 KB) stay resident in shared memory; the skip connection of conv2 is
// added on the tensor core by identity MMAs over the fp16 hi + lo residual stream, so the epilogue never reads the
// residual (its A stages are loaded with the same x = -1 origin and read one row in).
// ------------------------------------------------------------------------------------------------
namespace yr {
constexpr int NBOARD = 16;            // boards per CTA tile
constexpr int ASTAGES = 4;
constexpr int A_STAGE = 128 * 128;    // 128 rows x 64 fp16
constexpr int NACC = 4;               // TMEM accumulators (128 columns each)
constexpr int NUM_THREADS = 320;      // producer warp, MMA warp, 8 epilogue warps
constexpr int EPI_BYTES = 8 * 2048;   // two 1 KB store tiles per epilogue warp
struct Smem {
  uint8_t b[tc2::NCHUNK][tc2::B_CHUNK];
  uint8_t a[ASTAGES][A_STAGE];        // contiguous: rows 128.. of stage i are rows 0.. of stage i + 1
  uint8_t apad[1024];                 // zero rows after the last stage
  uint8_t epi[EPI_BYTES];
  uint8_t ident[256];
  uint64_t full[ASTAGES], empty[ASTAGES], tfull[NACC], tempty[NACC], bfull;
  uint32_t tmem_base;
};
// the contiguous unit range [u0, u1) of CTA pair `pair` (units = output board rows, 6 per 32-board group)
__device__ __forceinline__ void unit_range(int n_boards, int pair, int npairs, int& u0, int& u1) {
  const int groups = (n_boards + 2 * NBOARD - 1) / (2 * NBOARD);
  const long long U = 6LL * groups;
  u0 = (int)(U * pair / npairs);
  u1 = (int)(U * (pair + 1) / npairs);
}
}  // namespace yr

__device__ __forceinline__ void tma_load_4d_2sm(void* dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1, int c2, int c3) {
  asm volatile("cp.async.bulk.tensor.4d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
               ::"r"(smem_u32(dst)), "l"(map), "r"(smem_u32(bar) & 0xFEFFFFFFu), "r"(c0), "r"(c1), "r"(c2), "r"(c3) : "memory");
}
__device__ __forceinline__ void tma_store_4d(const CUtensorMap* map, const void* src, int c0, int c1, int c2, int c3) {
  asm volatile("cp.async.bulk.tensor.4d.global.shared::cta.bulk_group [%0, {%2, %3, %4, %5}], [%1];"
               ::"l"(map), "r"(smem_u32(src)), "r"(c0), "r"(c1), "r"(c2), "r"(c3) : "memory");
}

// stage sequence of one input row: conv1: C0 C1; conv2 with a residual: C0 Rhi0 Rhi1 C1 [Rlo0 Rlo1] -- a residual stage
// is consumed ~18x faster than a conv stage, so they are kept in pairs between the long stages (4-deep ring)
__device__ __forceinline__ void yrow_stage(int q, int nres, bool& isres, int& half, int& part) {
  if (nres == 0) { isres = false; half = q; part = 0; return; }
  isres = !(q == 0 || q == 3);
  if (!isres) { half = q == 0 ? 0 : 1; part = 0; return; }
  const int r = q < 3 ? q - 1 : q - 2;  // 0..3
  part = r >> 1; half = r & 1;
}

template <int EPI>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(yr::NUM_THREADS, 1)
az_k_conv_yrow(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmW,
               const __grid_constant__ CUtensorMap tmO16, const __grid_constant__ CUtensorMap tmOlo,
               const __grid_constant__ CUtensorMap tmRhi, const __grid_constant__ CUtensorMap tmRlo, GemmArgs ga) {
  using namespace tc2;
  constexpr int BN = 128, H = 6;
  constexpr int ASTAGES = yr::ASTAGES, NACC = yr::NACC, NB = yr::NBOARD;
  extern __shared__ __align__(1024) uint8_t smem_yr[];
  if ((smem_u32(smem_yr) & 1023u) != 0u) __trap();
  yr::Smem& s = *reinterpret_cast<yr::Smem*>(smem_yr);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const bool leader = rank == 0;
  int u0, u1;
  yr::unit_range(*ga.n_boards, blockIdx.x >> 1, gridDim.x >> 1, u0, u1);
  const bool has_work = u0 < u1;

  if (threadIdx.x == 0) {
    for (int i = 0; i < ASTAGES; i++) { mbar_init(&s.full[i], 1); mbar_init(&s.empty[i], 1); }
    for (int i = 0; i < NACC; i++) { mbar_init(&s.tfull[i], 1); mbar_init(&s.tempty[i], 16); }
    mbar_init(&s.bfull, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  // zero slots: row 0 of every stage (TMA only ever writes zeros there) and the rows after the last stage
  if (threadIdx.x < 64) {
    if (threadIdx.x < 8 * ASTAGES) *reinterpret_cast<uint4*>(s.a[threadIdx.x >> 3] + (threadIdx.x & 7) * 16) = make_uint4(0, 0, 0, 0);
    *reinterpret_cast<uint4*>(s.apad + threadIdx.x * 16) = make_uint4(0, 0, 0, 0);
    fence_proxy_async();
  }
  if (EPI == tc::EPI_CONV2 && threadIdx.x >= 192 && threadIdx.x < 192 + 64) {
    // this CTA's 8 x 16 slice of the 16 x 16 identity (B operand of the residual MMAs), un-swizzled K-major core matrices
    const int i = threadIdx.x - 192;
    const int n = (i & 31) >> 2, khalf = i >> 5, kk = (i & 3) * 2;
    const int k0 = khalf * 8 + kk, kone = (int)rank * 8 + n;
    const uint32_t w = (k0 == kone ? 0x3C00u : 0u) | (k0 + 1 == kone ? 0x3C000000u : 0u);
    *reinterpret_cast<uint32_t*>(s.ident + khalf * 128 + n * 16 + (i & 3) * 4) = w;
    fence_proxy_async();
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&s.tmem_base)), "r"(512u) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
  }
  tcgen05_fence_before();
  __syncthreads();
  cluster_sync_all();
  tcgen05_fence_after();
  const uint32_t tmem_base = s.tmem_base;
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");

  // Every role walks the same sequence: groups g intersecting [u0, u1), output rows [j_lo, j_hi) of the group, input
  // rows y = max(0, j_lo - 1) .. min(5, j_hi); `nbase` = running number of output rows before this group (accumulator
  // slot = number & 3, barrier phase = (number >> 2) & 1).
  if (warp == 0) {
    if (has_work) {  // ===== TMA producer (both CTAs) =====
      if (elect_one()) {
        if (leader) mbar_expect_tx(&s.bfull, 2 * NCHUNK * B_CHUNK);
        for (int ch = 0; ch < NCHUNK; ch++) tma_load_2d_2sm(s.b[ch], &tmW, &s.bfull, ch * BK, (int)rank * BNH);
      }
      __syncwarp();
      asm volatile("griddepcontrol.wait;" ::: "memory");
      int stage = 0;
      uint32_t phase = 0;
      for (int u = u0; u < u1;) {
        const int g = u / H, j_lo = u - g * H, j_hi = min(u1 - g * H, H);
        const int y_lo = max(0, j_lo - 1), y_hi = min(H - 1, j_hi);
        const int b0 = g * 2 * NB + (int)rank * NB;
        for (int y = y_lo; y <= y_hi; y++) {
          const int nres = (EPI == tc::EPI_CONV2 && y >= j_lo && y < j_hi) ? (ga.res_lo ? 4 : 2) : 0;
          for (int q = 0; q < 2 + nres; q++) {
            bool isres; int half, part;
            yrow_stage(q, nres, isres, half, part);
            mbar_wait(&s.empty[stage], phase ^ 1);
            if (elect_one()) {
              if (leader) mbar_expect_tx(&s.full[stage], 2 * yr::A_STAGE);
              tma_load_4d_2sm(s.a[stage], isres ? (part ? &tmRlo : &tmRhi) : &tmA, &s.full[stage], half * BK, -1, y, b0);
            }
            __syncwarp();
            if (++stage == ASTAGES) { stage = 0; phase ^= 1; }
          }
        }
        u = g * H + j_hi;
      }
    }
  } else if (warp == 1) {
    if (leader && has_work) {  // ===== MMA issuer (leader CTA only) =====
      constexpr uint32_t IDESC = (1u << 4) | ((uint32_t)(BN >> 3) << 17) | ((uint32_t)((2 * BM) >> 4) << 24);    // M = 256, N = 128
      constexpr uint32_t IDESC_R = (1u << 4) | ((uint32_t)(16 >> 3) << 17) | ((uint32_t)((2 * BM) >> 4) << 24);  // M = 256, N = 16
      const uint64_t idsc = umma_desc_interleave(smem_u32(s.ident), 128u, 256u);
      mbar_wait(&s.bfull, 0);
      tcgen05_fence_after();
      int stage = 0;
      uint32_t phase = 0;
      int nbase = 0;
      for (int u = u0; u < u1;) {
        const int g = u / H, j_lo = u - g * H, j_hi = min(u1 - g * H, H);
        const int y_lo = max(0, j_lo - 1), y_hi = min(H - 1, j_hi);
        for (int y = y_lo; y <= y_hi; y++) {
          // output rows first touched by this input row: j = y + 1, and j = 0 when y == 0 -- wait until the epilogue has
          // drained the accumulator slot they take
          for (int j = (y == 0 ? 0 : y + 1); j <= y + 1; j++) {
            if (j < j_lo || j >= j_hi) continue;
            const int n = nbase + (j - j_lo);
            mbar_wait(&s.tempty[n & 3], ((uint32_t)(n >> 2) & 1u) ^ 1u);
          }
          tcgen05_fence_after();
          const int nres = (EPI == tc::EPI_CONV2 && y >= j_lo && y < j_hi) ? (ga.res_lo ? 4 : 2) : 0;
          for (int q = 0; q < 2 + nres; q++) {
            bool isres; int half, part;
            yrow_stage(q, nres, isres, half, part);
            mbar_wait(&s.full[stage], phase);
            tcgen05_fence_after();
            const uint32_t abase = smem_u32(s.a[stage]);
            if (elect_one()) {
              if (isres) {  // skip connection (resnet.jl:55-62): acc[j = y][:, half*64 + k*16 ..] += A[:, k*16 ..] . I16
                const uint32_t tmem_d = tmem_base + (uint32_t)(((nbase + (y - j_lo)) & 3) * BN);
                const uint64_t adesc = umma_desc_sw128(abase + 128u);  // cell x sits in slot x + 1
#pragma unroll
                for (int k = 0; k < BK / 16; k++)
                  umma_f16_2sm(tmem_d + (uint32_t)(half * BK + k * 16), adesc + (uint64_t)(k * 2), idsc, IDESC_R, 1u);
              } else {
#pragma unroll
                for (int dj = 1; dj >= -1; dj--) {  // output row j = y + dj uses the vertical tap ky = dj + 1
                  const int j = y + dj;
                  if (j < j_lo || j >= j_hi) continue;
                  const int ky = dj + 1;
                  const uint32_t tmem_d = tmem_base + (uint32_t)(((nbase + (j - j_lo)) & 3) * BN);
                  const bool first = (half == 0) && (y == (j > 0 ? j - 1 : 0));  // first stage of the first input row of j
#pragma unroll
                  for (int kx = 0; kx < 3; kx++) {  // input x = x_out + 1 - kx lives in slot x_out + 2 - kx
                    const uint64_t adesc = umma_desc_sw128(abase + (uint32_t)(2 - kx) * 128u);
                    const uint64_t bdesc = umma_desc_sw128(smem_u32(s.b[(ky * 3 + kx) * 2 + half]));
#pragma unroll
                    for (int k = 0; k < BK / 16; k++)
                      umma_f16_2sm(tmem_d, adesc + (uint64_t)(k * 2), bdesc + (uint64_t)(k * 2), IDESC, (first && kx == 0 && k == 0) ? 0u : 1u);
                  }
                }
              }
              umma_commit_2sm(&s.empty[stage]);
            }
            __syncwarp();
            if (++stage == ASTAGES) { stage = 0; phase ^= 1; }
          }
          // output rows completed by this input row: j = y - 1, and j = 5 after y = 5
          if (elect_one()) {
            if (y - 1 >= j_lo && y - 1 < j_hi) umma_commit_2sm(&s.tfull[(nbase + (y - 1 - j_lo)) & 3]);
            if (y == H - 1 && j_hi == H) umma_commit_2sm(&s.tfull[(nbase + (H - 1 - j_lo)) & 3]);
          }
          __syncwarp();
        }
        nbase += j_hi - j_lo;
        u = g * H + j_hi;
      }
    }
  } else {  // ===== epilogue warps 2..9 (both CTAs): 128 rows (16 boards x 8 x-slots) x 128 channels per output row =====
    asm volatile("griddepcontrol.wait;" ::: "memory");
    const int quarter = warp & 3;
    const int colhalf = (warp - 2) >> 2;
    const int sw = (lane >> 2) & 1;  // SWIZZLE_32B: 16-byte chunk index ^= bit 7 of the byte address (row >> 2)
    uint8_t* tiles = s.epi + (warp - 2) * 2048;
    int ring = 0;
    int n = 0;
    const float* __restrict__ bias_g = ga.bias + colhalf * 64;
    for (int u = u0; u < u1; u++, n++) {
      const int g = u / H, j = u - g * H;
      const int bq = g * 2 * NB + (int)rank * NB + quarter * 4;  // first of this warp's 4 boards
      const int slot = n & 3;
      mbar_wait(&s.tfull[slot], (uint32_t)(n >> 2) & 1u);
      tcgen05_fence_after();
#pragma unroll
      for (int sc = 0; sc < 4; sc++) {
        const int col = colhalf * 64 + sc * 16;
        uint32_t v[16];
        tmem_ld16(tmem_base + slot * BN + col + ((uint32_t)(quarter * 32) << 16), v);
        uint4 oh4[2], ol4[2];
        __half2* oh = reinterpret_cast<__half2*>(oh4);
        __half2* ol = reinterpret_cast<__half2*>(ol4);
#pragma unroll
        for (int jj = 0; jj < 8; jj++) {
          const float2 bb = __ldg(reinterpret_cast<const float2*>(bias_g + sc * 16) + jj);
          const float x0 = fmaxf(__uint_as_float(v[2 * jj]) + bb.x, 0.f);
          const float x1 = fmaxf(__uint_as_float(v[2 * jj + 1]) + bb.y, 0.f);
          const __half2 h = __floats2half2_rn(x0, x1);
          oh[jj] = h;
          if (EPI == tc::EPI_CONV2) {  // lo = fp16(y - hi): hi + lo carries ~22 significand bits of the skip path
            const float2 hf = __half22float2(h);
            ol[jj] = __floats2half2_rn(x0 - hf.x, x1 - hf.y);
          }
        }
#pragma unroll
        for (int part = 0; part < (EPI == tc::EPI_CONV2 ? 2 : 1); part++) {
          uint8_t* tile = tiles + ring * 1024;
          ring ^= 1;
          if (lane == 0) tma_store_wait_read<1>();  // the store issued two stores ago has finished reading this tile
          __syncwarp();
          const uint4* o = part ? ol4 : oh4;
          *reinterpret_cast<uint4*>(tile + lane * 32 + ((0 ^ sw) << 4)) = o[0];
          *reinterpret_cast<uint4*>(tile + lane * 32 + ((1 ^ sw) << 4)) = o[1];
          fence_proxy_async();
          __syncwarp();
          if (lane == 0) { tma_store_4d(part ? &tmOlo : &tmO16, tile, col, 0, j, bq); tma_store_commit(); }
        }
      }
      tcgen05_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive_cluster(&s.tempty[slot], 0);
    }
    if (lane == 0) tma_store_wait_all();
    __syncwarp();
  }
  tcgen05_fence_before();
  __syncthreads();
  cluster_sync_all();
  if (warp == 1) {
    tcgen05_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u) : "memory");
  }
}

// ------------------------------------------------------------------------------------------------
// Persistent whole-tower kernel (round 2): ONE launch runs all 2 x num_blocks conv layers of the y-row tower.
// The per-layer kernel above spends ~45 % of its elapsed time outside the tensor pipe (launch + CTA ramp, TMEM alloc,
// cluster sync, the 144 KB weight load before the first MMA, pipeline fill, and the drain of the last epilogue): with
// ~30 us of work per layer those fixed costs are paid 14 times per evaluation.  Here every CTA pair keeps its contiguous
// unit range [u0, u1) (the same for every layer, since the leaf count does not change inside an evaluation) and loops
// over the layers itself:
//   * dependencies are LOCAL: layer l+1's input row y of a 32-board group needs layer l's output rows y-1..y+1 of the
//     same group, i.e. rows of this pair plus ONE halo row of the pair before / after it when a range boundary falls
//     inside a group.  No grid-wide barrier: each pair publishes "layer l stored" in a global counter (16 epilogue
//     warps x 1 per layer, monotonic over launches: the base is read at kernel start) and a producer spins only on
//     its lower neighbour (start of the layer) and its upper neighbour (just before the top halo row).  All CTAs are
//     co-resident (one per SM), so spinning cannot deadlock.  The same waits order the in-place reuse of T / X.
//   * a pair's first and last segments (the only rows neighbours read) are processed FIRST in every layer and published as
//     soon as they are stored; the middle groups follow.  Inside a CTA the 8 epilogue warps count the units whose TMA
//     stores have completed (`stored[]`); the producer loads a segment of layer l+1 when the same segment of layer l
//     is in memory, so at a layer boundary the ring already holds the next layer's first stages.
//   * the weights of the next layer are (re)loaded into the resident 144 KB by warp 1 of both CTAs as soon as the last
//     MMA of the layer has retired (`wfree`, multicast tcgen05.commit); the A producer never waits for them.
//   * the TMEM accumulator ring, the A-stage ring and all barrier phases simply continue across layers.
// Weights of all layers live in ONE [L*128][1152] fp16 tensor (one tensor map), biases in one [L][128] array.
// ------------------------------------------------------------------------------------------------
namespace tw {
struct Smem {
  uint8_t b[tc2::NCHUNK][tc2::B_CHUNK];
  uint8_t a[yr::ASTAGES][yr::A_STAGE];
  uint8_t apad[1024];
  uint8_t epi[yr::EPI_BYTES];
  uint8_t ident[256];
  uint8_t ident8[512];   // lo8 mode: this CTA's 16 x 32 slice of 2^-14 * I32 in e5m2 (B operand of the fp8 residual MMAs)
  uint64_t full[yr::ASTAGES], empty[yr::ASTAGES], tfull[yr::NACC], tempty[yr::NACC], bfull[tc2::NCHUNK], wfree;
  uint32_t tmem_base;
  int stored[8];         // per epilogue warp: units (all layers, processing order) whose TMA stores have completed
};
// A pair's unit range [u0, u1) is a run of SEGMENTS = maximal runs of output rows inside one 32-board group.  Other pairs read
// exactly two of its rows as halo: the LAST row u1-1 (pair above: bottom halo of its first segment) and the FIRST row u0
// (pair below: top halo of its last segment).  Every layer therefore processes the last segment first (when the range ends
// inside a group), then the first one, then the middle groups (k = processing order), and publishes the two rows separately
// (`done[128 + pair]`: row u1-1, `done[pair]`: row u0): when a layer ends, everything the neighbours and this pair's own
// first segments of the next layer need has been in memory for about half a layer, the producer has already put the next
// layer's first A stages into the ring, and the only wait left at the boundary is the first weight chunk.
struct Seg { int g, j_lo, j_hi; };
__device__ __forceinline__ Seg segment(int k, int nseg, int u0, int u1) {
  int i = k;
  if (nseg >= 2 && u1 % 6 != 0) i = (k == 0) ? nseg - 1 : k - 1;   // (a range that ends on a group boundary has no
                                                                  // reader above: its first segment goes first)
  Seg sg;
  sg.g = u0 / 6 + i;
  sg.j_lo = (i == 0) ? u0 - sg.g * 6 : 0;
  sg.j_hi = min(u1 - sg.g * 6, 6);
  return sg;
}
__device__ __forceinline__ int ld_acquire_shared_s32(const int* p) {
  int v;
  asm volatile("ld.acquire.cta.shared::cta.s32 %0, [%1];" : "=r"(v) : "r"(smem_u32(p)) : "memory");
  return v;
}
__device__ __forceinline__ void st_release_shared_s32(int* p, int v) {
  asm volatile("st.release.cta.shared::cta.s32 [%0], %1;" ::"r"(smem_u32(p)), "r"(v) : "memory");
}
__device__ __forceinline__ unsigned long long ld_acquire_u64(const unsigned long long* p) {
  unsigned long long v;
  asm volatile("ld.acquire.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void red_release_add_u64(unsigned long long* p, unsigned long long v) {
  asm volatile("red.release.gpu.global.add.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
// stage sequence of one input row of a conv2 layer in lo8 mode: C0 Rhi0 Rhi1 C1 Rlo8 (the 8-bit low-order part covers all 128
// channels in ONE 16 KB stage); kind 0 = conv, 1 = residual hi (fp16), 2 = residual lo (fp16), 3 = residual lo (e4m3)
__device__ __forceinline__ void stage_of(int q, int nres, bool lo8, int& kind, int& half) {
  if (!lo8 || nres < 3) {
    bool isres; int part;
    yrow_stage(q, nres, isres, half, part);
    kind = !isres ? 0 : (part ? 2 : 1);
    return;
  }
  if (q == 0) { kind = 0; half = 0; }
  else if (q == 1) { kind = 1; half = 0; }
  else if (q == 2) { kind = 1; half = 1; }
  else if (q == 3) { kind = 0; half = 1; }
  else { kind = 3; half = 0; }
}
__device__ __forceinline__ void umma_f8_2sm(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f8f6f4 [%0], %1, %2, %3, p;\n\t"
      "}" ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
// two floats -> two e4m3 bytes (first argument in the LOW byte = lower address)
__device__ __forceinline__ uint32_t cvt_e4m3x2(float lo_elem, float hi_elem) {
  uint16_t r;
  asm("cvt.rn.satfinite.e4m3x2.f32 %0, %1, %2;" : "=h"(r) : "f"(hi_elem), "f"(lo_elem));
  return (uint32_t)r;
}
constexpr float LO8_SCALE = 16384.0f;   // lo is stored as e4m3(lo * 2^14) (4 significant bits over 17 octaves, |lo| < 0.027); the
                                        // identity of its MMA is 2^-14 (e5m2 0x04), so the product is lo again, exactly
}  // namespace tw

__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(yr::NUM_THREADS, 1)
az_k_tower_yrow(const __grid_constant__ CUtensorMap tmX, const __grid_constant__ CUtensorMap tmT, const __grid_constant__ CUtensorMap tmXL,
                const __grid_constant__ CUtensorMap tmW, const __grid_constant__ CUtensorMap tmXo, const __grid_constant__ CUtensorMap tmTo,
                const __grid_constant__ CUtensorMap tmXLo, const __grid_constant__ CUtensorMap tmXL8, const __grid_constant__ CUtensorMap tmXL8o,
                GemmArgs ga, int num_layers, unsigned long long* __restrict__ done) {
  using namespace tc2;
  constexpr int BN = 128, H = 6;
  constexpr int ASTAGES = yr::ASTAGES, NB = yr::NBOARD;
  extern __shared__ __align__(1024) uint8_t smem_tw[];
  if ((smem_u32(smem_tw) & 1023u) != 0u) __trap();
  tw::Smem& s = *reinterpret_cast<tw::Smem*>(smem_tw);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const bool leader = rank == 0;
  const int pair = blockIdx.x >> 1, npairs = gridDim.x >> 1;
  const bool lo8 = ga.lo8 != 0;          // low-order part of the skip stream as e4m3 bytes (default) or fp16 (AZ_LO=16)

  if (threadIdx.x == 0) {
    for (int i = 0; i < ASTAGES; i++) { mbar_init(&s.full[i], 1); mbar_init(&s.empty[i], 1); }
    for (int i = 0; i < yr::NACC; i++) { mbar_init(&s.tfull[i], 1); mbar_init(&s.tempty[i], 16); }
    for (int i = 0; i < NCHUNK; i++) mbar_init(&s.bfull[i], 1);
    mbar_init(&s.wfree, 1);
    for (int i = 0; i < 8; i++) s.stored[i] = 0;
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (threadIdx.x < 64) {
    if (threadIdx.x < 8 * ASTAGES) *reinterpret_cast<uint4*>(s.a[threadIdx.x >> 3] + (threadIdx.x & 7) * 16) = make_uint4(0, 0, 0, 0);
    *reinterpret_cast<uint4*>(s.apad + threadIdx.x * 16) = make_uint4(0, 0, 0, 0);
    fence_proxy_async();
  }
  if (threadIdx.x >= 192 && threadIdx.x < 192 + 64) {  // this CTA's 8 x 16 slice of the 16 x 16 identity (residual MMAs)
    const int i = threadIdx.x - 192;
    const int n = (i & 31) >> 2, khalf = i >> 5, kk = (i & 3) * 2;
    const int k0 = khalf * 8 + kk, kone = (int)rank * 8 + n;
    const uint32_t w = (k0 == kone ? 0x3C00u : 0u) | (k0 + 1 == kone ? 0x3C000000u : 0u);
    *reinterpret_cast<uint32_t*>(s.ident + khalf * 128 + n * 16 + (i & 3) * 4) = w;
    fence_proxy_async();
  }
  if (threadIdx.x < 128) {  // e5m2 2^-14 * I32, this CTA's rows n = rank*16 + i: byte (i, k) at (i>>3)*256 + (k>>4)*128 + (i&7)*16 + (k&15)
    const int i = threadIdx.x >> 3, k4 = (threadIdx.x & 7) * 4;   // 4 k-bytes per thread
    uint32_t w = 0;
#pragma unroll
    for (int j = 0; j < 4; j++) if (k4 + j == (int)rank * 16 + i) w |= 0x04u << (8 * j);
    *reinterpret_cast<uint32_t*>(s.ident8 + (i >> 3) * 256 + (k4 >> 4) * 128 + (i & 7) * 16 + (k4 & 15)) = w;
    fence_proxy_async();
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&s.tmem_base)), "r"(512u) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
  }
  tcgen05_fence_before();
  __syncthreads();
  cluster_sync_all();
  tcgen05_fence_after();
  const uint32_t tmem_base = s.tmem_base;
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  // everything below reads data of earlier kernels (leaf count, activations, the flag counters of the previous launch)
  asm volatile("griddepcontrol.wait;" ::: "memory");

  int u0, u1;
  yr::unit_range(*ga.n_boards, pair, npairs, u0, u1);
  const bool has_work = u0 < u1;
  // flag protocol: every pair adds 16 per layer (one per epilogue warp) to each of its two counters (first row stored /
  // last row stored); counters are never reset, the value a pair finds in its own counter at kernel start is the base of
  // this launch (identical for all pairs and for both counters)
  const unsigned long long base = done[pair];
  // neighbours whose rows this pair reads as halo (only when the range boundary falls inside a 32-board group)
  int q_lo = -1, q_hi = -1;
  if (has_work) {
    if (u0 % H != 0) { q_lo = pair - 1; for (;;) { int a, b; yr::unit_range(*ga.n_boards, q_lo, npairs, a, b); if (a < b) break; q_lo--; } }
    if (u1 % H != 0) { q_hi = pair + 1; for (;;) { int a, b; yr::unit_range(*ga.n_boards, q_hi, npairs, a, b); if (a < b) break; q_hi++; } }
  }
  const int Up = u1 - u0;                                         // units per layer
  const int nseg = has_work ? (u1 - 1) / H - u0 / H + 1 : 0;
  unsigned long long* const done_up = done + 128;                 // row u1-1 of a layer stored (read by the pair above); `done`: row u0
  cluster_sync_all();  // `base` is read by both CTAs before any warp of the pair can add to the counter

  if (!has_work) {
    // idle pair (fewer units than pairs): keep the counter in step so that its base stays equal to everybody else's
    if (threadIdx.x == 0 && leader) {
      tw::red_release_add_u64(done + pair, 16ull * (unsigned long long)num_layers);
      tw::red_release_add_u64(done + 128 + pair, 16ull * (unsigned long long)num_layers);
    }
  } else if (warp == 0) {
    // ===== TMA producer (both CTAs): A stages only (the weights are loaded by warp 1), so it runs ahead across layer boundaries =====
    int stage = 0;
    uint32_t phase = 0;
    // (Tried and removed: starting pair p p*skew cycles late so that half the pairs are in an L2-hungry conv2 layer while the
    // others are in a conv1 layer -- 0 / 350 / 700 / 1400 / 2800 cycles per pair gave 5.58 / 5.56 / 5.47 / 5.29 / 4.95 M
    // expansions/s on one box: the average demand of a block is already at the chip's L2 limit, staggering only adds ramp.)
    for (int l = 0; l < num_layers; l++) {
      const bool conv2 = (l & 1) != 0;
      const CUtensorMap* mA = conv2 ? &tmT : &tmX;
      int cum = 0;   // units of this layer's segments up to and including the current one (processing order)
      for (int k = 0; k < nseg; k++) {
        const tw::Seg sg = tw::segment(k, nseg, u0, u1);
        const int g = sg.g, j_lo = sg.j_lo, j_hi = sg.j_hi;
        cum += j_hi - j_lo;
        const bool lo_halo = q_lo >= 0 && g * H + j_lo == u0;   // bottom halo row: produced by the pair below in layer l-1
        bool hi_ok = (l == 0) || !(q_hi >= 0 && g * H + j_hi == u1);
        if (l > 0) {
          // the rows of layer l-1 this segment reads: the same segment of this CTA (its 8 epilogue warps count the units whose
          // stores have completed, same processing order in every layer) ...
          const int need = (l - 1) * Up + cum;
          for (;;) {
            const int v = tw::ld_acquire_shared_s32(&s.stored[lane & 7]);
            if (__all_sync(0xFFFFFFFFu, v >= need)) break;
            __nanosleep(64);
          }
          // ... plus the halo row below = the LAST row of the lower neighbour in layer l-1
          if (lo_halo) {
            if (lane == 0) { while (tw::ld_acquire_u64(done_up + q_lo) < base + 16ull * (unsigned long long)l) {} }
            __syncwarp();
          }
          fence_proxy_async();
        }
        const int y_lo = max(0, j_lo - 1), y_hi = min(H - 1, j_hi);
        const int b0 = g * 2 * NB + (int)rank * NB;
        for (int y = y_lo; y <= y_hi; y++) {
          if (!hi_ok && y == j_hi) {  // top halo row = the FIRST row of the next pair in layer l-1
            if (lane == 0) { while (tw::ld_acquire_u64(done + q_hi) < base + 16ull * (unsigned long long)l) {} }
            __syncwarp();
            fence_proxy_async();
            hi_ok = true;
          }
          const int nres = (conv2 && y >= j_lo && y < j_hi) ? (l > 1 ? (lo8 ? 3 : 4) : 2) : 0;
          for (int q = 0; q < 2 + nres; q++) {
            int kind, half;
            tw::stage_of(q, nres, lo8, kind, half);
            mbar_wait(&s.empty[stage], phase ^ 1);
            if (elect_one()) {
              if (leader) mbar_expect_tx(&s.full[stage], 2 * yr::A_STAGE);
              const CUtensorMap* m = kind == 0 ? mA : (kind == 1 ? &tmX : (kind == 2 ? &tmXL : &tmXL8));
              tma_load_4d_2sm(s.a[stage], m, &s.full[stage], half * BK, -1, y, b0);
            }
            __syncwarp();
            if (++stage == ASTAGES) { stage = 0; phase ^= 1; }
          }
        }
      }
    }
  } else if (warp == 1) {
    // this CTA's half of layer l's weights: one barrier per 8 KB chunk, requested in the order the layer's first MMAs use them
    // (K half 0 first; vertical taps ky = 2, 1, 0), so the tensor pipe restarts when the first taps have landed, not after all
    // 144 KB.  Issued by warp 1 of BOTH CTAs as soon as every MMA of the previous layer has retired (`wfree`, multicast commit)
    auto load_weights = [&](int l) {
      if (elect_one()) {
        for (int half = 0; half < 2; half++)
          for (int ky = 2; ky >= 0; ky--)
            for (int kx = 0; kx < 3; kx++) {
              const int ch = (ky * 3 + kx) * 2 + half;
              if (leader) mbar_expect_tx(&s.bfull[ch], 2 * B_CHUNK);
              tma_load_2d_2sm(s.b[ch], &tmW, &s.bfull[ch], ch * BK, l * 128 + (int)rank * BNH);
            }
      }
      __syncwarp();
    };
    // (Tried and removed: the six ky = 2 chunks are free one input row before a layer ends and are what the next layer's first
    // input row needs; requesting them from the producer's wait loops on an extra `wearly` commit gave 27.93 vs 27.88 us per
    // layer -- the first weight chunk's latency is not what is left of the layer boundary.)
    load_weights(0);
    if (!leader) {
      for (int l = 1; l < num_layers; l++) {
        mbar_wait(&s.wfree, (uint32_t)(l - 1) & 1u);   // every MMA of layer l-1 (reads both CTAs' weights) has retired
        load_weights(l);
      }
    } else {  // ===== MMA issuer (leader CTA only) =====
      constexpr uint32_t IDESC = (1u << 4) | ((uint32_t)(BN >> 3) << 17) | ((uint32_t)((2 * BM) >> 4) << 24);    // M = 256, N = 128
      constexpr uint32_t IDESC_R = (1u << 4) | ((uint32_t)(16 >> 3) << 17) | ((uint32_t)((2 * BM) >> 4) << 24);  // M = 256, N = 16
      const uint64_t idsc = umma_desc_interleave(smem_u32(s.ident), 128u, 256u);
      // fp8 residual MMA: A = e4m3 (format 0), B = e5m2 (format 1), M = 256, N = 32, K = 32
      constexpr uint32_t IDESC_R8 = (1u << 4) | (1u << 10) | ((uint32_t)(32 >> 3) << 17) | ((uint32_t)((2 * BM) >> 4) << 24);
      const uint64_t idsc8 = umma_desc_interleave(smem_u32(s.ident8), 128u, 256u);
      int stage = 0;
      uint32_t phase = 0;
      int nbase = 0;
      for (int l = 0; l < num_layers; l++) {
        const bool conv2 = (l & 1) != 0;
        uint32_t wready = 0;   // bit ch: this layer's weight chunk ch has been waited for
        for (int k = 0; k < nseg; k++) {
          const tw::Seg sg = tw::segment(k, nseg, u0, u1);
          const int j_lo = sg.j_lo, j_hi = sg.j_hi;
          const int y_lo = max(0, j_lo - 1), y_hi = min(H - 1, j_hi);
          for (int y = y_lo; y <= y_hi; y++) {
            for (int j = (y == 0 ? 0 : y + 1); j <= y + 1; j++) {
              if (j < j_lo || j >= j_hi) continue;
              const int n = nbase + (j - j_lo);
              mbar_wait(&s.tempty[n & 3], ((uint32_t)(n >> 2) & 1u) ^ 1u);
            }
            tcgen05_fence_after();
            const int nres = (conv2 && y >= j_lo && y < j_hi) ? (l > 1 ? (lo8 ? 3 : 4) : 2) : 0;
            for (int q = 0; q < 2 + nres; q++) {
              int kind, half;
              tw::stage_of(q, nres, lo8, kind, half);
              const bool isres = kind != 0;
              mbar_wait(&s.full[stage], phase);
              tcgen05_fence_after();
              const uint32_t abase = smem_u32(s.a[stage]);
              if (!isres && wready != 0x3FFFFu) {  // first uses of this layer's weight chunks (warp-uniform)
#pragma unroll
                for (int dj = 1; dj >= -1; dj--) {
                  const int j = y + dj;
                  if (j < j_lo || j >= j_hi) continue;
#pragma unroll
                  for (int kx = 0; kx < 3; kx++) {
                    const int ch = ((dj + 1) * 3 + kx) * 2 + half;
                    if (!((wready >> ch) & 1u)) { mbar_wait(&s.bfull[ch], (uint32_t)l & 1u); wready |= 1u << ch; }
                  }
                }
                tcgen05_fence_after();
              }
              if (elect_one()) {
                if (kind == 3) {  // 8-bit low-order part: acc[:, 32k .. 32k+31] += A8[:, 32k ..] . (2^-14 I32), 4 x K = 32
                  const uint32_t tmem_d = tmem_base + (uint32_t)(((nbase + (y - j_lo)) & 3) * BN);
                  const uint64_t adesc = umma_desc_sw128(abase + 128u);
#pragma unroll
                  for (int k = 0; k < 4; k++)
                    tw::umma_f8_2sm(tmem_d + (uint32_t)(k * 32), adesc + (uint64_t)(k * 2), idsc8, IDESC_R8, 1u);
                } else if (isres) {
                  const uint32_t tmem_d = tmem_base + (uint32_t)(((nbase + (y - j_lo)) & 3) * BN);
                  const uint64_t adesc = umma_desc_sw128(abase + 128u);
#pragma unroll
                  for (int k = 0; k < BK / 16; k++)
                    umma_f16_2sm(tmem_d + (uint32_t)(half * BK + k * 16), adesc + (uint64_t)(k * 2), idsc, IDESC_R, 1u);
                } else {
#pragma unroll
                  for (int dj = 1; dj >= -1; dj--) {
                    const int j = y + dj;
                    if (j < j_lo || j >= j_hi) continue;
                    const int ky = dj + 1;
                    const uint32_t tmem_d = tmem_base + (uint32_t)(((nbase + (j - j_lo)) & 3) * BN);
                    const bool first = (half == 0) && (y == (j > 0 ? j - 1 : 0));
#pragma unroll
                    for (int kx = 0; kx < 3; kx++) {
                      const uint64_t adesc = umma_desc_sw128(abase + (uint32_t)(2 - kx) * 128u);
                      const uint64_t bdesc = umma_desc_sw128(smem_u32(s.b[(ky * 3 + kx) * 2 + half]));
#pragma unroll
                      for (int k = 0; k < BK / 16; k++)
                        umma_f16_2sm(tmem_d, adesc + (uint64_t)(k * 2), bdesc + (uint64_t)(k * 2), IDESC, (first && kx == 0 && k == 0) ? 0u : 1u);
                    }
                  }
                }
                umma_commit_2sm(&s.empty[stage]);
              }
              __syncwarp();
              if (++stage == ASTAGES) { stage = 0; phase ^= 1; }
            }
            if (elect_one()) {
              if (y - 1 >= j_lo && y - 1 < j_hi) umma_commit_2sm(&s.tfull[(nbase + (y - 1 - j_lo)) & 3]);
              if (y == H - 1 && j_hi == H) umma_commit_2sm(&s.tfull[(nbase + (H - 1 - j_lo)) & 3]);
            }
            __syncwarp();
          }
          nbase += j_hi - j_lo;
        }
        if (elect_one()) umma_commit_2sm(&s.wfree);  // the resident weights may be replaced
        __syncwarp();
        if (l + 1 < num_layers) {
          mbar_wait(&s.wfree, (uint32_t)l & 1u);
          load_weights(l + 1);
        }
      }
    }
  } else {  // ===== epilogue warps 2..9 (both CTAs) =====
    const int quarter = warp & 3;
    const int colhalf = (warp - 2) >> 2;
    uint8_t* tile = s.epi + (warp - 2) * 2048;   // one 32-row x 64-byte tile per warp (SWIZZLE_64B: 16-byte chunk ^= (row >> 1) & 3)
    const int sw = (lane >> 1) & 3;
    int n = 0;
    for (int l = 0; l < num_layers; l++) {
      const bool conv2 = (l & 1) != 0;
      const bool want_lo = conv2 && l != num_layers - 1;   // nobody reads the low-order part of the last block's output
      const float* __restrict__ bias_g = ga.bias + (size_t)l * 128 + colhalf * 64;
      const CUtensorMap* mO = conv2 ? &tmXo : &tmTo;
      for (int k = 0; k < nseg; k++) {
        const tw::Seg sg = tw::segment(k, nseg, u0, u1);
        const int g = sg.g;
        for (int j = sg.j_lo; j < sg.j_hi; j++, n++) {
          const int bq = g * 2 * NB + (int)rank * NB + quarter * 4;
          const int slot = n & 3;
          mbar_wait(&s.tfull[slot], (uint32_t)(n >> 2) & 1u);
          tcgen05_fence_after();
          uint4 l8[4];   // lo8 mode: this row's 64 low-order bytes of the OUTPUT, filled over the two 32-column steps
          uint32_t* l8w = reinterpret_cast<uint32_t*>(l8);
  #pragma unroll
          for (int sc = 0; sc < 2; sc++) {
            const int col = colhalf * 64 + sc * 32;
            uint32_t v[32];
            tmem_ld32(tmem_base + slot * BN + col + ((uint32_t)(quarter * 32) << 16), v);
            uint4 oh4[4], ol4[4];
            __half2* oh = reinterpret_cast<__half2*>(oh4);
            __half2* ol = reinterpret_cast<__half2*>(ol4);
  #pragma unroll
            for (int jj = 0; jj < 16; jj++) {
              const float2 bb = __ldg(reinterpret_cast<const float2*>(bias_g + sc * 32) + jj);
              const float x0 = fmaxf(__uint_as_float(v[2 * jj]) + bb.x, 0.f);
              const float x1 = fmaxf(__uint_as_float(v[2 * jj + 1]) + bb.y, 0.f);
              const __half2 h = __floats2half2_rn(x0, x1);
              oh[jj] = h;
              if (want_lo) {  // lo = y - hi: hi + lo carries ~22 (fp16 lo) / ~15 (e4m3 lo) significant bits of the skip path
                const float2 hf = __half22float2(h);
                if (lo8) {
                  const uint32_t b2 = tw::cvt_e4m3x2((x0 - hf.x) * tw::LO8_SCALE, (x1 - hf.y) * tw::LO8_SCALE);
                  if (jj & 1) l8w[sc * 8 + (jj >> 1)] |= b2 << 16; else l8w[sc * 8 + (jj >> 1)] = b2;
                } else {
                  ol[jj] = __floats2half2_rn(x0 - hf.x, x1 - hf.y);
                }
              }
            }
            const int nparts = (want_lo && !lo8) ? 2 : 1;
            for (int part = 0; part < nparts; part++) {
              if (lane == 0) tma_store_wait_read<0>();  // the previous store has finished reading the tile
              __syncwarp();
              const uint4* o = part ? ol4 : oh4;
  #pragma unroll
              for (int c = 0; c < 4; c++) *reinterpret_cast<uint4*>(tile + lane * 64 + ((c ^ sw) << 4)) = o[c];
              fence_proxy_async();
              __syncwarp();
              if (lane == 0) { tma_store_4d(part ? &tmXLo : mO, tile, col, 0, j, bq); tma_store_commit(); }
            }
          }
          if (want_lo && lo8) {  // one 32-row x 64-byte tile of e4m3 bytes (channels colhalf*64 .. +63)
            if (lane == 0) tma_store_wait_read<0>();
            __syncwarp();
  #pragma unroll
            for (int c = 0; c < 4; c++) *reinterpret_cast<uint4*>(tile + lane * 64 + ((c ^ sw) << 4)) = l8[c];
            fence_proxy_async();
            __syncwarp();
            if (lane == 0) { tma_store_4d(&tmXL8o, tile, colhalf * 64, 0, j, bq); tma_store_commit(); }
          }
          tcgen05_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive_cluster(&s.tempty[slot], 0);
          // this unit's rows are in memory once the warp's stores have completed: count it for this CTA's producer, and tell
          // the neighbouring pairs when it is one of the two rows they read
          if (lane == 0) {
            tma_store_wait_all();
            fence_proxy_async();
            tw::st_release_shared_s32(&s.stored[warp - 2], n + 1);
            if (g * H + j == u0) tw::red_release_add_u64(done + pair, 1ull);
            if (g * H + j == u1 - 1) tw::red_release_add_u64(done_up + pair, 1ull);
          }
          __syncwarp();
        }
      }
    }
  }
  tcgen05_fence_before();
  __syncthreads();
  cluster_sync_all();
  if (warp == 1) {
    tcgen05_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u) : "memory");
  }
}

// ------------------------------------------------------------------------------------------------
// Stem (round 2): leaf states -> first conv (3x3, C_in -> 128, folded BN, ReLU; K = 9*C_in = 27 for Connect Four, padded
// to one 64-wide K block), ONE kernel, straight from the game's vectorize_state (no host round trip; replaces
// GI.vectorize_state + Flux.batch + convert_input, src/networks/network.jl:310-312).  The im2col rows are never written to HBM: four builder
// warps (one thread per tile row) assemble the 128 x 64 fp16 A tile of the first conv directly in shared memory in the
// SWIZZLE_128B K-major layout the tensor core reads (a row is exactly one 128-byte swizzle row), double buffered
// against the MMA (4 x tcgen05.mma M=128,N=128,K=16 per tile) and the epilogue of the previous tile.  Saves the 15 MB
// im2col write + read and one launch per evaluation (the im2col + GEMM pair took 13 + 17 us at ~2750 leaves).
// ------------------------------------------------------------------------------------------------
template <class G, bool HP = G::HAS_PLANE> struct AzPlane { __device__ static float get(const AzEnv&, int, int, int) { return 0.0f; } };
template <class G> struct AzPlane<G, true> { __device__ static float get(const AzEnv& e, int col, int row, int c) { return G::plane(e, col, row, c); } };
template <class G> __device__ __forceinline__ float az_plane_of(const AzEnv& e, int col, int row, int c) { return AzPlane<G>::get(e, col, row, c); }

namespace st {
constexpr int NUM_THREADS = 320;   // B loader, MMA, 4 builder warps, 4 epilogue warps
constexpr int NBMAX = 12;          // boards a 128-row tile can touch
template <int NX>
struct Smem {
  uint8_t b[128 * 128];            // weights Wt[co][64]
  uint8_t a[2][128 * 128];
  uint8_t epi[4][2048];            // one 32-row x 64-byte store tile per epilogue warp (SWIZZLE_64B)
  float xs[2][NBMAX][NX];
  uint64_t bfull, afull[2], aempty[2], tfull[2], tempty[2];
  uint32_t tmem_base;
  float bias[128];
};
}  // namespace st

template <class G>
__global__ void __launch_bounds__(st::NUM_THREADS, 2)   // two CTAs per SM (71 KB smem, 256 TMEM columns, <= 102 registers each): their latencies overlap
az_k_stem(const AzEnv* __restrict__ envs, const __grid_constant__ CUtensorMap tmW, const __grid_constant__ CUtensorMap tmO, GemmArgs ga, int dense) {
  constexpr int W = G::XW, H = G::XH, C = G::XC, NX = W * H * C, BN = 128, F = 128;
  using SmemT = st::Smem<NX>;
  extern __shared__ uint8_t smem_st[];
  SmemT& s = *reinterpret_cast<SmemT*>((reinterpret_cast<uintptr_t>(smem_st) + 1023) & ~(uintptr_t)1023);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int RS = dense ? W : W + 1, BS = dense ? W * H : (W + 1) * (H + 1);
  if (threadIdx.x == 0) {
    mbar_init(&s.bfull, 1);
    for (int i = 0; i < 2; i++) { mbar_init(&s.afull[i], 128); mbar_init(&s.aempty[i], 1); mbar_init(&s.tfull[i], 1); mbar_init(&s.tempty[i], 4); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (threadIdx.x >= 64 && threadIdx.x - 64 < BN) s.bias[threadIdx.x - 64] = ga.bias[threadIdx.x - 64];
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&s.tmem_base)), "r"((uint32_t)(2 * BN)) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem_base = s.tmem_base;
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  if (warp == 0) {  // the weights do not depend on earlier kernels
    if (elect_one()) { mbar_expect_tx(&s.bfull, 128 * 128); tma_load_2d(s.b, &tmW, &s.bfull, 0, 0); }
    __syncwarp();
  }
  asm volatile("griddepcontrol.wait;" ::: "memory");
  const int n_boards = *ga.n_boards;
  const int rows_used = n_boards * BS;
  const int num_tiles = (rows_used + 127) / 128;

  if (warp == 1) {  // ===== MMA issuer =====
    mbar_wait(&s.bfull, 0);
    int it = 0;
    for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x, it++) {
      const int buf = it & 1;
      const uint32_t ph = (it >> 1) & 1;
      mbar_wait(&s.tempty[buf], ph ^ 1);
      mbar_wait(&s.afull[buf], ph);
      tcgen05_fence_after();
      const uint64_t adesc = umma_desc_sw128(smem_u32(s.a[buf]));
      const uint64_t bdesc = umma_desc_sw128(smem_u32(s.b));
      if (elect_one()) {
#pragma unroll
        for (int k = 0; k < 4; k++)
          umma_f16(tmem_base + buf * BN, adesc + (uint64_t)(k * 2), bdesc + (uint64_t)(k * 2), tc::idesc<BN>(), k ? 1u : 0u);
        umma_commit(&s.aempty[buf]);
        umma_commit(&s.tfull[buf]);
      }
      __syncwarp();
    }
  } else if (warp >= 2 && warp < 6) {  // ===== builders: thread t owns row t of the tile =====
    const int t = threadIdx.x - 64;
    int it = 0;
    for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x, it++) {
      const int buf = it & 1;
      const uint32_t ph = (it >> 1) & 1;
      mbar_wait(&s.aempty[buf], ph ^ 1);
      const int r0 = tile * 128;
      const int b_first = r0 / BS;
      const int b_last = min((r0 + 127) / BS, n_boards - 1);
      if (!G::HAS_PLANE) {
        // vectorize_state of the tile's boards: board slot k is done by lane k / 4 of builder warp k % 4
        const int k = (t & 31) * 4 + (t >> 5);
        if (k <= b_last - b_first && k < st::NBMAX) G::vectorize(envs[b_first + k], s.xs[buf][k]);
        asm volatile("bar.sync 1, 128;" ::: "memory");
      }
      const int r = r0 + t;
      uint4 chunk[8];
      __half* hv = reinterpret_cast<__half*>(chunk);
#pragma unroll
      for (int k = 0; k < 64; k++) hv[k] = __float2half_rn(0.0f);
      if (r < rows_used) {
        const int b = r / BS, rr = r - b * BS, yy = rr / RS, xx = rr - yy * RS;
        if (yy < H && xx < W) {
          const float* x = s.xs[buf][b - b_first];
          AzEnv eb;
          if (G::HAS_PLANE) eb = envs[b];
#pragma unroll
          for (int k = 0; k < 9 * C; k++) {   // k = tap*C + c; Flux Conv is a true convolution: tap (kx,ky) reads (x + 1 - kx, y + 1 - ky)
            const int tap = k / C, c = k % C, ky = tap / 3, kx = tap % 3;
            const int ix = xx + 1 - kx, iy = yy + 1 - ky;
            if (ix >= 0 && ix < W && iy >= 0 && iy < H)
              hv[k] = __float2half_rn(G::HAS_PLANE ? az_plane_of<G>(eb, ix, iy, c) : x[ix + W * iy + W * H * c]);
          }
        }
      }
      uint8_t* row = s.a[buf] + t * 128;
#pragma unroll
      for (int q = 0; q < 8; q++) *reinterpret_cast<uint4*>(row + ((q ^ (t & 7)) << 4)) = chunk[q];
      fence_proxy_async();
      mbar_arrive(&s.afull[buf]);   // (xs[buf] is rewritten two tiles later, i.e. after the next tile's bar.sync: every row is built by then)
    }
  } else if (warp >= 6) {  // ===== epilogue warps 6..9: TMEM lane quarter = warp % 4 =====
    // fp16 rows leave through 32-row x 64-byte SWIZZLE_64B tiles and TMA bulk-tensor stores (a row-per-thread STG epilogue
    // touches 32 different 128-byte lines per warp instruction and is LSU-tag bound: it took 3/4 of the stem's time)
    const int quarter = warp & 3;
    uint8_t* tile = s.epi[quarter];
    const int sw = (lane >> 1) & 3;
    int it = 0;
    for (int tile_i = blockIdx.x; tile_i < num_tiles; tile_i += gridDim.x, it++) {
      const int buf = it & 1;
      const uint32_t ph = (it >> 1) & 1;
      mbar_wait(&s.tfull[buf], ph);
      tcgen05_fence_after();
      const int p0 = tile_i * 128 + quarter * 32;
      const int p = p0 + lane;
      const int rr = p % ga.g.board_rows;
      const bool valid = (p < rows_used) && (rr < ga.g.valid_rows) && ((rr % ga.g.row_stride) != ga.g.wcols);
      const bool in_alloc = p < ga.alloc_rows;
#pragma unroll 1
      for (int c = 0; c < BN / 32; c++) {
        uint32_t v[32];
        tmem_ld32(tmem_base + buf * BN + c * 32 + ((uint32_t)(quarter * 32) << 16), v);
        float x[32];
#pragma unroll
        for (int j = 0; j < 32; j++) x[j] = valid ? fmaxf(__uint_as_float(v[j]) + s.bias[c * 32 + j], 0.0f) : 0.0f;
        if (ga.out32 != nullptr && in_alloc) {
          float4* op = reinterpret_cast<float4*>(ga.out32 + (size_t)p * F + c * 32);
#pragma unroll
          for (int j = 0; j < 8; j++) op[j] = make_float4(x[4 * j], x[4 * j + 1], x[4 * j + 2], x[4 * j + 3]);
        }
        uint4 o[4];
        __half2* oh = reinterpret_cast<__half2*>(o);
#pragma unroll
        for (int j = 0; j < 16; j++) oh[j] = __floats2half2_rn(x[2 * j], x[2 * j + 1]);
        if (lane == 0) tma_store_wait_read<0>();
        __syncwarp();
#pragma unroll
        for (int q = 0; q < 4; q++) *reinterpret_cast<uint4*>(tile + lane * 64 + ((q ^ sw) << 4)) = o[q];
        fence_proxy_async();
        __syncwarp();
        if (lane == 0 && p0 < ga.alloc_rows) { tma_store_2d(&tmO, tile, c * 32, p0); tma_store_commit(); }   // rows past the allocation are clipped
      }
      tcgen05_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&s.tempty[buf]);
    }
    if (lane == 0) tma_store_wait_all();
    __syncwarp();
  }
  tcgen05_fence_before();
  __syncthreads();
  if (warp == 1) {
    tcgen05_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)(2 * BN)) : "memory");
  }
}

// ------------------------------------------------------------------------------------------------
// Head 1x1 convs (round 2): both heads' Conv1x1(128 -> 32) + BatchNorm + ReLU as one N = 64 GEMM over the tower's output rows.
// Unlike the generic GEMM kernel, the 16 KB of weights stay resident (loaded once per CTA), the A ring
// holds four 16 KB stages (two tiles in flight), the fp16 feature rows leave as 2 KB bulk copies (a feature row is 64
// contiguous bytes, so 32 rows of a head are one contiguous chunk), and at 80 KB of shared memory two CTAs share an SM.
// ------------------------------------------------------------------------------------------------
namespace hc {
constexpr int NUM_THREADS = 192, ASTAGES = 4;
struct Smem {
  uint8_t b[2][64 * 128];           // Wt[64 co][2 x 64 k]
  uint8_t a[ASTAGES][128 * 128];
  uint8_t epi[4][2][2048];          // per epilogue warp: policy / value tile, 32 rows x 64 B, linear
  uint64_t bfull, full[ASTAGES], empty[ASTAGES], tfull[2], tempty[2];
  uint32_t tmem_base;
  float bias[64];
};
}  // namespace hc
__device__ __forceinline__ void bulk_store(void* gdst, const void* ssrc, uint32_t bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gdst), "r"(smem_u32(ssrc)), "r"(bytes) : "memory");
}
__global__ void __launch_bounds__(hc::NUM_THREADS, 2)
az_k_head_conv(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmW, GemmArgs ga) {
  using namespace hc;
  constexpr int BN = 64;
  extern __shared__ uint8_t smem_hc[];
  Smem& s = *reinterpret_cast<Smem*>((reinterpret_cast<uintptr_t>(smem_hc) + 1023) & ~(uintptr_t)1023);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    mbar_init(&s.bfull, 1);
    for (int i = 0; i < ASTAGES; i++) { mbar_init(&s.full[i], 1); mbar_init(&s.empty[i], 1); }
    for (int i = 0; i < 2; i++) { mbar_init(&s.tfull[i], 1); mbar_init(&s.tempty[i], 4); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (threadIdx.x >= 64 && threadIdx.x - 64 < BN) s.bias[threadIdx.x - 64] = ga.bias[threadIdx.x - 64];
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&s.tmem_base)), "r"(128u) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem_base = s.tmem_base;
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  if (warp == 0) {  // the weights do not depend on earlier kernels
    if (elect_one()) {
      mbar_expect_tx(&s.bfull, 2 * 64 * 128);
      tma_load_2d(s.b[0], &tmW, &s.bfull, 0, 0);
      tma_load_2d(s.b[1], &tmW, &s.bfull, 64, 0);
    }
    __syncwarp();
  }
  asm volatile("griddepcontrol.wait;" ::: "memory");
  const int rows_used = (*ga.n_boards) * ga.rows_per_board;
  const int num_tiles = (rows_used + 127) / 128;
  if (warp == 0) {
    int stage = 0;
    uint32_t phase = 0;
    for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x)
      for (int kb = 0; kb < 2; kb++) {
        mbar_wait(&s.empty[stage], phase ^ 1);
        if (elect_one()) { mbar_expect_tx(&s.full[stage], 128 * 128); tma_load_2d(s.a[stage], &tmA, &s.full[stage], kb * 64, tile * 128); }
        __syncwarp();
        if (++stage == ASTAGES) { stage = 0; phase ^= 1; }
      }
  } else if (warp == 1) {
    constexpr uint32_t IDESC = (1u << 4) | ((uint32_t)(BN >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
    mbar_wait(&s.bfull, 0);
    int stage = 0, it = 0;
    uint32_t phase = 0;
    for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x, it++) {
      const int acc = it & 1;
      mbar_wait(&s.tempty[acc], (((uint32_t)it >> 1) & 1u) ^ 1u);
      tcgen05_fence_after();
      for (int kb = 0; kb < 2; kb++) {
        mbar_wait(&s.full[stage], phase);
        tcgen05_fence_after();
        const uint64_t adesc = umma_desc_sw128(smem_u32(s.a[stage]));
        const uint64_t bdesc = umma_desc_sw128(smem_u32(s.b[kb]));
        if (elect_one()) {
#pragma unroll
          for (int k = 0; k < 4; k++) umma_f16(tmem_base + acc * BN, adesc + (uint64_t)(k * 2), bdesc + (uint64_t)(k * 2), IDESC, (kb | k) ? 1u : 0u);
          umma_commit(&s.empty[stage]);
          if (kb == 1) umma_commit(&s.tfull[acc]);
        }
        __syncwarp();
        if (++stage == ASTAGES) { stage = 0; phase ^= 1; }
      }
    }
  } else {
    const int quarter = warp & 3;
    int it = 0;
    for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x, it++) {
      const int acc = it & 1;
      mbar_wait(&s.tfull[acc], ((uint32_t)it >> 1) & 1u);
      tcgen05_fence_after();
      const int p0 = tile * 128 + quarter * 32, p = p0 + lane;
      const int rr = p % ga.g.board_rows;
      const bool valid = (p < rows_used) && (rr < ga.g.valid_rows) && ((rr % ga.g.row_stride) != ga.g.wcols);
      if (lane == 0) tma_store_wait_read<0>();   // the previous tile's two copies have left the staging tiles
      __syncwarp();
#pragma unroll
      for (int c = 0; c < 2; c++) {   // c = 0: policy features, 1: value features
        uint32_t v[32];
        tmem_ld32(tmem_base + acc * BN + c * 32 + ((uint32_t)(quarter * 32) << 16), v);
        uint4 o[4];
        __half2* oh = reinterpret_cast<__half2*>(o);
#pragma unroll
        for (int j = 0; j < 16; j++) {
          const float x0 = valid ? fmaxf(__uint_as_float(v[2 * j]) + s.bias[c * 32 + 2 * j], 0.0f) : 0.0f;
          const float x1 = valid ? fmaxf(__uint_as_float(v[2 * j + 1]) + s.bias[c * 32 + 2 * j + 1], 0.0f) : 0.0f;
          oh[j] = __floats2half2_rn(x0, x1);
        }
        uint8_t* t = s.epi[quarter][c] + lane * 64;
#pragma unroll
        for (int q = 0; q < 4; q++) *reinterpret_cast<uint4*>(t + q * 16) = o[q];
      }
      fence_proxy_async();
      __syncwarp();
      if (lane == 0 && p0 + 32 <= ga.alloc_rows) {
        bulk_store(ga.out16a + (size_t)p0 * 32, s.epi[quarter][0], 2048);
        bulk_store(ga.out16b + (size_t)p0 * 32, s.epi[quarter][1], 2048);
        tma_store_commit();
      }
      tcgen05_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&s.tempty[acc]);
    }
    if (lane == 0) tma_store_wait_all();
    __syncwarp();
  }
  tcgen05_fence_before();
  __syncthreads();
  if (warp == 1) {
    tcgen05_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(128u) : "memory");
  }
}

// ------------------------------------------------------------------------------------------------
// Fused head outputs (round 2): the value head's Dense(K -> 128) + relu + Dense(128 -> 1) + tanh and the policy head's
// Dense(K -> A) + softmax + legal-action mask + renormalisation (resnet.jl:75-90, network.jl:264-271) in ONE launch
// instead of two GEMM launches and a finalize kernel: even CTAs run value tiles (N = 128), odd CTAs policy tiles (N = 64,
// A used); the epilogue thread that owns a board row reduces its TMEM row in registers, so the hidden layer and the
// logits never touch HBM.
// ------------------------------------------------------------------------------------------------
struct HeadArgs {
  const int32_t* n_boards;
  int kblocks;            // K / 64
  const float* bias_v;    // [128] value dense bias
  const float* wv2;       // [128]
  const float* bv2;       // [1]
  const float* bias_p;    // [64] policy dense bias (A used)
  float* logit_out;       // parity hook or null
  float* vpre_out;        // parity hook or null
};
template <class G>
__global__ void __launch_bounds__(tc::NUM_THREADS, 1)
az_k_heads_dense(const __grid_constant__ CUtensorMap tmHv, const __grid_constant__ CUtensorMap tmWd, const __grid_constant__ CUtensorMap tmHp,
                 const __grid_constant__ CUtensorMap tmWp, HeadArgs ha, const AzEnv* __restrict__ envs, float* __restrict__ P,
                 float* __restrict__ V, float* __restrict__ Pinv) {
  using namespace tc;
  constexpr int A = G::A;
  using SmemT = Smem<128>;
  extern __shared__ uint8_t smem_hd[];
  SmemT& s = *reinterpret_cast<SmemT*>((reinterpret_cast<uintptr_t>(smem_hd) + 1023) & ~(uintptr_t)1023);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const bool policy = (blockIdx.x & 1) != 0;
  const int BN = policy ? 64 : 128;
  const uint32_t b_bytes = (uint32_t)BN * BK * 2;
  const CUtensorMap* mA = policy ? &tmHp : &tmHv;
  const CUtensorMap* mB = policy ? &tmWp : &tmWd;
  const int kblocks = ha.kblocks;
  if (threadIdx.x == 0) {
    for (int i = 0; i < STAGES; i++) { mbar_init(&s.full[i], 1); mbar_init(&s.empty[i], 1); }
    for (int i = 0; i < 2; i++) { mbar_init(&s.tfull[i], 1); mbar_init(&s.tempty[i], 4); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (threadIdx.x >= 64 && threadIdx.x - 64 < BN) s.bias[threadIdx.x - 64] = (policy ? ha.bias_p : ha.bias_v)[threadIdx.x - 64];
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&s.tmem_base)), "r"(256u) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem_base = s.tmem_base;
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  asm volatile("griddepcontrol.wait;" ::: "memory");
  const int n_boards = *ha.n_boards;
  const int num_tiles = (n_boards + BM - 1) / BM;
  const int first = blockIdx.x >> 1, stride = max(1, (int)gridDim.x >> 1);
  const uint32_t idesc_rt = (1u << 4) | ((uint32_t)(BN >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);

  if (warp == 0) {
    int stage = 0;
    uint32_t phase = 0;
    for (int tile = first; tile < num_tiles; tile += stride) {
      for (int kb = 0; kb < kblocks; kb++) {
        mbar_wait(&s.empty[stage], phase ^ 1);
        if (elect_one()) {
          mbar_expect_tx(&s.full[stage], A_BYTES + b_bytes);
          tma_load_2d(s.a[stage], mA, &s.full[stage], kb * BK, tile * BM);
          tma_load_2d(s.b[stage], mB, &s.full[stage], kb * BK, 0);
        }
        __syncwarp();
        if (++stage == STAGES) { stage = 0; phase ^= 1; }
      }
    }
  } else if (warp == 1) {
    int stage = 0;
    uint32_t phase = 0;
    int it = 0;
    for (int tile = first; tile < num_tiles; tile += stride, it++) {
      const int acc = it & 1;
      mbar_wait(&s.tempty[acc], (((uint32_t)it >> 1) & 1u) ^ 1u);
      tcgen05_fence_after();
      const uint32_t tmem_d = tmem_base + acc * 128;
      for (int kb = 0; kb < kblocks; kb++) {
        mbar_wait(&s.full[stage], phase);
        tcgen05_fence_after();
        const uint64_t adesc = umma_desc_sw128(smem_u32(s.a[stage]));
        const uint64_t bdesc = umma_desc_sw128(smem_u32(s.b[stage]));
        if (elect_one()) {
#pragma unroll
          for (int k = 0; k < BK / 16; k++) umma_f16(tmem_d, adesc + (uint64_t)(k * 2), bdesc + (uint64_t)(k * 2), idesc_rt, (kb | k) ? 1u : 0u);
          umma_commit(&s.empty[stage]);
          if (kb == kblocks - 1) umma_commit(&s.tfull[acc]);
        }
        __syncwarp();
        if (++stage == STAGES) { stage = 0; phase ^= 1; }
      }
    }
  } else {
    const int quarter = warp & 3;
    int it = 0;
    for (int tile = first; tile < num_tiles; tile += stride, it++) {
      const int acc = it & 1;
      mbar_wait(&s.tfull[acc], ((uint32_t)it >> 1) & 1u);
      tcgen05_fence_after();
      const int b = tile * BM + quarter * 32 + lane;
      const bool valid = b < n_boards;
      if (!policy) {  // value: tanh(w2 . relu(W1 h + b1) + b2), summed in column order
        float vacc = 0.0f;
#pragma unroll 1
        for (int c = 0; c < 4; c++) {
          uint32_t v[32];
          tmem_ld32(tmem_base + acc * 128 + c * 32 + ((uint32_t)(quarter * 32) << 16), v);
#pragma unroll
          for (int j = 0; j < 32; j++) vacc += fmaxf(__uint_as_float(v[j]) + s.bias[c * 32 + j], 0.0f) * __ldg(ha.wv2 + c * 32 + j);
        }
        if (valid) {
          const float vpre = vacc + __ldg(ha.bv2);
          V[b] = tanhf(vpre);
          if (ha.vpre_out) ha.vpre_out[b] = vpre;
        }
      } else {  // policy: softmax over all A logits, then mask + renormalise (eps(Float32), network.jl:268)
        uint32_t v[32];
        tmem_ld32(tmem_base + acc * 128 + ((uint32_t)(quarter * 32) << 16), v);
        if (valid) {
          float lg[A], m = -3.0e38f;
#pragma unroll
          for (int a = 0; a < A; a++) { lg[a] = __uint_as_float(v[a]) + s.bias[a]; m = fmaxf(m, lg[a]); }
          if (ha.logit_out) {
#pragma unroll
            for (int a = 0; a < A; a++) ha.logit_out[(size_t)b * A + a] = lg[a];
          }
          float se = 0.0f;
#pragma unroll
          for (int a = 0; a < A; a++) { lg[a] = expf(lg[a] - m); se += lg[a]; }
          const uint32_t legal = G::legal_mask(envs[b]);
          float sp = 0.0f;
#pragma unroll
          for (int a = 0; a < A; a++) { lg[a] = ((legal >> a) & 1u) ? lg[a] / se : 0.0f; sp += lg[a]; }
#pragma unroll
          for (int a = 0; a < A; a++) P[(size_t)b * A + a] = lg[a] / (sp + 1.1920929e-07f);
          if (Pinv) Pinv[b] = 1.0f - sp;
        }
      }
      tcgen05_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&s.tempty[acc]);
    }
  }
  tcgen05_fence_before();
  __syncthreads();
  if (warp == 1) {
    tcgen05_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(256u) : "memory");
  }
}

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------
typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                    const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                    CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static PFN_encodeTiled get_encode_fn() {
  static PFN_encodeTiled fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
      fn = (PFN_encodeTiled)p;
  }
  return fn;
}
// fp16 matrix [outer][inner] with a row pitch in bytes; box = [box_outer][box_inner], SWIZZLE_128B (box_inner = 64 elements)
static int make_map_2d(az_ctx* ctx, CUtensorMap* m, void* base, uint64_t inner, uint64_t outer, uint64_t pitch_bytes,
                       uint32_t box_inner, uint32_t box_outer, CUtensorMapSwizzle swz = CU_TENSOR_MAP_SWIZZLE_128B,
                       CUtensorMapDataType dt = CU_TENSOR_MAP_DATA_TYPE_FLOAT16) {
  PFN_encodeTiled fn = get_encode_fn();
  if (!fn) { ctx->err = "cuTensorMapEncodeTiled not available"; return AZ_ECUDA; }
  cuuint64_t dims[2] = {inner, outer};
  cuuint64_t strides[1] = {pitch_bytes};
  cuuint32_t box[2] = {box_inner, box_outer};
  cuuint32_t es[2] = {1, 1};
  CUresult r = fn(m, dt, 2, base, dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                  swz, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) { ctx->err = "cuTensorMapEncodeTiled failed: " + std::to_string((int)r); return AZ_ECUDA; }
  return AZ_OK;
}

// launch with programmatic stream serialization (PDL): the kernel may start while its predecessor in the stream is
// still draining; it must execute griddepcontrol.wait before touching data the predecessor produces
template <class... KArgs, class... Args>
static cudaError_t launch_pdl(void (*kernel)(KArgs...), int grid, int block, size_t smem, cudaStream_t st, Args... args) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(grid); cfg.blockDim = dim3(block); cfg.dynamicSmemBytes = smem; cfg.stream = st;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at; cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kernel, args...);
}

// ------------------------------------------------------------------------------------------------
// Weight folding ON THE DEVICE (round 2): the Flux-order fp32 parameter blob -> the kernels' fp16 layouts with BatchNorm
// (test mode) folded in, so that a network trained on the same GPU (alphazero.jl_b200/learning.py, or Flux through CUDA.jl)
// hands its parameters over without a host round trip (az_net_load_device); az_net_load uploads the host blob once and
// takes the same path.  Arithmetic = the host fold it replaces, one rounding per operation (no FMA contraction):
//   scale = gamma / sqrt(sigma2 + eps),  W' = fp16(W * scale),  b' = (b - mu) * scale + beta.
// ------------------------------------------------------------------------------------------------
// conv (k x k, Flux W[kx, ky, cin, cout] column-major) -> dst[o * dst_stride + tap * tap_stride + c], tap = ky * k + kx
__global__ void az_k_fold_conv(const float* __restrict__ w, const float* __restrict__ b, const float* __restrict__ bn, int cout, int cin, int k,
                               __half* __restrict__ dst, int dst_stride, int tap_stride, int row0, float* __restrict__ bias_out) {
  const int total = cout * k * k * cin;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    const int c = i % cin, tap = (i / cin) % (k * k), o = i / (cin * k * k);
    const int ky = tap / k, kx = tap % k;
    const float sc = __fdiv_rn(bn[o], __fsqrt_rn(__fadd_rn(bn[3 * cout + o], 1e-5f)));
    dst[(size_t)(row0 + o) * dst_stride + tap * tap_stride + c] = __float2half_rn(__fmul_rn(w[kx + k * (ky + k * (c + (size_t)cin * o))], sc));
    if (c == 0 && tap == 0) bias_out[row0 + o] = __fadd_rn(__fmul_rn(__fsub_rn(b[o], bn[2 * cout + o]), sc), bn[cout + o]);
  }
}
// dense over the flattened (W, H, 32) head features (Flux W[out, in] column-major, in = x + W*y + W*H*c)
//   -> dst[o * KD + (y * RS + x) * 32 + c]
__global__ void az_k_fold_dense(const float* __restrict__ w1, int outs, int nc, int W, int H, int RS, int KD, __half* __restrict__ dst) {
  const int total = outs * nc * H * W;   // nc <= 32 head channels; the destination keeps 32 per position
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    const int o = i % outs, pos = (i / outs) % (W * H), c = i / (outs * W * H);
    const int x = pos % W, y = pos / W;
    dst[(size_t)o * KD + (size_t)(y * RS + x) * 32 + c] = __float2half_rn(w1[o + (size_t)outs * (pos + (size_t)W * H * c)]);
  }
}

template <class G>
struct ResNetImpl : az_net {
  az_resnet_hp hp{};
  static constexpr int F = 128, W = G::XW, H = G::XH, C = G::XC, A = G::A, WH = W * H;
  // activation row layout, fixed at init(): DENSE rows (b*W*H + y*W + x) for the Connect-Four tower kernels
  // (C4_TOWER && num_blocks > 0), otherwise padded NHWC (row stride W+1, one zero row per board) for the generic 9-tap kernel
  bool dense = false;
  int RS = W + 1;                                              // rows per board row
  int BS = (W + 1) * (H + 1);                                  // rows per board
  int VR = (W + 1) * H;                                        // rows of a board up to (excluding) the pad row
  int KP = (W + 1) * H * 32;                                   // policy / value feature length (pad columns carry zero weights)
  int KD = ((W + 1) * H * 32 + 63) / 64 * 64;                  // value-dense K rounded to the 64-wide K block
  // device weights
  __half* d_wstem = nullptr; float* d_bstem = nullptr;   // stem weights Wt[co][64] (k = tap*C + c, zero padded)
  __half* d_wpol = nullptr; float* d_bpol = nullptr;     // policy dense as a GEMM: Wt[64 (A used)][KD]
  CUtensorMap mapWstem{}, mapWpol{}, mapHp{};
  std::vector<__half*> d_wconv; std::vector<float*> d_bconv;   // per-layer views into d_wall / d_ball
  __half* d_wall = nullptr; float* d_ball = nullptr;            // all tower layers: Wt[l][co][tap*F + ci], bias[l][co]
  unsigned long long* d_done = nullptr;                          // persistent tower: per-pair layer counters (never reset)
  CUtensorMap mapWall{};                                         // [L*128][1152] fp16, 64 x 64 boxes
  bool persistent = true;      // AZ_TOWER=layer: one launch per conv layer (the reference kernel) instead of the whole-tower kernel
  size_t smem_tower = 0, smem_stem = 0;
  __half *d_wh = nullptr, *d_wd = nullptr;
  float *d_bh = nullptr, *d_bd = nullptr, *d_wv2 = nullptr, *d_bv2 = nullptr;
  std::vector<CUtensorMap> mapW;
  CUtensorMap mapWh{}, mapWd{};
  // activations (allocated for max_rows on first use)
  int act_boards = 0, alloc_rows = 0, alloc_boards = 0;
  float* d_x32 = nullptr;                 // generic tower: fp32 residual stream
  __half *d_x16 = nullptr, *d_t16 = nullptr, *d_hp = nullptr, *d_hv = nullptr;
  CUtensorMap mapX{}, mapT{}, mapHv{};
  __half* d_xl16 = nullptr;              // Connect-Four tower: low-order part of the block outputs (x = X16 + XL16)
  std::vector<CUtensorMap> mapW2;        // 64co x 64k weight boxes
  // y-row tower: 4-D (channel, x, y, board) views of the dense activations
  CUtensorMap map4X{}, map4T{}, map4XL{};        // loads: box (64 ch, 8 x, 1 y, 16 boards), SWIZZLE_128B, zero fill outside
  CUtensorMap map4Xo{}, map4To{}, map4XLo{};     // stores: box (16 ch, 8 x, 1 y, 4 boards), SWIZZLE_32B (per-layer kernels)
  uint8_t* d_xl8 = nullptr;                        // persistent tower, lo8 mode: low-order part of the block outputs as e4m3(lo * 2^14)
  CUtensorMap map4XL8{}, map4XL8o{};               // u8 views: load box (128 B, 8 x, 1 y, 16 boards) SWIZZLE_128B; store box (64 B, 8 x, 1 y, 4 boards) SWIZZLE_64B
  bool lo8 = true;                                 // AZ_LO=16: keep the low-order part in fp16 (XL16) like the per-layer kernels
  CUtensorMap mapXo64{};                           // stem stores: 2-D [rows][128] fp16, box (32 ch, 32 rows), SWIZZLE_64B
  CUtensorMap map4Xo64{}, map4To64{}, map4XLo64{};  // stores of the persistent kernel: box (32 ch, 8 x, 1 y, 4 boards), SWIZZLE_64B
  static constexpr bool C4_TOWER = (W + 1) == 8 && H == 6;
  size_t smem_yrow = 0;
  ConvGeom geom{};
  bool loaded = false;
  size_t smem128 = 0;
  // profiling: 4 events per evaluation (start, tower begin, tower end, end)
  // The event ring is drained (stream sync + accumulate) whenever it fills, so EVERY evaluation of a profiled pass is
  // counted whatever its length (round 1 truncated at the ring size and overstated the roofline for long passes).
  static constexpr int PROF_SLOTS = 2048;
  bool profiling = false;
  std::vector<cudaEvent_t> pev;
  int64_t prof_evals = 0;                       // evaluations currently in the ring
  double prof_tower_ms = 0, prof_total_ms = 0;  // drained sums
  int64_t prof_drained = 0;
  void prof_drain() {
    cudaStreamSynchronize(ctx->stream);
    for (int64_t i = 0; i < prof_evals; i++) {
      float a = 0, b = 0;
      cudaEventElapsedTime(&a, pev[i * 4 + 1], pev[i * 4 + 2]);
      cudaEventElapsedTime(&b, pev[i * 4 + 0], pev[i * 4 + 3]);
      prof_tower_ms += a; prof_total_ms += b;
    }
    prof_drained += prof_evals;
    prof_evals = 0;
  }

  uint64_t gen = 1;
  uint64_t generation() override { return gen; }
  bool capturable() override { return !profiling && act_boards > 0; }
  int set_profiling(int enable) override {
    if (enable && pev.empty()) {
      pev.resize((size_t)PROF_SLOTS * 4);
      for (auto& e : pev) if (cudaEventCreate(&e) != cudaSuccess) { ctx->err = "cudaEventCreate failed"; return AZ_ECUDA; }
    }
    cudaStreamSynchronize(ctx->stream);
    profiling = enable != 0;
    prof_evals = 0; prof_drained = 0; prof_tower_ms = prof_total_ms = 0;
    return AZ_OK;
  }
  int get_profile(double* tower_ms, int64_t* tower_launches, double* total_ms, int64_t* evals) override {
    prof_drain();
    if (tower_ms) *tower_ms = prof_tower_ms;
    if (tower_launches) *tower_launches = prof_drained * ((dense && persistent) ? 1 : 2 * hp.num_blocks);
    if (total_ms) *total_ms = prof_total_ms;
    if (evals) *evals = prof_drained;
    prof_drained = 0; prof_tower_ms = prof_total_ms = 0;
    return AZ_OK;
  }

  template <class K> int set_smem(K kernel, size_t bytes) {
    cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
    if (e != cudaSuccess) { ctx->err = std::string("cudaFuncSetAttribute(smem): ") + cudaGetErrorString(e); return AZ_ECUDA; }
    return AZ_OK;
  }
  int init() {
    // The kernels are written for 128 tower channels and 32 + 32 head channels.  Narrower networks (the reference's
    // profiling scripts use 64 filters) are the same arithmetic with zero weights and zero biases in the unused channels:
    // ReLU(0) = 0 and adding 0.0f to an fp32 accumulator is exact, so the outputs are those of the narrow network; the
    // padding is written by load_device() when it folds the parameters.  Such a network costs what a 128-filter one costs.
    if (hp.num_filters < 1 || hp.num_filters > F || hp.conv_kernel_size[0] != 3 || hp.conv_kernel_size[1] != 3) {
      ctx->err = "ResNet: this build supports 1 <= num_filters <= 128 and conv_kernel_size = (3, 3)";
      return AZ_EUNSUPPORTED;
    }
    if (hp.num_policy_head_filters < 1 || hp.num_policy_head_filters > 32 || hp.num_value_head_filters < 1 || hp.num_value_head_filters > 32) {
      ctx->err = "ResNet: this build supports 1 <= num_policy_head_filters, num_value_head_filters <= 32";
      return AZ_EUNSUPPORTED;
    }
    if (hp.num_blocks < 0) { ctx->err = "ResNet: num_blocks must be >= 0"; return AZ_EINVAL; }
    dense = C4_TOWER && hp.num_blocks > 0;
    if (dense) { RS = W; BS = W * H; VR = W * H; KP = W * H * 32; KD = (KP + 63) / 64 * 64; }
    geom.row_stride = RS; geom.board_rows = BS; geom.valid_rows = VR; geom.wcols = dense ? RS : W;  // dense: every row is a cell
    for (int ky = 0; ky < 3; ky++)
      for (int kx = 0; kx < 3; kx++) geom.off[ky * 3 + kx] = (1 - ky) * (W + 1) + (1 - kx);
    smem128 = sizeof(tc::Smem<128>) + 1024;
    AZ_TRY2(set_smem(az_k_gemm_tc<128, tc::EPI_CONV1>, smem128));
    AZ_TRY2(set_smem(az_k_gemm_tc<128, tc::EPI_CONV2>, smem128));
    smem_yrow = sizeof(yr::Smem);
    static_assert(sizeof(yr::Smem) <= 232448, "y-row tower kernel exceeds the 227 KB shared-memory limit");
    AZ_TRY2(set_smem(az_k_conv_yrow<tc::EPI_CONV1>, smem_yrow));
    AZ_TRY2(set_smem(az_k_conv_yrow<tc::EPI_CONV2>, smem_yrow));
    smem_tower = sizeof(tw::Smem);
    static_assert(sizeof(tw::Smem) <= 232448, "persistent tower kernel exceeds the 227 KB shared-memory limit");
    AZ_TRY2(set_smem(az_k_tower_yrow, smem_tower));
    smem_stem = sizeof(st::Smem<W * H * C>) + 1024;
    AZ_TRY2(set_smem(az_k_stem<G>, smem_stem));
    AZ_TRY2(set_smem(az_k_heads_dense<G>, smem128));
    AZ_TRY2(set_smem(az_k_head_conv, sizeof(hc::Smem) + 1024));
    // AZ_TOWER=layer and AZ_LO=16 select the per-layer reference form of the Connect-Four tower (see az_k_conv_yrow)
    { const char* e = getenv("AZ_TOWER"); persistent = !(e && e[0] == 'l'); }          // AZ_TOWER=layer
    { const char* e = getenv("AZ_LO"); lo8 = !(e && e[0] == '1'); }                    // AZ_LO=16: fp16 low-order residual part
    if (cudaMalloc((void**)&d_done, 256 * sizeof(unsigned long long)) != cudaSuccess) { cudaGetLastError(); ctx->err = "cudaMalloc (tower flags) failed"; return AZ_ENOMEM; }
    cudaMemset(d_done, 0, 256 * sizeof(unsigned long long));
    return AZ_OK;
  }
  int64_t num_params() override {
    const int npf = hp.num_policy_head_filters, nvf = hp.num_value_head_filters;
    const int64_t Fr = hp.num_filters;
    int64_t n = 0;
    n += 9LL * C * Fr + Fr + 4 * Fr;                                   // stem conv + BN
    n += (int64_t)hp.num_blocks * 2 * (9LL * Fr * Fr + Fr + 4 * Fr);   // blocks
    n += Fr * nvf + nvf + 4 * nvf + (int64_t)WH * nvf * Fr + Fr + Fr + 1;  // vhead
    n += Fr * npf + npf + 4 * npf + (int64_t)WH * npf * A + A;             // phead
    return n;
  }
  template <class T> int up(T** dst, const std::vector<T>& v) {
    cudaError_t e = cudaMalloc((void**)dst, v.size() * sizeof(T));
    if (e != cudaSuccess) { ctx->err = "cudaMalloc (weights) failed"; return AZ_ENOMEM; }
    e = cudaMemcpy(*dst, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice);
    if (e != cudaSuccess) { ctx->err = "cudaMemcpy (weights) failed"; return AZ_ECUDA; }
    return AZ_OK;
  }
  void free_weights() {
    cudaFree(d_wstem); cudaFree(d_bstem);
    cudaFree(d_wall); cudaFree(d_ball); d_wall = nullptr; d_ball = nullptr;
    d_wconv.clear(); d_bconv.clear(); mapW.clear(); mapW2.clear();
    cudaFree(d_wh); cudaFree(d_wd); cudaFree(d_bh); cudaFree(d_bd); cudaFree(d_wv2); cudaFree(d_bv2);
    cudaFree(d_wpol); cudaFree(d_bpol); d_wpol = nullptr; d_bpol = nullptr;
    d_bstem = d_bh = d_bd = d_wv2 = d_bv2 = nullptr; d_wh = d_wd = d_wstem = nullptr;
  }
  void free_act() {
    cudaFree(d_x32); cudaFree(d_x16); cudaFree(d_t16); cudaFree(d_hp); cudaFree(d_hv);
    cudaFree(d_xl16); cudaFree(d_xl8); d_xl8 = nullptr;
    d_x32 = nullptr; d_x16 = d_t16 = d_hp = d_hv = d_xl16 = nullptr;
  }
  ~ResNetImpl() override { free_weights(); free_act(); cudaFree(d_done); for (auto e : pev) cudaEventDestroy(e); }

  // blob -> folded device weights.  Flux order: Conv W[kw,kh,cin,cout] (kw fastest), b; BatchNorm gamma, beta, mu, sigma2;
  // Dense W[out,in] (out fastest), b.  Order: common (stem, blocks), vhead, phead.
  int load(const float* blob, int64_t n) override {
    if (n != num_params()) { ctx->err = "az_net_load: blob has " + std::to_string(n) + " floats, expected " + std::to_string(num_params()); return AZ_EINVAL; }
    float* d_blob = nullptr;
    if (cudaMalloc((void**)&d_blob, (size_t)n * sizeof(float)) != cudaSuccess) { cudaGetLastError(); ctx->err = "cudaMalloc (parameter blob) failed"; return AZ_ENOMEM; }
    if (cudaMemcpy(d_blob, blob, (size_t)n * sizeof(float), cudaMemcpyHostToDevice) != cudaSuccess) {
      cudaGetLastError(); cudaFree(d_blob); ctx->err = "cudaMemcpy (parameter blob) failed"; return AZ_ECUDA;
    }
    const int st = load_device(d_blob, n);
    cudaFree(d_blob);
    return st;
  }
  template <class T> int dzalloc(T** dst, size_t count) {
    if (cudaMalloc((void**)dst, count * sizeof(T)) != cudaSuccess) { cudaGetLastError(); ctx->err = "cudaMalloc (weights) failed"; return AZ_ENOMEM; }
    cudaMemsetAsync(*dst, 0, count * sizeof(T), ctx->stream);
    return AZ_OK;
  }
  // d_blob: DEVICE pointer to the Flux-order parameters.  Flux order: Conv W[kw,kh,cin,cout] (kw fastest), b; BatchNorm gamma,
  // beta, mu, sigma2; Dense W[out,in] (out fastest), b.  Order: common (stem, blocks), vhead, phead.
  int load_device(const float* d_blob, int64_t n) override {
    if (n != num_params()) { ctx->err = "az_net_load_device: blob has " + std::to_string(n) + " floats, expected " + std::to_string(num_params()); return AZ_EINVAL; }
    cudaStream_t st = ctx->stream;
    cudaStreamSynchronize(st);
    gen++;
    free_weights();
    loaded = false;
    const float* q = d_blob;
    const int Fr = hp.num_filters, npf = hp.num_policy_head_filters, nvf = hp.num_value_head_filters;   // real widths; the
    // destination layouts keep F = 128 channels / 32 head channels and start zeroed (dzalloc): unused channels stay zero
    auto grid_for = [](size_t total) { return (int)std::min<size_t>((total + 255) / 256, 4096); };
    {  // stem
      const float* w = q; q += 9 * C * Fr;
      const float* b = q; q += Fr;
      const float* bn = q; q += 4 * Fr;
      static_assert(9 * C <= 64, "stem K must fit one 64-wide K block");
      AZ_TRY2(dzalloc(&d_wstem, (size_t)F * 64)); AZ_TRY2(dzalloc(&d_bstem, (size_t)F));
      az_k_fold_conv<<<grid_for((size_t)Fr * 9 * C), 256, 0, st>>>(w, b, bn, Fr, C, 3, d_wstem, 64, C, 0, d_bstem);
      AZ_TRY2(make_map_2d(ctx, &mapWstem, d_wstem, 64, F, 64 * 2, tc::BK, 128));
    }
    const int L = 2 * hp.num_blocks;
    if (L > 0) {
      AZ_TRY2(dzalloc(&d_wall, (size_t)L * F * 9 * F)); AZ_TRY2(dzalloc(&d_ball, (size_t)L * F));
      AZ_TRY2(make_map_2d(ctx, &mapWall, d_wall, 9 * F, (uint64_t)L * F, 9 * F * 2, tc2::BK, tc2::BNH));
    }
    for (int l = 0; l < L; l++) {
      const float* w = q; q += 9LL * Fr * Fr;
      const float* b = q; q += Fr;
      const float* bn = q; q += 4 * Fr;
      __half* dw = d_wall + (size_t)l * F * 9 * F; float* db = d_ball + (size_t)l * F;   // Wt[co][tap*F + ci]
      az_k_fold_conv<<<grid_for((size_t)Fr * 9 * Fr), 256, 0, st>>>(w, b, bn, Fr, Fr, 3, dw, 9 * F, F, 0, db);
      d_wconv.push_back(dw); d_bconv.push_back(db);
      CUtensorMap m;
      AZ_TRY2(make_map_2d(ctx, &m, dw, 9 * F, F, 9 * F * 2, tc::BK, 128));
      mapW.push_back(m);
      AZ_TRY2(make_map_2d(ctx, &m, dw, 9 * F, F, 9 * F * 2, tc2::BK, tc2::BNH));
      mapW2.push_back(m);
    }
    // head 1x1 convs: rows 0..31 policy filters, 32..63 value filters
    AZ_TRY2(dzalloc(&d_wh, (size_t)64 * F)); AZ_TRY2(dzalloc(&d_bh, (size_t)64));
    {  // vhead: Conv1x1 F->32, BN, Dense(WH*32 -> F), Dense(F -> 1)
      const float* w = q; q += (int64_t)Fr * nvf;
      const float* b = q; q += nvf;
      const float* bn = q; q += 4 * nvf;
      az_k_fold_conv<<<grid_for((size_t)nvf * Fr), 256, 0, st>>>(w, b, bn, nvf, Fr, 1, d_wh, F, F, 32, d_bh);
      const float* w1 = q; q += (int64_t)WH * nvf * Fr;
      const float* b1 = q; q += Fr;
      AZ_TRY2(dzalloc(&d_wd, (size_t)F * KD));   // Wd[o][k'], k' = (y*RS + x)*32 + c; pad positions stay zero
      az_k_fold_dense<<<grid_for((size_t)Fr * nvf * WH), 256, 0, st>>>(w1, Fr, nvf, W, H, RS, KD, d_wd);
      AZ_TRY2(dzalloc(&d_bd, (size_t)F));
      cudaMemcpyAsync(d_bd, b1, Fr * sizeof(float), cudaMemcpyDeviceToDevice, st);
      AZ_TRY2(make_map_2d(ctx, &mapWd, d_wd, KD, F, (uint64_t)KD * 2, tc::BK, 128));
      const float* w2 = q; q += Fr;
      const float* b2 = q; q += 1;
      AZ_TRY2(dzalloc(&d_wv2, (size_t)F)); AZ_TRY2(dzalloc(&d_bv2, (size_t)1));
      cudaMemcpyAsync(d_wv2, w2, Fr * sizeof(float), cudaMemcpyDeviceToDevice, st);
      cudaMemcpyAsync(d_bv2, b2, sizeof(float), cudaMemcpyDeviceToDevice, st);
    }
    {  // phead: Conv1x1 F->32, BN, Dense(WH*32 -> A)
      const float* w = q; q += (int64_t)Fr * npf;
      const float* b = q; q += npf;
      const float* bn = q; q += 4 * npf;
      az_k_fold_conv<<<grid_for((size_t)npf * Fr), 256, 0, st>>>(w, b, bn, npf, Fr, 1, d_wh, F, F, 0, d_bh);
      const float* w1 = q; q += (int64_t)WH * npf * A;
      const float* b1 = q; q += A;
      AZ_TRY2(dzalloc(&d_wpol, (size_t)64 * KD));   // Wt[a][k'], rows >= A and pad positions zero
      az_k_fold_dense<<<grid_for((size_t)A * npf * WH), 256, 0, st>>>(w1, A, npf, W, H, RS, KD, d_wpol);
      AZ_TRY2(dzalloc(&d_bpol, (size_t)64));
      cudaMemcpyAsync(d_bpol, b1, A * sizeof(float), cudaMemcpyDeviceToDevice, st);
      AZ_TRY2(make_map_2d(ctx, &mapWpol, d_wpol, KD, 64, (uint64_t)KD * 2, tc::BK, 64));
    }
    AZ_TRY2(make_map_2d(ctx, &mapWh, d_wh, F, 64, F * 2, tc::BK, 64));
    cudaError_t e = cudaStreamSynchronize(st);   // the caller may free / overwrite d_blob as soon as this returns
    if (e == cudaSuccess) e = cudaGetLastError();
    if (e != cudaSuccess) { ctx->err = std::string("az_net_load_device: ") + cudaGetErrorString(e); return AZ_ECUDA; }
    ctx->launches += 3 + L + 4;
    loaded = true;
    return AZ_OK;
  }
  template <class T> int dmalloc(T** p, size_t n) {
    if (cudaMalloc((void**)p, n * sizeof(T)) != cudaSuccess) { ctx->err = "cudaMalloc (activations) failed"; cudaGetLastError(); return AZ_ENOMEM; }
    cudaMemsetAsync(*p, 0, n * sizeof(T), ctx->stream);
    return AZ_OK;
  }
  // dense activations [boards][H][W][128] fp16 as a 4-D tensor (channel, x, y, board); box = (bc, bx, 1, bb)
  int make_map_4d(az_ctx* c, CUtensorMap* m, void* base, int boards, uint32_t bc, uint32_t bx, uint32_t bb, CUtensorMapSwizzle swz,
                  bool u8 = false) {
    PFN_encodeTiled fn = get_encode_fn();
    if (!fn) { c->err = "cuTensorMapEncodeTiled not available"; return AZ_ECUDA; }
    const cuuint64_t eb = u8 ? 1 : 2;
    cuuint64_t dims[4] = {(cuuint64_t)F, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)boards};
    cuuint64_t strides[3] = {(cuuint64_t)F * eb, (cuuint64_t)W * F * eb, (cuuint64_t)W * H * F * eb};
    cuuint32_t box[4] = {bc, bx, 1, bb};
    cuuint32_t es[4] = {1, 1, 1, 1};
    CUresult r = fn(m, u8 ? CU_TENSOR_MAP_DATA_TYPE_UINT8 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 4, base, dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE, swz,
                    CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { c->err = "cuTensorMapEncodeTiled (4-D) failed: " + std::to_string((int)r); return AZ_ECUDA; }
    return AZ_OK;
  }
  int ensure_act(int max_boards) {
    if (max_boards <= act_boards) return AZ_OK;
    cudaStreamSynchronize(ctx->stream);
    gen++;
    free_act();
    alloc_rows = ((max_boards * BS + 127) / 128) * 128 + 128;
    alloc_boards = alloc_rows / BS;
    if (!dense) AZ_TRY2(dmalloc(&d_x32, (size_t)alloc_rows * F));
    else AZ_TRY2(dmalloc(&d_xl16, (size_t)alloc_rows * F));
    AZ_TRY2(dmalloc(&d_x16, (size_t)alloc_rows * F));
    AZ_TRY2(dmalloc(&d_t16, (size_t)alloc_rows * F)); AZ_TRY2(dmalloc(&d_hp, (size_t)alloc_rows * 32));
    AZ_TRY2(dmalloc(&d_hv, (size_t)alloc_rows * 32));
    AZ_TRY2(make_map_2d(ctx, &mapHp, d_hp, (uint64_t)BS * 32, alloc_boards, (uint64_t)BS * 32 * 2, tc::BK, tc::BM));
    AZ_TRY2(make_map_2d(ctx, &mapX, d_x16, F, alloc_rows, F * 2, tc::BK, tc::BM));
    AZ_TRY2(make_map_2d(ctx, &mapT, d_t16, F, alloc_rows, F * 2, tc::BK, tc::BM));
    AZ_TRY2(make_map_2d(ctx, &mapXo64, d_x16, F, alloc_rows, F * 2, 32, 32, CU_TENSOR_MAP_SWIZZLE_64B));
    AZ_TRY2(make_map_2d(ctx, &mapHv, d_hv, (uint64_t)BS * 32, alloc_boards, (uint64_t)BS * 32 * 2, tc::BK, tc::BM));
    if (dense) {
      const CUtensorMapSwizzle s128 = CU_TENSOR_MAP_SWIZZLE_128B, s32 = CU_TENSOR_MAP_SWIZZLE_32B;
      AZ_TRY2(make_map_4d(ctx, &map4X, d_x16, alloc_boards, 64, 8, yr::NBOARD, s128));
      AZ_TRY2(make_map_4d(ctx, &map4T, d_t16, alloc_boards, 64, 8, yr::NBOARD, s128));
      AZ_TRY2(make_map_4d(ctx, &map4XL, d_xl16, alloc_boards, 64, 8, yr::NBOARD, s128));
      AZ_TRY2(make_map_4d(ctx, &map4Xo, d_x16, alloc_boards, 16, 8, 4, s32));
      AZ_TRY2(make_map_4d(ctx, &map4To, d_t16, alloc_boards, 16, 8, 4, s32));
      AZ_TRY2(make_map_4d(ctx, &map4XLo, d_xl16, alloc_boards, 16, 8, 4, s32));
      const CUtensorMapSwizzle s64 = CU_TENSOR_MAP_SWIZZLE_64B;
      AZ_TRY2(make_map_4d(ctx, &map4Xo64, d_x16, alloc_boards, 32, 8, 4, s64));
      AZ_TRY2(make_map_4d(ctx, &map4To64, d_t16, alloc_boards, 32, 8, 4, s64));
      AZ_TRY2(make_map_4d(ctx, &map4XLo64, d_xl16, alloc_boards, 32, 8, 4, s64));
      AZ_TRY2(dmalloc(&d_xl8, (size_t)alloc_rows * F));
      AZ_TRY2(make_map_4d(ctx, &map4XL8, d_xl8, alloc_boards, 128, 8, yr::NBOARD, s128, true));
      AZ_TRY2(make_map_4d(ctx, &map4XL8o, d_xl8, alloc_boards, 64, 8, 4, s64, true));
    }
    act_boards = max_boards;
    return AZ_OK;
  }
  // the persistent whole-tower kernel: cooperative launch (all CTA pairs co-resident: its neighbour spin-waits must never
  // wait for a pair that cannot be scheduled, e.g. when two engines share a GPU) + programmatic stream serialization
  int launch_tower(int grid, cudaStream_t st, const GemmArgs& ga) {
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3(grid); cfg.blockDim = dim3(yr::NUM_THREADS); cfg.dynamicSmemBytes = smem_tower; cfg.stream = st;
    cudaLaunchAttribute at[2];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization; at[0].val.programmaticStreamSerializationAllowed = 1;
    at[1].id = cudaLaunchAttributeCooperative; at[1].val.cooperative = 1;
    cfg.attrs = at; cfg.numAttrs = 2;
    const int L = 2 * hp.num_blocks;
    GemmArgs g2 = ga;
    g2.lo8 = lo8 ? 1 : 0;
    cudaError_t e = cudaLaunchKernelEx(&cfg, az_k_tower_yrow, map4X, map4T, map4XL, mapWall, map4Xo64, map4To64, map4XLo64, map4XL8, map4XL8o, g2, L, d_done);
    if (e != cudaSuccess) { ctx->err = std::string("persistent tower launch: ") + cudaGetErrorString(e); cudaGetLastError(); return AZ_ECUDA; }
    return AZ_OK;
  }
  int eval(const AzEnv* envs, const int32_t* n_rows, int max_rows, float* P, float* V) override {
    return eval_with_pinv(envs, n_rows, max_rows, P, V, nullptr);
  }
  int reserve(int max_rows) override { return ensure_act(max_rows); }
  int eval_with_pinv(const AzEnv* envs, const int32_t* n_rows, int max_rows, float* P, float* V, float* Pinv) override {
    if (!loaded) { ctx->err = "ResNet: az_net_load must be called before the network is used"; return AZ_ESTATE; }
    AZ_TRY2(ensure_act(max_rows));
    cudaStream_t st = ctx->stream;
    if (profiling && prof_evals == PROF_SLOTS) prof_drain();
    const bool prof = profiling;
    cudaEvent_t* pe = prof ? &pev[(size_t)prof_evals * 4] : nullptr;
    if (prof) cudaEventRecord(pe[0], st);
    const int row_tiles = (max_rows * BS + tc::BM - 1) / tc::BM;
    GemmArgs ga{};
    ga.n_boards = n_rows; ga.g = geom; ga.alloc_rows = alloc_rows; ga.rows_per_board = BS;
    ga.bias = d_bstem; ga.out16a = d_x16; ga.out32 = dense ? nullptr : d_x32;
    launch_pdl(az_k_stem<G>, std::min(row_tiles, 2 * ctx->num_sms), st::NUM_THREADS, smem_stem, st, envs, mapWstem, mapXo64, ga, dense ? 1 : 0);
    if (prof) cudaEventRecord(pe[1], st);
    const int grid_yr = ctx->num_sms & ~1;  // persistent: one CTA pair per SM pair, balanced unit ranges (idle pairs exit)
    if (dense && persistent) {
      ga.bias = d_ball;
      AZ_TRY2(launch_tower(grid_yr, st, ga));
    }
    for (int blk = 0; dense && !persistent && blk < hp.num_blocks; blk++) {
      ga.bias = d_bconv[2 * blk]; ga.res_lo = 0;
      if (blk > 0) launch_pdl(az_k_conv_yrow<tc::EPI_CONV1>, grid_yr, yr::NUM_THREADS, smem_yrow, st, map4X, mapW2[2 * blk], map4To, map4XLo, map4X, map4XL, ga);
      else az_k_conv_yrow<tc::EPI_CONV1><<<grid_yr, yr::NUM_THREADS, smem_yrow, st>>>(map4X, mapW2[2 * blk], map4To, map4XLo, map4X, map4XL, ga);
      ga.bias = d_bconv[2 * blk + 1];
      ga.res_lo = blk > 0 ? 1 : 0;  // block 0: the residual is the fp16 stem output, no low-order part yet
      launch_pdl(az_k_conv_yrow<tc::EPI_CONV2>, grid_yr, yr::NUM_THREADS, smem_yrow, st, map4T, mapW2[2 * blk + 1], map4Xo, map4XLo, map4X, map4XL, ga);
    }
    const int grid = std::min(row_tiles, ctx->num_sms);
    for (int blk = 0; !dense && blk < hp.num_blocks; blk++) {
      ga.kblocks = 18; ga.bias = d_bconv[2 * blk]; ga.out16a = d_t16;
      az_k_gemm_tc<128, tc::EPI_CONV1><<<grid, tc::NUM_THREADS, smem128, st>>>(mapX, mapW[2 * blk], ga);
      ga.bias = d_bconv[2 * blk + 1]; ga.resid32 = d_x32; ga.out32 = d_x32; ga.out16a = d_x16;
      az_k_gemm_tc<128, tc::EPI_CONV2><<<grid, tc::NUM_THREADS, smem128, st>>>(mapT, mapW[2 * blk + 1], ga);
    }
    if (prof) cudaEventRecord(pe[2], st);
    // heads: both 1x1 convs (N = 64), then the value / policy dense layers and outputs
    ga.bias = d_bh; ga.out16a = d_hp; ga.out16b = d_hv;
    launch_pdl(az_k_head_conv, std::min(row_tiles, 2 * ctx->num_sms), hc::NUM_THREADS, sizeof(hc::Smem) + 1024, st, mapX, mapWh, ga);
    const int board_tiles = (max_rows + tc::BM - 1) / tc::BM;
    HeadArgs ha{n_rows, KD / 64, d_bd, d_wv2, d_bv2, d_bpol, dbg_logit, dbg_vpre};
    const int hgrid = 2 * std::max(1, std::min(board_tiles, ctx->num_sms / 2));
    launch_pdl(az_k_heads_dense<G>, hgrid, tc::NUM_THREADS, smem128, st, mapHv, mapWd, mapHp, mapWpol, ha, envs, P, V, Pinv);
    if (prof) { cudaEventRecord(pe[3], st); prof_evals++; }
    ctx->launches += 3 + ((dense && persistent) ? 1 : 2 * hp.num_blocks);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) { ctx->err = std::string("network launch: ") + cudaGetErrorString(e); return AZ_ECUDA; }
    return AZ_OK;
  }
};

az_net* az_make_resnet(az_ctx* ctx, int game, const az_resnet_hp* hp, int* status) {
  az_net* n = nullptr;
  int st = AZ_OK;
  auto mk = [&](auto* impl) {
    impl->ctx = ctx; impl->kind = AZ_NET_RESNET; impl->game = game; impl->hp = *hp;
    st = impl->init();
    if (st != AZ_OK) { delete impl; return (az_net*)nullptr; }
    return (az_net*)impl;
  };
  switch (game) {
    case 0: n = mk(new ResNetImpl<GameC4>()); break;
    case 1: n = mk(new ResNetImpl<GameTTT>()); break;
    case 2: n = mk(new ResNetImpl<GameMancala>()); break;
    case 3: n = mk(new ResNetImpl<GameGW>()); break;
    default: ctx->err = "az_net_create_resnet: unknown game"; st = AZ_EINVAL;
  }
  *status = st;
  return n;
}

// ------------------------------------------------------------------------------------------------
// SimpleNet (src/networks/architectures/simplenet.jl:37-64): dense two-head MLP, fp32 on CUDA cores (0.1-0.7 MFLOP per
// leaf: launch-latency bound, one fused kernel).  BatchNorm (test mode) is folded into the preceding Dense at load.
// ------------------------------------------------------------------------------------------------
struct MlpLayer { const float* w; const float* b; int in, out, relu; };
struct MlpArgs {
  MlpLayer common[10]; int n_common;
  MlpLayer vhead[6]; int n_vhead;
  MlpLayer phead[6]; int n_phead;
  int width;
};
template <int NB>
__device__ __forceinline__ void mlp_layer(const MlpLayer& L, const float* __restrict__ xin, int xstride, float* __restrict__ xout,
                                          int ostride, int nb) {
  for (int o = threadIdx.x; o < L.out; o += blockDim.x) {
    float acc[NB];
#pragma unroll
    for (int j = 0; j < NB; j++) acc[j] = L.b[o];
    for (int i = 0; i < L.in; i++) {
      const float w = L.w[(size_t)o + (size_t)L.out * i];  // Flux Dense W[out,in], column-major: coalesced over o
#pragma unroll
      for (int j = 0; j < NB; j++) acc[j] += w * xin[j * xstride + i];
    }
#pragma unroll
    for (int j = 0; j < NB; j++)
      if (j < nb) xout[j * ostride + o] = L.relu ? fmaxf(acc[j], 0.0f) : acc[j];
  }
  __syncthreads();
}
template <class G, int NB>
__global__ void __launch_bounds__(256) az_k_simplenet(const AzEnv* __restrict__ envs, const int32_t* __restrict__ n_boards, MlpArgs m,
                                                      float* __restrict__ P, float* __restrict__ V, float* __restrict__ Pinv,
                                                      float* __restrict__ logit_out, float* __restrict__ vpre_out) {
  constexpr int A = G::A, NX = G::XW * G::XH * G::XC, MAXW = 256;
  __shared__ float x0[NB][NX];
  __shared__ float ha[NB][MAXW], hb[NB][MAXW], hc[NB][MAXW];
  __shared__ float outp[NB][A + 1];
  const int b0 = blockIdx.x * NB;
  const int nb = min(NB, *n_boards - b0);
  if (nb <= 0) return;
  for (int j = 0; j < NB; j++) {
    if (threadIdx.x == j && j < nb) G::vectorize(envs[b0 + j], x0[j]);
    if (j >= nb) for (int i = threadIdx.x; i < NX; i += blockDim.x) x0[j][i] = 0.0f;
  }
  __syncthreads();
  // common trunk: ping-pong ha <-> hb
  float* cur = &ha[0][0];
  float* nxt = &hb[0][0];
  mlp_layer<NB>(m.common[0], &x0[0][0], NX, cur, MAXW, NB);
  for (int l = 1; l < m.n_common; l++) {
    mlp_layer<NB>(m.common[l], cur, MAXW, nxt, MAXW, NB);
    float* t = cur; cur = nxt; nxt = t;
  }
  float* trunk = cur;           // keep the trunk output; heads use the other two buffers
  float* s1 = nxt;
  float* s2 = &hc[0][0];
  // value head
  const float* in = trunk;
  for (int l = 0; l < m.n_vhead - 1; l++) {
    float* o = (l & 1) ? s2 : s1;
    mlp_layer<NB>(m.vhead[l], in, MAXW, o, MAXW, NB);
    in = o;
  }
  {
    const MlpLayer& L = m.vhead[m.n_vhead - 1];  // Dense(width, 1, tanh)
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    for (int j = warp; j < nb; j += (blockDim.x >> 5)) {
      float acc = 0.0f;
      for (int i = lane; i < L.in; i += 32) acc += L.w[i] * in[j * MAXW + i];
#pragma unroll
      for (int off = 16; off >= 1; off >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, off);
      if (lane == 0) { outp[j][A] = tanhf(acc + L.b[0]); if (vpre_out) vpre_out[b0 + j] = acc + L.b[0]; }
    }
  }
  __syncthreads();
  // policy head
  in = trunk;
  for (int l = 0; l < m.n_phead - 1; l++) {
    float* o = (l & 1) ? s2 : s1;
    mlp_layer<NB>(m.phead[l], in, MAXW, o, MAXW, NB);
    in = o;
  }
  mlp_layer<NB>(m.phead[m.n_phead - 1], in, MAXW, &outp[0][0], A + 1, nb);  // logits (relu = 0), A outputs per board
  if (threadIdx.x < nb) {
    const int j = threadIdx.x, row = b0 + j;
    float lg[A], mx = -3.0e38f;
#pragma unroll
    for (int a = 0; a < A; a++) { lg[a] = outp[j][a]; mx = fmaxf(mx, lg[a]); }
    if (logit_out) {
#pragma unroll
      for (int a = 0; a < A; a++) logit_out[(size_t)row * A + a] = lg[a];
    }
    float se = 0.0f;
#pragma unroll
    for (int a = 0; a < A; a++) { lg[a] = expf(lg[a] - mx); se += lg[a]; }
    const uint32_t legal = G::legal_mask(envs[row]);
    float sp = 0.0f;
#pragma unroll
    for (int a = 0; a < A; a++) { lg[a] = ((legal >> a) & 1u) ? lg[a] / se : 0.0f; sp += lg[a]; }
#pragma unroll
    for (int a = 0; a < A; a++) P[(size_t)row * A + a] = lg[a] / (sp + 1.1920929e-07f);
    V[row] = outp[j][A];
    if (Pinv) Pinv[row] = 1.0f - sp;
  }
}

template <class G>
struct SimpleNetImpl : az_net {
  az_simplenet_hp hp{};
  static constexpr int NX = G::XW * G::XH * G::XC, A = G::A, NB = 4;
  std::vector<float*> bufs;
  MlpArgs margs{};
  bool loaded = false;
  uint64_t gen = 1;
  uint64_t generation() override { return gen; }
  int init() {
    if (hp.width < 1 || hp.width > 256) { ctx->err = "SimpleNet: this build supports 1 <= width <= 256"; return AZ_EUNSUPPORTED; }
    if (hp.depth_common < 0 || hp.depth_common > 9 || hp.depth_phead < 0 || hp.depth_phead > 5 || hp.depth_vhead < 0 || hp.depth_vhead > 5) {
      ctx->err = "SimpleNet: depth_common <= 9, depth_phead/depth_vhead <= 5"; return AZ_EUNSUPPORTED;
    }
    return AZ_OK;
  }
  int64_t dense_size(int in, int out) const { return (int64_t)in * out + out + (hp.use_batch_norm ? 4 * out : 0); }
  int64_t num_params() override {
    const int w = hp.width;
    int64_t n = dense_size(NX, w) + (int64_t)hp.depth_common * dense_size(w, w);
    n += (int64_t)hp.depth_vhead * dense_size(w, w) + ((int64_t)w + 1);
    n += (int64_t)hp.depth_phead * dense_size(w, w) + ((int64_t)w * A + A);
    return n;
  }
  void free_all() { for (auto p : bufs) cudaFree(p); bufs.clear(); }
  ~SimpleNetImpl() override { free_all(); }
  int upload(const std::vector<float>& v, const float** out) {
    float* d = nullptr;
    if (cudaMalloc((void**)&d, v.size() * sizeof(float)) != cudaSuccess) { ctx->err = "cudaMalloc (weights) failed"; return AZ_ENOMEM; }
    cudaMemcpy(d, v.data(), v.size() * sizeof(float), cudaMemcpyHostToDevice);
    bufs.push_back(d);
    *out = d;
    return AZ_OK;
  }
  // make_dense (simplenet.jl:39-47): Dense(in,out) [+ BatchNorm(out, relu)] or Dense(in,out,relu)
  int take_dense(const float*& q, int in, int out, bool hidden, MlpLayer* L) {
    std::vector<float> w(q, q + (size_t)in * out); q += (size_t)in * out;
    std::vector<float> b(q, q + out); q += out;
    if (hidden && hp.use_batch_norm) {
      const float* bn = q; q += 4 * out;
      for (int o = 0; o < out; o++) {
        const float sc = bn[o] / std::sqrt(bn[3 * out + o] + 1e-5f);
        for (int i = 0; i < in; i++) w[(size_t)o + (size_t)out * i] *= sc;
        b[o] = (b[o] - bn[2 * out + o]) * sc + bn[out + o];
      }
    }
    L->in = in; L->out = out; L->relu = hidden ? 1 : 0;
    AZ_TRY2(upload(w, &L->w));
    AZ_TRY2(upload(b, &L->b));
    return AZ_OK;
  }
  int load(const float* blob, int64_t n) override {
    if (n != num_params()) { ctx->err = "az_net_load: blob has " + std::to_string(n) + " floats, expected " + std::to_string(num_params()); return AZ_EINVAL; }
    cudaStreamSynchronize(ctx->stream);
    gen++;
    free_all();
    const float* q = blob;
    const int w = hp.width;
    margs = MlpArgs{};
    margs.width = w;
    AZ_TRY2(take_dense(q, NX, w, true, &margs.common[0]));
    for (int l = 0; l < hp.depth_common; l++) AZ_TRY2(take_dense(q, w, w, true, &margs.common[1 + l]));
    margs.n_common = 1 + hp.depth_common;
    for (int l = 0; l < hp.depth_vhead; l++) AZ_TRY2(take_dense(q, w, w, true, &margs.vhead[l]));
    AZ_TRY2(take_dense(q, w, 1, false, &margs.vhead[hp.depth_vhead]));
    margs.n_vhead = hp.depth_vhead + 1;
    for (int l = 0; l < hp.depth_phead; l++) AZ_TRY2(take_dense(q, w, w, true, &margs.phead[l]));
    AZ_TRY2(take_dense(q, w, A, false, &margs.phead[hp.depth_phead]));
    margs.n_phead = hp.depth_phead + 1;
    loaded = true;
    return AZ_OK;
  }
  int eval(const AzEnv* envs, const int32_t* n_rows, int max_rows, float* P, float* V) override {
    return eval_with_pinv(envs, n_rows, max_rows, P, V, nullptr);
  }
  int eval_with_pinv(const AzEnv* envs, const int32_t* n_rows, int max_rows, float* P, float* V, float* Pinv) override {
    if (!loaded) { ctx->err = "SimpleNet: az_net_load must be called before the network is used"; return AZ_ESTATE; }
    az_k_simplenet<G, NB><<<(max_rows + NB - 1) / NB, 256, 0, ctx->stream>>>(envs, n_rows, margs, P, V, Pinv, dbg_logit, dbg_vpre);
    ctx->launches++;
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) { ctx->err = std::string("SimpleNet launch: ") + cudaGetErrorString(e); return AZ_ECUDA; }
    return AZ_OK;
  }
};

az_net* az_make_simplenet(az_ctx* ctx, int game, const az_simplenet_hp* hp, int* status) {
  az_net* n = nullptr;
  int st = AZ_OK;
  auto mk = [&](auto* impl) {
    impl->ctx = ctx; impl->kind = AZ_NET_SIMPLENET; impl->game = game; impl->hp = *hp;
    st = impl->init();
    if (st != AZ_OK) { delete impl; return (az_net*)nullptr; }
    return (az_net*)impl;
  };
  switch (game) {
    case 0: n = mk(new SimpleNetImpl<GameC4>()); break;
    case 1: n = mk(new SimpleNetImpl<GameTTT>()); break;
    case 2: n = mk(new SimpleNetImpl<GameMancala>()); break;
    case 3: n = mk(new SimpleNetImpl<GameGW>()); break;
    default: ctx->err = "az_net_create_simplenet: unknown game"; st = AZ_EINVAL;
  }
  *status = st;
  return n;
}
