// conv_tc.cu — tcgen05 / TMEM / TMA implicit-GEMM convolution for sm_100a, fp32-grade through a THREE-PRODUCT SPLIT.
//
// fprop / dgrad / attention GEMMs (conv_tc_ps_kernel): 3 x FP16.  Every operand is scaled by a power of two taken from its "amax slot"
// (an upper bound of max|v|: dp_amax for activations / gradients, dp_pack_conv_weight_tc for weights) so that |s*v| < 2^14, then
//     s*v = hi + lo,   hi = fp16(s*v) (11 significant bits),  lo' = fp16((s*v - hi) * 2^11)            (22 bits kept, as 3xTF32 does)
//     x*w ~= [hi(x)*hi(w)] + 2^-11 * [hi(x)*lo'(w) + lo'(x)*hi(w)]
// with both brackets accumulated in fp32 in TMEM (main | correction accumulator) by tcgen05.mma kind::f16 — twice the rate of
// kind::tf32 and half the shared-memory operand bytes, which is what bounded the 3xTF32 kernel (profiles/r02_experiments.md).  Elements
// more than 2^28 below the tensor's maximum lose RELATIVE precision (absolute error <= 2^-50 of the maximum): below fp32 round-off of any
// sum they take part in.
// The weight gradient (wgrad_tc_kernel) uses the same split with both operands scaled by their own slots.
//
// GEMM view: M = N*H*W output pixels (tile of 128 = one TMA box of the NHWC activation), N = output channels, K = taps x input
// channels, one pipeline stage = (one tap, 64 channels).  The activation box is im2col-free: the tap shift is a coordinate offset,
// image borders are TMA out-of-bounds zero fill, stride 2 is a TMA element stride.
//
// Kernels:
//   conv_tc_ps_kernel     fprop / dgrad / NT GEMM: persistent (1 CTA per SM loops over (tile, K split) work items), the raw fp32 A boxes
//                         are split IN PLACE into fp16 hi | lo' tiles by 4 warps, B = pre-split fp16 weights by TMA, 3 x 64 KB stages,
//                         two TMEM accumulator sets (the epilogue of tile i overlaps the main loop of tile i+1), and
//                         a_hi x [b_hi | b_lo'] issued as ONE N=256 instruction into [main | correction]
//   splitk_epilogue_kernel  fixed-order sum of the K splits + the epilogue (small-M launches)
//   wgrad_tc_kernel       weight gradient: dY^T split into TMEM (TS mode), X split in place in shared memory, both MN-major, 64-pixel
//                         stages, split-K over pixels
//   pack / split / transpose helpers; dp_gemm_nt_tc runs the attention GEMMs on the persistent kernel.
// History (git tags): `lab-kernels-r01` round-1 experimental variants; `lab-pair-kernel-r02` the cta_group::2 CTA-pair kernel (correct,
// 1.4x slower); `tf32x3-r02` the all-3xTF32 build this file replaced.
#include <cuda.h>
#include <cuda_fp16.h>
#include <mutex>
#include "common.cuh"

namespace {

constexpr int BM = 128, BK = 64;          // pixel tile, K elements (channels of one tap) per pipeline stage
constexpr int A_BYTES = BM * 32 * 4;      // 16 KB: one raw fp32 TMA box of 32 channels = one fp16 tile of 64 channels

struct TcParams {
  int Nimg, H, W;
  int Nout;            // GEMM N (valid output channels)
  int kchunks;         // ceil(Kg / 64)
  int bw, bh, bn, tiles_w, tiles_h;
  float* y; long long ldy;
  const float* bias;
  const float* rowadd; long long ld_rowadd;
  const float* residual; long long ld_res;
  int accumulate;
  int vec4;            // all epilogue pointers / strides are 16-byte aligned
  // generalised tap table (stride-2 dgrad runs as 4 parity classes with 1/2/2/4 taps each) and output pixel mapping
  int ntaps;
  signed char dh[9], dw[9], wt[9];
  int os, oa, ob, Ho, Wo;   // output pixel = (p*os + oa, q*os + ob) on an [Ho][Wo] grid
  int in_stride;            // strided fprop: input pixel = in_stride * output pixel + tap offset (the A map traverses W, H with that stride)
  float alpha;              // epilogue scale of the accumulator (attention logits); 1 for convolutions
  int b_from_img;           // batched GEMM: the B tile index is the tile's image (bn == 1) instead of a filter tap
  const uint32_t* amax_a;   // amax slots of the A operand (activation / gradient view) and of the B operand (weights / split activation)
  const uint32_t* amax_b;
  uint32_t* amax_out;       // optional amax slot of the output tensor
  // split-K (persistent kernel, launches with fewer tiles than half the SMs: the 4x4 / 8x8 / 16x16 levels): work item = (tile, K split);
  // a split walks `it_per_split` pipeline stages of the tile and writes its raw accumulator to ws[split][row][channel]
  // (row = tile_m * 128 + TMEM lane, pitch ws_ld); splitk_epilogue_kernel sums the splits in fixed order and applies the epilogue
  int ksplit, it_per_split;
  float* ws; long long ws_split_stride; int ws_ld;
  int ld_split;             // pre-split A (conv_tc_ps_kernel<false, true>): fp16 elements from a pixel's hi channels to its lo' channels
};

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  uint32_t done;
  do {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done)
        : "r"(bar), "r"(parity)
        : "memory");
  } while (!done);
}
__device__ __forceinline__ void tma_load_4d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1, int c2, int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
      ::"r"(dst), "l"(reinterpret_cast<uint64_t>(map)), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}
__device__ __forceinline__ void tma_load_3d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
      ::"r"(dst), "l"(reinterpret_cast<uint64_t>(map)), "r"(bar), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
// K-major, 128B-swizzled operand tile descriptor (cute::UMMA::SmemDescriptor): start>>4 | LBO(1)<<16 | SBO(1024B>>4)<<32
// | version(1)<<46 | layout SWIZZLE_128B(2)<<61
__device__ __forceinline__ uint64_t umma_desc(uint32_t saddr) {
  return (uint64_t)((saddr & 0x3FFFF) >> 4) | (1ull << 16) | (64ull << 32) | (1ull << 46) | (2ull << 61);
}
__device__ __forceinline__ void umma_f16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t acc) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(acc)
      : "memory");
}
// A operand from TENSOR memory (packed fp16 pairs, 8 columns per 16-element K step)
__device__ __forceinline__ void umma_f16_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t bdesc, uint32_t idesc, uint32_t acc) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}"
      ::"r"(tmem_d), "r"(tmem_a), "l"(bdesc), "r"(idesc), "r"(acc)
      : "memory");
}
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
// warp-converged single-lane election (elect.sync): lets ptxas keep descriptors / barrier addresses in UNIFORM registers and emit
// straight-line UTCHMMA / UTMALDG; a plain `if (lane == 0)` makes it wrap every such instruction in an ELECT / BRA.U.ANY loop.
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile("{\n\t.reg .pred P1;\n\telect.sync _|P1, 0xffffffff;\n\tselp.u32 %0, 1, 0, P1;\n\t}" : "=r"(pred));
  return pred != 0;
}
// A whole (converged) warp waits on a barrier (every lane polls: hardware-suspended try_wait; lane-0-only polling measured 14 % slower).
__device__ __forceinline__ void mbar_wait_warp(uint32_t bar, uint32_t parity) { mbar_wait(bar, parity); }
__device__ __forceinline__ void tmem_st32(uint32_t taddr, const uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
      "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};"
      ::"r"(taddr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]), "r"(v[8]), "r"(v[9]),
        "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15]), "r"(v[16]), "r"(v[17]), "r"(v[18]), "r"(v[19]),
        "r"(v[20]), "r"(v[21]), "r"(v[22]), "r"(v[23]), "r"(v[24]), "r"(v[25]), "r"(v[26]), "r"(v[27]), "r"(v[28]), "r"(v[29]),
        "r"(v[30]), "r"(v[31])
      : "memory");
}
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};"
      ::"r"(taddr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]), "r"(v[8]), "r"(v[9]),
        "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15])
      : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32]) {   // caller issues tcgen05.wait::ld
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
        "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]),
        "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]),
        "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr));
}

// ------------------------------------------------------------------------------------------------ persistent variant
// One CTA per SM loops over (tile, K split) work items (static stride), 10 warps: TMA producer | MMA issuer | 4 splitter warps |
// 4 epilogue warps.  Stage in shared memory = [A box k 0..31 | A box k 32..63 | b_hi | b_lo'] x 16 KB.  Splitter thread <-> pixel row
// reads its 64 raw floats (2 x 128 B, TMA 128B-swizzled: conflict-free for a quarter warp), scales and splits them.  Two operand paths:
//   TS = false  the row's 64 fp16 hi / 64 lo' values overwrite the same two 128-byte rows IN PLACE (K-major SWIZZLE_128B tiles, no
//               second buffer, no cross-thread hazard); SS-mode MMA.  TMEM = two accumulator sets (2 x [main 128 | correction 128]),
//               so the epilogue of tile i overlaps the main loop of tile i+1.  Shared-memory traffic per stage: 64 KB TMA writes + 64 KB
//               splitter + 80 KB MMA operand reads (measured: L1/TEX 72 % busy — the limiter, profiles/r02_experiments.md).
//   TS = true   hi / lo' go to TENSOR memory with tcgen05.st (thread = TMEM lane) and the MMA takes A from TMEM: 64 + 32 + 48 KB per
//               stage.  The A stages take the TMEM columns of the second accumulator set ([0,256) accumulators | 256 + 64 s: a_hi 32
//               a_lo' 32), so the epilogue drains the single set into registers first and hands it back before touching global memory.
// launch_tc picks TS for long K loops (>= 9 stages per work item: the 3x3 convolutions, + 7-15 % on the big layers) and the
// double-buffered SS form for short ones (1x1 convolutions / linears: 4-stage tiles lose more to the accumulator hand-over than they gain).
//   PRE = true  (TS = false) the A operand arrives split (DP_CONV_X_SPLIT, written by dp_groupnorm_fwd_split): TMA loads the hi box
//               and the lo' box ([128 px][64 ch] fp16, SWIZZLE_128B — the layout the in-place split leaves) into the same two 16 KB
//               slots, the MMA warp waits on the TMA barrier directly and the splitter warps idle.  A stage's chain is TMA -> MMA;
//               the double-buffered SS accumulators, as there is no hand-over to avoid.
constexpr int PS_THREADS = 320, PS_STAGES = 3;
constexpr int PS_TS_MIN_STAGES = 9;     // K-loop length (stages per work item) from which the TS operand path wins

template <bool TS, bool PRE>
__global__ void __launch_bounds__(PS_THREADS, 1)
conv_tc_ps_kernel(const __grid_constant__ CUtensorMap mapA, const __grid_constant__ CUtensorMap mapBh,
                  const __grid_constant__ CUtensorMap mapBl, const TcParams p, const int tiles_m, const int total_tiles) {
  const int total_work = total_tiles * p.ksplit;     // work item wi = split * total_tiles + tile (the splits of one tile run on different SMs)
  constexpr int BN = 128;
  constexpr int B_BYTES = BN * BK * 2;
  constexpr int STAGE_BYTES = 2 * A_BYTES + 2 * B_BYTES;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw = smem_u32(smem_raw);
  const uint32_t pad_to = ((raw + 1023u) & ~1023u) - raw;
  uint8_t* smem = smem_raw + pad_to;
  const uint32_t sbase = raw + pad_to;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + PS_STAGES * STAGE_BYTES);
  const uint32_t bar0 = sbase + PS_STAGES * STAGE_BYTES;
  auto full_bar = [&](int s) { return bar0 + 8u * s; };
  auto conv_bar = [&](int s) { return bar0 + 8u * (PS_STAGES + s); };
  auto empty_bar = [&](int s) { return bar0 + 8u * (2 * PS_STAGES + s); };
  auto tfull_bar = [&](int b) { return bar0 + 8u * (3 * PS_STAGES + b); };
  auto tempty_bar = [&](int b) { return bar0 + 8u * (3 * PS_STAGES + 2 + b); };
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 3 * PS_STAGES + 4);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    for (int s = 0; s < PS_STAGES; ++s) { mbar_init(full_bar(s), 1); mbar_init(conv_bar(s), 128); mbar_init(empty_bar(s), 1); }
    for (int b = 0; b < 2; ++b) { mbar_init(tfull_bar(b), 1); mbar_init(tempty_bar(b), 128); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem_base = *tmem_slot;
  const int iters_per_tile = p.ntaps * p.kchunks;

  auto tile_coords = [&](int tile, int& q0, int& p0, int& n0, int& nblk) {
    nblk = tile / tiles_m;
    const int tile_m = tile - nblk * tiles_m;
    const int tw = tile_m % p.tiles_w;
    const int th = (tile_m / p.tiles_w) % p.tiles_h;
    const int tn = tile_m / (p.tiles_w * p.tiles_h);
    q0 = tw * p.bw; p0 = th * p.bh; n0 = tn * p.bn;
  };

  if (warp == 0) {
    if (lane == 0) {
      asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&mapA)) : "memory");
      asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&mapBh)) : "memory");
      asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&mapBl)) : "memory");
      uint32_t g = 0;
      for (int wi = blockIdx.x; wi < total_work; wi += gridDim.x) {
        const int tile = wi % total_tiles, it0 = (wi / total_tiles) * p.it_per_split, it1 = min(iters_per_tile, it0 + p.it_per_split);
        int q0, p0, n0, nblk;
        tile_coords(tile, q0, p0, n0, nblk);
        for (int it = it0; it < it1; ++it, ++g) {
          const int s = g % PS_STAGES;
          const uint32_t ph = (g / PS_STAGES) & 1u;
          mbar_wait(empty_bar(s), ph ^ 1u);
          mbar_expect_tx(full_bar(s), 2 * A_BYTES + 2 * B_BYTES);
          const int tap = it / p.kchunks, kc = it - tap * p.kchunks;
          const uint32_t st = sbase + s * STAGE_BYTES;
          const int aw = q0 * p.in_stride + p.dw[tap], ah = p0 * p.in_stride + p.dh[tap];
          if constexpr (PRE) {       // hi channels [64 kc, 64 kc + 64) and their lo' at + ld_split (past the row: TMA zero fill)
            tma_load_4d(st, &mapA, full_bar(s), kc * BK, aw, ah, n0);
            tma_load_4d(st + A_BYTES, &mapA, full_bar(s), p.ld_split + kc * BK, aw, ah, n0);
          } else {
            tma_load_4d(st, &mapA, full_bar(s), kc * BK, aw, ah, n0);
            tma_load_4d(st + A_BYTES, &mapA, full_bar(s), kc * BK + 32, aw, ah, n0);     // past the last channel: TMA zero fill
          }
          const int tapb = p.b_from_img ? n0 : p.wt[tap];
          tma_load_3d(st + 2 * A_BYTES, &mapBh, full_bar(s), kc * BK, nblk * BN, tapb);
          tma_load_3d(st + 2 * A_BYTES + B_BYTES, &mapBl, full_bar(s), kc * BK, nblk * BN, tapb);
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      uint32_t g = 0, tl = 0;
      for (int wi = blockIdx.x; wi < total_work; wi += gridDim.x, ++tl) {
        const int tile = wi % total_tiles, it0 = (wi / total_tiles) * p.it_per_split, it1 = min(iters_per_tile, it0 + p.it_per_split);
        const int nblk = tile / tiles_m;
        const int n_valid = min(BN, p.Nout - nblk * BN);
        const uint32_t n_instr = (uint32_t)((n_valid + 15) & ~15);
        // kind::f16 instruction descriptor: D = fp32 (bit 4), A / B format 0 = fp16, both K-major, N >> 3 at bit 17, M >> 4 at bit 24
        const uint32_t idesc = (1u << 4) | ((n_instr >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);
        const uint32_t idesc256 = (1u << 4) | ((256u >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);
        if constexpr (TS) {
          mbar_wait(tempty_bar(0), (tl & 1u) ^ 1u);           // epilogue has drained the accumulators of the previous tile
          asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
          const uint32_t acc = tmem_base;
          for (int it = it0; it < it1; ++it, ++g) {
            const int s = g % PS_STAGES;
            const uint32_t ph = (g / PS_STAGES) & 1u;
            mbar_wait(conv_bar(s), ph);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            const uint32_t st = sbase + s * STAGE_BYTES;
  #pragma unroll
            const uint32_t a_t = tmem_base + 256u + 64u * (uint32_t)s;
  #pragma unroll
            for (int k = 0; k < BK / 16; ++k) {      // one instruction = 16 fp16 along K = 8 packed TMEM columns of A, 32 bytes of every B row
              const uint64_t b_hi = umma_desc(st + 2 * A_BYTES + k * 32);
              const uint32_t first = (it > it0 || k > 0) ? 1u : 0u;
              // a_hi x [b_hi | b_lo'] -> [main | correction] as ONE N=256 instruction (the two B tiles are adjacent in shared memory)
              umma_f16_ts(acc, a_t + k * 8, b_hi, idesc256, first);
              umma_f16_ts(acc + 128, a_t + 32 + k * 8, b_hi, idesc, 1u);
            }
            umma_commit(empty_bar(s));
          }
          umma_commit(tfull_bar(0));
        } else {
          const uint32_t b = tl & 1u, use = tl >> 1;
          mbar_wait(tempty_bar(b), (use & 1u) ^ 1u);          // epilogue has drained this accumulator set
          asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
          const uint32_t acc = tmem_base + b * 256u;
          for (int it = it0; it < it1; ++it, ++g) {
            const int s = g % PS_STAGES;
            const uint32_t ph = (g / PS_STAGES) & 1u;
            mbar_wait(PRE ? full_bar(s) : conv_bar(s), ph);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            const uint32_t st = sbase + s * STAGE_BYTES;
  #pragma unroll
            for (int k = 0; k < BK / 16; ++k) {      // one instruction = 16 fp16 along K = 32 bytes of every 128-byte row
              const uint64_t a_hi = umma_desc(st + k * 32), a_lo = umma_desc(st + A_BYTES + k * 32);
              const uint64_t b_hi = umma_desc(st + 2 * A_BYTES + k * 32);
              const uint32_t first = (it > it0 || k > 0) ? 1u : 0u;
              // a_hi x [b_hi | b_lo'] -> [main | correction] as ONE N=256 instruction (the two B tiles are adjacent in shared memory):
              // 8 instead of 12 instructions per stage and 5/6 of the operand reads
              umma_f16(acc, a_hi, b_hi, idesc256, first);
              umma_f16(acc + 128, a_lo, b_hi, idesc, 1u);
            }
            umma_commit(empty_bar(s));
          }
          umma_commit(tfull_bar(b));
        }
      }
    }
  } else if (warp < 6) {
    if constexpr (PRE) {
      // ---- nothing to split
    } else if constexpr (TS) {
      // ---- splitter warps 2..5 (TMEM lane quarter = warp & 3)
      const int r = (warp & 3) * 32 + lane;            // pixel row of the tile = TMEM lane
      const uint32_t lane_addr = (uint32_t)((warp & 3) * 32) << 16;
      const uint32_t sw = (uint32_t)(r & 7);           // 128B swizzle: 16-byte chunk c of row r sits at chunk position c ^ (r & 7)
      const float sa = scale_up(amax_exponent(p.amax_a));
      uint32_t g = 0;
      for (int wi = blockIdx.x; wi < total_work; wi += gridDim.x) {
        const int it0 = (wi / total_tiles) * p.it_per_split, it1 = min(iters_per_tile, it0 + p.it_per_split);
        for (int it = it0; it < it1; ++it, ++g) {
          const int s = g % PS_STAGES;
          const uint32_t ph = (g / PS_STAGES) & 1u;
          mbar_wait(full_bar(s), ph);
          const uint8_t* a0 = smem + s * STAGE_BYTES + r * 128;      // row r of the k 0..31 box
          const uint8_t* a1 = a0 + A_BYTES;                          // row r of the k 32..63 box
          uint32_t hi[32], lo[32];                                   // column j = K elements (2j, 2j+1)
  #pragma unroll
          for (int c = 0; c < 8; ++c) {       // a quarter warp (8 consecutive rows) touches 8 distinct chunk positions: conflict-free
            const float4 x0 = *reinterpret_cast<const float4*>(a0 + ((c ^ sw) << 4));
            const float4 x1 = *reinterpret_cast<const float4*>(a1 + ((c ^ sw) << 4));
            split2(x0.x * sa, x0.y * sa, hi[2 * c], lo[2 * c]);
            split2(x0.z * sa, x0.w * sa, hi[2 * c + 1], lo[2 * c + 1]);
            split2(x1.x * sa, x1.y * sa, hi[16 + 2 * c], lo[16 + 2 * c]);
            split2(x1.z * sa, x1.w * sa, hi[16 + 2 * c + 1], lo[16 + 2 * c + 1]);
          }
          const uint32_t a_t = tmem_base + lane_addr + 256u + 64u * (uint32_t)s;
          tmem_st32(a_t, hi);
          tmem_st32(a_t + 32, lo);
          asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
          asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
          mbar_arrive(conv_bar(s));
        }
      }
    } else {
      // ---- splitter warps 2..5
      const int r = threadIdx.x - 64;                  // pixel row of the tile
      const uint32_t sw = (uint32_t)(r & 7);           // 128B swizzle: 16-byte chunk c of row r sits at chunk position c ^ (r & 7)
      const float sa = scale_up(amax_exponent(p.amax_a));
      uint32_t g = 0;
      for (int wi = blockIdx.x; wi < total_work; wi += gridDim.x) {
        const int it0 = (wi / total_tiles) * p.it_per_split, it1 = min(iters_per_tile, it0 + p.it_per_split);
        for (int it = it0; it < it1; ++it, ++g) {
          const int s = g % PS_STAGES;
          const uint32_t ph = (g / PS_STAGES) & 1u;
          mbar_wait(full_bar(s), ph);
          uint8_t* a0 = smem + s * STAGE_BYTES + r * 128;      // row r of the k 0..31 box  -> row r of a_hi
          uint8_t* a1 = a0 + A_BYTES;                          // row r of the k 32..63 box -> row r of a_lo'
          float4 v[16];
  #pragma unroll
          for (int c = 0; c < 8; ++c) {       // a quarter warp (8 consecutive rows) touches 8 distinct chunk positions: conflict-free
            v[c] = *reinterpret_cast<const float4*>(a0 + ((c ^ sw) << 4));
            v[8 + c] = *reinterpret_cast<const float4*>(a1 + ((c ^ sw) << 4));
          }
  #pragma unroll
          for (int c = 0; c < 8; ++c) {       // output chunk c = k 8c .. 8c+7
            const float4 x0 = v[2 * c], x1 = v[2 * c + 1];
            uint4 h, l;
            split2(x0.x * sa, x0.y * sa, h.x, l.x);
            split2(x0.z * sa, x0.w * sa, h.y, l.y);
            split2(x1.x * sa, x1.y * sa, h.z, l.z);
            split2(x1.z * sa, x1.w * sa, h.w, l.w);
            *reinterpret_cast<uint4*>(a0 + ((c ^ sw) << 4)) = h;
            *reinterpret_cast<uint4*>(a1 + ((c ^ sw) << 4)) = l;
          }
          asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
          mbar_arrive(conv_bar(s));
        }
      }
    }
  } else {
    // ---- epilogue warps 6..9 (TMEM lane quarter = warp & 3)
    const int q = warp & 3;
    const int row = q * 32 + lane;
    const uint32_t lane_addr = (uint32_t)(q * 32) << 16;
    const int w_l = row % p.bw, h_l = (row / p.bw) % p.bh, n_l = row / (p.bw * p.bh);
    // accumulators hold (s_a s_b) x the products: f1 * f2 undoes the two power-of-two operand scales (two factors: their product may underflow)
    const float f1 = scale_dn(amax_exponent(p.amax_a)), f2 = scale_dn(amax_exponent(p.amax_b)) * p.alpha;
    auto fin = [&](uint32_t main, uint32_t corr) { return fmaf(__uint_as_float(corr), LO_UNSCALE, __uint_as_float(main)) * f1 * f2; };
    float amax = 0.f;         // max |value written| by this thread (split launches: splitk_epilogue_kernel writes, and tracks, the outputs)
    uint32_t tl = 0;
    for (int wi = blockIdx.x; wi < total_work; wi += gridDim.x, ++tl) {
      const int tile = wi % total_tiles;
      int q0, p0, n0, nblk;
      tile_coords(tile, q0, p0, n0, nblk);
      if constexpr (TS) {
        mbar_wait(tfull_bar(0), tl & 1u);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        const int img = n0 + n_l;
        const bool row_ok = img < p.Nimg;
        const long long m = ((long long)img * p.Ho + ((p0 + h_l) * p.os + p.oa)) * p.Wo + ((q0 + w_l) * p.os + p.ob);
        float* yrow = p.y + m * p.ldy;
        const float* rrow = p.residual ? p.residual + m * p.ld_res : nullptr;
        const float* arow2 = p.rowadd ? p.rowadd + (long long)img * p.ld_rowadd : nullptr;
        float out[BN];          // this thread's row of the tile: drained before anything else so the MMA warp can start the next tile
  #pragma unroll
        for (int j = 0; j < BN / 32; ++j) {
          uint32_t v[32], u[32];
          const uint32_t taddr = tmem_base + lane_addr + (uint32_t)(j * 32);
          tmem_ld32(taddr, v);
          tmem_ld32(taddr + 128u, u);
          asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
  #pragma unroll
          for (int i = 0; i < 32; ++i) out[j * 32 + i] = fin(v[i], u[i]);
        }
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        mbar_arrive(tempty_bar(0));
  #pragma unroll
        for (int j = 0; j < BN / 32; ++j) {
          const float* oj = out + j * 32;
          if (p.ksplit > 1) {   // split-K: partial sums into this split's slab of the (padded) workspace; splitk_epilogue_kernel finishes
            float* wrow = p.ws + (long long)(wi / total_tiles) * p.ws_split_stride + ((long long)(tile - nblk * tiles_m) * BM + row) * p.ws_ld + nblk * BN + j * 32;
  #pragma unroll
            for (int i = 0; i < 32; i += 4)
              *reinterpret_cast<float4*>(wrow + i) = make_float4(oj[i], oj[i + 1], oj[i + 2], oj[i + 3]);
          } else if (row_ok) {
            const int c0 = nblk * BN + j * 32;
            if (p.vec4 && c0 + 32 <= p.Nout) {
  #pragma unroll
              for (int i = 0; i < 32; i += 4) {
                float4 o = make_float4(oj[i], oj[i + 1], oj[i + 2], oj[i + 3]);
                if (p.bias) { float4 t = __ldg(reinterpret_cast<const float4*>(p.bias + c0 + i)); o.x += t.x; o.y += t.y; o.z += t.z; o.w += t.w; }
                if (arow2) { float4 t = __ldg(reinterpret_cast<const float4*>(arow2 + c0 + i)); o.x += t.x; o.y += t.y; o.z += t.z; o.w += t.w; }
                if (rrow) { float4 t = __ldg(reinterpret_cast<const float4*>(rrow + c0 + i)); o.x += t.x; o.y += t.y; o.z += t.z; o.w += t.w; }
                float4* dst = reinterpret_cast<float4*>(yrow + c0 + i);
                if (p.accumulate) { float4 t = *dst; o.x += t.x; o.y += t.y; o.z += t.z; o.w += t.w; }
                *dst = o;
                amax = fmaxf(fmaxf(amax, fmaxf(fabsf(o.x), fabsf(o.y))), fmaxf(fabsf(o.z), fabsf(o.w)));
              }
            } else {
  #pragma unroll
              for (int i = 0; i < 32; ++i) {
                const int c = c0 + i;
                if (c < p.Nout) {
                  float o = oj[i];
                  if (p.bias) o += __ldg(p.bias + c);
                  if (arow2) o += __ldg(arow2 + c);
                  if (rrow) o += __ldg(rrow + c);
                  if (p.accumulate) o += yrow[c];
                  yrow[c] = o;
                  amax = fmaxf(amax, fabsf(o));
                }
              }
            }
          }
        }
      } else {
        const uint32_t b = tl & 1u, use = tl >> 1;
        mbar_wait(tfull_bar(b), use & 1u);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        const int img = n0 + n_l;
        const bool row_ok = img < p.Nimg;
        const long long m = ((long long)img * p.Ho + ((p0 + h_l) * p.os + p.oa)) * p.Wo + ((q0 + w_l) * p.os + p.ob);
        float* yrow = p.y + m * p.ldy;
        const float* rrow = p.residual ? p.residual + m * p.ld_res : nullptr;
        const float* arow2 = p.rowadd ? p.rowadd + (long long)img * p.ld_rowadd : nullptr;
  #pragma unroll 1
        for (int j = 0; j < BN / 32; ++j) {
          uint32_t v[32], u[32];
          const uint32_t taddr = tmem_base + lane_addr + b * 256u + (uint32_t)(j * 32);
          asm volatile(
              "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
              "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
              "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
              : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
                "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]),
                "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]),
                "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
              : "r"(taddr));
          asm volatile(
              "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
              "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
              "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
              : "=r"(u[0]), "=r"(u[1]), "=r"(u[2]), "=r"(u[3]), "=r"(u[4]), "=r"(u[5]), "=r"(u[6]), "=r"(u[7]), "=r"(u[8]),
                "=r"(u[9]), "=r"(u[10]), "=r"(u[11]), "=r"(u[12]), "=r"(u[13]), "=r"(u[14]), "=r"(u[15]), "=r"(u[16]),
                "=r"(u[17]), "=r"(u[18]), "=r"(u[19]), "=r"(u[20]), "=r"(u[21]), "=r"(u[22]), "=r"(u[23]), "=r"(u[24]),
                "=r"(u[25]), "=r"(u[26]), "=r"(u[27]), "=r"(u[28]), "=r"(u[29]), "=r"(u[30]), "=r"(u[31])
              : "r"(taddr + 128u));
          asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
          if (j == BN / 32 - 1) {   // accumulators are in registers: hand the TMEM set back to the MMA warp
            asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
            mbar_arrive(tempty_bar(b));
          }
          if (p.ksplit > 1) {   // split-K: raw partial sums into this split's slab of the (padded) workspace; splitk_epilogue_kernel finishes
            float* wrow = p.ws + (long long)(wi / total_tiles) * p.ws_split_stride + ((long long)(tile - nblk * tiles_m) * BM + row) * p.ws_ld + nblk * BN + j * 32;
  #pragma unroll
            for (int i = 0; i < 32; i += 4)
              *reinterpret_cast<float4*>(wrow + i) = make_float4(fin(v[i], u[i]), fin(v[i + 1], u[i + 1]), fin(v[i + 2], u[i + 2]), fin(v[i + 3], u[i + 3]));
          } else if (row_ok) {
            const int c0 = nblk * BN + j * 32;
            if (p.vec4 && c0 + 32 <= p.Nout) {
  #pragma unroll
              for (int i = 0; i < 32; i += 4) {
                float4 o = make_float4(fin(v[i], u[i]), fin(v[i + 1], u[i + 1]), fin(v[i + 2], u[i + 2]), fin(v[i + 3], u[i + 3]));
                if (p.bias) { float4 t = __ldg(reinterpret_cast<const float4*>(p.bias + c0 + i)); o.x += t.x; o.y += t.y; o.z += t.z; o.w += t.w; }
                if (arow2) { float4 t = __ldg(reinterpret_cast<const float4*>(arow2 + c0 + i)); o.x += t.x; o.y += t.y; o.z += t.z; o.w += t.w; }
                if (rrow) { float4 t = __ldg(reinterpret_cast<const float4*>(rrow + c0 + i)); o.x += t.x; o.y += t.y; o.z += t.z; o.w += t.w; }
                float4* dst = reinterpret_cast<float4*>(yrow + c0 + i);
                if (p.accumulate) { float4 t = *dst; o.x += t.x; o.y += t.y; o.z += t.z; o.w += t.w; }
                *dst = o;
                amax = fmaxf(fmaxf(amax, fmaxf(fabsf(o.x), fabsf(o.y))), fmaxf(fabsf(o.z), fabsf(o.w)));
              }
            } else {
  #pragma unroll
              for (int i = 0; i < 32; ++i) {
                const int c = c0 + i;
                if (c < p.Nout) {
                  float o = fin(v[i], u[i]);
                  if (p.bias) o += __ldg(p.bias + c);
                  if (arow2) o += __ldg(arow2 + c);
                  if (rrow) o += __ldg(rrow + c);
                  if (p.accumulate) o += yrow[c];
                  yrow[c] = o;
                  amax = fmaxf(amax, fabsf(o));
                }
              }
            }
          }
        }
      }
    }
    if (p.amax_out && p.ksplit == 1) amax_commit(p.amax_out, amax);
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  }
  __syncthreads();
  if (warp == 1) {
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512) : "memory");
  }
}

// Sums the K splits of conv_tc_ps_kernel in fixed order (deterministic) and applies its epilogue: bias, per-image row, residual,
// accumulate, the (strided) output pixel mapping.  One thread per (GEMM row, 4 channels).
__global__ void __launch_bounds__(256) splitk_epilogue_kernel(const TcParams p, const int tiles_m) {
  const int c4 = (p.Nout + 3) >> 2;
  const long long total = (long long)tiles_m * BM * c4;
  float amax = 0.f;
  for (long long i = blockIdx.x * 256ll + threadIdx.x; i < total; i += (long long)gridDim.x * 256) {
    const long long grow = i / c4;
    const int c = (int)(i - grow * c4) << 2;
    const int tile_m = (int)(grow / BM), row = (int)(grow - (long long)tile_m * BM);
    const int tw = tile_m % p.tiles_w, th = (tile_m / p.tiles_w) % p.tiles_h, tn = tile_m / (p.tiles_w * p.tiles_h);
    const int w_l = row % p.bw, h_l = (row / p.bw) % p.bh, n_l = row / (p.bw * p.bh);
    const int img = tn * p.bn + n_l;
    if (img >= p.Nimg) continue;
    const float* src = p.ws + grow * p.ws_ld + c;
    float4 acc = *reinterpret_cast<const float4*>(src);
    for (int ks = 1; ks < p.ksplit; ++ks) {
      const float4 t = *reinterpret_cast<const float4*>(src + ks * p.ws_split_stride);
      acc.x += t.x; acc.y += t.y; acc.z += t.z; acc.w += t.w;
    }
    float o[4] = {acc.x, acc.y, acc.z, acc.w};     // the splits were written with the operand scales and alpha already undone
    const long long m = ((long long)img * p.Ho + ((th * p.bh + h_l) * p.os + p.oa)) * p.Wo + ((tw * p.bw + w_l) * p.os + p.ob);
    float* yrow = p.y + m * p.ldy;
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const int cc = c + e;
      if (cc < p.Nout) {
        float v = o[e];
        if (p.bias) v += __ldg(p.bias + cc);
        if (p.rowadd) v += __ldg(p.rowadd + (long long)img * p.ld_rowadd + cc);
        if (p.residual) v += __ldg(p.residual + m * p.ld_res + cc);
        if (p.accumulate) v += yrow[cc];
        yrow[cc] = v;
        amax = fmaxf(amax, fabsf(v));
      }
    }
  }
  if (p.amax_out) amax_commit(p.amax_out, amax);
}

// ------------------------------------------------------------------------------------------------ wgrad
// dW[k][tap][c] = sum_pixels dy[pix][k] * x[pix @ tap][c]: M = out-channels (128 per tile), N = in-channels of one tap (128 per tile),
// GEMM-K = pixels, 64 per pipeline stage.  Both operands are pixel-major fp32 activations, i.e. MN-major for this product:
//   dy: 4 raw TMA boxes [64 px][32 ch] (128-byte rows, SWIZZLE_128B).  Thread <-> out-channel reads its channel down the 64 pixel rows
//       (a warp reads one conflict-free 128 B row per instruction), scales, splits into fp16 hi / lo' and writes 2 x 32 packed columns
//       of TENSOR MEMORY with tcgen05.st: the MMA then runs in TS mode (A from TMEM), so dy never goes back to shared memory.
//   x:  4 raw boxes; the boxes of channels [64j, 64j+32) and [64j+32, 64j+64) land where the fp16 blocks x_hi[j] and x_lo'[j] will live
//       ([hi0 | hi1 | lo0 | lo1], 8 KB each = [64 px][64 ch] fp16, MN-major SWIZZLE_128B: LBO = 8 KB between 64-channel blocks, SBO = 1 KB
//       between 8-pixel K groups); splitter thread <-> (block j, pixel row) rewrites its two 128-byte rows in place.
//   a_hi x [x_hi | x_lo'] -> [main | correction] is ONE N=256 instruction, a_lo' x x_hi adds to the correction half.
// TMEM: [0,128) main acc | [128,256) correction acc | 256 + 64*s: a_hi (32 columns = 64 pixels) a_lo' (32) of stage s.
// grid = (k tiles * c tiles * taps, splits): split z covers pixel chunks [z*cps, (z+1)*cps) and writes its partial
// tile to workspace[z][k][tap*C + c]; dp_conv2d_wgrad_reduce sums splits in fixed order (deterministic).
struct WgParams {
  int Nimg, H, W, C, K;
  int R, S, pad;
  int bw, bh, bn, tiles_w, tiles_h;   // 64-pixel box of the dy grid
  int total_chunks, chunks_per_split;
  int c_tiles;
  float* ws;
  int in_stride;             // x pixel = in_stride * dy pixel + tap offset
  const uint32_t* amax_x; const uint32_t* amax_y;
  float* bias_ws;            // optional [splits][K]: column sums of dy over this split's pixels (written by the tap 0 / c-tile 0 CTAs)
  int ld_split;              // pre-split x (wgrad_tc_kernel<true>): fp16 elements from a pixel's hi channels to its lo' channels
};
constexpr int WG_KPIX = 64;                  // pixels per stage
constexpr int WG_BLK = WG_KPIX * 128;        // 8 KB: one raw fp32 box [64 px][32 ch] = one fp16 block [64 px][64 ch]
constexpr int WG_STAGES = 3, WG_STAGE_BYTES = 8 * WG_BLK;

// MN-major fp16 operand, 128B-swizzled (canonical ((8,n),(8,k)):((1,LBO),(8,SBO)) in 16-byte units): LBO = 8 KB between 64-channel
// blocks, SBO = 1 KB between 8-pixel K groups
__device__ __forceinline__ uint64_t umma_desc_mn(uint32_t saddr) {
  return (uint64_t)((saddr & 0x3FFFF) >> 4) | ((uint64_t)(WG_BLK >> 4) << 16) | (64ull << 32) | (1ull << 46) | (2ull << 61);
}

// warps: 0 TMA | 1, 6 MMA issuers (alternate stages) | 2-5 and 7-10: two half-groups of splitters that work on the SAME stage (pixels
// 0..31 / 32..63 of dy, first / second raw box of every x row) + epilogue.  The ring is latency bound — period ~ (TMA latency + split +
// MMA) / stages, r02_experiments.md section 13 — so halving the ~850-instruction split of a stage shortens every stage's chain; groups on
// ALTERNATE stages did not (same chain) and, visiting each barrier only every second phase of a 3-stage ring, could be lapped.
// PRE = true: x arrives split (DP_CONV_X_SPLIT): TMA loads its hi / lo' [64 px][64 ch] fp16 boxes straight into the x_hi / x_lo'
// blocks, and the splitters only split dy.
constexpr int WG_THREADS = 352;
template <bool PRE>
__global__ void __launch_bounds__(WG_THREADS, 1)
wgrad_tc_kernel(const __grid_constant__ CUtensorMap mapDy, const __grid_constant__ CUtensorMap mapX, const WgParams p) {
  constexpr int WSTAGES = WG_STAGES;
  constexpr int STAGE_BYTES = WG_STAGE_BYTES;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw = smem_u32(smem_raw);
  const uint32_t pad_to = ((raw + 1023u) & ~1023u) - raw;
  uint8_t* smem = smem_raw + pad_to;
  const uint32_t sbase = raw + pad_to;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + WSTAGES * STAGE_BYTES);
  const uint32_t bar0 = sbase + WSTAGES * STAGE_BYTES;
  auto full_bar = [&](int s) { return bar0 + 8u * s; };
  auto conv_bar = [&](int s) { return bar0 + 8u * (WSTAGES + s); };
  auto empty_bar = [&](int s) { return bar0 + 8u * (2 * WSTAGES + s); };
  const uint32_t tmem_full_bar = bar0 + 8u * (3 * WSTAGES);
  auto iss_bar = [&](int s) { return bar0 + 8u * (3 * WSTAGES + 1 + s); };
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 4 * WSTAGES + 1);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    for (int s = 0; s < WSTAGES; ++s) { mbar_init(full_bar(s), 1); mbar_init(conv_bar(s), 256); mbar_init(empty_bar(s), 1); mbar_init(iss_bar(s), 1); }
    mbar_init(tmem_full_bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem_base = *tmem_slot;

  const int T = p.R * p.S;
  int tile = blockIdx.x;
  const int tap = tile % T; tile /= T;
  const int ct = tile % p.c_tiles;
  const int kt = tile / p.c_tiles;
  const int r = tap / p.S, sx = tap - r * p.S;
  const int chunk0 = blockIdx.y * p.chunks_per_split;
  const int chunk1 = min(p.total_chunks, chunk0 + p.chunks_per_split);
  const int num_iters = max(0, chunk1 - chunk0);   // 0 for a trailing empty split: its workspace tile is zero-filled
  // 32-channel boxes that hold valid channels (pruned widths: 96 / 179 / 358 ...): boxes past the last channel are neither loaded nor
  // split — their accumulator rows / columns are never stored, so whatever the stage buffers still hold there is harmless
  const int dy_boxes = min(4, (p.K - kt * 128 + 31) >> 5), x_boxes = min(4, (p.C - ct * 128 + 31) >> 5);
  const int x_blocks = min(2, (p.C - ct * 128 + 63) >> 6);    // pre-split x: 64-channel hi / lo' block pairs holding valid channels

  if (warp == 0) {
    if (lane == 0) {
      asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&mapDy)) : "memory");
      asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&mapX)) : "memory");
      for (int it = 0; it < num_iters; ++it) {
        const int s = it % WSTAGES;
        const uint32_t ph = (uint32_t)(it / WSTAGES) & 1u;
        mbar_wait(empty_bar(s), ph ^ 1u);
        mbar_expect_tx(full_bar(s), (uint32_t)((dy_boxes + (PRE ? 2 * x_blocks : x_boxes)) * WG_BLK));
        const int chunk = chunk0 + it;
        const int tw = chunk % p.tiles_w;
        const int th = (chunk / p.tiles_w) % p.tiles_h;
        const int tn = chunk / (p.tiles_w * p.tiles_h);
        const int q0 = tw * p.bw, p0 = th * p.bh, n0 = tn * p.bn;
        const uint32_t st = sbase + s * STAGE_BYTES;
        const int xw = q0 * p.in_stride + sx - p.pad, xh = p0 * p.in_stride + r - p.pad;
#pragma unroll
        for (int b = 0; b < 4; ++b)     // dy: up to 4 boxes of 32 out-channels
          if (b < dy_boxes) tma_load_4d(st + b * WG_BLK, &mapDy, full_bar(s), kt * 128 + b * 32, q0, p0, n0);
#pragma unroll
        for (int j = 0; j < 2; ++j) {
          if constexpr (PRE) {          // x: hi channels [64j, 64j+64) -> x_hi[j], their lo' -> x_lo'[j]
            if (j < x_blocks) {
              tma_load_4d(st + (4 + j) * WG_BLK, &mapX, full_bar(s), ct * 128 + 64 * j, xw, xh, n0);
              tma_load_4d(st + (6 + j) * WG_BLK, &mapX, full_bar(s), p.ld_split + ct * 128 + 64 * j, xw, xh, n0);
            }
          } else {                      // x: channels [64j, 64j+32) -> future x_hi[j], [64j+32, 64j+64) -> future x_lo'[j]
            if (2 * j < x_boxes) tma_load_4d(st + (4 + j) * WG_BLK, &mapX, full_bar(s), ct * 128 + 64 * j, xw, xh, n0);
            if (2 * j + 1 < x_boxes) tma_load_4d(st + (6 + j) * WG_BLK, &mapX, full_bar(s), ct * 128 + 64 * j + 32, xw, xh, n0);
          }
        }
      }
    }
  } else if (warp == 1 || warp == 6) {
    // two issuer warps on alternate stages (a lone issuer cannot run ahead of the tensor queue, profiles/r01_experiments.md),
    // warp-converged with one elected lane
    const uint32_t mw = (warp == 1) ? 0u : 1u;
    // kind::f16, D = fp32, A = fp16 from TMEM, B = fp16 MN-major (bit 16)
    const uint32_t idesc = (1u << 4) | (1u << 16) | ((uint32_t)(128 >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
    const uint32_t idesc256 = (1u << 4) | (1u << 16) | ((uint32_t)(256 >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
    if (num_iters == 0 && mw == 0) {   // empty split: release the epilogue (it writes zeros)
      if (elect_one()) umma_commit(tmem_full_bar);
      __syncwarp();
    }
    for (int it = 0; it < num_iters; ++it) {
      if (((uint32_t)it & 1u) != mw) continue;
      const int s = it % WSTAGES;
      const uint32_t ph = (uint32_t)(it / WSTAGES) & 1u;
      mbar_wait_warp(conv_bar(s), ph);
      mbar_wait_warp(full_bar(s), ph);
      if (it > 0) mbar_wait_warp(iss_bar((it - 1) % WSTAGES), (uint32_t)((it - 1) / WSTAGES) & 1u);
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      const uint32_t st = sbase + s * STAGE_BYTES;
      const uint32_t a_t = tmem_base + 256u + 64u * s;
      if (elect_one()) {
#pragma unroll
        for (int k = 0; k < WG_KPIX / 16; ++k) {     // 16 pixels per instruction = 8 packed TMEM columns of A, two 8-pixel groups (2 KB) of B
          const uint64_t b_hi = umma_desc_mn(st + 4 * WG_BLK + k * 2048);
          const uint32_t first = (it > 0 || k > 0) ? 1u : 0u;
          umma_f16_ts(tmem_base, a_t + k * 8, b_hi, idesc256, first);
          umma_f16_ts(tmem_base + 128, a_t + 32 + k * 8, b_hi, idesc, 1u);
        }
        umma_commit(empty_bar(s));
        if (it == num_iters - 1) umma_commit(tmem_full_bar);
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        mbar_arrive(iss_bar(s));
      }
      __syncwarp();
    }
  } else {
    const int half = warp > 6 ? 1 : 0;        // splitter half-group
    const int tid = threadIdx.x - (half ? 224 : 64);
    const int q = warp & 3;                   // TMEM lane quarter == 32-channel box of dy (each half-group covers the four quarters)
    const uint32_t lane_addr = (uint32_t)(q * 32) << 16;
    const int Ey = amax_exponent(p.amax_y), Ex = amax_exponent(p.amax_x);
    const float sy = scale_up(Ey), sxs = scale_up(Ex);
    const int xj = tid >> 6, xp = tid & 63;   // x task of this thread: 64-channel block, pixel row; `half` picks the raw box of the row
    const uint32_t xsw = (uint32_t)(xp & 7);
    float bsum = 0.f;                         // sum of this thread's out-channel of dy over its pixels of the split (bias gradient)
    float* bsh = reinterpret_cast<float*>(tmem_slot + 2);      // 128 floats behind the barriers: the halves' bias sums meet here
    for (int it = 0; it < num_iters; ++it) {
      const int s = it % WSTAGES;
      const uint32_t ph = (uint32_t)(it / WSTAGES) & 1u;
      mbar_wait(full_bar(s), ph);
      // (1) dy^T -> TMEM: channel `lane` of box q, pixel rows 32 half .. 32 half + 31; 16-byte chunk j of row `pix` sits at position j ^ (pix & 7)
      if (q < dy_boxes) {
        const uint8_t* blk = smem + s * STAGE_BYTES + q * WG_BLK + half * 32 * 128 + (lane & 3) * 4;
        uint32_t hi[16], lo[16];
        float ssum = 0.f;
#pragma unroll
        for (int j = 0; j < 16; ++j) {
          const float v0 = *reinterpret_cast<const float*>(blk + (2 * j) * 128 + ((((lane >> 2) ^ (2 * j)) & 7) << 4));
          const float v1 = *reinterpret_cast<const float*>(blk + (2 * j + 1) * 128 + ((((lane >> 2) ^ (2 * j + 1)) & 7) << 4));
          split2(v0 * sy, v1 * sy, hi[j], lo[j]);      // TMEM column 16 half + j = pixels (2j, 2j+1) of this half, low half first
          ssum += v0 + v1;
        }
        bsum += ssum;
        const uint32_t a_t = tmem_base + lane_addr + 256u + 64u * s + 16u * half;
        tmem_st16(a_t, hi);
        tmem_st16(a_t + 32, lo);
      }
      // (2) x: row xp of block xj.  This thread reads the row's raw box `half` (channels 32 half .. 32 half + 31 of the block); once BOTH
      //     halves have read, it writes chunks 4 half .. 4 half + 3 of the fp16 x_hi row (over box 0) and of the x_lo' row (over box 1)
      if constexpr (!PRE) {
        uint8_t* a0 = smem + s * STAGE_BYTES + (4 + xj) * WG_BLK + xp * 128;
        uint8_t* a1 = a0 + 2 * WG_BLK;
        const uint8_t* src = half ? a1 : a0;
        const bool x_valid = 2 * xj + half < x_boxes;
        float4 v[8];
        if (x_valid) {
#pragma unroll
          for (int c = 0; c < 8; ++c) v[c] = *reinterpret_cast<const float4*>(src + ((c ^ xsw) << 4));
        }
        asm volatile("bar.sync 1, 256;" ::: "memory");
        if (x_valid)
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          const float4 x0 = v[2 * c], x1 = v[2 * c + 1];
          uint4 h, l;
          split2(x0.x * sxs, x0.y * sxs, h.x, l.x);
          split2(x0.z * sxs, x0.w * sxs, h.y, l.y);
          split2(x1.x * sxs, x1.y * sxs, h.z, l.z);
          split2(x1.z * sxs, x1.w * sxs, h.w, l.w);
          const uint32_t pos = (uint32_t)(((4 * half + c) ^ xsw) << 4);
          *reinterpret_cast<uint4*>(a0 + pos) = h;
          *reinterpret_cast<uint4*>(a1 + pos) = l;
        }
      }
      asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
      mbar_arrive(conv_bar(s));
    }
    if (half) bsh[q * 32 + lane] = bsum;
    asm volatile("bar.sync 1, 256;" ::: "memory");
    if (!half) bsum += bsh[q * 32 + lane];
    mbar_wait(tmem_full_bar, 0);
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const float f1 = scale_dn(Ey), f2 = scale_dn(Ex);
    const int row = q * 32 + lane;            // k_out within the tile
    const int kout = kt * 128 + row;
    const long long TC_ = (long long)T * p.C;
    float* wrow = p.ws + ((long long)blockIdx.y * p.K + kout) * TC_ + (long long)tap * p.C;
    if (p.bias_ws && !half && tap == 0 && ct == 0 && kout < p.K) p.bias_ws[(long long)blockIdx.y * p.K + kout] = bsum;   // 0 for an empty split
    // epilogue: half-group 0 drains accumulator columns [0, 64), half-group 1 [64, 128)
    if (num_iters == 0) {                     // nothing was accumulated (TMEM holds garbage): this split contributes zeros
      if (kout < p.K)
        for (int c = ct * 128 + half * 64; c < min(p.C, ct * 128 + half * 64 + 64); ++c) wrow[c] = 0.f;
    } else
#pragma unroll 1
    for (int j = 2 * half; j < 2 * half + 2; ++j) {
      uint32_t v[32], u[32];
      const uint32_t taddr = tmem_base + lane_addr + (uint32_t)(j * 32);
      tmem_ld32(taddr, v);
      tmem_ld32(taddr + 128u, u);
      asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
      if (kout < p.K) {
        const int c0 = ct * 128 + j * 32;
#pragma unroll
        for (int i = 0; i < 32; ++i)
          if (c0 + i < p.C) wrow[c0 + i] = fmaf(__uint_as_float(u[i]), LO_UNSCALE, __uint_as_float(v[i])) * f1 * f2;
      }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  }
  __syncthreads();
  if (warp == 1) {
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512) : "memory");
  }
}

// ------------------------------------------------------------------------------------------------ host side
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn g_encode = nullptr;
int g_tc_state = -1;  // -1 unknown, 0 unavailable, 1 ok
int g_num_sms = 148;
std::mutex g_tc_mutex;
constexpr int PS_SMEM = PS_STAGES * (2 * A_BYTES + 2 * 128 * BK * 2) + 2048;
constexpr int WG_SMEM = WG_STAGES * WG_STAGE_BYTES + 2048;

// Row length (fp16 elements) of the packed weight tiles (dp_pack_conv_weight_tc): rows longer than 64 are zero-padded to a multiple of
// 64 elements (128 B) so that every 64-element TMA box row is exactly one aligned 128-byte line; short rows to a multiple of 8 (the TMA
// 16-byte stride rule).  With 16-byte padding only, pruned widths (90 / 179 input channels) ran 20-25 % slower (round 1, 3xTF32 rows).
static int wrow(int c) { return c > 64 ? ((c + 63) & ~63) : ((c + 7) & ~7); }

int tc_init() {
  std::lock_guard<std::mutex> lk(g_tc_mutex);
  if (g_tc_state >= 0) return g_tc_state;
  g_tc_state = 0;
  int dev = 0, major = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) { (void)cudaGetLastError(); return 0; }
  if (cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev) != cudaSuccess || major != 10) { (void)cudaGetLastError(); return 0; }
  void* fn = nullptr;
  cudaDriverEntryPointQueryResult qres;
  if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres) != cudaSuccess || !fn ||
      qres != cudaDriverEntryPointSuccess) { (void)cudaGetLastError(); return 0; }
  g_encode = (EncodeTiledFn)fn;
  bool ok = cudaFuncSetAttribute(conv_tc_ps_kernel<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, PS_SMEM) == cudaSuccess;
  ok = ok && cudaFuncSetAttribute(conv_tc_ps_kernel<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, PS_SMEM) == cudaSuccess;
  ok = ok && cudaFuncSetAttribute(conv_tc_ps_kernel<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, PS_SMEM) == cudaSuccess;
  ok = ok && cudaFuncSetAttribute(wgrad_tc_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, WG_SMEM) == cudaSuccess;
  ok = ok && cudaFuncSetAttribute(wgrad_tc_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, WG_SMEM) == cudaSuccess;
  cudaDeviceGetAttribute(&g_num_sms, cudaDevAttrMultiProcessorCount, dev);
  if (!ok) { (void)cudaGetLastError(); return 0; }
  (void)cudaGetLastError();
  g_tc_state = 1;
  return 1;
}

// pix_stride > 1 (strided convolution): dims 1 and 2 (W, H) are traversed with that element stride; the caller passes the box
// extents in traversed elements (box = loaded pixels x pix_stride)
bool make_map(CUtensorMap* m, const void* base, int rank, const cuuint64_t* dims, const cuuint64_t* strides_bytes,
              const cuuint32_t* box, CUtensorMapSwizzle swz = CU_TENSOR_MAP_SWIZZLE_128B, int pix_stride = 1,
              CUtensorMapDataType dtype = CU_TENSOR_MAP_DATA_TYPE_FLOAT32) {
  cuuint32_t estr[5] = {1, (cuuint32_t)pix_stride, (cuuint32_t)pix_stride, 1, 1};
  CUresult r = g_encode(m, dtype, (cuuint32_t)rank, const_cast<void*>(base), dims, strides_bytes, box, estr,
                        CU_TENSOR_MAP_INTERLEAVE_NONE, swz, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS;
}

// 128-pixel box of an [N][H][W] grid
bool pick_box(int N, int H, int W, int& bw, int& bh, int& bn) {
  if (W >= BM) {
    if (W % BM) return false;
    bw = BM; bh = 1; bn = 1; return true;
  }
  if (BM % W) return false;
  bw = W;
  int rem = BM / W;
  if (H >= rem) {
    if (H % rem) return false;
    bh = rem; bn = 1; return true;
  }
  if (rem % H) return false;
  bh = H; bn = rem / H;
  return true;
}

struct TapTable { int n; signed char dh[9], dw[9], wt[9]; };
// K splits of a persistent-kernel launch with `tiles` output tiles of `iters` pipeline stages each: enough work items to fill the SMs,
// at least 4 stages per split, none when the tiles already cover half the machine
static int pick_ksplit(int tiles, int iters, int& it_per_split) {
  it_per_split = iters;
  if (tiles * 2 > g_num_sms || iters < 8) return 1;
  int ks = g_num_sms / tiles;
  if (ks > iters / 4) ks = iters / 4;
  if (ks > 16) ks = 16;
  if (ks < 2) return 1;
  it_per_split = (iters + ks - 1) / ks;
  return (iters + it_per_split - 1) / it_per_split;      // no empty split
}

// Shared launcher.  act: [Nimg][H][W][Kg] fp32 view (ld_act) = A operand on whose pixel grid the M tiles live, amax_a its amax slot;
// w_hi / w_lo: fp16 [T][Nout][ldb] with the scale of slot amax_b; out: [Nimg][Ho][Wo][Nout] view, output pixel = (p*os+oa, q*os+ob).
// ws: optional split-K workspace (dp_conv_splitk_workspace_floats floats); *ws_need != nullptr: only report the floats a split launch needs.
// act_split: the A operand already split (DP_CONV_X_SPLIT layout, hi -> lo' distance ld_split fp16 elements): read instead of act
int launch_tc(const float* act, long long ld_act, const uint32_t* amax_a, int Nimg, int H, int W, int Kg, const void* w_hi, const void* w_lo,
              const uint32_t* amax_b, int Nout, int T, const TapTable& taps, int os, int oa, int ob, int Ho, int Wo, float* out,
              long long ld_out, const float* bias, const float* rowadd, long long ld_rowadd, const float* residual, long long ld_res,
              int accumulate, cudaStream_t st, float alpha = 1.0f, int b_from_img = 0, int in_stride = 1, int ldb = -1, float* ws = nullptr,
              long long* ws_need = nullptr, uint32_t* amax_out = nullptr, const void* act_split = nullptr, long long ld_split = 0) {
  if (ldb < 0) ldb = wrow(Kg);   // packed conv weights; batched GEMM callers pass their own row pitch
  if (!tc_init()) return DP_ERR_UNSUPPORTED;
  if (!ws_need && (!w_hi || !w_lo || !amax_a || !amax_b)) return DP_ERR_UNSUPPORTED;
  if (!ws_need && !act_split && (ld_act % 4 || ((uintptr_t)act & 15))) return DP_ERR_UNSUPPORTED;
  if (!ws_need && (((uintptr_t)w_hi & 15) || ((uintptr_t)w_lo & 15))) return DP_ERR_UNSUPPORTED;
  if (act_split && (in_stride != 1 || ld_split < Kg || ld_split % 8 || ((uintptr_t)act_split & 15))) return DP_ERR_UNSUPPORTED;
  int bw, bh, bn;
  if (!pick_box(Nimg, H, W, bw, bh, bn)) return DP_ERR_UNSUPPORTED;
  constexpr int BN = 128;
  if (ws_need) {     // geometry-only query
    *ws_need = 0;
    if (b_from_img) return DP_OK;
    const int tiles_m = (W / bw) * (H / bh) * ((Nimg + bn - 1) / bn), n_tiles = (Nout + 127) / 128;
    int ips;
    const int ks = pick_ksplit(tiles_m * n_tiles, taps.n * ((Kg + BK - 1) / BK), ips);
    if (ks > 1) *ws_need = (long long)ks * tiles_m * BM * n_tiles * 128;
    return DP_OK;
  }
  if (b_from_img && bn != 1) return DP_ERR_UNSUPPORTED;
  CUtensorMap mA, mBh, mBl;
  {
    // strided fprop: the M tiles live on the OUTPUT grid [H][W]; the activation is [H*in_stride][W*in_stride] and the box picks every
    // in_stride-th pixel (TMA element strides), so a tile is still one 128-pixel box
    const cuuint64_t Hin = (cuuint64_t)H * in_stride, Win = (cuuint64_t)W * in_stride;
    cuuint64_t dims[4] = {(cuuint64_t)Kg, Win, Hin, (cuuint64_t)Nimg};
    cuuint64_t str[3] = {(cuuint64_t)ld_act * 4, Win * ld_act * 4, Hin * Win * ld_act * 4};
    cuuint32_t box[4] = {32u, (cuuint32_t)(bw * in_stride), (cuuint32_t)(bh * in_stride), (cuuint32_t)bn};   // two boxes of 32 fp32 channels per stage
    if (box[1] > 256 || box[2] > 256) return DP_ERR_UNSUPPORTED;
    if (act_split) {   // [pixel][hi | lo'] fp16 rows of 2 ld_split elements: boxes of 64 channels (128 bytes)
      cuuint64_t sdims[4] = {(cuuint64_t)(2 * ld_split), Win, Hin, (cuuint64_t)Nimg};
      cuuint64_t sstr[3] = {(cuuint64_t)ld_split * 4, Win * ld_split * 4, Hin * Win * ld_split * 4};
      box[0] = (cuuint32_t)BK;
      if (!make_map(&mA, act_split, 4, sdims, sstr, box, CU_TENSOR_MAP_SWIZZLE_128B, 1, CU_TENSOR_MAP_DATA_TYPE_FLOAT16)) return DP_ERR_UNSUPPORTED;
    } else if (!make_map(&mA, act, 4, dims, str, box, CU_TENSOR_MAP_SWIZZLE_128B, in_stride)) return DP_ERR_UNSUPPORTED;
  }
  {
    const cuuint64_t Kp = (cuuint64_t)ldb;
    if (Kp % 8) return DP_ERR_UNSUPPORTED;
    cuuint64_t dims[3] = {Kp, (cuuint64_t)Nout, (cuuint64_t)T};
    cuuint64_t str[2] = {Kp * 2, (cuuint64_t)Nout * Kp * 2};
    cuuint32_t box[3] = {(cuuint32_t)BK, (cuuint32_t)BN, 1};
    if (!make_map(&mBh, w_hi, 3, dims, str, box, CU_TENSOR_MAP_SWIZZLE_128B, 1, CU_TENSOR_MAP_DATA_TYPE_FLOAT16) ||
        !make_map(&mBl, w_lo, 3, dims, str, box, CU_TENSOR_MAP_SWIZZLE_128B, 1, CU_TENSOR_MAP_DATA_TYPE_FLOAT16)) return DP_ERR_UNSUPPORTED;
  }
  TcParams p{};
  p.Nimg = Nimg; p.H = H; p.W = W; p.Nout = Nout;
  p.ntaps = taps.n;
  for (int i = 0; i < 9; ++i) { p.dh[i] = taps.dh[i]; p.dw[i] = taps.dw[i]; p.wt[i] = taps.wt[i]; }
  p.os = os; p.oa = oa; p.ob = ob; p.Ho = Ho; p.Wo = Wo;
  p.alpha = alpha; p.b_from_img = b_from_img; p.in_stride = in_stride; p.amax_a = amax_a; p.amax_b = amax_b; p.amax_out = amax_out;
  p.kchunks = (Kg + BK - 1) / BK;
  p.bw = bw; p.bh = bh; p.bn = bn; p.tiles_w = W / bw; p.tiles_h = H / bh;
  p.y = out; p.ldy = ld_out; p.bias = bias; p.rowadd = rowadd; p.ld_rowadd = ld_rowadd; p.residual = residual; p.ld_res = ld_res;
  p.accumulate = accumulate;
  auto al16 = [](const void* q, long long ld) { return q == nullptr || ((((uintptr_t)q) & 15) == 0 && (ld % 4) == 0); };
  p.vec4 = (al16(out, ld_out) && al16(bias, 0) && al16(rowadd, ld_rowadd) && al16(residual, ld_res)) ? 1 : 0;
  const int tiles_n = (Nimg + bn - 1) / bn;
  dim3 grid((unsigned)(p.tiles_w * p.tiles_h * tiles_n), (unsigned)((Nout + BN - 1) / BN));
  p.ksplit = 1; p.it_per_split = p.ntaps * p.kchunks;
  p.ld_split = (int)ld_split;
  {
    const int tiles_m = (int)grid.x, total = (int)(grid.x * grid.y);
    if (ws && !b_from_img) {
      p.ksplit = pick_ksplit(total, p.ntaps * p.kchunks, p.it_per_split);
      p.ws = ws; p.ws_ld = (int)grid.y * 128; p.ws_split_stride = (long long)tiles_m * BM * p.ws_ld;
    }
    const int work = total * p.ksplit;
    const int ctas = work < g_num_sms ? work : g_num_sms;
    if (act_split) conv_tc_ps_kernel<false, true><<<ctas, PS_THREADS, PS_SMEM, st>>>(mA, mBh, mBl, p, tiles_m, total);
    else if (p.it_per_split >= PS_TS_MIN_STAGES) conv_tc_ps_kernel<true, false><<<ctas, PS_THREADS, PS_SMEM, st>>>(mA, mBh, mBl, p, tiles_m, total);
    else conv_tc_ps_kernel<false, false><<<ctas, PS_THREADS, PS_SMEM, st>>>(mA, mBh, mBl, p, tiles_m, total);
    if (p.ksplit > 1) {
      int rc = dp_check_launch();
      if (rc) return rc;
      const long long items = (long long)tiles_m * BM * ((Nout + 3) / 4);
      long long blocks = (items + 255) / 256;
      if (blocks > g_num_sms * 8) blocks = g_num_sms * 8;
      splitk_epilogue_kernel<<<(int)blocks, 256, 0, st>>>(p, tiles_m);
    }
  }
  return dp_check_launch();
}

// one scaled fp32 value -> fp16 hi and lo' = (v - hi) * 2^11
__device__ __forceinline__ void split1(float v, __half& h, __half& l) {
  h = __float2half_rn(v);
  l = __float2half_rn((v - __half2float(h)) * LO_SCALE);
}
__global__ void pack_tc_kernel(const float* __restrict__ w, int K, int C, int RS, int Cp, int Kp, __half* __restrict__ kc_hi,
                               __half* __restrict__ kc_lo, __half* __restrict__ ck_hi, __half* __restrict__ ck_lo,
                               const uint32_t* __restrict__ amax) {
  // rows are zero-padded to Cp = dp_tc_weight_row(C), Kp = dp_tc_weight_row(K): kc [RS][K][Cp] (fprop B), ck [RS][C][Kp] (dgrad B)
  const float sw = scale_up(amax_exponent(amax));
  const long long na = (long long)RS * K * Cp, nb = (long long)RS * C * Kp;
  const long long total = na > nb ? na : nb;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    if (i < na && kc_hi) {
      int c = (int)(i % Cp); long long t = i / Cp; int k = (int)(t % K), tap = (int)(t / K);
      split1(c < C ? w[((long long)k * C + c) * RS + tap] * sw : 0.f, kc_hi[i], kc_lo[i]);
    }
    if (i < nb && ck_hi) {
      int k = (int)(i % Kp); long long t = i / Kp; int c = (int)(t % C), tap = (int)(t / C);
      split1(k < K ? w[((long long)k * C + c) * RS + tap] * sw : 0.f, ck_hi[i], ck_lo[i]);
    }
  }
}
// fp16 hi / lo' split of a batched [rows][cols] fp32 matrix, dense output rows of `pitch` = round8(cols) elements: 8 columns per thread
// (two float4 loads, one 16-byte store per output)
__global__ void split_h3_rows_kernel(const float* __restrict__ x, long long ld, long long bs, int rows, int cols, int pitch, int vec,
                                     __half* __restrict__ hi, __half* __restrict__ lo, const uint32_t* __restrict__ amax) {
  const float sx = scale_up(amax_exponent(amax));
  const int groups = pitch >> 3;
  const long long total = (long long)rows * groups;
  const float* xb = x + (long long)blockIdx.y * bs;
  __half* hb = hi + (long long)blockIdx.y * rows * pitch;
  __half* lb = lo + (long long)blockIdx.y * rows * pitch;
  for (long long i = blockIdx.x * 256ll + threadIdx.x; i < total; i += (long long)gridDim.x * 256) {
    const long long r = i / groups;
    const int c0 = (int)(i - r * groups) << 3;
    const float* src = xb + r * ld + c0;
    float v[8];
    if (vec && c0 + 8 <= cols) {
      const float4 a = __ldg(reinterpret_cast<const float4*>(src)), b = __ldg(reinterpret_cast<const float4*>(src + 4));
      v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
    } else {
#pragma unroll
      for (int j = 0; j < 8; ++j) v[j] = (c0 + j < cols) ? __ldg(src + j) : 0.f;
    }
    uint4 h, l;
    split2(v[0] * sx, v[1] * sx, h.x, l.x); split2(v[2] * sx, v[3] * sx, h.y, l.y);
    split2(v[4] * sx, v[5] * sx, h.z, l.z); split2(v[6] * sx, v[7] * sx, h.w, l.w);
    *reinterpret_cast<uint4*>(hb + r * pitch + c0) = h;
    *reinterpret_cast<uint4*>(lb + r * pitch + c0) = l;
  }
}
// transposed form: out[b][c][r] (rows of round8(rows) elements).  A 64 (r) x 64 (c) tile through shared memory: float4 reads along c
// (256 bytes per 16 threads), then every thread owns one output row segment of 16 consecutive r: two 16-byte stores per array
__global__ void __launch_bounds__(256) split_h3_t_kernel(const float* __restrict__ x, long long ld, long long bs, int rows, int cols, int vec,
                                                         __half* __restrict__ hi, __half* __restrict__ lo, const uint32_t* __restrict__ amax) {
  __shared__ float t[64][65];
  const float sx = scale_up(amax_exponent(amax));
  const int b = blockIdx.z, r0 = blockIdx.y * 64, c0 = blockIdx.x * 64, tid = threadIdx.x;
  const float* xb = x + (long long)b * bs;
  {
    const int cc = (tid & 15) * 4, c = c0 + cc;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int rr = (tid >> 4) + 16 * i, r = r0 + rr;
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (r < rows) {
        const float* src = xb + (long long)r * ld + c;
        if (vec && c + 4 <= cols) v = __ldg(reinterpret_cast<const float4*>(src));
        else {
          if (c < cols) v.x = __ldg(src);
          if (c + 1 < cols) v.y = __ldg(src + 1);
          if (c + 2 < cols) v.z = __ldg(src + 2);
          if (c + 3 < cols) v.w = __ldg(src + 3);
        }
      }
      t[rr][cc] = v.x * sx; t[rr][cc + 1] = v.y * sx; t[rr][cc + 2] = v.z * sx; t[rr][cc + 3] = v.w * sx;
    }
  }
  __syncthreads();
  const int rows8 = (rows + 7) & ~7;
  const int c = c0 + (tid >> 2), rs = (tid & 3) * 16;
  if (c < cols) {
    const long long o = ((long long)b * cols + c) * rows8 + r0 + rs;
#pragma unroll
    for (int h8 = 0; h8 < 2; ++h8) {
      if (r0 + rs + 8 * h8 + 8 <= rows8) {         // rows8 and the segments are multiples of 8: a segment is inside or outside as a whole
        uint4 h, l;
        const int rb = rs + 8 * h8, cl = tid >> 2;
        split2(t[rb][cl], t[rb + 1][cl], h.x, l.x); split2(t[rb + 2][cl], t[rb + 3][cl], h.y, l.y);
        split2(t[rb + 4][cl], t[rb + 5][cl], h.z, l.z); split2(t[rb + 6][cl], t[rb + 7][cl], h.w, l.w);
        *reinterpret_cast<uint4*>(hi + o + 8 * h8) = h;
        *reinterpret_cast<uint4*>(lo + o + 8 * h8) = l;
      }
    }
  }
}
// out[b][c][r] = in[b][r][c]: 64 x 64 tiles, float4 on both sides when the extents allow it
__global__ void __launch_bounds__(256) transpose_batched_kernel(const float* __restrict__ in, float* __restrict__ out, int rows, int cols, int vec) {
  __shared__ float t[64][65];
  const int b = blockIdx.z, r0 = blockIdx.y * 64, c0 = blockIdx.x * 64, tid = threadIdx.x;
  const float* ib = in + (long long)b * rows * cols;
  float* ob = out + (long long)b * rows * cols;
  const int q4 = (tid & 15) * 4, l16 = tid >> 4;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int rr = l16 + 16 * i, r = r0 + rr, c = c0 + q4;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (r < rows) {
      const float* src = ib + (long long)r * cols + c;
      if (vec && c + 4 <= cols) v = __ldg(reinterpret_cast<const float4*>(src));
      else {
        if (c < cols) v.x = __ldg(src);
        if (c + 1 < cols) v.y = __ldg(src + 1);
        if (c + 2 < cols) v.z = __ldg(src + 2);
        if (c + 3 < cols) v.w = __ldg(src + 3);
      }
    }
    t[rr][q4] = v.x; t[rr][q4 + 1] = v.y; t[rr][q4 + 2] = v.z; t[rr][q4 + 3] = v.w;
  }
  __syncthreads();
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int cc = l16 + 16 * i, c = c0 + cc, r = r0 + q4;
    if (c < cols) {
      float* dst = ob + (long long)c * rows + r;
      if (vec && r + 4 <= rows) *reinterpret_cast<float4*>(dst) = make_float4(t[q4][cc], t[q4 + 1][cc], t[q4 + 2][cc], t[q4 + 3][cc]);
      else {
        if (r < rows) dst[0] = t[q4][cc];
        if (r + 1 < rows) dst[1] = t[q4 + 1][cc];
        if (r + 2 < rows) dst[2] = t[q4 + 2][cc];
        if (r + 3 < rows) dst[3] = t[q4 + 3][cc];
      }
    }
  }
}
}  // namespace

extern "C" int dp_split_h3(const float* x, int64_t ld, int64_t bs, int32_t batch, int32_t rows, int32_t cols, int32_t transpose,
                           const uint32_t* amax, void* hi, void* lo, dp_stream_t stream) {
  DP_REQUIRE(x && hi && lo && amax, DP_ERR_NULL);
  DP_REQUIRE(batch > 0 && rows > 0 && cols > 0 && ld >= cols && batch <= 65535, DP_ERR_SHAPE);
  if (!transpose) {
    const int pitch = (cols + 7) & ~7;
    const int vec = ((((uintptr_t)x) & 15) == 0 && ld % 4 == 0 && bs % 4 == 0) ? 1 : 0;
    long long blocks = ((long long)rows * (pitch >> 3) + 255) / 256;
    if (blocks > 148 * 8) blocks = 148 * 8;
    split_h3_rows_kernel<<<dim3((unsigned)blocks, (unsigned)batch), 256, 0, (cudaStream_t)stream>>>(x, ld, bs, rows, cols, pitch, vec, (__half*)hi,
                                                                                                (__half*)lo, amax);
  } else {
    // the padded tail of a row (rows8) must be covered by the grid: round the covered extent up
    const int vec = ((((uintptr_t)x) & 15) == 0 && ld % 4 == 0 && bs % 4 == 0) ? 1 : 0;
    DP_REQUIRE((((uintptr_t)hi) & 15) == 0 && (((uintptr_t)lo) & 15) == 0, DP_ERR_ALIGN);
    dim3 grid((cols + 63) / 64, (((rows + 7) & ~7) + 63) / 64, batch);
    split_h3_t_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(x, ld, bs, rows, cols, vec, (__half*)hi, (__half*)lo, amax);
  }
  return dp_check_launch();
}
extern "C" int dp_transpose_batched(const float* in, float* out, int32_t batch, int32_t rows, int32_t cols, dp_stream_t stream) {
  DP_REQUIRE(in && out, DP_ERR_NULL);
  DP_REQUIRE(batch > 0 && rows > 0 && cols > 0 && batch <= 65535, DP_ERR_SHAPE);
  const int vec = ((((uintptr_t)in) & 15) == 0 && (((uintptr_t)out) & 15) == 0 && rows % 4 == 0 && cols % 4 == 0) ? 1 : 0;
  dim3 grid((cols + 63) / 64, (rows + 63) / 64, batch);
  transpose_batched_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(in, out, rows, cols, vec);
  return dp_check_launch();
}
extern "C" int dp_gemm_nt_tc(const dp_gemm_nt_args* a, dp_stream_t stream) {
  DP_REQUIRE(a && a->A && a->b_hi && a->b_lo && a->C, DP_ERR_NULL);
  DP_REQUIRE(a->batch > 0 && a->H > 0 && a->W > 0 && a->Kg > 0 && a->N > 0 && a->ld_a >= a->Kg && a->ldc >= a->N, DP_ERR_SHAPE);
  if (a->batch > 127) { /* the B "tap" index travels in a signed char table only for real taps; images use n0 directly */ }
  TapTable t{};
  t.n = 1;
  return launch_tc(a->A, a->ld_a, a->amax_a, a->batch, a->H, a->W, a->Kg, a->b_hi, a->b_lo, a->amax_b, a->N, a->batch, t, 1, 0, 0, a->H,
                   a->W, a->C, a->ldc, nullptr, nullptr, 0, nullptr, 0, 0, (cudaStream_t)stream, a->alpha, 1, 1, (a->Kg + 7) & ~7, nullptr,
                   nullptr, a->amax_out);
}

int dp_tc_runtime_ok() { return tc_init(); }

static TapTable dense_taps(int R, int S, int pad, bool flip) {
  TapTable t{};
  t.n = R * S;
  for (int r = 0; r < R; ++r)
    for (int s = 0; s < S; ++s) {
      int i = r * S + s;
      t.dh[i] = (signed char)(r - pad); t.dw[i] = (signed char)(s - pad);
      t.wt[i] = (signed char)(flip ? (R * S - 1 - i) : i);
    }
  return t;
}

int dp_conv2d_fprop_tc(const dp_conv_args* a, dp_stream_t stream) {
  if (!a || !a->x || !a->y) return DP_ERR_UNSUPPORTED;   // let the SIMT entry produce the precise error
  const bool pre = (a->flags & DP_CONV_X_SPLIT) != 0;
  if (a->R != a->S || (a->R != 1 && a->R != 3) || a->pad_l != a->pad_t) return DP_ERR_UNSUPPORTED;
  // stride 1: 'same' padding.  stride 2: 3x3 with pad 1, or pad 0 + the (0,1,0,1) zero border of Downsample2D (resnet.py:213-218) which
  // TMA out-of-bounds zero fill provides for free
  if (!((a->stride == 1 && a->pad_t == (a->R - 1) / 2) || (a->stride == 2 && a->R == 3 && (a->pad_t == 0 || a->pad_t == 1)))) return DP_ERR_UNSUPPORTED;
  if (a->P * a->stride != a->H || a->Q * a->stride != a->W) return DP_ERR_UNSUPPORTED;   // stride 2: even extents, out = in / 2 (Downsample2D, pad 1)
  if (a->N <= 0 || a->H <= 0 || a->W <= 0 || a->C <= 0 || a->K <= 0 || (!pre && a->ldx < a->C) || a->ldy < a->K) return DP_ERR_UNSUPPORTED;
  return launch_tc(pre ? nullptr : (const float*)a->x, a->ldx, a->amax_x, a->N, a->P, a->Q, a->C, a->w_tc_hi, a->w_tc_lo, a->amax_w, a->K,
                   a->R * a->S, dense_taps(a->R, a->S, a->pad_t, false), 1, 0, 0, a->P, a->Q, (float*)a->y, a->ldy, a->bias, a->rowadd,
                   a->ld_rowadd, a->residual, a->ld_res, (a->flags & DP_CONV_ACCUMULATE) ? 1 : 0, (cudaStream_t)stream, 1.0f, 0, a->stride, -1,
                   a->workspace, nullptr, a->amax_out, pre ? a->x : nullptr, pre ? a->ldx : 0);
}

// stride-1 dgrad == fprop of dy with the taps flipped and the (K,C) roles swapped: dx[n,h,w,c] = sum dy[n,h+1-r,w+1-s,k] W[k,c,r,s].
// stride-2 dgrad: dx[2i+a, 2j+b] only sees taps with (a+pad-r), (b+pad-s) even -> 4 parity classes, each a dense GEMM over the
// dy grid with 1/2/2/4 taps and a strided output mapping (no MACs wasted on structural zeros).
int dp_conv2d_dgrad_tc(const dp_conv_args* a, dp_stream_t stream) {
  if (!a || !a->x || !a->y) return DP_ERR_UNSUPPORTED;
  if (a->N <= 0 || a->H <= 0 || a->W <= 0 || a->C <= 0 || a->K <= 0 || a->ldx < a->C || a->ldy < a->K) return DP_ERR_UNSUPPORTED;
  if (a->R != a->S || (a->R != 1 && a->R != 3)) return DP_ERR_UNSUPPORTED;
  const int acc = (a->flags & DP_CONV_ACCUMULATE) ? 1 : 0;
  if (a->stride == 1) {
    if (a->pad_t != (a->R - 1) / 2 || a->pad_l != a->pad_t || a->P != a->H || a->Q != a->W) return DP_ERR_UNSUPPORTED;
    return launch_tc((const float*)a->y, a->ldy, a->amax_y, a->N, a->H, a->W, a->K, a->w_tc_hi, a->w_tc_lo, a->amax_w, a->C, a->R * a->S,
                     dense_taps(a->R, a->S, a->pad_t, true), 1, 0, 0, a->H, a->W, (float*)a->x, a->ldx, nullptr, nullptr, 0, nullptr, 0,
                     acc, (cudaStream_t)stream, 1.0f, 0, 1, -1, a->workspace, nullptr, a->amax_out);
  }
  if (a->stride != 2 || a->R != 3 || a->H != 2 * a->P || a->W != 2 * a->Q) return DP_ERR_UNSUPPORTED;
  TapTable cls[4];
  for (int ca = 0; ca < 2; ++ca)
    for (int cb = 0; cb < 2; ++cb) {
      TapTable& t = cls[ca * 2 + cb];
      t = TapTable{};
      for (int r = 0; r < 3; ++r)
        for (int s = 0; s < 3; ++s) {
          int nh = ca + a->pad_t - r, nw = cb + a->pad_l - s;
          if ((nh & 1) || (nw & 1)) continue;
          t.dh[t.n] = (signed char)(nh / 2); t.dw[t.n] = (signed char)(nw / 2); t.wt[t.n] = (signed char)(r * 3 + s);
          ++t.n;
        }
      if (t.n == 0) return DP_ERR_UNSUPPORTED;
    }
  for (int ca = 0; ca < 2; ++ca)
    for (int cb = 0; cb < 2; ++cb) {
      int rc = launch_tc((const float*)a->y, a->ldy, a->amax_y, a->N, a->P, a->Q, a->K, a->w_tc_hi, a->w_tc_lo, a->amax_w, a->C, 9, cls[ca * 2 + cb], 2, ca, cb,
                         a->H, a->W, (float*)a->x, a->ldx, nullptr, nullptr, 0, nullptr, 0, acc, (cudaStream_t)stream, 1.0f, 0, 1, -1,
                         a->workspace, nullptr, a->amax_out);
      if (rc != DP_OK) return (ca == 0 && cb == 0) ? rc : (rc == DP_ERR_UNSUPPORTED ? DP_ERR_SHAPE : rc);
    }
  return DP_OK;
}

// Floats of split-K workspace dp_conv2d_fprop (op 0) / dp_conv2d_dgrad (op 1) can use for this geometry (0: the launch fills the SMs
// without splitting).  With a->workspace == NULL the launch simply does not split.
extern "C" long long dp_conv_splitk_workspace_floats(const dp_conv_args* a, int op) {
  if (!a || a->N <= 0 || a->H <= 0 || a->W <= 0 || a->C <= 0 || a->K <= 0 || a->R != a->S || (a->R != 1 && a->R != 3)) return 0;
  long long need = 0;
  TapTable t{};
  if (op == 0) {
    t.n = a->R * a->S;
    launch_tc(nullptr, 0, nullptr, a->N, a->P, a->Q, a->C, nullptr, nullptr, nullptr, a->K, t.n, t, 1, 0, 0, a->P, a->Q, nullptr, 0, nullptr,
              nullptr, 0, nullptr, 0, 0, nullptr, 1.0f, 0, a->stride, -1, nullptr, &need);
  } else if (a->stride == 1) {
    t.n = a->R * a->S;
    launch_tc(nullptr, 0, nullptr, a->N, a->H, a->W, a->K, nullptr, nullptr, nullptr, a->C, t.n, t, 1, 0, 0, a->H, a->W, nullptr, 0, nullptr,
              nullptr, 0, nullptr, 0, 0, nullptr, 1.0f, 0, 1, -1, nullptr, &need);
  } else {
    for (int taps = 1; taps <= 4; taps *= 2) {     // the parity classes of a stride-2 3x3 dgrad have 1 / 2 / 2 / 4 taps and run back to back
      long long n = 0;
      t.n = taps;
      launch_tc(nullptr, 0, nullptr, a->N, a->P, a->Q, a->K, nullptr, nullptr, nullptr, a->C, 9, t, 2, 0, 0, a->H, a->W, nullptr, 0, nullptr,
                nullptr, 0, nullptr, 0, 0, nullptr, 1.0f, 0, 1, -1, nullptr, &n);
      if (n > need) need = n;
    }
  }
  return need;
}

// 64-pixel K-chunk box of an [N][H][W] grid
static bool pick_box64(int H, int W, int& bw, int& bh, int& bn) {
  if (W >= WG_KPIX) { if (W % WG_KPIX) return false; bw = WG_KPIX; bh = 1; bn = 1; return true; }
  if (WG_KPIX % W) return false;
  bw = W;
  int rem = WG_KPIX / W;
  if (H >= rem) { if (H % rem) return false; bh = rem; bn = 1; return true; }
  if (rem % H) return false;
  bh = H; bn = rem / H;
  return true;
}

int dp_conv2d_wgrad_tc(const dp_conv_args* a, dp_stream_t stream) {
  if (!a || !a->x || !a->y || !a->workspace) return DP_ERR_UNSUPPORTED;
  if (!tc_init()) return DP_ERR_UNSUPPORTED;
  if (a->R != a->S || (a->R != 1 && a->R != 3) || a->pad_l != a->pad_t) return DP_ERR_UNSUPPORTED;
  // stride 1: 'same' padding.  stride 2: 3x3 with pad 1, or pad 0 + the (0,1,0,1) zero border of Downsample2D (resnet.py:213-218) which
  // TMA out-of-bounds zero fill provides for free
  if (!((a->stride == 1 && a->pad_t == (a->R - 1) / 2) || (a->stride == 2 && a->R == 3 && (a->pad_t == 0 || a->pad_t == 1)))) return DP_ERR_UNSUPPORTED;
  if (a->P * a->stride != a->H || a->Q * a->stride != a->W || a->splits < 1) return DP_ERR_UNSUPPORTED;
  const bool pre = (a->flags & DP_CONV_X_SPLIT) != 0;
  if (a->ldy % 4 || ((uintptr_t)a->y & 15)) return DP_ERR_UNSUPPORTED;
  if (!pre && (a->ldx % 4 || ((uintptr_t)a->x & 15))) return DP_ERR_UNSUPPORTED;
  if (pre && (a->stride != 1 || a->ldx < a->C || a->ldx % 8 || ((uintptr_t)a->x & 15))) return DP_ERR_UNSUPPORTED;
  int bw, bh, bn;
  if (!a->amax_x || !a->amax_y) return DP_ERR_UNSUPPORTED;
  if (!pick_box64(a->P, a->Q, bw, bh, bn)) return DP_ERR_UNSUPPORTED;   // 64-pixel chunks of the dy (output) grid; images past the batch
  const int img_boxes = (a->N + bn - 1) / bn;                           // in the last box are TMA zero fill: they add nothing
  CUtensorMap mDy, mX;
  {
    cuuint64_t dims[4] = {(cuuint64_t)a->K, (cuuint64_t)a->Q, (cuuint64_t)a->P, (cuuint64_t)a->N};
    cuuint64_t str[3] = {(cuuint64_t)a->ldy * 4, (cuuint64_t)a->Q * a->ldy * 4, (cuuint64_t)a->P * a->Q * a->ldy * 4};
    cuuint32_t box[4] = {32, (cuuint32_t)bw, (cuuint32_t)bh, (cuuint32_t)bn};
    if (!make_map(&mDy, a->y, 4, dims, str, box)) return DP_ERR_UNSUPPORTED;
  }
  if (pre) {   // [pixel][hi | lo'] fp16 rows of 2 ldx elements: [64 px][64 ch] boxes
    cuuint64_t dims[4] = {(cuuint64_t)(2 * a->ldx), (cuuint64_t)a->W, (cuuint64_t)a->H, (cuuint64_t)a->N};
    cuuint64_t str[3] = {(cuuint64_t)a->ldx * 4, (cuuint64_t)a->W * a->ldx * 4, (cuuint64_t)a->H * a->W * a->ldx * 4};
    cuuint32_t box[4] = {64, (cuuint32_t)bw, (cuuint32_t)bh, (cuuint32_t)bn};
    if (!make_map(&mX, a->x, 4, dims, str, box, CU_TENSOR_MAP_SWIZZLE_128B, 1, CU_TENSOR_MAP_DATA_TYPE_FLOAT16)) return DP_ERR_UNSUPPORTED;
  } else {   // x is sampled at stride * (output pixel) + tap offset: TMA element strides on W, H
    cuuint64_t dims[4] = {(cuuint64_t)a->C, (cuuint64_t)a->W, (cuuint64_t)a->H, (cuuint64_t)a->N};
    cuuint64_t str[3] = {(cuuint64_t)a->ldx * 4, (cuuint64_t)a->W * a->ldx * 4, (cuuint64_t)a->H * a->W * a->ldx * 4};
    cuuint32_t box[4] = {32, (cuuint32_t)(bw * a->stride), (cuuint32_t)(bh * a->stride), (cuuint32_t)bn};
    if (box[1] > 256 || box[2] > 256) return DP_ERR_UNSUPPORTED;
    if (!make_map(&mX, a->x, 4, dims, str, box, CU_TENSOR_MAP_SWIZZLE_128B, a->stride)) return DP_ERR_UNSUPPORTED;
  }
  WgParams p{};
  p.Nimg = a->N; p.H = a->P; p.W = a->Q; p.C = a->C; p.K = a->K; p.R = a->R; p.S = a->S; p.pad = a->pad_t; p.in_stride = a->stride;
  p.bw = bw; p.bh = bh; p.bn = bn; p.tiles_w = a->Q / bw; p.tiles_h = a->P / bh;
  p.total_chunks = p.tiles_w * p.tiles_h * img_boxes;
  p.amax_x = a->amax_x; p.amax_y = a->amax_y; p.bias_ws = a->bias_ws; p.ld_split = pre ? (int)a->ldx : 0;
  p.chunks_per_split = (p.total_chunks + a->splits - 1) / a->splits;
  p.c_tiles = (a->C + 127) / 128;
  p.ws = a->workspace;
  const int k_tiles = (a->K + 127) / 128;
  dim3 grid((unsigned)(k_tiles * p.c_tiles * a->R * a->S), (unsigned)a->splits);
  if (pre) wgrad_tc_kernel<true><<<grid, WG_THREADS, WG_SMEM, (cudaStream_t)stream>>>(mDy, mX, p);
  else wgrad_tc_kernel<false><<<grid, WG_THREADS, WG_SMEM, (cudaStream_t)stream>>>(mDy, mX, p);
  return dp_check_launch();
}

extern "C" int dp_conv_presplit_eligible(const dp_conv_args* a) {
  if (!a || !tc_init()) return DP_ERR_UNSUPPORTED;
  if (a->N <= 0 || a->H <= 0 || a->W <= 0 || a->C <= 0 || a->K <= 0) return DP_ERR_UNSUPPORTED;
  if (a->R != a->S || (a->R != 1 && a->R != 3) || a->stride != 1 || a->pad_t != (a->R - 1) / 2 || a->pad_l != a->pad_t) return DP_ERR_UNSUPPORTED;
  if (a->P != a->H || a->Q != a->W) return DP_ERR_UNSUPPORTED;
  int bw, bh, bn;
  if (!pick_box(a->N, a->H, a->W, bw, bh, bn) || !pick_box64(a->H, a->W, bw, bh, bn)) return DP_ERR_UNSUPPORTED;   // fprop / wgrad tiles
  return DP_OK;
}

extern "C" int dp_pack_conv_weight_tc(const float* w, int32_t K, int32_t C, int32_t R, int32_t S, void* kc_hi, void* kc_lo,
                                      void* ck_hi, void* ck_lo, uint32_t* amax_w, dp_stream_t stream) {
  DP_REQUIRE(w && amax_w, DP_ERR_NULL);
  DP_REQUIRE((kc_hi == nullptr) == (kc_lo == nullptr) && (ck_hi == nullptr) == (ck_lo == nullptr), DP_ERR_NULL);
  DP_REQUIRE(K > 0 && C > 0 && R > 0 && S > 0, DP_ERR_SHAPE);
  // the weight's own amax slot first (one scale per tensor), then both fp16 hi / lo' orientations with that scale
  if (cudaMemsetAsync(amax_w, 0, sizeof(uint32_t), (cudaStream_t)stream) != cudaSuccess) return dp_check_launch();
  int rc = dp_amax(w, (int64_t)C * R * S, K, C * R * S, amax_w, stream);
  if (rc) return rc;
  const int Cp = wrow(C), Kp = wrow(K);
  long long total = (long long)R * S * ((long long)K * Cp > (long long)C * Kp ? (long long)K * Cp : (long long)C * Kp);
  int blocks = (int)((total + 255) / 256);
  if (blocks > 148 * 16) blocks = 148 * 16;
  pack_tc_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(w, K, C, R * S, Cp, Kp, (__half*)kc_hi, (__half*)kc_lo, (__half*)ck_hi, (__half*)ck_lo,
                                                           amax_w);
  return dp_check_launch();
}

extern "C" int dp_tc_weight_row(int channels) { return channels > 0 ? wrow(channels) : 0; }
