// Implicit-GEMM NHWC convolution on the 5th-gen tensor cores (tcgen05 + TMEM + TMA), sm_100a only.
//
// Replaces every nn.Conv2d + BatchNorm2d (+ReLU, +residual add) of the reference network
// (/root/reference/acr/model.py: BasicBlock :470-499, Bottleneck :501-539, transition / fuse convs
// :620-663, :703-736, SegmNet :374-463, head stacks :288-313, contact conv :227-235), which the
// reference dispatches to cuDNN + separate ATen elementwise kernels.
//
// GEMM view:  D[M = 128 output pixels][N = cout_pad] += A[M][K] * B[N][K],  K = taps * cin_pad.
//   * Work unit = a 16x16-pixel SUPER-TILE of one image = two M = 128 UMMA tiles (left / right 8 columns; an M tile is
//     16 image rows x 8 pixels, i.e. 16 swizzle atoms of 8 pixels at a uniform stride).  One CTA computes all output
//     channels of its tile (N <= 256 per instruction; wider layers and the MMA-bound 256->256 layers as "virtual tiles" of
//     N / nsplit channels, ConvTcParams::nsplit), so activations are never re-read across N tiles.
//   * A operand by TMA, the conv padding by TMA's out-of-bounds zero fill.  3x3 stride-1 convs with 64-channel chunks load
//     ONE haloed box {64, 24, 18} per chunk and address all nine taps inside it through UMMA descriptors whose start is
//     NOT aligned to the swizzle repeat (MODE_P1; the 128B swizzle follows the absolute shared-memory address, see
//     tools/umma_shift_probe.cu); narrower chunks use three kx-shifted boxes {CK, 16, 18} with the ky taps as row offsets
//     (MODE_PATCH).  Dense 32-channel tensors are convolved as x-pairs (two pixels per 128-byte row): stride 1 as a
//     64->64 conv with block-sparse weights whose side taps are 32x32 corners (MODE_XPAIR), stride 2 from two row-parity
//     boxes with taps = row offset + pair-column offset + K half (MODE_S2X).  Other stride-2 convs read four parity views
//     (even/odd rows x columns, own tensor maps), 1x1 convs a single tap.
//   * B operand: packed weights [cout_pad][taps*cin_pad] (BN folded), 2-D TMA boxes {CK, N}; resident in shared memory for
//     the whole kernel when they fit (all 32/64-channel layers), otherwise streamed through their own mbarrier ring.
//   * Both land in shared memory in the canonical K-major swizzled layout (128B / 64B / 32B swizzle for CK = 64 / 32 / 16)
//     that UMMA shared-memory descriptors address directly.
//   * Persistent CTAs (one per SM): warp 0 = TMA producer; warps 1..2 = MMA issuers, ONE PER HALF of the super-tile (each an
//     elected thread issuing tcgen05.mma into its own fp32 accumulator in TMEM, double buffered when 4 N <= 512 columns);
//     8 epilogue warps (tcgen05.ld -> +bias (+residual) (ReLU) -> 16-bit / fp32 NHWC) overlapping the next tile's main
//     loop -- either with direct 256-bit global accesses or, where it measured faster (every layer with a residual, all
//     N = 64 layers, wide convs of narrow inputs), STAGED: 4 KB slabs per warp, the residual prefetched by TMA loads and the
//     result written by TMA stores, synchronised per warp only.
//     -DACR_DUAL_ISSUER=0 builds the single-issuer form (A/B measurements; two issuers bought 6 %: the N = 64 MMAs are
//     bound by the shared-memory bandwidth of their operand reads, profiles/r2_conv_ncu_summary.md).
#include <cuda.h>
#include <stdlib.h>

#include "ops.cuh"

namespace acr {

// ------------------------------------------------------------------------------- PTX wrappers
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n.reg .pred p;\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
      "selp.u32 %0, 1, 0, p;\n}"
      : "=r"(ok)
      : "r"(bar), "r"(parity)
      : "memory");
  return ok != 0;
}
// bounded wait: a protocol bug must fail the launch, not hang the GPU box
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  for (uint32_t spin = 0; !mbar_try_wait(bar, parity); ++spin)
    if (spin > (1u << 26)) {
      printf("conv_tc: mbarrier timeout (block %d,%d thread %d bar %u parity %u)\n", blockIdx.x, blockIdx.y,
             threadIdx.x, bar, parity);
      __trap();
    }
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
// one lane of a converged warp (the pattern CUTLASS uses so that tcgen05/TMA issue stays on the uniform
// datapath without per-lane emulation loops)
__device__ __forceinline__ bool elect_one_sync() {
  uint32_t pred;
  asm volatile("{\n.reg .pred p;\nelect.sync _|p, 0xffffffff;\nselp.u32 %0, 1, 0, p;\n}" : "=r"(pred));
  return pred != 0;
}
// Programmatic dependent launch: a kernel launched with the programmatic-stream-serialisation attribute may
// start while its predecessor is still draining; everything that touches the predecessor's outputs (or
// writes memory the predecessor may still read) comes after pdl_wait().
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

__device__ __forceinline__ void tma_load_4d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1,
                                            int c2, int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
      ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}
// TMA store of one [16 rows][8 px][64 ch] slab (shared -> global, bulk async-group completion)
__device__ __forceinline__ void tma_store_4d(const CUtensorMap* map, uint32_t src, int c0, int c1, int c2, int c3) {
  asm volatile("cp.async.bulk.tensor.4d.global.shared::cta.bulk_group [%0, {%2, %3, %4, %5}], [%1];"
               ::"l"(map), "r"(src), "r"(c0), "r"(c1), "r"(c2), "r"(c3) : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_read0() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
template <int N> __device__ __forceinline__ void bulk_wait_read() { asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory"); }
__device__ __forceinline__ void bulk_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void named_bar_sync(int id, int nthreads) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory"); }
__device__ __forceinline__ uint4 lds128(uint32_t addr) {
  uint4 v;
  asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr) : "memory");
  return v;
}
__device__ __forceinline__ void sts128(uint32_t addr, const uint4& v) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* map) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(map) : "memory");
}

__device__ __forceinline__ void tmem_alloc(uint32_t dst_smem, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dst_smem), "r"(ncols) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void umma_f16(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                         uint32_t accumulate) {
  asm volatile(
      "{\n.reg .pred p;\nsetp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n}"
      ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// same, with the 64-bit descriptors passed as (lo, hi) register pairs: the issuing thread only adds
// small constants to the 32-bit `lo` words between MMAs (the issue loop is a single thread, so every
// integer instruction in it is on the tensor pipe's critical path)
__device__ __forceinline__ void umma_f16_lohi(uint32_t tmem_d, uint32_t a_lo, uint32_t a_hi, uint32_t b_lo, uint32_t b_hi,
                                              uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n.reg .pred p;\n.reg .b64 da, db;\n"
      "mov.b64 da, {%1, %2};\nmov.b64 db, {%3, %4};\n"
      "setp.ne.b32 p, %6, 0;\n"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %5, p;\n}"
      ::"r"(tmem_d), "r"(a_lo), "r"(a_hi), "r"(b_lo), "r"(b_hi), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t* r) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// UMMA shared-memory descriptor, K-major swizzled operand (cute::UMMA::SmemDescriptor bit layout):
//   [0,14) start>>4 | [16,30) LBO>>4 (=1, unused for swizzled K-major) | [32,46) SBO>>4 |
//   [46,48) version=1 | [61,64) layout (2=128B, 4=64B, 6=32B swizzle)
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t saddr, uint32_t sbo_bytes, uint32_t layout) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr >> 4) & 0x3FFF);
  d |= (uint64_t)1 << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)layout << 61;
  return d;
}

// ------------------------------------------------------------------------------------ kernel
// Measured on B200 (tools/tma_bench.cu, 148 CTAs): a 4-D TMA box costs ~620 clk per SM whatever its
// size (4 KB .. 72 KB), a 2-D box ~320 clk.  So the CTA works on 16x16-pixel super-tiles: ONE box per
// (channel chunk, kx) feeds two M=128 UMMA tiles (left / right 8 columns) and three ky taps.
constexpr int TILE_Y = 16, TILE_X = 16, HALF_X = 8, TILE_M = 128;
#ifndef ACR_DUAL_ISSUER
#define ACR_DUAL_ISSUER 1
#endif
constexpr bool DUAL = ACR_DUAL_ISSUER != 0;
constexpr int ISSUERS = DUAL ? 2 : 1;        // MMA-issuing warps (one per half-tile accumulator when 2)
constexpr int EPI_WARP0 = 1 + ISSUERS;       // first epilogue warp
constexpr int EPI_WARPS = 8;
constexpr int TC_THREADS = 32 * (EPI_WARP0 + EPI_WARPS);
constexpr int SMEM_BUDGET = 224 * 1024;

struct ConvTcParams {
  CUtensorMap tmA[4];
  CUtensorMap tmB;
  CUtensorMap tmOut;   // output as {C, W, H, B}, box {64, 8, 16, 1} (tma_out) or {64, 8, 4, 1} (epi_staged), 128B swizzle
  CUtensorMap tmRes;   // residual, box {64, 8, 4, 1}, 128B swizzle (epi_staged)
  const void* ext[3];  // extra terms added before the activation (folded fuse sums), read at (oy >> shift, ox >> shift)
  int n_ext, ext_shift[3], ext_stride[3], ext_W[3], ext_H[3];
  int epi_staged;      // N % 64 == 0, 16-bit output: every epilogue warp stages 32 px x 128 B slabs in shared memory, TMA in/out
  int epi_nb;          // staging buffers per epilogue warp (ring depth, 1..3)
  const float* bias;
  const void* res;
  void* out;
  int taps, ksz, stride, cchunks, cin_pad, npad, relu, has_res, out_f32, bias_per_image, pow11_ch0;
  uint32_t bias_bytes;  // shared-memory bias region: 1 KB up to 256 output channels, more for the N-split layers beyond
  int nsplit, nsub;   // N split: every super-tile is computed as nsplit "virtual tiles" of nsub = npad / nsplit output channels
                      // (N = 256 would need all 512 TMEM columns for ONE tile: with two halves of 128 the accumulators are
                      // double buffered again and the epilogue of one half overlaps the MMAs of the other; also lifts N > 256)
  int xpair;    // x-paired 32->32 conv run as 64->64 (see below): side taps are quarter blocks
  uint32_t idesc_half;
  int debug;    // MODE_DIAG bits (0 in the product path)
  int tma_out;  // epilogue stages 64-channel slabs in shared memory and stores them with TMA (16-bit, cout_pad % 64 == 0)
  uint32_t stage_out_bytes;
  int vec256;   // output / residual rows are 32-byte aligned: 256-bit epilogue accesses
  int ksteps;   // k16 steps of a chunk that hold real channels (the rest are TMA zero fill: skipped)
  int patch_mode, b_resident, SA, SB;
  int patch1;   // MODE_P1: ONE 24-wide haloed box per channel chunk, kx shifts = unaligned descriptor starts
  int s2x;      // MODE_S2X: 3x3 stride-2 conv of a dense 32-channel tensor read as x-pairs: two row-parity boxes per tile
  uint32_t a_stage_bytes, b_block_bytes, b_region_bytes;
  int tmem_cols, acc_stride, nbuf;
  int tiles_x, tiles_per_img, total_tiles, Ho, Wo, out_stride, res_stride;
  uint32_t idesc;
};

// kx served by the i-th A patch of a channel chunk.  x-paired convs take the centre tap first: it is the only
// one that writes all N columns, so it must be the MMA that zero-initialises the accumulator.
__device__ __forceinline__ int patch_kx(int i, int xpair) { return xpair ? (i == 0 ? 1 : (i == 1 ? 0 : 2)) : i; }

template <int CK>
struct SwizzleCfg {
  static constexpr uint32_t kRowBytes = CK * 2;
  static constexpr uint32_t kAtom = 8 * kRowBytes;          // 8 pixels of one image row = one swizzle atom
  static constexpr uint32_t kSBO_A = TILE_X * kRowBytes;    // next image row of the 16-wide box
  static constexpr uint32_t kLayout = CK == 64 ? 2u : (CK == 32 ? 4u : 6u);
};

// MODE bits (compile-time specialisation of the single-thread MMA issue loop)
constexpr int MODE_PATCH = 1, MODE_RESIDENT = 2, MODE_XPAIR = 4;
// MODE_P1 (with MODE_PATCH, CK = 64): the whole haloed input patch of a super-tile is ONE TMA box {64, 24, 18} per channel
// chunk (x0-1 .. x0+22, y0-1 .. y0+16; the row pitch of 24 pixels keeps every image row on a swizzle-atom boundary).
// The nine taps are nine UMMA descriptors into it: ky moves the start by whole image rows, kx by single pixels --
// a start address that is NOT aligned to the 1024-byte swizzle repeat.  tools/umma_shift_probe.cu established how
// the tensor core treats that (B200, profiles/r2_umma_shift_probe.log): the 128-byte swizzle is a function of the
// ABSOLUTE shared-memory address bits (chunk ^= (addr >> 7) & 7), exactly like the TMA unit wrote the box, so any
// 128-byte-aligned start works with base offset 0; a non-zero base-offset field XORs the chunk order once more (it is
// for layouts whose swizzle pattern is relative to the tile, not ours).  One box instead of three: a third of the
// TMA issues, half the L2 -> smem bytes, half the shared memory per tile (a whole tile of look-ahead fits next to
// resident weights).
constexpr int MODE_P1 = 16;
constexpr int P1_PITCH = 24;   // pixels per image row of the single box
// MODE_S2X (CK = 64): 3x3 STRIDE-2 conv whose input is a dense 32-channel tensor, viewed as (H, W/2, 64): one 128-byte
// row = an even pixel's 32 channels followed by its odd neighbour's.  Output pixel (oy, ox) reads input columns
// 2ox-1, 2ox, 2ox+1 = [pair ox-1, odd half], [pair ox, even half], [pair ox, odd half] and rows 2oy-1, 2oy, 2oy+1 =
// odd-row view row oy-1, even-row view row oy, odd-row view row oy+1.  So a 16x16 output tile needs TWO boxes
// {64, 24 pair columns from x0-1, 17 rows} (even rows from y0, odd rows from y0-1) instead of nine 64-byte-row
// boxes of four parity views: the nine taps are descriptor starts inside them (row offset 0/1, pair-column offset
// 0/1 = an unaligned start, K half 0/1 = k-steps {0,1} or {2,3}).  The packed weights carry the 32 input channels
// of tap (ky,kx) at K offset 32*(kx != 1) (engine._pack_conv(s2x=True)).
constexpr int MODE_S2X = 32;
// MODE_DIAG: diagnostic instances (tools/conv_bench.py, ACR_B200_CONV_DIAG=bits): 1 = the issuer skips the MMAs,
// 2 = the epilogue only recycles the accumulator, 4 = the epilogue reads TMEM but skips math and stores.  Timing
// floors of each warp role; never launched by the product path (debug == 0).
constexpr int MODE_DIAG = 8;

template <int CK, typename T, int MODE>
__global__ void __launch_bounds__(TC_THREADS, 1) conv_tc_kernel(const __grid_constant__ ConvTcParams P) {
  using Cfg = SwizzleCfg<CK>;
  constexpr bool PATCH = (MODE & MODE_PATCH) != 0, RESIDENT = (MODE & MODE_RESIDENT) != 0, XPAIR = (MODE & MODE_XPAIR) != 0;
  constexpr bool P1 = (MODE & MODE_P1) != 0, S2X = (MODE & MODE_S2X) != 0;
  static_assert(!P1 || (PATCH && CK == 64), "the single-box form exists for CK = 64 patch convs");
  static_assert(!S2X || (!PATCH && !P1 && !XPAIR && CK == 64), "the x-paired stride-2 form is a CK = 64 mode of its own");
  constexpr bool DIAG = (MODE & MODE_DIAG) != 0;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw = smem_u32(smem_raw);
  const uint32_t base = (raw + 1023u) & ~1023u;  // swizzle atoms need 1024-byte alignment
  const int SA = P.SA, SB = P.SB;
  const uint32_t b_base = base;
  const uint32_t a_base = base + P.b_region_bytes;
  const uint32_t stage_base = a_base + (uint32_t)SA * P.a_stage_bytes;  // epilogue staging: 2 halves x [128 px][128 B]
  const uint32_t bias_base = stage_base + P.stage_out_bytes;            // fp32 bias[npad] (<= 1 KB)
  const uint32_t bar_base = bias_base + P.bias_bytes;
  // barrier map: fullA[SA] emptyA[SA] fullB[SB] emptyB[SB] bres tmem_full[buf][half] tmem_empty[buf][half] | tmem_ptr
  auto fullA = [&](int s) { return bar_base + 8u * s; };
  auto emptyA = [&](int s) { return bar_base + 8u * (SA + s); };
  auto fullB = [&](int s) { return bar_base + 8u * (2 * SA + s); };
  auto emptyB = [&](int s) { return bar_base + 8u * (2 * SA + SB + s); };
  const uint32_t bres_bar = bar_base + 8u * (2 * SA + 2 * SB);
  auto tmem_full = [&](int b, int h) { return bres_bar + 8u * (1 + b * 2 + h); };
  auto tmem_empty = [&](int b, int h) { return bres_bar + 8u * (5 + b * 2 + h); };
  const uint32_t tmem_ptr_addr = bres_bar + 8u * 9;
  auto res_full = [&](int i) { return bres_bar + 8u * (10 + i); };   // staged epilogue: residual slab in buffer i % 3 of warp i / 3 has landed
  volatile uint32_t* tmem_ptr_gen = reinterpret_cast<volatile uint32_t*>(smem_raw + (tmem_ptr_addr - raw));
  float* s_bias = reinterpret_cast<float*>(smem_raw + (bias_base - raw));

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int nA = P.s2x ? 2 : (P.patch1 ? P.cchunks : (P.patch_mode ? P.cchunks * 3 : P.taps * P.cchunks));  // A loads per super-tile
  const int nsub = P.patch1 ? 9 : (P.patch_mode ? 3 : 1);                                     // taps served by one A load
  const int nbuf = P.nbuf;

  if (threadIdx.x == 0) {
    // a stage is free again once EVERY issuer's MMAs have read it (tcgen05.commit tracks the issuing thread's MMAs only)
    for (int s = 0; s < SA; ++s) { mbar_init(fullA(s), 1); mbar_init(emptyA(s), ISSUERS); }
    for (int s = 0; s < SB; ++s) { mbar_init(fullB(s), 1); mbar_init(emptyB(s), ISSUERS); }
    mbar_init(bres_bar, 1);
    for (int b = 0; b < 2; ++b)
      for (int h = 0; h < 2; ++h) { mbar_init(tmem_full(b, h), 1); mbar_init(tmem_empty(b, h), EPI_WARPS / 2); }
    for (int i = 0; i < EPI_WARPS * 3; ++i) mbar_init(res_full(i), 1);
    fence_barrier_init();
    tma_prefetch_desc(&P.tmB);
    tma_prefetch_desc(&P.tmA[0]);
    if (P.tma_out || P.epi_staged) tma_prefetch_desc(&P.tmOut);
    if (P.epi_staged && P.has_res) tma_prefetch_desc(&P.tmRes);
  }
  if (!P.bias_per_image)
    for (int i = threadIdx.x; i < P.npad; i += TC_THREADS) s_bias[i] = P.bias[i];
  if (warp == 1) tmem_alloc(tmem_ptr_addr, (uint32_t)P.tmem_cols);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_gen;
  // let the next kernel of the stream begin its own prologue (barrier init, TMEM alloc, weight loads) as
  // soon as SMs drain; our own prologue above touched nothing the previous kernel produces
  pdl_launch_dependents();

  if (warp == 0) {
    // ===================================================================== TMA producer
    // (whole warp stays converged; one elected lane issues)
    {
      if (P.b_resident && elect_one_sync()) {  // whole weight tensor once per CTA
        const int nblk = P.taps * P.cchunks;
        mbar_expect_tx(bres_bar, (uint32_t)nblk * P.b_block_bytes);
        for (int i = 0; i < nblk; ++i)
          tma_load_2d(b_base + (uint32_t)i * P.b_block_bytes, &P.tmB, bres_bar, (i / P.cchunks) * P.cin_pad + (i % P.cchunks) * CK, 0);
      }
      __syncwarp();
      pdl_wait();   // weights are constants; the activations below are the previous kernel's output
      int sa = 0, sb = 0;
      uint32_t pha = 0, phb = 0;
      for (int vt = blockIdx.x; vt < P.total_tiles * P.nsplit; vt += gridDim.x) {
        const int tile = vt / P.nsplit, n_off = (vt - tile * P.nsplit) * P.nsub;
        const int n = tile / P.tiles_per_img, rem = tile % P.tiles_per_img;
        const int y0 = (rem / P.tiles_x) * TILE_Y, x0 = (rem % P.tiles_x) * TILE_X;
        for (int a = 0; a < nA; ++a) {
          int cc, view = 0, dy = 0, dx = 0, tap0;
          int nsub_a = nsub;
          if (P.s2x) {                  // a = row parity: even rows from y0 (taps ky=1), odd rows from y0-1 (ky=0,2)
            cc = 0; view = a; dy = a ? -1 : 0; dx = -1; tap0 = 0; nsub_a = a ? 6 : 3;
          } else if (P.patch1) {        // one 18x24 box per channel chunk: rows y0-1 .. y0+16, columns x0-1 .. x0+22
            cc = a; dy = -1; dx = -1; tap0 = 0;
          } else if (P.patch_mode) {    // one 18x16 box per (channel chunk, kx); rows y0-1 .. y0+16
            cc = a / 3; const int kx = patch_kx(a % 3, P.xpair);
            dy = -1; dx = kx - 1; tap0 = kx;
          } else {
            const int tap = a / P.cchunks; cc = a % P.cchunks; tap0 = tap;
            if (P.ksz == 3) {
              const int ky = tap / 3, kx = tap % 3;
              if (P.stride == 1) { dy = ky - 1; dx = kx - 1; }
              else {  // input row 2*oy + ky - 1 = 2*(oy + dy) + py
                const int py = (ky == 1) ? 0 : 1, px = (kx == 1) ? 0 : 1;
                dy = (ky == 0) ? -1 : 0; dx = (kx == 0) ? -1 : 0;
                view = py * 2 + px;
              }
            }
          }
          mbar_wait(emptyA(sa), pha ^ 1u);
          if (elect_one_sync()) {
            mbar_expect_tx(fullA(sa), P.a_stage_bytes);
            tma_load_4d(a_base + (uint32_t)sa * P.a_stage_bytes, &P.tmA[view], fullA(sa), cc * CK, x0 + dx, y0 + dy, n);
          }
          __syncwarp();
          if (++sa == SA) { sa = 0; pha ^= 1u; }
          if (!P.b_resident) {
            for (int sub = 0; sub < nsub_a; ++sub) {
              // weight block order = the issuer's tap order (single box: ky-major, kx 1,0,2 for x-paired convs;
              // stride-2 pairs: ky=1 with the even-row box, then ky=0 and ky=2 with the odd-row box)
              const int tap = P.s2x ? (a == 0 ? 3 + sub : (sub < 3 ? sub : 3 + sub))
                                    : (P.patch1 ? (sub / 3) * 3 + patch_kx(sub % 3, P.xpair) : (P.patch_mode ? sub * 3 + tap0 : tap0));
              mbar_wait(emptyB(sb), phb ^ 1u);
              if (elect_one_sync()) {
                mbar_expect_tx(fullB(sb), P.b_block_bytes);
                tma_load_2d(b_base + (uint32_t)sb * P.b_block_bytes, &P.tmB, fullB(sb), tap * P.cin_pad + cc * CK, n_off);
              }
              __syncwarp();
              if (++sb == SB) { sb = 0; phb ^= 1u; }
            }
          }
        }
      }
    }
  } else if (warp < EPI_WARP0) {
    // ====================================================================== MMA issuer(s)
    // ONE elected thread per issuing warp runs the whole issue loop.  It is a single dependent instruction stream, so
    // every integer / branch instruction in it sits on the tensor pipe's critical path (ncu source view: the issuing
    // warp never waited for data, it spent its time on its own bookkeeping).  Hence: mode flags are template
    // constants, the tap / k-step loops are fully unrolled, descriptors advance by adding constants to one 32-bit
    // word -- and with DUAL the two halves of the super-tile have an issuer each (warp 1: left 8 columns, warp 2:
    // right 8 columns), each with its own accumulator and its own full/empty barriers towards the epilogue.
    if (RESIDENT) { mbar_wait(bres_bar, 0); tc_fence_after(); }
    if (elect_one_sync()) {
      constexpr int NH = DUAL ? 1 : 2;                 // halves issued by this thread
      const int h0 = DUAL ? warp - 1 : 0;              // first half issued by this thread
      // descriptor words that never change (see make_smem_desc): hi = SBO | version | layout, lo = addr>>4 | LBO
      const uint32_t hi_a = (Cfg::kSBO_A >> 4) | (1u << 14) | (Cfg::kLayout << 29);
      const uint32_t hi_b = (Cfg::kAtom >> 4) | (1u << 14) | (Cfg::kLayout << 29);
      const uint32_t lo_flags = 1u << 16;
      const uint32_t idesc = P.idesc, idesc_half = P.idesc_half, acc_stride = (uint32_t)P.acc_stride;
      const uint32_t b_block16 = P.b_block_bytes >> 4, a_stage16 = P.a_stage_bytes >> 4;
      // the right half's rows start one swizzle atom (8 pixels) into every image row of the box
      const uint32_t a_lo_base = (((a_base >> 4) & 0x3FFF) | lo_flags) + (uint32_t)h0 * (Cfg::kAtom >> 4);
      const uint32_t b_lo_base = ((b_base >> 4) & 0x3FFF) | lo_flags;   // (shadowed per virtual tile below)
      const int cchunks = P.cchunks, ksteps = P.ksteps, taps = P.taps;
      const bool full_k = ksteps == CK / 16;
      int sa = 0, sb = 0;
      uint32_t pha = 0, phb = 0;
      int it = 0;
      // the MMAs of one (A stage, tap): this thread's half / halves of the super-tile, every k16 step of the chunk
      auto issue_hi = [&](uint32_t d0, uint32_t a_tap, uint32_t hi_a, uint32_t b_lo, uint32_t first, int kx) {
        if (DIAG && (P.debug & 1)) return;
        if (XPAIR && kx != 1) {
          // side taps of the x-paired conv connect ONE pixel of the neighbouring pair to ONE of ours: a 32x32
          // corner of the 64x64 block.  left pair (kx 0): K 32..63 -> N 0..31; right pair (kx 2): K 0..31 -> N 32..63
          const int ks0 = kx == 0 ? 2 : 0;
          const uint32_t dcol = kx == 0 ? 0u : 32u, brow = kx == 0 ? 0u : ((32u * Cfg::kRowBytes) >> 4);
#pragma unroll
          for (int ks = ks0; ks < ks0 + 2; ++ks) {
            const uint32_t f = (ks == ks0) ? first : 1u;
#pragma unroll
            for (int hh = 0; hh < NH; ++hh)
              umma_f16_lohi(d0 + hh * acc_stride + dcol, a_tap + hh * (Cfg::kAtom >> 4) + ks * 2, hi_a, b_lo + brow + ks * 2, hi_b, idesc_half, f);
          }
        } else if (full_k) {   // one straight-line block: nothing between the MMAs but descriptor adds
#pragma unroll
          for (int ks = 0; ks < CK / 16; ++ks) {
            const uint32_t f = (ks == 0) ? first : 1u;
#pragma unroll
            for (int hh = 0; hh < NH; ++hh)
              umma_f16_lohi(d0 + hh * acc_stride, a_tap + hh * (Cfg::kAtom >> 4) + ks * 2, hi_a, b_lo + ks * 2, hi_b, idesc, f);
          }
        } else {               // 33/34-channel inputs: the zero-filled tail of the chunk is skipped
#pragma unroll
          for (int ks = 0; ks < CK / 16; ++ks) {
            if (ks < ksteps) {
              const uint32_t f = (ks == 0) ? first : 1u;
#pragma unroll
              for (int hh = 0; hh < NH; ++hh)
                umma_f16_lohi(d0 + hh * acc_stride, a_tap + hh * (Cfg::kAtom >> 4) + ks * 2, hi_a, b_lo + ks * 2, hi_b, idesc, f);
            }
          }
        }
      };
      auto issue = [&](uint32_t d0, uint32_t a_tap, uint32_t b_lo, uint32_t first, int kx) { issue_hi(d0, a_tap, hi_a, b_lo, first, kx); };
      const uint32_t b_lo_base0 = b_lo_base;
      for (int vt = blockIdx.x; vt < P.total_tiles * P.nsplit; vt += gridDim.x, ++it) {
        const int buf = nbuf == 2 ? (it & 1) : 0;
        const uint32_t use = nbuf == 2 ? ((uint32_t)it >> 1) : (uint32_t)it;   // how often this buffer was used before
#pragma unroll
        for (int hh = 0; hh < NH; ++hh) mbar_wait(tmem_empty(buf, h0 + hh), (use & 1u) ^ 1u);  // epilogue drained the accumulator(s)
        tc_fence_after();
        const uint32_t d0 = tmem_base + (uint32_t)(buf * 2 + h0) * acc_stride;
        // resident weights hold all N rows: this virtual tile multiplies rows [n_off, n_off + nsub)
        const uint32_t b_lo_base = b_lo_base0 + (RESIDENT ? (uint32_t)((vt % P.nsplit) * P.nsub) * (Cfg::kRowBytes >> 4) : 0u);
        if (S2X) {
          // two A stages per tile (even-row box, odd-row box); tap (ky,kx): row offset (ky == 2), pair-column offset
          // (kx != 0), K half (kx != 1) -> k-steps {0,1} or {2,3} of the 64-wide row, same k-steps of the weight block
          constexpr uint32_t SBO1 = P1_PITCH * Cfg::kRowBytes;
          const uint32_t hi1 = (SBO1 >> 4) | (1u << 14) | (Cfg::kLayout << 29);
#pragma unroll
          for (int v = 0; v < 2; ++v) {
            mbar_wait(fullA(sa), pha);
            tc_fence_after();
            const uint32_t a_lo = a_lo_base + (uint32_t)sa * a_stage16;
#pragma unroll
            for (int t9 = 0; t9 < 6; ++t9) {
              if (v == 0 && t9 >= 3) continue;
              const int ky = v == 0 ? 1 : (t9 < 3 ? 0 : 2), kx = t9 % 3;
              uint32_t b_lo;
              if (RESIDENT) b_lo = b_lo_base + (uint32_t)(ky * 3 + kx) * b_block16;
              else { mbar_wait(fullB(sb), phb); tc_fence_after(); b_lo = b_lo_base + (uint32_t)sb * b_block16; }
              const uint32_t a_tap = a_lo + (uint32_t)((ky == 2 ? P1_PITCH : 0) + (kx != 0 ? 1 : 0)) * (Cfg::kRowBytes >> 4);
              const int ks0 = kx == 1 ? 0 : 2;
              if (!(DIAG && (P.debug & 1))) {
#pragma unroll
                for (int ks = ks0; ks < ks0 + 2; ++ks) {
                  const uint32_t f = (v == 0 && t9 == 0 && ks == ks0) ? 0u : 1u;
#pragma unroll
                  for (int hh = 0; hh < NH; ++hh)
                    umma_f16_lohi(d0 + hh * acc_stride, a_tap + hh * (Cfg::kAtom >> 4) + ks * 2, hi1, b_lo + ks * 2, hi_b, idesc, f);
                }
              }
              if (!RESIDENT) { umma_commit(emptyB(sb)); if (++sb == SB) { sb = 0; phb ^= 1u; } }
            }
            umma_commit(emptyA(sa));
            if (++sa == SA) { sa = 0; pha ^= 1u; }
          }
        } else if (P1) {
          // one A stage per channel chunk; tap (ky,kx) starts (ky * 24 + kx) pixels into it (+ 8 for the right half)
          constexpr uint32_t SBO1 = P1_PITCH * Cfg::kRowBytes;
          for (int cc = 0; cc < cchunks; ++cc) {
            mbar_wait(fullA(sa), pha);
            tc_fence_after();
            const uint32_t a_lo = a_lo_base + (uint32_t)sa * a_stage16;
#pragma unroll
            for (int ky = 0; ky < 3; ++ky) {
#pragma unroll
              for (int i = 0; i < 3; ++i) {
                const int kx = XPAIR ? (i == 0 ? 1 : (i == 1 ? 0 : 2)) : i;
                uint32_t b_lo;
                if (RESIDENT) b_lo = b_lo_base + (uint32_t)((ky * 3 + kx) * cchunks + cc) * b_block16;
                else { mbar_wait(fullB(sb), phb); tc_fence_after(); b_lo = b_lo_base + (uint32_t)sb * b_block16; }
                const uint32_t first = (ky == 0 && i == 0) ? (cc != 0 ? 1u : 0u) : 1u;
                // base offset 0: the swizzle phase comes from the absolute address (see MODE_P1 above)
                const uint32_t hi1 = (SBO1 >> 4) | (1u << 14) | (Cfg::kLayout << 29);
                issue_hi(d0, a_lo + (uint32_t)(ky * P1_PITCH + kx) * (Cfg::kRowBytes >> 4), hi1, b_lo, first, kx);
                if (!RESIDENT) { umma_commit(emptyB(sb)); if (++sb == SB) { sb = 0; phb ^= 1u; } }
              }
            }
            umma_commit(emptyA(sa));
            if (++sa == SA) { sa = 0; pha ^= 1u; }
          }
        } else if (PATCH) {
          // one A stage per (channel chunk, kx): rows y0-1 .. y0+16, the three ky taps are 16-pixel row shifts
          for (int cc = 0; cc < cchunks; ++cc) {
#pragma unroll
            for (int i = 0; i < 3; ++i) {
              const int kx = XPAIR ? (i == 0 ? 1 : (i == 1 ? 0 : 2)) : i;
              mbar_wait(fullA(sa), pha);
              tc_fence_after();
              const uint32_t a_lo = a_lo_base + (uint32_t)sa * a_stage16;
#pragma unroll
              for (int sub = 0; sub < 3; ++sub) {
                uint32_t b_lo;
                if (RESIDENT) b_lo = b_lo_base + (uint32_t)((sub * 3 + kx) * cchunks + cc) * b_block16;
                else { mbar_wait(fullB(sb), phb); tc_fence_after(); b_lo = b_lo_base + (uint32_t)sb * b_block16; }
                const uint32_t first = (i == 0 && sub == 0) ? (cc != 0 ? 1u : 0u) : 1u;
                issue(d0, a_lo + (uint32_t)sub * (Cfg::kSBO_A >> 4), b_lo, first, kx);
                if (!RESIDENT) { umma_commit(emptyB(sb)); if (++sb == SB) { sb = 0; phb ^= 1u; } }
              }
              umma_commit(emptyA(sa));  // this issuer's MMAs have read the A stage
              if (++sa == SA) { sa = 0; pha ^= 1u; }
            }
          }
        } else {
          // one A stage per (tap, channel chunk)
          uint32_t first = 0u, b_res = b_lo_base;
          for (int tap = 0; tap < taps; ++tap) {
            for (int cc = 0; cc < cchunks; ++cc) {
              mbar_wait(fullA(sa), pha);
              tc_fence_after();
              uint32_t b_lo;
              if (RESIDENT) { b_lo = b_res; b_res += b_block16; }
              else { mbar_wait(fullB(sb), phb); tc_fence_after(); b_lo = b_lo_base + (uint32_t)sb * b_block16; }
              issue(d0, a_lo_base + (uint32_t)sa * a_stage16, b_lo, first, 1);
              first = 1u;
              if (!RESIDENT) { umma_commit(emptyB(sb)); if (++sb == SB) { sb = 0; phb ^= 1u; } }
              umma_commit(emptyA(sa));
              if (++sa == SA) { sa = 0; pha ^= 1u; }
            }
          }
        }
#pragma unroll
        for (int hh = 0; hh < NH; ++hh) umma_commit(tmem_full(buf, h0 + hh));  // this thread's accumulator(s) complete
      }
    }
    __syncwarp();
  } else {
    // ========================================================================= epilogue
    const int q = warp & 3;                // TMEM lane quadrant this warp may access
    const int h = (warp - EPI_WARP0) >> 2; // which half (accumulator) of the super-tile
    const int r = q * 32 + lane;
    // TMA-store path: a warp's direct stores put every lane on its own 128-byte line (32 LSU wavefronts per
    // instruction -- ncu: l1tex data pipe 77 % busy, the epilogue was the bound of the N = 64 layers); staging
    // the slab in swizzled shared memory costs 4 wavefronts per instruction and the TMA unit writes whole lines.
    const bool tma_out = P.tma_out != 0;
    const uint32_t stage_row = stage_base + (uint32_t)h * 16384u + (uint32_t)r * 128u;
    const uint32_t stage_sw = (uint32_t)(r & 7);
    int it = 0;
    pdl_wait();   // residual / per-image bias reads and every output write wait for the previous kernel
    if (P.epi_staged && !DIAG) {
      // ------------------------------------------------- staged epilogue (N multiple of 64, 16-bit output, shared bias)
      // Direct global accesses put every lane of a warp on its own 128-byte line (32 LSU wavefronts per instruction,
      // ncu: l1tex data pipe 77 % busy) and keep the residual's DRAM latency inside the per-tile critical path.
      // Here the unit of work is a SLAB = the warp's 32 pixels (4 rows x 8 columns of the half tile) x 64 channels =
      // 4 KB, the 128B-swizzled image of a TMA box {64, 8, 4}.  Every epilogue warp owns a ring of NB such buffers and
      // walks the slabs of its tiles in order (slab k = (tile k / G, channels 64 (k % G) ..), G = N / 64):
      //   * the residual of slab k is fetched into buffer k % NB by a TMA load (asynchronous, its own mbarrier) as soon
      //     as the store that last used that buffer has finished reading it -- up to NB-1 slabs ahead, i.e. the DRAM
      //     latency of the residual overlaps the processing of the previous slabs / the next tile's MMAs;
      //   * a thread reads / rewrites only its own 128-byte row (conflict-free 16-byte accesses);
      //   * the finished slab leaves with one TMA store.
      // Synchronisation is per warp only: __syncwarp + proxy fences, bulk-group waits, no CTA-wide barrier.
      const int wi = warp - EPI_WARP0;
      const int NB = P.epi_nb, G = P.nsub >> 6;
      const uint32_t my_stage = stage_base + (uint32_t)(wi * NB) * 4096u;
      const uint32_t sw = (uint32_t)(lane & 7);
      const bool has_res = P.has_res != 0;
      const int vtiles = P.total_tiles * P.nsplit;
      const int my_tiles = ((int)blockIdx.x < vtiles) ? (vtiles - 1 - (int)blockIdx.x) / (int)gridDim.x + 1 : 0;
      const int total_slabs = my_tiles * G;
      // slab k -> image n, pixel origin (tx, ty), tensor channel cg (for TMA) -- cg includes the virtual tile's N offset
      auto slab_xy = [&](int k, int& n, int& tx, int& ty, int& cg) {
        const int vt = (int)blockIdx.x + (k / G) * (int)gridDim.x;
        const int tile = vt / P.nsplit;
        cg = (vt - tile * P.nsplit) * P.nsub + (k % G) * 64;
        n = tile / P.tiles_per_img;
        const int rem = tile % P.tiles_per_img;
        ty = (rem / P.tiles_x) * TILE_Y + 4 * q;
        tx = (rem % P.tiles_x) * TILE_X + h * HALF_X;
      };
      auto load_res = [&](int k) {    // lane 0 only
        int n, tx, ty, cg;
        slab_xy(k, n, tx, ty, cg);
        const int b = k % NB;
        mbar_expect_tx(res_full(wi * 3 + b), 4096u);
        tma_load_4d(my_stage + (uint32_t)b * 4096u, &P.tmRes, res_full(wi * 3 + b), cg, tx, ty, n);
      };
      const int ahead = NB > 1 ? NB - 1 : 1;     // residual loads in flight beyond the slab being processed
      if (has_res && lane == 0)
        for (int k = 0; k < ahead && k < total_slabs; ++k) load_res(k);
      int k = 0;
      for (int vt = blockIdx.x; vt < vtiles; vt += gridDim.x, ++it) {
        const int buf = nbuf == 2 ? (it & 1) : 0;
        const uint32_t use = nbuf == 2 ? ((uint32_t)it >> 1) : (uint32_t)it;
        mbar_wait(tmem_full(buf, h), use & 1u);
        tc_fence_after();
        const uint32_t t_row = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)((buf * 2 + h) * P.acc_stride);
        for (int g = 0; g < G; ++g, ++k) {
          int n, tx, ty, cg;
          slab_xy(k, n, tx, ty, cg);
          const int c0 = g * 64;                                 // column inside the accumulator
          const int b = k % NB;
          const uint32_t row = my_stage + (uint32_t)b * 4096u + (uint32_t)lane * 128u;
          uint32_t v[4][16];
#pragma unroll
          for (int c = 0; c < 4; ++c) tmem_ld16(t_row + (uint32_t)(c0 + c * 16), v[c]);
          tmem_ld_wait();
          if (g == G - 1) {                                      // all TMEM reads of this tile done: accumulator back
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(tmem_empty(buf, h));
          }
          if (has_res) {
            mbar_wait(res_full(wi * 3 + b), (uint32_t)(k / NB) & 1u);   // this slab's residual box has landed
          } else {
            if (lane == 0) {                                     // the store that last used this buffer has read it
              if (NB == 1) bulk_wait_read0(); else if (NB == 2) bulk_wait_read<1>(); else bulk_wait_read<2>();
            }
            __syncwarp();
          }
#pragma unroll
          for (int c = 0; c < 4; ++c) {
            float f[16];
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              const float4 b4 = *reinterpret_cast<const float4*>(s_bias + cg + c * 16 + 4 * i);
              f[4 * i + 0] = __uint_as_float(v[c][4 * i + 0]) + b4.x; f[4 * i + 1] = __uint_as_float(v[c][4 * i + 1]) + b4.y;
              f[4 * i + 2] = __uint_as_float(v[c][4 * i + 2]) + b4.z; f[4 * i + 3] = __uint_as_float(v[c][4 * i + 3]) + b4.w;
            }
            const uint32_t a0 = row + ((((uint32_t)(2 * c)) ^ sw) << 4), a1 = row + ((((uint32_t)(2 * c + 1)) ^ sw) << 4);
            if (has_res) {
              float x[16];
              unpack8<T>(lds128(a0), x);
              unpack8<T>(lds128(a1), x + 8);
#pragma unroll
              for (int i = 0; i < 16; ++i) f[i] += x[i];
            }
            if (P.relu) {
#pragma unroll
              for (int i = 0; i < 16; ++i) f[i] = fmaxf(f[i], 0.f);
            }
            sts128(a0, pack8<T>(f));
            sts128(a1, pack8<T>(f + 8));
          }
          fence_proxy_async_smem();                              // generic-proxy writes -> visible to the TMA unit
          __syncwarp();
          if (lane == 0) {
            tma_store_4d(&P.tmOut, my_stage + (uint32_t)b * 4096u, cg, tx, ty, n);
            bulk_commit();
            const int kn = k + ahead;                            // next residual to fetch
            if (has_res && kn < total_slabs) {
              // its buffer was last used by the store of slab kn - NB: everything but the newest NB-1 groups (the
              // store just committed included) must have finished reading shared memory
              if (NB == 1) bulk_wait_read0(); else if (NB == 2) bulk_wait_read<1>(); else bulk_wait_read<1>();
              load_res(kn);
            }
          }
          __syncwarp();
        }
      }
      if (lane == 0) bulk_wait_all();                            // staging must outlive the stores
    } else
    for (int vt = blockIdx.x; vt < P.total_tiles * P.nsplit; vt += gridDim.x, ++it) {
      const int buf = nbuf == 2 ? (it & 1) : 0;
      const uint32_t use = nbuf == 2 ? ((uint32_t)it >> 1) : (uint32_t)it;
      const int tile = vt / P.nsplit, n_off = (vt - tile * P.nsplit) * P.nsub;   // output channels [n_off, n_off + nsub)
      const int n = tile / P.tiles_per_img, rem = tile % P.tiles_per_img;
      const int oy = (rem / P.tiles_x) * TILE_Y + (r >> 3), ox = (rem % P.tiles_x) * TILE_X + h * HALF_X + (r & 7);
      const size_t pix = ((size_t)n * P.Ho + oy) * P.Wo + ox;
      const int ty0 = (rem / P.tiles_x) * TILE_Y, tx0 = (rem % P.tiles_x) * TILE_X + h * HALF_X;
      const T* resp = P.has_res ? reinterpret_cast<const T*>(P.res) + pix * P.res_stride + n_off : nullptr;
      // bias: per CTA from shared memory, or (folded part-head conv) one row per image from global
      const float* bsrc = P.bias_per_image ? P.bias + (size_t)n * P.npad : s_bias + n_off;
      uint4 rr[4][2];
      if (resp) {   // prefetch the first 64 residual channels while the MMAs are still running
#pragma unroll
        for (int c = 0; c < 4; ++c)
          if (c * 16 < P.nsub) {
            if (P.vec256) ldg256(resp + c * 16, rr[c][0], rr[c][1]);
            else {
              rr[c][0] = *reinterpret_cast<const uint4*>(resp + c * 16);
              rr[c][1] = *reinterpret_cast<const uint4*>(resp + c * 16 + 8);
            }
          }
      }
      mbar_wait(tmem_full(buf, h), use & 1u);
      tc_fence_after();
      if (DIAG && (P.debug & 2)) {
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(tmem_empty(buf, h));
        continue;
      }
      const uint32_t t_row = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)((buf * 2 + h) * P.acc_stride);
      for (int g0 = 0; g0 < P.nsub; g0 += 64) {
        const int nch = min(4, (P.nsub - g0) >> 4);  // 16-column chunks in this group (warp-uniform)
        uint32_t v[4][16];
#pragma unroll
        for (int c = 0; c < 4; ++c)
          if (c < nch) tmem_ld16(t_row + (uint32_t)(g0 + c * 16), v[c]);
        tmem_ld_wait();
        if (g0 + 64 >= P.nsub) {  // all TMEM reads of this tile done: hand the accumulator back
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(tmem_empty(buf, h));
        }
        if (DIAG && (P.debug & 4)) continue;
        if (tma_out) {            // the previous slab's TMA store must have finished READING the staging buffer
          if (r == 0) bulk_wait_read0();
          named_bar_sync(1 + h, 128);
        }
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          if (c >= nch) continue;
          const int c0 = g0 + c * 16;
          float f[16];
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const float4 b4 = P.bias_per_image ? *reinterpret_cast<const float4*>(bsrc + c0 + 4 * i)
                                               : *reinterpret_cast<const float4*>(s_bias + n_off + c0 + 4 * i);   // LDS, not a generic load
            f[4 * i + 0] = __uint_as_float(v[c][4 * i + 0]) + b4.x; f[4 * i + 1] = __uint_as_float(v[c][4 * i + 1]) + b4.y;
            f[4 * i + 2] = __uint_as_float(v[c][4 * i + 2]) + b4.z; f[4 * i + 3] = __uint_as_float(v[c][4 * i + 3]) + b4.w;
          }
          if (P.pow11_ch0 && c0 + n_off == 0) f[0] = powf(1.1f, f[0]);   // cam scale channel (acr/model.py:95-96)
          if (resp) {
            float x[16];
            unpack8<T>(rr[c][0], x);
            unpack8<T>(rr[c][1], x + 8);
#pragma unroll
            for (int i = 0; i < 16; ++i) f[i] += x[i];
            // this chunk's residual registers are free again: fetch the same chunk of the NEXT 64-channel group now,
            // so that its DRAM round trip overlaps the rest of this group (wide layers are HBM bound)
            if (c0 + 64 < P.nsub) {
              if (P.vec256) ldg256(resp + c0 + 64, rr[c][0], rr[c][1]);
              else {
                rr[c][0] = *reinterpret_cast<const uint4*>(resp + c0 + 64);
                rr[c][1] = *reinterpret_cast<const uint4*>(resp + c0 + 64 + 8);
              }
            }
          }
          for (int e = 0; e < P.n_ext; ++e) {   // folded fuse sum: the other terms, nearest-upsampled (warp-uniform loop)
            const T* xp = reinterpret_cast<const T*>(P.ext[e]) +
                          (((size_t)n * P.ext_H[e] + (oy >> P.ext_shift[e])) * P.ext_W[e] + (ox >> P.ext_shift[e])) * P.ext_stride[e] + n_off + c0;
            uint4 u0, u1;
            ldg256(xp, u0, u1);
            float x[16];
            unpack8<T>(u0, x);
            unpack8<T>(u1, x + 8);
#pragma unroll
            for (int i = 0; i < 16; ++i) f[i] += x[i];
          }
          if (P.relu) {
#pragma unroll
            for (int i = 0; i < 16; ++i) f[i] = fmaxf(f[i], 0.f);
          }
          if (P.out_f32) {
            float* o = reinterpret_cast<float*>(P.out) + pix * P.out_stride + n_off + c0;
#pragma unroll
            for (int i = 0; i < 4; ++i) reinterpret_cast<float4*>(o)[i] = make_float4(f[4 * i], f[4 * i + 1], f[4 * i + 2], f[4 * i + 3]);
          } else {
            T* o = reinterpret_cast<T*>(P.out) + pix * P.out_stride + n_off + c0;
            if (tma_out) {
              sts128(stage_row + ((((uint32_t)(2 * c)) ^ stage_sw) << 4), pack8<T>(f));
              sts128(stage_row + ((((uint32_t)(2 * c + 1)) ^ stage_sw) << 4), pack8<T>(f + 8));
            } else if (P.vec256) stg256(o, pack8<T>(f), pack8<T>(f + 8));
            else {
              reinterpret_cast<uint4*>(o)[0] = pack8<T>(f);
              reinterpret_cast<uint4*>(o)[1] = pack8<T>(f + 8);
            }
          }
        }
        if (tma_out) {   // slab complete in shared memory: one thread hands it to the TMA unit
          fence_proxy_async_smem();
          named_bar_sync(1 + h, 128);
          if (r == 0) {
            tma_store_4d(&P.tmOut, stage_base + (uint32_t)h * 16384u, n_off + g0, tx0, ty0, n);
            bulk_commit();
          }
        }
      }
    }
  }
  if (warp >= EPI_WARP0 && P.tma_out && ((warp & 3) * 32 + (threadIdx.x & 31)) == 0) bulk_wait_all();  // staging must outlive the stores
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, (uint32_t)P.tmem_cols);
  }
}

// --------------------------------------------------------------------------------- host side
struct ConvTcPlan {
  ConvTcParams p;
  int ck, act_dtype, grid;
  size_t smem;
};

typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static PFN_encodeTiled get_encode() {
  static PFN_encodeTiled fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<PFN_encodeTiled>(p);
  }
  return fn;
}

static int num_sms() {
  static int n = 0;
  if (!n) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
  }
  return n;
}

static int encode(CUtensorMap* m, int act_dtype, int rank, const void* ptr, const cuuint64_t* dims,
                  const cuuint64_t* strides, const cuuint32_t* box, int ck) {
  PFN_encodeTiled fn = get_encode();
  if (!fn) { set_error("conv_tc: cuTensorMapEncodeTiled unavailable (no CUDA driver?)"); return ACR_B200_ECUDA; }
  cuuint32_t es[5] = {1, 1, 1, 1, 1};
  const CUtensorMapSwizzle sw = ck == 64 ? CU_TENSOR_MAP_SWIZZLE_128B : (ck == 32 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_32B);
  const CUtensorMapDataType dt = act_dtype == ACR_DT_BF16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16;
  CUresult r = fn(m, dt, (cuuint32_t)rank, const_cast<void*>(ptr), dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE, sw,
                  CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) { set_error("conv_tc: cuTensorMapEncodeTiled failed (%d)", (int)r); return ACR_B200_ECUDA; }
  return ACR_B200_OK;
}

// Output tensor map of the staged epilogues: NHWC tensor as {C, W, H, B}, box {64 channels, 8 px, 4 rows, 1}, 128B swizzle
// (one epilogue warp's 32-pixel slab).  Shared with stem_tc.cu.
int encode_slab_store_map(void* tmap, const TensorRef& out, int channels, int batch, int act_dtype) {
  const cuuint64_t esz = 2;
  cuuint32_t box[4] = {64, 8, 4, 1};
  cuuint64_t dims[4] = {(cuuint64_t)channels, (cuuint64_t)out.W, (cuuint64_t)out.H, (cuuint64_t)batch};
  cuuint64_t str[3] = {(cuuint64_t)out.pix_stride * esz, (cuuint64_t)out.W * out.pix_stride * esz, (cuuint64_t)out.H * out.W * out.pix_stride * esz};
  return encode(static_cast<CUtensorMap*>(tmap), act_dtype, 4, out.ptr, dims, str, box, 64);
}

// The TMA-store epilogue is opt-in (ACR_B200_TMA_OUT=1, read at plan creation): on B200 it measured 2 % slower per
// step than direct 256-bit stores (two named barriers per slab and one A stage less outweigh the saved LSU
// wavefronts), see DESIGN.md section 6.  It stays as a tested path for wider-N / store-bound layers.
static bool tma_out_disabled() {
  const char* e = getenv("ACR_B200_TMA_OUT");
  return !(e && atoi(e) != 0);
}

// The single-box A operand (MODE_P1) is on by default; ACR_B200_P1=0 (read at plan creation) selects the three
// kx-shifted boxes again (A/B timing).
static bool p1_enabled() {
  const char* e = getenv("ACR_B200_P1");
  return !(e && atoi(e) == 0);
}

// ACR_B200_NSPLIT=0 (read at plan creation) computes N = 256 layers as one 256-column accumulator per half tile again
// (single-buffered TMEM): A/B timing of the two-halves form.
static bool nsplit_enabled() {
  const char* e = getenv("ACR_B200_NSPLIT");
  return !(e && atoi(e) == 0);
}

// ACR_B200_EPI (read at plan creation): 0 = direct-store epilogue everywhere, 1 (default) = staged epilogue where it
// measured faster (profiles/r2_conv_ab_epilogue.log, r2_conv_ab_singlebox.log): every layer with a residual -- its
// DRAM latency leaves the critical path: 64->256 1x1 + residual 1123 -> 730 us = the HBM copy rate --, every N = 64
// layer (with the single-box operand there is room for the staging buffers next to a whole tile of look-ahead:
// x-paired 32->32 114 -> 101 us) and the wide convs of narrow inputs, 2 = every eligible layer (A/B timing).
static int epi_staged_level() {
  const char* e = getenv("ACR_B200_EPI");
  return e ? atoi(e) : 1;
}

// ACR_B200_CONV_MAX_CTAS=n (read at plan creation, testing only): at most n persistent CTAs, so that small test
// convs run several virtual tiles per CTA (TMEM buffer alternation, barrier phases and staging rings carried
// across tiles, an odd grid for the N split).  Unset or <= 0: one CTA per SM.
static int conv_max_ctas() {
  const char* e = getenv("ACR_B200_CONV_MAX_CTAS");
  return e ? atoi(e) : 0;
}

int conv_tc_prepare(const ConvArgs& a, int act_dtype, ConvTcPlan** out) {
  ACR_CHECK_ARG(a.out.H % TILE_Y == 0 && a.out.W % TILE_X == 0, "conv_tc: output %dx%d is not a multiple of the 16x16 super-tile", a.out.H, a.out.W);
  ACR_CHECK_ARG(a.in.pix_stride % 8 == 0 && a.cin_pad % 16 == 0 && a.cout_pad % 16 == 0 && a.cout_pad <= 1024,
                "conv_tc: channel alignment");
  ACR_CHECK_ARG(a.in.dtype == act_dtype, "conv_tc: input dtype mismatch");
  ACR_CHECK_ARG(!(a.k == 1 && a.stride != 1), "conv_tc: 1x1 stride-2 unsupported");
  ACR_CHECK_ARG(!a.xpair || (a.k == 3 && a.stride == 1 && a.cin_pad == 64 && a.cout_pad == 64 && a.in.pix_stride >= 64),
                "conv_tc: the x-paired form is a 3x3 stride-1 64->64 conv");
  ACR_CHECK_ARG(!a.s2x || (a.k == 3 && a.stride == 2 && a.cin_pad == 64 && a.in.pix_stride == 64 && a.in.C == 64 && !a.xpair &&
                           a.in.H == 2 * a.out.H && a.in.W == a.out.W),
                "conv_tc: the x-paired stride-2 form reads a dense 32-channel tensor as (H, W/2, 64)");
  const int ck = (a.cin_pad % 64 == 0) ? 64 : ((a.cin_pad % 32 == 0) ? 32 : 16);
  ConvTcPlan* pl = new ConvTcPlan();
  ConvTcParams& p = pl->p;
  pl->ck = ck; pl->act_dtype = act_dtype;
  p.patch_mode = (a.k == 3 && a.stride == 1) ? 1 : 0;
  p.patch1 = (p.patch_mode && ck == 64 && p1_enabled()) ? 1 : 0;
  p.s2x = a.s2x ? 1 : 0;
  const cuuint32_t box_rows = p.s2x ? TILE_Y + 1 : (p.patch_mode ? TILE_Y + 2 : TILE_Y);
  const cuuint32_t box_cols = (p.patch1 || p.s2x) ? P1_PITCH : TILE_X;
  const cuuint64_t esz = 2;
  const cuuint64_t dim0 = (cuuint64_t)(a.cin_pad < a.in.pix_stride ? a.cin_pad : a.in.pix_stride);
  int rc = ACR_B200_OK;
  if (a.s2x) {   // two row-parity views of the x-paired input (H, W/2, 64): rows 2r + py
    for (int v = 0; v < 2 && !rc; ++v) {
      const char* ptr = static_cast<const char*>(a.in.ptr) + (size_t)v * a.in.W * a.in.pix_stride * esz;
      cuuint64_t dims[4] = {dim0, (cuuint64_t)a.in.W, (cuuint64_t)a.in.H / 2, (cuuint64_t)a.batch};
      cuuint64_t str[3] = {(cuuint64_t)a.in.pix_stride * esz, (cuuint64_t)2 * a.in.W * a.in.pix_stride * esz,
                           (cuuint64_t)a.in.H * a.in.W * a.in.pix_stride * esz};
      cuuint32_t box[4] = {(cuuint32_t)ck, box_cols, box_rows, 1};
      rc = encode(&p.tmA[v], act_dtype, 4, ptr, dims, str, box, ck);
    }
    for (int v = 2; v < 4 && !rc; ++v) p.tmA[v] = p.tmA[0];
  } else if (a.stride == 1) {
    cuuint64_t dims[4] = {dim0, (cuuint64_t)a.in.W, (cuuint64_t)a.in.H, (cuuint64_t)a.batch};
    cuuint64_t str[3] = {(cuuint64_t)a.in.pix_stride * esz, (cuuint64_t)a.in.W * a.in.pix_stride * esz,
                         (cuuint64_t)a.in.H * a.in.W * a.in.pix_stride * esz};
    cuuint32_t box[4] = {(cuuint32_t)ck, box_cols, box_rows, 1};
    rc = encode(&p.tmA[0], act_dtype, 4, a.in.ptr, dims, str, box, ck);
    for (int v = 1; v < 4 && !rc; ++v) p.tmA[v] = p.tmA[0];
  } else {
    for (int v = 0; v < 4 && !rc; ++v) {
      const int py = v >> 1, px = v & 1;
      const char* ptr = static_cast<const char*>(a.in.ptr) + ((size_t)py * a.in.W + px) * a.in.pix_stride * esz;
      cuuint64_t dims[4] = {dim0, (cuuint64_t)a.in.W / 2, (cuuint64_t)a.in.H / 2, (cuuint64_t)a.batch};
      cuuint64_t str[3] = {(cuuint64_t)2 * a.in.pix_stride * esz, (cuuint64_t)2 * a.in.W * a.in.pix_stride * esz,
                           (cuuint64_t)a.in.H * a.in.W * a.in.pix_stride * esz};
      cuuint32_t box[4] = {(cuuint32_t)ck, TILE_X, box_rows, 1};
      rc = encode(&p.tmA[v], act_dtype, 4, ptr, dims, str, box, ck);
    }
  }
  // N split (see ConvTcParams::nsplit): mandatory above 256 output channels (one UMMA instruction / the TMEM columns),
  // chosen at 256 so that the accumulators are double buffered again (ACR_B200_NSPLIT=0 keeps N = 256 whole)
  int nsplit = 1;
  if (a.cout_pad > 256) {
    nsplit = (a.cout_pad + 255) / 256;
    while (a.cout_pad % nsplit || (a.cout_pad / nsplit) % 16) ++nsplit;
  } else if (a.cout_pad == 256 && a.cin_pad >= 256 && a.k == 3 && !a.bias_per_image && !a.pow11_ch0 && nsplit_enabled()) {
    // measured (profiles/r2_conv_ab_nsplit.log): the MMA-bound 256->256 3x3 layers gain 8-18 % from the double-buffered
    // halves; layers whose weights stream per tile with a short K (34->256, 64->256) lose (each half re-loads A and
    // issues twice the TMA boxes per unit of math), so they keep N = 256 whole
    nsplit = 2;
  }
  const int nsub = a.cout_pad / nsplit;
  ACR_CHECK_ARG(nsub <= 256 && nsub % 16 == 0 && (nsplit == 1 || !a.bias_per_image), "conv_tc: cannot split N = %d", a.cout_pad);
  const bool want_tma_out = a.out.dtype != ACR_DT_F32 && nsub % 64 == 0 && (uintptr_t)a.out.ptr % 16 == 0 &&
                            a.out.pix_stride % 8 == 0 && !tma_out_disabled();
  if (!rc && want_tma_out) {
    cuuint64_t dims[4] = {(cuuint64_t)a.cout_pad, (cuuint64_t)a.out.W, (cuuint64_t)a.out.H, (cuuint64_t)a.batch};
    cuuint64_t str[3] = {(cuuint64_t)a.out.pix_stride * esz, (cuuint64_t)a.out.W * a.out.pix_stride * esz,
                         (cuuint64_t)a.out.H * a.out.W * a.out.pix_stride * esz};
    cuuint32_t box[4] = {64, HALF_X, TILE_Y, 1};
    rc = encode(&p.tmOut, act_dtype, 4, a.out.ptr, dims, str, box, 64);
  }
  // staged epilogue (per-warp TMA store + TMA residual prefetch): N = 64, 16-bit output, shared bias
  const int epi_level = epi_staged_level();
  bool want_staged = !want_tma_out && a.out.dtype != ACR_DT_F32 && nsub % 64 == 0 && (uintptr_t)a.out.ptr % 16 == 0 &&
                     a.out.pix_stride % 8 == 0 && !a.bias_per_image && !a.pow11_ch0 && a.n_ext == 0 &&
                     (!a.has_res || ((uintptr_t)a.res.ptr % 16 == 0 && a.res.pix_stride % 8 == 0)) &&
                     (epi_level >= 2 || (epi_level == 1 && (a.has_res || a.cout_pad == 64 || (a.cout_pad >= 256 && a.cin_pad <= 64))));
  // ring depth per epilogue warp: one buffer when a tile is one slab (the next tile's MMAs hide the residual fetch),
  // otherwise as many (<= 3) as fit next to the operand stages
  int epi_nb = 0;
  if (want_staged) {
    const size_t a_st = (size_t)(box_rows * box_cols) * ck * 2, b_blk = (size_t)nsub * ck * 2;
    const size_t b_tot = a.cout_pad <= 256 ? (size_t)a.k * a.k * (a.cin_pad / ck) * a.cout_pad * ck * 2 : (size_t)1 << 40;
    const size_t min_a0 = (size_t)((p.patch_mode && !p.patch1) ? 3 : 2) * a_st;
    for (int nb = (nsub == 64 ? 1 : 3); nb >= 1 && !epi_nb; --nb) {
      const size_t fx = 1024 + (((size_t)a.cout_pad * 4 + 1023) & ~(size_t)1023) + 512 + (size_t)EPI_WARPS * nb * 4096;
      if (b_tot + min_a0 + fx <= (size_t)SMEM_BUDGET || 4 * b_blk + min_a0 + fx <= (size_t)SMEM_BUDGET) epi_nb = nb;
    }
    if (!epi_nb) want_staged = false;
  }
  if (!rc && want_staged) {
    cuuint32_t box[4] = {64, HALF_X, 4, 1};
    {
      cuuint64_t dims[4] = {(cuuint64_t)a.cout_pad, (cuuint64_t)a.out.W, (cuuint64_t)a.out.H, (cuuint64_t)a.batch};
      cuuint64_t str[3] = {(cuuint64_t)a.out.pix_stride * esz, (cuuint64_t)a.out.W * a.out.pix_stride * esz,
                           (cuuint64_t)a.out.H * a.out.W * a.out.pix_stride * esz};
      rc = encode(&p.tmOut, act_dtype, 4, a.out.ptr, dims, str, box, 64);
    }
    if (!rc && a.has_res) {
      cuuint64_t dims[4] = {(cuuint64_t)a.cout_pad, (cuuint64_t)a.res.W, (cuuint64_t)a.res.H, (cuuint64_t)a.batch};
      cuuint64_t str[3] = {(cuuint64_t)a.res.pix_stride * esz, (cuuint64_t)a.res.W * a.res.pix_stride * esz,
                           (cuuint64_t)a.res.H * a.res.W * a.res.pix_stride * esz};
      rc = encode(&p.tmRes, act_dtype, 4, a.res.ptr, dims, str, box, 64);
    }
  }
  if (rc) { delete pl; return rc; }
  p.epi_staged = want_staged ? 1 : 0;
  p.epi_nb = epi_nb;
  p.n_ext = a.n_ext;
  for (int e = 0; e < a.n_ext; ++e) {
    ACR_CHECK_ARG((uintptr_t)a.ext[e].ptr % 32 == 0 && a.ext[e].pix_stride % 16 == 0 && a.out.dtype != ACR_DT_F32,
                  "conv_tc: extra term %d must be a 16-bit tensor with 32-byte aligned rows", e);
    p.ext[e] = a.ext[e].ptr; p.ext_shift[e] = a.ext_shift[e]; p.ext_stride[e] = a.ext[e].pix_stride;
    p.ext_W[e] = a.ext[e].W; p.ext_H[e] = a.ext[e].H;
  }
  p.bias = a.bias; p.res = a.has_res ? a.res.ptr : nullptr; p.out = a.out.ptr;
  p.taps = a.k * a.k; p.ksz = a.k; p.stride = a.stride; p.cchunks = a.cin_pad / ck; p.cin_pad = a.cin_pad;
  p.ksteps = ck / 16;
  p.vec256 = (a.out.dtype != ACR_DT_F32) && ((uintptr_t)a.out.ptr % 32 == 0) && (a.out.pix_stride % 16 == 0) &&
             (!a.has_res || (((uintptr_t)a.res.ptr % 32 == 0) && (a.res.pix_stride % 16 == 0)));
  if (p.cchunks == 1 && (int)((dim0 + 15) / 16) < p.ksteps) p.ksteps = (int)((dim0 + 15) / 16);
  p.npad = a.cout_pad; p.nsplit = nsplit; p.nsub = nsub;
  p.relu = a.relu; p.has_res = a.has_res; p.out_f32 = a.out.dtype == ACR_DT_F32;
  p.bias_per_image = a.bias_per_image; p.pow11_ch0 = a.pow11_ch0;
  p.xpair = a.xpair;
  { const char* e = getenv("ACR_B200_CONV_DIAG"); p.debug = e ? atoi(e) : 0; }
  p.tiles_x = a.out.W / TILE_X; p.tiles_per_img = p.tiles_x * (a.out.H / TILE_Y);
  p.total_tiles = p.tiles_per_img * a.batch;
  p.Ho = a.out.H; p.Wo = a.out.W; p.out_stride = a.out.pix_stride;
  p.res_stride = a.has_res ? a.res.pix_stride : 0;
  // per super-tile two accumulators (left/right half) of acc_stride columns (power of two >= cout_pad);
  // double buffered when 4 of them fit the 512 TMEM columns
  p.acc_stride = 16;
  while (p.acc_stride < nsub) p.acc_stride *= 2;
  p.nbuf = (4 * p.acc_stride <= 512) ? 2 : 1;
  p.tmem_cols = p.nbuf * 2 * p.acc_stride < 32 ? 32 : p.nbuf * 2 * p.acc_stride;
  // instruction descriptor (cute::UMMA::InstrDescriptor): D=f32, A/B = bf16|f16, K-major both, N, M=128
  const uint32_t fmt = act_dtype == ACR_DT_BF16 ? 1u : 0u;
  p.idesc = (1u << 4) | (fmt << 7) | (fmt << 10) | ((uint32_t)(nsub >> 3) << 17) | ((uint32_t)(TILE_M >> 4) << 24);
  p.idesc_half = (1u << 4) | (fmt << 7) | (fmt << 10) | ((uint32_t)(32 >> 3) << 17) | ((uint32_t)(TILE_M >> 4) << 24);
  // shared-memory plan
  p.a_stage_bytes = (uint32_t)(box_rows * box_cols) * ck * 2;
  // resident weights: every output channel of a (tap, chunk) in one box (<= 256 rows); streamed: one virtual tile's rows
  const size_t b_total = a.cout_pad <= 256 ? (size_t)p.taps * p.cchunks * a.cout_pad * ck * 2 : (size_t)1 << 40;
  p.tma_out = want_tma_out ? 1 : 0;
  p.stage_out_bytes = p.tma_out ? 2u * 16384u : (p.epi_staged ? (uint32_t)(EPI_WARPS * p.epi_nb) * 4096u : 0u);
  p.bias_bytes = (uint32_t)(((size_t)a.cout_pad * 4 + 1023) & ~(size_t)1023);
  const size_t fixed = 1024 /*alignment slack*/ + p.bias_bytes + 512 /*barriers*/ + p.stage_out_bytes;
  const int nA = p.s2x ? 2 : (p.patch1 ? p.cchunks : (p.patch_mode ? p.cchunks * 3 : p.taps * p.cchunks));
  // stages that must fit next to resident weights: a tile's worth of kx patches (3) for 3x3 stride-1 convs, 2 otherwise
  const size_t min_a = (size_t)((p.patch_mode && !p.patch1) ? 3 : 2) * (size_t)p.a_stage_bytes;
  p.b_resident = (b_total + min_a + fixed <= (size_t)SMEM_BUDGET) ? 1 : 0;
  p.b_block_bytes = (uint32_t)(p.b_resident ? a.cout_pad : nsub) * ck * 2;
  {
    const int taps = a.k * a.k;
    cuuint64_t dims[2] = {(cuuint64_t)taps * a.cin_pad, (cuuint64_t)a.cout_pad};
    cuuint64_t str[1] = {(cuuint64_t)taps * a.cin_pad * esz};
    cuuint32_t box[2] = {(cuuint32_t)ck, (cuuint32_t)(p.b_resident ? a.cout_pad : nsub)};
    rc = encode(&p.tmB, act_dtype, 2, a.w, dims, str, box, ck);
    if (rc) { delete pl; return rc; }
  }
  if (p.b_resident) {
    p.b_region_bytes = (uint32_t)((b_total + 1023) & ~(size_t)1023);
    p.SB = 0;
  } else {
    p.SB = 4;
    while (p.SB > 2 && (size_t)p.SB * p.b_block_bytes + min_a + fixed > (size_t)SMEM_BUDGET) --p.SB;
    p.b_region_bytes = (uint32_t)(((size_t)p.SB * p.b_block_bytes + 1023) & ~(size_t)1023);
  }
  int SA = (int)(((size_t)SMEM_BUDGET - fixed - p.b_region_bytes) / p.a_stage_bytes);
  if (SA > 8) SA = 8;
  if (SA > 2 * nA && !p.patch1) SA = 2 * nA;  // no point in more stages than two super-tiles' worth of loads
  if ((p.patch1 || p.s2x) && SA > 4) SA = 4;
  if (SA < 2) { set_error("conv_tc: shared memory plan does not fit (cout_pad %d, ck %d)", a.cout_pad, ck); delete pl; return ACR_B200_EINVAL; }
  p.SA = SA;
  pl->smem = fixed + p.b_region_bytes + (size_t)SA * p.a_stage_bytes;
  pl->grid = p.total_tiles * nsplit < num_sms() ? p.total_tiles * nsplit : num_sms();
  const int cap = conv_max_ctas();
  if (cap > 0 && pl->grid > cap) pl->grid = cap;
  *out = pl;
  return ACR_B200_OK;
}

static bool pdl_enabled() {   // ACR_B200_PDL=0 disables programmatic dependent launch (A/B timing, debugging)
  static int v = -1;
  if (v < 0) { const char* e = getenv("ACR_B200_PDL"); v = e ? atoi(e) : 1; }
  return v != 0;
}

template <int CK, typename T, int MODE>
static int launch_inst(const ConvTcPlan* pl, cudaStream_t st) {
  static unsigned long long configured = 0;
  ACR_CHECK_CUDA(ensure_dynamic_smem(conv_tc_kernel<CK, T, MODE>, SMEM_BUDGET, &configured));
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(pl->grid); cfg.blockDim = dim3(TC_THREADS); cfg.dynamicSmemBytes = pl->smem; cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr; cfg.numAttrs = pdl_enabled() ? 1 : 0;
  ACR_CHECK_CUDA(cudaLaunchKernelEx(&cfg, conv_tc_kernel<CK, T, MODE>, pl->p));
  return ACR_B200_OK;
}

// MODE bits of the kernel instance that runs a plan, or -1 (error set) when no instance exists for it
static int plan_mode(const ConvTcPlan* pl) {
  const ConvTcParams& p = pl->p;
  const int mode = (p.patch_mode ? MODE_PATCH : 0) | (p.b_resident ? MODE_RESIDENT : 0);
  if (pl->ck == 64 && p.s2x) {
    if (p.debug) { set_error("conv_tc: no diagnostic instance of the x-paired stride-2 form"); return -1; }
    return MODE_S2X | (p.b_resident ? MODE_RESIDENT : 0);
  }
  if (pl->ck == 64 && p.patch1) {
    if (p.debug) { set_error("conv_tc: diagnostic instances exist for the three-box form only (ACR_B200_P1=0)"); return -1; }
    if (p.xpair && !p.b_resident) { set_error("conv_tc: x-paired conv needs resident weights"); return -1; }
    return mode | MODE_P1 | (p.xpair ? MODE_XPAIR : 0);
  }
  if (p.debug) {
    if (pl->ck != 64 || mode != (MODE_PATCH | MODE_RESIDENT)) { set_error("conv_tc: diagnostic instances exist for CK=64 patch/resident only"); return -1; }
    return mode | MODE_DIAG | (p.xpair ? MODE_XPAIR : 0);
  }
  if (pl->ck == 64 && p.xpair) {
    if (mode != (MODE_PATCH | MODE_RESIDENT)) { set_error("conv_tc: x-paired conv needs resident weights"); return -1; }
    return mode | MODE_XPAIR;
  }
  return mode;
}

template <int CK, typename T>
static int launch_mode(const ConvTcPlan* pl, cudaStream_t st) {
  constexpr int PR = MODE_PATCH | MODE_RESIDENT;
  switch (plan_mode(pl)) {
    case -1: return ACR_B200_EINVAL;
    case 0: return launch_inst<CK, T, 0>(pl, st);
    case MODE_PATCH: return launch_inst<CK, T, MODE_PATCH>(pl, st);
    case MODE_RESIDENT: return launch_inst<CK, T, MODE_RESIDENT>(pl, st);
    case PR: return launch_inst<CK, T, PR>(pl, st);
    // the remaining forms exist for CK = 64 only (plan_mode never picks them otherwise)
    case MODE_S2X: return launch_inst<64, T, MODE_S2X>(pl, st);
    case MODE_S2X | MODE_RESIDENT: return launch_inst<64, T, MODE_RESIDENT | MODE_S2X>(pl, st);
    case MODE_PATCH | MODE_P1: return launch_inst<64, T, MODE_PATCH | MODE_P1>(pl, st);
    case PR | MODE_P1: return launch_inst<64, T, PR | MODE_P1>(pl, st);
    case PR | MODE_XPAIR | MODE_P1: return launch_inst<64, T, PR | MODE_XPAIR | MODE_P1>(pl, st);
    case PR | MODE_XPAIR: return launch_inst<64, T, PR | MODE_XPAIR>(pl, st);
    case PR | MODE_DIAG: return launch_inst<64, T, PR | MODE_DIAG>(pl, st);
    case PR | MODE_XPAIR | MODE_DIAG: return launch_inst<64, T, PR | MODE_XPAIR | MODE_DIAG>(pl, st);
    default: set_error("conv_tc: no kernel instance for MODE %d", plan_mode(pl)); return ACR_B200_EINVAL;
  }
}

int conv_tc_launch(const ConvTcPlan* pl, cudaStream_t st) {
  const bool bf = pl->act_dtype == ACR_DT_BF16;
  switch (pl->ck) {
    case 64: return bf ? launch_mode<64, __nv_bfloat16>(pl, st) : launch_mode<64, __half>(pl, st);
    case 32: return bf ? launch_mode<32, __nv_bfloat16>(pl, st) : launch_mode<32, __half>(pl, st);
    default: return bf ? launch_mode<16, __nv_bfloat16>(pl, st) : launch_mode<16, __half>(pl, st);
  }
}

int conv_tc_describe(const ConvTcPlan* pl, int32_t* info, int n_info) {
  const int mode = plan_mode(pl);
  if (mode < 0) return ACR_B200_EINVAL;
  const ConvTcParams& p = pl->p;
  int32_t v[ACR_CONV_INFO_N] = {};
  v[ACR_CONV_INFO_CK] = pl->ck;
  v[ACR_CONV_INFO_MODE] = mode;
  v[ACR_CONV_INFO_B_RESIDENT] = p.b_resident;
  v[ACR_CONV_INFO_NSPLIT] = p.nsplit;
  v[ACR_CONV_INFO_NSUB] = p.nsub;
  v[ACR_CONV_INFO_NBUF] = p.nbuf;
  v[ACR_CONV_INFO_EPILOGUE] = p.tma_out ? 2 : (p.epi_staged ? 1 : 0);
  v[ACR_CONV_INFO_EPI_NB] = p.epi_nb;
  v[ACR_CONV_INFO_SA] = p.SA;
  v[ACR_CONV_INFO_SB] = p.SB;
  v[ACR_CONV_INFO_GRID] = pl->grid;
  v[ACR_CONV_INFO_VTILES] = p.total_tiles * p.nsplit;
  for (int i = 0; i < n_info && i < ACR_CONV_INFO_N; ++i) info[i] = v[i];
  return ACR_B200_OK;
}

void conv_tc_free(ConvTcPlan* p) { delete p; }

}  // namespace acr
