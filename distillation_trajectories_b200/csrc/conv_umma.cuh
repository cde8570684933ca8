// tcgen05 / TMA implicit-GEMM convolution for sm_100a (DTRAJ_PREC_F16, DTRAJ_PREC_TF32, DTRAJ_PREC_TF32X3).
//
// GEMM view of one conv layer (models.py:48-57):  D[M, N] = A[M, K] * B[K, N]
//   M = n_img*H*W output pixels, N = coutp, K = ntaps * (c0p + c1p).
// A is never materialised: with NHWC feature maps a 3x3 tap is a SHIFTED 4-d box of the
// input tensor, so one TMA box load {128 bytes of channels, W, Hb, Nb} at coordinates
// {c0, dx, y0+dy, img0} delivers the 128-row im2col tile of tap (dy,dx) straight into the
// 128-byte-swizzled K-major layout tcgen05.mma reads; out-of-bounds rows/columns (the
// conv's zero padding) are zero-filled by the TMA unit.  The channel concat of the decoder
// blocks (models.py:206,211,216) is two tensor maps feeding consecutive K blocks.  A K block
// (128 bytes per row) is 32 fp32 channels (kind::tf32) or 64 fp16 channels (kind::f16).
//
// Roles (320 threads, one persistent CTA per SM, optionally CTA pairs with cta_group::2):
// warp 0 = TMA producer + TMEM allocator, warp 1 = MMA issuer (one elected lane), warps 2-9 =
// epilogue (TMEM -> registers -> bias / ReLU / time-bias / residual / fused tails -> swizzled
// ring buffer -> TMA store).  A `stages`-deep mbarrier ring connects producer and issuer; two
// fp32 accumulator sets (128 lanes x N columns) live in TMEM so that the epilogue of tile i
// overlaps the MMAs of tile i+1.
//
// 3xTF32 (DTRAJ_PREC_TF32X3): the K loop runs three passes  A_hi*B_hi + A_hi*B_lo + A_lo*B_hi
// (the two cross terms into a separate accumulator), where x_lo = x - trunc_tf32(x) is kept in a
// second plane by every producer of an activation (ACT_SPLIT) and the weights are split on the host.
#pragma once
#include <type_traits>
#include <cstdlib>
#include <cuda_fp16.h>
#include "common.cuh"
#include "conv_simt.cuh"

namespace dtraj {

// Device-side error words (bit 0: a pipeline role timed out on an mbarrier -- it would otherwise hang the GPU; bit 1:
// fp16 mode, an activation left the fp16 range).  Every dtraj_unet handle owns one word (ConvLayer::err, Enc1*Params::err), so
// that two models running on two streams can tell whose launch failed; launches without a handle (dtraj_test_conv,
// dtraj_bench_conv) report to this library-wide word.
__device__ unsigned int g_umma_error = 0;
#ifdef DTRAJ_PROBES
// Probe build only (tools/timeline.py): SM-clock stamps of CTA 0's issuer and two of its epilogue warps over its first 16 tiles of a
// 256-column CONV_RESACC + CONV_POOL layer at 8x8 -- [this kernel | k_enc1_f16][tile][issuer | epilogue warp 2 | epilogue warp 6][event].
__device__ long long g_timeline[2][16][3][16];
__device__ int g_tl_select[4] = {CONV_RESACC | CONV_POOL, CONV_RESACC | CONV_POOL, 256, 8};     // {flag mask, flag value, coutp, W} of the recorded layer
#define DTRAJ_TL(who, ev) do { if (tl_on && tl_tile < 16) g_timeline[tl_slot][tl_tile][who][ev] = clock64(); } while (0)
#else
#define DTRAJ_TL(who, ev) do { } while (0)
#endif

struct UmmaConv {
    ConvLayer L;               // epilogue parameters + shapes (wpk unused here)
    int npass;                 // 1 (TF32) or 3 (TF32X3)
    int stages;
    int tmem_cols;             // total TMEM columns allocated (power of two): acc_stages x acc_cols
    int acc_cols;              // columns of one accumulator set (x2 for 3 passes: main + correction accumulator)
    int acc_stages;            // 2 when two accumulator sets fit in 512 columns, else 1
    int corr_col;              // offset of the correction accumulator inside a set (3 passes), else 0
    int res_col;               // offset of the residual-conv accumulator inside a set (CONV_RESACC), else 0
    int nch0, nch;             // K chunks (one 128-byte K block per pixel: 32 fp32 / 64 fp16 channels) of source 0 / of both sources
    uint32_t half_mask;        // fp16 mode: bit c set = chunk c holds only 32 real channels (a source padded to an odd multiple of
                               // 32: TMA zero-fills the rest of the box, the weights are zero there, and only 2 of the 4 K = 16
                               // MMAs are issued)
    int r_nch0, r_nch;         // the same counts for the residual conv's sources (CONV_RESACC)
    uint32_t r_half_mask;
    int n_tiles;               // 128-row output tiles
    int n_split;               // column split of a tile when there are fewer tiles than SMs (power of two)
    int ncols;                 // coutp / n_split: columns per work item (multiple of 32)
    int n_work;                // n_tiles * n_split work items; CTA b handles b, b + gridDim.x, ...
    int pair;                  // 1: CTA pairs run tcgen05.mma.cta_group::2 -- M = 256 (two 128-row tiles, one per CTA), each CTA
                               //    stages only ITS half of the weight tile, the leader CTA issues for both
    int kbs;                   // K blocks per pipeline stage (2 when both sources have an even number of them); halo mode: weight tiles (taps) per stage, 1 / 3 / 9
    int epi_bufs;              // epilogue ring depth per warp (1 when the freed 32 KB buy another operand stage)
    int posm;                  // position-major tiles (fp16, maps of <= 4x4): a tile = ONE output position of 128 images, K loop over
                               //    the taps that fall inside the map only; nblk_img = tiles per position
    int nblk_img;
    int epi_kind;              // fp16 epilogue: 1..4 = one of the flag sets compiled as straight-line code (epi_kind_of), 0 = generic
    int box_h, box_n;          // A box = {32, W, box_h, box_n}
    int tiles_per_img;         // >= 1
    int b_lo_row;              // row offset of the low-plane weights inside the B tensor map
    int cb;                    // epilogue column block: 128, 64 or 32 (largest that divides coutp)
    int log2_hw;               // H*W is a power of two: image index of output row m is m >> log2_hw
    int log2_wh;               // log2(W / 2) (CONV_POOL)
    int f16;                   // 1: DTRAJ_PREC_F16 -- fp16 feature maps / weights (64 channels per 128-byte K block), kind::f16 MMAs
    int halo;                  // HALO mode (fp16, 3x3): a tile's pixels arrive ONCE per 64-channel chunk as a halo box, the nine taps are
                               //    descriptor views of it.  1: 8x8 maps, a tile = two images, halos [10 rows][2 images][10 pixels] through
                               //    the permuted dimensions {c, x, image, y};  2: 16x16 and 32x32 maps, a tile = 16 rows x 8 columns of one
                               //    image, halo [18 rows][10 pixels] through the standard dimensions {c, x, y, image}
    int n_hb;                  // halo ring depth
    int hlg_x, hlg_t;          // halo mode 2: log2 of the 8-column groups per image (1 at 16x16, 2 at 32x32) and of the tiles per image
                               //    (1, 3): tile t covers image t >> hlg_t, columns from (t & (2^hlg_x - 1)) * 8, rows from the band above
};

// halo mode 2: image, first row and first column of tile `t`
__device__ __forceinline__ void halo2_tile(const UmmaConv& p, int t, int& img, int& y0, int& x0) {
    img = t >> p.hlg_t;
    x0 = (t & ((1 << p.hlg_x) - 1)) * 8;
    y0 = ((t & ((1 << p.hlg_t) - 1)) >> p.hlg_x) * 16;
}

constexpr uint32_t kHaloBytes = 26624;     // 200 halo pixels x 128 B, rounded up to 1024
constexpr uint32_t kHaloTx = 200 * 128;    // bytes one halo box delivers

struct UmmaMaps {              // 64-byte aligned tensor maps, passed as __grid_constant__
    CUtensorMap a[4];          // [src0 hi, src1 hi, src0 lo, src1 lo]
    CUtensorMap b;
    CUtensorMap out;           // [M, coutp] output, box {32 ch, 32 rows}   (epilogue TMA store)
    CUtensorMap out_lo;        // low plane of the output (3xTF32)
    CUtensorMap res;           // [M, coutp] residual, same box             (epilogue TMA load)
    CUtensorMap ra[2];         // CONV_RESACC: the block's input maps (A operand of the fused 1x1 residual conv)
    CUtensorMap rb;            //              its packed weights
};

namespace ptx {
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
    return pred != 0;
}
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
// bounded wait: a protocol bug must surface as an error flag, never as a hung GPU
__device__ __forceinline__ uint32_t mbar_try(uint32_t bar, uint32_t parity) {
    uint32_t ok;
    asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
                 "selp.u32 %0, 1, 0, p;\n\t}"
                 : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
    return ok;
}
__device__ __noinline__ bool mbar_wait_slow(unsigned int* err, uint32_t bar, uint32_t parity) {
#pragma unroll 1
    for (uint32_t i = 0; i < (1u << 22); ++i)
        if (mbar_try(bar, parity)) return true;
    atomicOr(err, 1u);
    return false;
}
__device__ __forceinline__ bool mbar_wait(unsigned int* err, uint32_t bar, uint32_t parity) {
    if (mbar_try(bar, parity)) return true;
    return mbar_wait_slow(err, bar, parity);
}
__device__ __forceinline__ void tma_load_4d(uint32_t dst, const CUtensorMap* map, uint32_t bar,
                                            int c0, int c1, int c2, int c3) {
    asm volatile("cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes "
                 "[%0], [%1, {%3, %4, %5, %6}], [%2];"
                 ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3) : "memory");
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1) {
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes "
                 "[%0], [%1, {%3, %4}], [%2];"
                 ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* map, uint32_t src, int c0, int c1) {
    asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];"
                 ::"l"(map), "r"(src), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void tma_store_4d(const CUtensorMap* map, uint32_t src, int c0, int c1, int c2, int c3) {
    asm volatile("cp.async.bulk.tensor.4d.global.shared::cta.bulk_group [%0, {%2, %3, %4, %5}], [%1];"
                 ::"l"(map), "r"(src), "r"(c0), "r"(c1), "r"(c2), "r"(c3) : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void bulk_wait_read() { asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
// ---- CTA-pair (cta_group::2) forms
__device__ __forceinline__ void tma_load_4d_2sm(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1, int c2, int c3) {
    asm volatile("cp.async.bulk.tensor.4d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes "
                 "[%0], [%1, {%3, %4, %5, %6}], [%2];"
                 ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3) : "memory");
}
__device__ __forceinline__ void tma_load_2d_2sm(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1) {
    asm volatile("cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes "
                 "[%0], [%1, {%3, %4}], [%2];"
                 ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void mma_tf32_2sm(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t acc) {
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
                 "tcgen05.mma.cta_group::2.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
                 ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(acc) : "memory");
}
__device__ __forceinline__ void tc_commit_2sm(uint32_t bar, uint16_t mask) {
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
                 ::"r"(bar), "h"(mask) : "memory");
}
// shared::cluster address of `addr` (a shared::cta address of this CTA) in CTA `rank` of the cluster
__device__ __forceinline__ uint32_t map_to_cta(uint32_t addr, uint32_t rank) {
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
    return r;
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
    asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
// The same arrival WITHOUT release semantics, for barriers that hand over TMEM only ("accumulator drained": the tcgen05.ld results are
// in registers after tcgen05.wait::ld, and tcgen05.fence::before_thread_sync / ::after_thread_sync order the tensor-memory accesses
// around the barrier).  The .release.cluster form compiles to MEMBAR.ALL.GPU + ERRBAR in front of the arrive and waited there for the
// warp's global pool stores: 9 % of the epilogue's stall samples and ~1500 cycles between a tile's last TMEM load and the issuer
// seeing the accumulator free (profiles/r02i_timeline.txt, r02i_epilogue_stalls.txt).
__device__ __forceinline__ void mbar_arrive_cluster_relaxed(uint32_t cluster_addr) {
    asm volatile("mbarrier.arrive.relaxed.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
// ... and with CTA-scope release, for barriers that hand over SHARED MEMORY written by this CTA's threads to the pair's tensor core:
// every writer has executed fence.proxy.async on its stores and been synchronised with the arriving thread (named barrier /
// __syncwarp), so the remote arrival only has to stay behind that synchronisation -- no MEMBAR.ALL.GPU.
__device__ __forceinline__ void mbar_arrive_cluster_cta(uint32_t cluster_addr) {
    asm volatile("mbarrier.arrive.release.cta.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void prefetch_tmap(const CUtensorMap* map) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(map) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mma_tf32(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t acc) {
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
                 "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
                 ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(acc) : "memory");
}
__device__ __forceinline__ void mma_f16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t acc) {
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
                 "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
                 ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(acc) : "memory");
}
__device__ __forceinline__ void mma_f16_2sm(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t acc) {
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
                 "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
                 ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(acc) : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t* v) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x32.b32 "
                 "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
                 "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
                   "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]),
                   "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]),
                   "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
                 : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
}  // namespace ptx

// K-major, 128-byte swizzle shared-memory matrix descriptor (cute::UMMA::SmemDescriptor):
// start>>4 [0,14) | LBO>>4 = 1 [16,30) | SBO>>4 = 1024B/16 [32,46) | version 1 [46,48) | SWIZZLE_128B = 2 [61,64)
__device__ __forceinline__ uint64_t umma_desc_sw128(uint32_t smem_addr) {
    return (uint64_t)((smem_addr >> 4) & 0x3fffu) | ((uint64_t)1 << 16) | ((uint64_t)64 << 32) |
           ((uint64_t)1 << 46) | ((uint64_t)2 << 61);
}
// kind::tf32 instruction descriptor (cute::UMMA::InstrDescriptor): D fp32, A/B tf32, both K-major, M=128
__host__ __device__ inline uint32_t umma_idesc_tf32(int n) {
    return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
}

// kind::f16 instruction descriptor: D fp32, A/B fp16 (format 0), both K-major, M=128; K = 16 per instruction
__host__ __device__ inline uint32_t umma_idesc_f16(int n) {
    return (1u << 4) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
}

constexpr int kEpiWarps = 8;             // two per TMEM lane quarter, each takes every other 32-column chunk
constexpr int kUmmaThreads = 64 + 32 * kEpiWarps;
constexpr int kEpiBufsMax = 2;           // per-warp ring of 4 KB (32 rows x 32 columns) epilogue buffers: 1 or 2
constexpr int kATileBytes = 128 * 128;   // 128 rows x 32 fp32

// Persistent kernel: one CTA per SM walks tiles blockIdx.x, blockIdx.x + gridDim.x, ...  The three roles
// run decoupled: the producer streams operands for tile i+1 while the issuer is still on tile i, and the
// epilogue warps drain accumulator buffer `acc` while the issuer fills the other one (TMEM holds two
// accumulators whenever 2 x columns-per-tile <= 512), so neither the epilogue's latency nor its
// instruction count sits on the tensor pipe's critical path.
template <bool kPair, bool kF16>
__global__ void __launch_bounds__(kUmmaThreads, 1)
k_conv_umma_t(const __grid_constant__ UmmaMaps maps, const UmmaConv p) {
    constexpr int kCh = kF16 ? 64 : 32;      // channels of one 128-byte K block
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    // carve: [stages x (A 16 KB | B coutp*128 B)] [epilogue ring kEpiWarps x kEpiBufs x 4 KB (2 KB in fp16 mode)] [barriers]
    const uint32_t base = (ptx::smem_u32(smem_raw) + 1023u) & ~1023u;
    const int coutp = p.L.coutp;
    const int ncols = p.ncols;                                 // columns this CTA computes per work item (coutp / n_split)
    const int n_rows = ncols;                                  // rows of the N operand tile (UMMA N)
    const uint32_t b_bytes = (uint32_t)(kPair ? n_rows / 2 : n_rows) * 128u;   // N-operand bytes staged in THIS CTA
    // halo mode: a stage holds ONE weight tile (a tap of a chunk); the pixels live in the halo ring behind the stages
    const uint32_t stage_bytes = p.halo ? (uint32_t)p.kbs * b_bytes : (uint32_t)p.kbs * (kATileBytes + b_bytes);   // kbs x [M tile 16 KB] then kbs x [N tile]; halo mode: kbs weight tiles (taps)
    const uint32_t halo_base = base + p.stages * stage_bytes;
    const uint32_t ring_base = halo_base + (p.halo ? (uint32_t)p.n_hb * kHaloBytes : 0u);
    const int kEpiBufs = p.epi_bufs;
    // (an epilogue buffer is [32 rows][32 columns]: 4 KB of floats, 2 KB of halfs -- the fp16 kernels give the other half to the operand ring)
    constexpr uint32_t kEpiBufBytes = kF16 ? 2048u : 4096u;
    const uint32_t bar_base = ring_base + (uint32_t)(kEpiWarps * kEpiBufs) * kEpiBufBytes;
    auto full_bar = [&](int s) { return bar_base + 8u * s; };
    auto empty_bar = [&](int s) { return bar_base + 8u * (p.stages + s); };
    const uint32_t acc_full0 = bar_base + 16u * p.stages;      // [2] accumulator ready   (issuer -> epilogue)
    const uint32_t acc_empty0 = acc_full0 + 16u;               // [2] accumulator drained (epilogue -> issuer)
    const uint32_t res_bar0 = acc_empty0 + 16u;                // [kEpiWarps][kEpiBufs] residual-chunk barriers
    const uint32_t tmem_slot = res_bar0 + 8u * kEpiWarps * kEpiBufsMax;
    const uint32_t hfull0 = tmem_slot + 16u;                   // [4] halo buffer loaded   (TMA -> issuer)
    const uint32_t hempty0 = hfull0 + 32u;                     // [4] halo buffer consumed (issuer -> TMA)
    const uint32_t fin_base = hempty0 + 32u;                   // CONV_FINAL partial sums [4 quarters][32 lanes][4]
    // Per-channel epilogue constants, staged ONCE per CTA: rows of coutp floats [bias | residual-conv bias | time bias x 3 variants |
    // final-1x1 weights x finC].  Read from global memory at their point of use they were the epilogue's bottleneck: with 227 KB of
    // shared memory the L1 keeps ~28 KB, every chunk's ~20 dependent LDGs went to an L2 busy streaming operands at 5 TB/s, and the
    // epilogue warps of the 256-wide residual layers were busy 78 % of the kernel (ncu source view, profiles/r02b_resacc_ab.txt).
    const uint32_t cst_base = fin_base + ((p.L.flags & CONV_FINAL) ? 2048u : 0u);
    float* const cst = reinterpret_cast<float*>(smem_raw + (cst_base - ptx::smem_u32(smem_raw)));
    volatile uint32_t* tmem_slot_ptr = reinterpret_cast<volatile uint32_t*>(
        smem_raw + (tmem_slot - ptx::smem_u32(smem_raw)));

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    unsigned int* const errw = p.L.err ? p.L.err : &g_umma_error;
#ifdef DTRAJ_PROBES
    const bool tl_on = blockIdx.x == 0 && (threadIdx.x & 31) == 0 && (p.L.flags & g_tl_select[0]) == g_tl_select[1] &&
                       p.L.coutp == g_tl_select[2] && p.L.W == g_tl_select[3];
    const int tl_slot = 0;        // (slot 1: k_enc1_f16)
    int tl_tile = 0;
#endif
    const int crank = kPair ? (int)ptx::cluster_ctarank() : 0;
    const uint16_t cmask = kPair ? 3 : 1;
    const int work0 = (int)blockIdx.x - crank;   // first work item of this CTA's cluster; all its CTAs loop alike
    const int nch0 = p.nch0, nch = p.nch;
    const int iters_per_pass = p.L.ntaps * nch;

    if (warp == 0) {
        if (ptx::elect_one()) {
            ptx::prefetch_tmap(&maps.a[0]);
            ptx::prefetch_tmap(&maps.b);
            if (p.L.c1p) ptx::prefetch_tmap(&maps.a[1]);
            for (int s = 0; s < p.stages; ++s) { ptx::mbar_init(full_bar(s), 1); ptx::mbar_init(empty_bar(s), 1); }
            for (int i = 0; i < 2; ++i) {
                ptx::mbar_init(acc_full0 + 8u * i, 1);
                ptx::mbar_init(acc_empty0 + 8u * i, kEpiWarps * (kPair ? 2 : 1));   // pair: both CTAs' epilogues report to the leader
            }
            for (int i = 0; i < kEpiWarps * kEpiBufsMax; ++i) ptx::mbar_init(res_bar0 + 8u * i, 1);
            for (int i = 0; i < 4; ++i) { ptx::mbar_init(hfull0 + 8u * i, 1); ptx::mbar_init(hempty0 + 8u * i, 1); }
            if (!(p.L.flags & CONV_NOSTORE)) ptx::prefetch_tmap(&maps.out);
            if (p.L.flags & CONV_RESID) ptx::prefetch_tmap(&maps.res);
            asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        }
        __syncwarp();
        if constexpr (!kPair) {
            asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;"
                         ::"r"(tmem_slot), "r"((uint32_t)p.tmem_cols) : "memory");
            asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
        } else {
            asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;"
                         ::"r"(tmem_slot), "r"((uint32_t)p.tmem_cols) : "memory");
            asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
        }
    }
    {   // (weights and tables only: nothing here was written by the preceding kernel, so it may run before pdl_wait)
        const int coutp_ = p.L.coutp, fl_ = p.L.flags;
        for (int i = threadIdx.x; i < coutp_; i += blockDim.x) {
            cst[i] = p.L.bias[i];
            if (fl_ & CONV_RESACC) cst[coutp_ + i] = p.L.rbias[i];
            if ((fl_ & CONV_TBIAS) && !p.L.tb_rows)
                for (int v = 0; v < 3; ++v) cst[(2 + v) * coutp_ + i] = p.L.tbias[(size_t)v * p.L.tb_var_stride + i];
        }
        if (fl_ & CONV_FINAL)
            for (int i = threadIdx.x; i < p.L.finC * coutp_; i += blockDim.x) cst[5 * coutp_ + i] = p.L.finw[i];
    }
    ptx::tc_fence_before();
    __syncthreads();
    if constexpr (kPair) ptx::cluster_sync_all(); // the peer's barriers exist before anything arrives on them
    ptx::tc_fence_after();
    const uint32_t tmem_base = *tmem_slot_ptr;
    const float* const bias_s = cst;                           // generic pointers into shared memory
    const float* const rbias_s = cst + p.L.coutp;
    const float* const finw_s = cst + 5 * p.L.coutp;
    pdl_launch_dependents();                   // the next kernel of the stream / graph may start its prologue
    pdl_wait();                                // ... and this one touches activations only after its predecessor is complete
    auto arrive_acc_empty = [&](int acc) {     // "accumulator drained": to this CTA's issuer, or to the pair leader's
        if constexpr (!kPair) ptx::mbar_arrive(acc_empty0 + 8u * acc);
        else ptx::mbar_arrive_cluster_relaxed(ptx::map_to_cta(acc_empty0 + 8u * acc, 0));
    };

    if (warp == 0) {
        // ------------------------------------------------------------ TMA producer
        // One thread.  Its instruction stream, not the memory system, paces short MMAs (ncu: ~750 cycles per
        // iteration of the first persistent version against 128 cycles of MMA work at N = 64), so every index
        // is carried incrementally and a stage holds `kbs` (1 or 2) 32-channel K blocks per barrier round trip.
        if (ptx::elect_one()) {
            const int w_half = kPair ? ncols / 2 : ncols;      // weight rows this CTA fetches (pair: its half of the tile)
            // pair: the LEADER's barrier collects the bytes of both CTAs' loads
            const uint32_t tx_bytes = (uint32_t)p.kbs * ((uint32_t)kATileBytes + b_bytes) * (kPair ? 2u : 1u);
            const uint32_t w_base_off = (uint32_t)p.kbs * kATileBytes;      // the N (weight) slots follow the M (pixel) slots
            int s = 0;
            uint32_t ph = 0;
            bool ok = true;
            if constexpr (kF16) if (p.halo) {
                // ---- halo mode: per 64-channel chunk ONE box {64 ch, 10, 2 images, 10} over the permuted dimensions
                // {c, x, image, y} (out-of-bounds rows / columns zero-filled = the conv's padding), then the nine weight tiles
                int hb = 0;
                uint32_t hph = 0;
                // one stage = `n` weight tiles (taps b_row, b_row + row_step, ...) behind ONE barrier round trip: this thread's
                // instruction stream, not the memory system, paces the N <= 128 layers (an issuer that sends one of the four MMAs
                // of a K block is only 17 % faster on dec1.conv1, 7 % on the sf 0.5 student's: profiles/r02q_ring_ab.txt)
                auto weight_stage = [&](const CUtensorMap* wm, int b_row) -> bool {
                    if (!ptx::mbar_wait(errw, empty_bar(s), ph ^ 1u)) return false;
                    uint32_t fb = full_bar(s);
                    if constexpr (kPair) fb = ptx::map_to_cta(fb, 0);
                    if (!kPair || crank == 0) ptx::mbar_expect_tx(full_bar(s), b_bytes * (kPair ? 2u : 1u));
                    if constexpr (kPair) ptx::tma_load_2d_2sm(base + s * stage_bytes, wm, fb, 0, b_row);
                    else ptx::tma_load_2d(base + s * stage_bytes, wm, fb, 0, b_row);
                    if (++s == p.stages) { s = 0; ph ^= 1u; }
                    return true;
                };
                // kb = 3 or 9 taps' weight tiles (rows b_row, + row_step, ...) behind ONE barrier round trip: the instruction streams of this
                // thread and of the issuer, not the memory system, pace the N <= 128 layers (an issuer that sends one of the four MMAs of
                // a K block is only 17 % faster on dec1.conv1, 7 % on the sf 0.5 student's: profiles/r02q_ring_ab.txt)
                auto weight_stage_n = [&](auto KB, const CUtensorMap* wm, int b_row, int row_step) -> bool {
                    constexpr int kb = decltype(KB)::value;
                    if (!ptx::mbar_wait(errw, empty_bar(s), ph ^ 1u)) return false;
                    uint32_t fb = full_bar(s);
                    if constexpr (kPair) fb = ptx::map_to_cta(fb, 0);
                    if (!kPair || crank == 0) ptx::mbar_expect_tx(full_bar(s), (uint32_t)kb * b_bytes * (kPair ? 2u : 1u));
                    const uint32_t dst = base + s * stage_bytes;
#pragma unroll
                    for (int j = 0; j < kb; ++j) {
                        if constexpr (kPair) ptx::tma_load_2d_2sm(dst + (uint32_t)j * b_bytes, wm, fb, 0, b_row + j * row_step);
                        else ptx::tma_load_2d(dst + (uint32_t)j * b_bytes, wm, fb, 0, b_row + j * row_step);
                    }
                    if (++s == p.stages) { s = 0; ph ^= 1u; }
                    return true;
                };
                // `tile`: this CTA's tile; xy0 = -1: the halo box of a 3x3 tap set, 0: the un-shifted 128 pixels (residual conv)
                auto pixel_box = [&](const CUtensorMap* am, int c0, int xy0, int tile, uint32_t bytes) -> bool {
                    if (!ptx::mbar_wait(errw, hempty0 + 8u * hb, hph ^ 1u)) return false;
                    uint32_t fb = hfull0 + 8u * hb;
                    if constexpr (kPair) fb = ptx::map_to_cta(fb, 0);
                    if (!kPair || crank == 0) ptx::mbar_expect_tx(hfull0 + 8u * hb, bytes * (kPair ? 2u : 1u));
                    // mode 1: dims {c, x, image, y}, two images from 2 * tile;  mode 2: dims {c, x, y, image}, 16 x 8 pixels from (y0, x0)
                    int k1 = xy0, k2 = 2 * tile, k3 = xy0;
                    if (p.halo == 2) { int ty, tx; halo2_tile(p, tile, k3, ty, tx); k1 = tx + xy0; k2 = ty + xy0; }
                    if constexpr (kPair) ptx::tma_load_4d_2sm(halo_base + hb * kHaloBytes, am, fb, c0, k1, k2, k3);
                    else ptx::tma_load_4d(halo_base + hb * kHaloBytes, am, fb, c0, k1, k2, k3);
                    if (++hb == p.n_hb) { hb = 0; hph ^= 1u; }
                    return true;
                };
                const uint32_t halo_tx = p.halo == 1 ? kHaloTx : 180u * 128u;
                for (int wk = work0; wk < p.n_work && ok; wk += gridDim.x) {
                    const int img0 = wk + crank;                   // this CTA's tile (a padding tile loads zeros)
                    for (int chunk = 0; chunk < nch && ok; ++chunk) {
                        const bool second = chunk >= nch0;
                        ok = pixel_box(second ? &maps.a[1] : &maps.a[0], (second ? chunk - nch0 : chunk) * kCh, -1, img0, halo_tx);
                        if (p.kbs == 9) ok = weight_stage_n(std::integral_constant<int, 9>{}, &maps.b, chunk * coutp + crank * w_half, nch * coutp);
                        else if (p.kbs == 3) for (int tap = 0; tap < 9 && ok; tap += 3) ok = weight_stage_n(std::integral_constant<int, 3>{}, &maps.b, (tap * nch + chunk) * coutp + crank * w_half, nch * coutp);
                        else for (int tap = 0; tap < 9 && ok; ++tap) ok = weight_stage(&maps.b, (tap * nch + chunk) * coutp + crank * w_half);
                    }
                    if (p.L.flags & CONV_RESACC) {                 // 1x1 residual conv: the un-shifted 128 pixels of the block input
                        // (its weight tiles also share a stage -- up to 3, or 4 where a stage has room for 9 -- one pixel box per K block)
                        const int rk = p.kbs >= 9 ? 4 : p.kbs >= 3 ? 3 : 1;
                        for (int rc = 0; rc < p.r_nch && ok;) {
                            const int n = p.r_nch - rc < rk ? p.r_nch - rc : rk;
                            const int b_row = rc * coutp + crank * w_half;
                            if (n == 4) ok = weight_stage_n(std::integral_constant<int, 4>{}, &maps.rb, b_row, coutp);
                            else if (n == 3) ok = weight_stage_n(std::integral_constant<int, 3>{}, &maps.rb, b_row, coutp);
                            else if (n == 2) ok = weight_stage_n(std::integral_constant<int, 2>{}, &maps.rb, b_row, coutp);
                            else ok = weight_stage(&maps.rb, b_row);
                            for (int j = 0; j < n && ok; ++j, ++rc) {
                                const bool second = rc >= p.r_nch0;
                                ok = pixel_box(second ? &maps.ra[1] : &maps.ra[0], (second ? rc - p.r_nch0 : rc) * kCh, 0, img0, (uint32_t)kATileBytes);
                            }
                        }
                    }
                }
                ok = false;                                        // (skip the im2col loop below)
            }
            if (p.posm) {
                // ---- position-major tiles: rows = 128 images at one output position (px, py); a tap (dy, dx) that leaves the map is
                // all zeros for every row of the tile and is skipped -- 4 of 9 taps remain on a 2x2 map, 6.25 on average on 4x4, 1 on 1x1
                for (int wk = work0; wk < p.n_work && ok; wk += gridDim.x) {
                    const int work = wk + crank;
                    const int tile = work / p.n_split, n0 = (work % p.n_split) * ncols;
                    const int pos = tile / p.nblk_img, img0 = (tile - pos * p.nblk_img) * 128;
                    const int py = pos / p.L.W, px = pos - py * p.L.W;
                    // one stage = kbs (1 or 2) K blocks of ONE source at one tap: consecutive 64-channel chunks, their weight tiles
                    // coutp rows apart -- laid out [kbs pixel tiles][kbs weight tiles] as the generic issuer loop expects
                    auto stage1 = [&](const CUtensorMap* am, const CUtensorMap* wm, int c0, int x, int y, int b_row) -> bool {
                        if (!ptx::mbar_wait(errw, empty_bar(s), ph ^ 1u)) return false;
                        const uint32_t st0 = base + s * stage_bytes;
                        uint32_t fb = full_bar(s);
                        if constexpr (kPair) fb = ptx::map_to_cta(fb, 0);
                        if (!kPair || crank == 0) ptx::mbar_expect_tx(full_bar(s), tx_bytes);
                        for (int j = 0; j < p.kbs; ++j) {
                            if constexpr (!kPair) {
                                ptx::tma_load_4d(st0 + (uint32_t)j * kATileBytes, am, fb, c0 + j * kCh, x, y, img0);
                                ptx::tma_load_2d(st0 + w_base_off + (uint32_t)j * b_bytes, wm, fb, 0, b_row + j * coutp);
                            } else {
                                ptx::tma_load_4d_2sm(st0 + (uint32_t)j * kATileBytes, am, fb, c0 + j * kCh, x, y, img0);
                                ptx::tma_load_2d_2sm(st0 + w_base_off + (uint32_t)j * b_bytes, wm, fb, 0, b_row + j * coutp);
                            }
                        }
                        if (++s == p.stages) { s = 0; ph ^= 1u; }
                        return true;
                    };
                    for (int pass = 0; pass < p.npass && ok; ++pass) {       // 3xTF32: hi x hi, hi x lo weights, lo x hi
                        const int am = pass == 2 ? 2 : 0, b_pass = (pass == 1 ? p.b_lo_row : 0) + n0 + crank * w_half;
                        for (int tap = 0; tap < 9 && ok; ++tap) {
                            const int y = py + tap / 3 - 1, x = px + tap % 3 - 1;
                            if (y < 0 || y >= p.L.H || x < 0 || x >= p.L.W) continue;
                            for (int chunk = 0; chunk < nch && ok; chunk += p.kbs) {
                                const bool second = chunk >= nch0;
                                ok = stage1(&maps.a[am + (second ? 1 : 0)], &maps.b, (second ? chunk - nch0 : chunk) * kCh, x, y,
                                            (tap * nch + chunk) * coutp + b_pass);
                            }
                        }
                    }
                    if (p.L.flags & CONV_RESACC)
                        for (int rc = 0; rc < p.r_nch && ok; rc += p.kbs) {
                            const bool second = rc >= p.r_nch0;
                            ok = stage1(second ? &maps.ra[1] : &maps.ra[0], &maps.rb, (second ? rc - p.r_nch0 : rc) * kCh, px, py, rc * coutp + n0 + crank * w_half);
                        }
                }
                ok = false;                                        // (skip the im2col loop below)
            }
            for (int wk = work0; wk < p.n_work && ok; wk += gridDim.x) {
                const int work = wk + crank;                   // may be a padding item past n_work: loads hit OOB zeros
                const int tile = work / p.n_split, n0 = (work % p.n_split) * ncols;
                int img0, y0;
                if (p.tiles_per_img > 1) { img0 = tile / p.tiles_per_img; y0 = (tile % p.tiles_per_img) * p.box_h; }
                else { img0 = tile * p.box_n; y0 = 0; }
                // one pipeline stage: kbs K blocks = (activation box at tap (dx, dy), weight rows) pairs
                auto fill_stage = [&](const CUtensorMap* am0, const CUtensorMap* am1, const CUtensorMap* wm, int n_first,
                                      int& chunk, int n_chunks, int& dx, int& dy, int& b_row) -> bool {
                    if (!ptx::mbar_wait(errw, empty_bar(s), ph ^ 1u)) return false;
                    const uint32_t st0 = base + s * stage_bytes;
                    // pair: complete_tx goes to the leader's barrier (same offset, CTA 0 of the cluster)
                    uint32_t fb = full_bar(s);
                    if constexpr (kPair) fb = ptx::map_to_cta(fb, 0);
                    if (!kPair || crank == 0) ptx::mbar_expect_tx(full_bar(s), tx_bytes);
                    for (int j = 0; j < p.kbs; ++j) {
                        const bool second = chunk >= n_first;
                        const int c0 = (second ? chunk - n_first : chunk) * kCh;
                        if constexpr (!kPair) {
                            ptx::tma_load_4d(st0 + j * kATileBytes, second ? am1 : am0, fb, c0, dx, y0 + dy, img0);
                            ptx::tma_load_2d(st0 + w_base_off + j * b_bytes, wm, fb, 0, b_row);
                        } else {
                            ptx::tma_load_4d_2sm(st0 + j * kATileBytes, second ? am1 : am0, fb, c0, dx, y0 + dy, img0);
                            ptx::tma_load_2d_2sm(st0 + w_base_off + j * b_bytes, wm, fb, 0, b_row);
                        }
                        b_row += coutp;
                        if (++chunk == n_chunks) { chunk = 0; if (++dx == 2) { dx = -1; ++dy; } }
                    }
                    if (++s == p.stages) { s = 0; ph ^= 1u; }
                    return true;
                };
                for (int pass = 0; pass < p.npass && ok; ++pass) {
                    const CUtensorMap* am0 = &maps.a[pass == 2 ? 2 : 0];
                    const CUtensorMap* am1 = &maps.a[pass == 2 ? 3 : 1];
                    int b_row = (pass == 1 ? p.b_lo_row : 0) + n0 + crank * w_half;
                    int dy = p.L.ntaps == 9 ? -1 : 0, dx = dy, chunk = 0;
                    for (int it = 0; it < iters_per_pass && ok; it += p.kbs) ok = fill_stage(am0, am1, &maps.b, nch0, chunk, nch, dx, dy, b_row);
                }
                if (p.L.flags & CONV_RESACC) {     // the block's 1x1 residual conv: centre tap of the block INPUT maps
                    int b_row = n0 + crank * w_half, dy = 0, dx = 0, chunk = 0;
                    for (int it = 0; it < p.r_nch && ok; it += p.kbs) {
                        dx = dy = 0;
                        ok = fill_stage(&maps.ra[0], &maps.ra[1], &maps.rb, p.r_nch0, chunk, p.r_nch + 1, dx, dy, b_row);
                    }
                }
            }
        }
    } else if (warp == 1) {
        // ------------------------------------------------------------ MMA issuer
        if (ptx::elect_one() && (!kPair || crank == 0)) {
            const uint32_t idesc = (kF16 ? umma_idesc_f16(n_rows) : umma_idesc_tf32(n_rows)) + (kPair ? ((uint32_t)(128 >> 4) << 24) : 0u);   // pair: M = 256
            // descriptors differ between stages / K blocks only in their 14-bit start-address field
            const uint64_t desc0 = umma_desc_sw128(base);
            const uint32_t stage16 = stage_bytes >> 4;
            const uint32_t m_step16 = kATileBytes >> 4, n_step16 = b_bytes >> 4, n_off16 = ((uint32_t)p.kbs * kATileBytes) >> 4;
            int s = 0, acc = 0;
            uint32_t ph = 0, acc_ph = 0;
            bool ok = true;
            if constexpr (kF16) if (p.halo) {
                // ---- halo mode: tap (dy, dx) of a chunk = view of the halo buffer starting (dy*20 + dx) pixel rows in, 8-row groups
                // (one image row of 8 pixels) 10 pixel rows = 1280 B apart: [halo row][image][halo column] makes that uniform
                const uint64_t hdesc0 = ((uint64_t)1 << 16) | ((uint64_t)(1280 >> 4) << 32) | ((uint64_t)1 << 46) | ((uint64_t)2 << 61);
                int hb = 0;
                uint32_t hph = 0;
                const int tap_rows = p.halo == 1 ? 20 : 10;         // halo rows (of 128 B) one image row down
                auto mma4 = [&](uint32_t d_tmem, uint64_t ad, uint64_t bd, uint32_t& accum, int nk) {
#pragma unroll
                    for (int k = 0; k < 4; ++k) {
                        if (k >= nk) break;
                        if constexpr (!kPair) ptx::mma_f16(d_tmem, ad + 2u * k, bd + 2u * k, idesc, accum);
                        else ptx::mma_f16_2sm(d_tmem, ad + 2u * k, bd + 2u * k, idesc, accum);
                        accum = 1u;
                    }
                };
                auto free_stage = [&]() {
                    if constexpr (kPair) ptx::tc_commit_2sm(empty_bar(s), cmask); else ptx::tc_commit(empty_bar(s));
                    if (++s == p.stages) { s = 0; ph ^= 1u; }
                };
                auto free_halo = [&]() {
                    if constexpr (kPair) ptx::tc_commit_2sm(hempty0 + 8u * hb, cmask); else ptx::tc_commit(hempty0 + 8u * hb);
                    if (++hb == p.n_hb) { hb = 0; hph ^= 1u; }
                };
                for (int wk = work0; wk < p.n_work && ok; wk += gridDim.x) {
                    DTRAJ_TL(0, 0);
                    ok = ptx::mbar_wait(errw, acc_empty0 + 8u * acc, acc_ph ^ 1u);
                    ptx::tc_fence_after();
                    DTRAJ_TL(0, 1);
                    const uint32_t d_set = tmem_base + (uint32_t)(acc * p.acc_cols);
                    uint32_t accum = 0u;
                    for (int chunk = 0; chunk < nch && ok; ++chunk) {
                        ok = ptx::mbar_wait(errw, hfull0 + 8u * hb, hph);
                        ptx::tc_fence_after();
                        const uint32_t hbuf = halo_base + (uint32_t)hb * kHaloBytes;
                        int dy = 0, dx = 0;
                        const int nk = ((p.half_mask >> chunk) & 1u) ? 2 : 4;
                        if (p.kbs > 1) {                                  // a stage holds the weight tiles of 3 taps (one tap row) or of all 9
                            const uint64_t ha = hdesc0 | (uint64_t)((hbuf >> 4) & 0x3fffu);
                            const uint32_t w16 = b_bytes >> 4;                // (descriptor addresses count 16 bytes)
                            auto run_taps = [&](auto KB) {
                                constexpr int kb = decltype(KB)::value;
                                for (int g = 0; g < 9 / kb && ok; ++g) {
                                    ok = ptx::mbar_wait(errw, full_bar(s), ph);
                                    ptx::tc_fence_after();
                                    const uint64_t wd = umma_desc_sw128(base + s * stage_bytes);
                                    const uint64_t hr = ha + (uint64_t)(uint32_t)(g * tap_rows * 8);     // kb = 3: g is the tap row
#pragma unroll
                                    for (int j = 0; j < kb; ++j)
                                        mma4(d_set, hr + (uint64_t)(uint32_t)((j / 3) * tap_rows * 8 + (j % 3) * 8), wd + (uint64_t)(w16 * (uint32_t)j), accum, nk);
                                    free_stage();
                                }
                            };
                            if (p.kbs == 9) run_taps(std::integral_constant<int, 9>{});
                            else run_taps(std::integral_constant<int, 3>{});
                        } else
                        for (int tap = 0; tap < 9 && ok; ++tap) {
                            ok = ptx::mbar_wait(errw, full_bar(s), ph);
                            ptx::tc_fence_after();
                            const uint32_t a_addr = hbuf + (uint32_t)(dy * tap_rows + dx) * 128u;
                            mma4(d_set, hdesc0 | (uint64_t)((a_addr >> 4) & 0x3fffu), umma_desc_sw128(base + s * stage_bytes), accum, nk);
                            free_stage();
                            if (++dx == 3) { dx = 0; ++dy; }
                        }
                        free_halo();
                    }
                    if (p.L.flags & CONV_RESACC) {
                        uint32_t accum_r = 0u;
                        const int rk = p.kbs >= 9 ? 4 : p.kbs >= 3 ? 3 : 1;     // residual weight tiles per stage (as the producer packs them)
                        for (int rc = 0; rc < p.r_nch && ok;) {
                            const int n = p.r_nch - rc < rk ? p.r_nch - rc : rk;
                            ok = ptx::mbar_wait(errw, full_bar(s), ph);
                            const uint64_t wd = umma_desc_sw128(base + s * stage_bytes);
                            for (int j = 0; j < n && ok; ++j, ++rc) {
                                ok = ptx::mbar_wait(errw, hfull0 + 8u * hb, hph);
                                ptx::tc_fence_after();
                                mma4(d_set + (uint32_t)p.res_col, umma_desc_sw128(halo_base + (uint32_t)hb * kHaloBytes), wd + (uint64_t)((b_bytes >> 4) * (uint32_t)j), accum_r,
                                     ((p.r_half_mask >> rc) & 1u) ? 2 : 4);
                                free_halo();
                            }
                            free_stage();
                        }
                    }
                    if constexpr (kPair) ptx::tc_commit_2sm(acc_full0 + 8u * acc, cmask); else ptx::tc_commit(acc_full0 + 8u * acc);
                    DTRAJ_TL(0, 2);
#ifdef DTRAJ_PROBES
                    ++tl_tile;
#endif
                    if (++acc == p.acc_stages) { acc = 0; acc_ph ^= 1u; }
                }
                ok = false;                                        // (skip the im2col loop below)
            }
            for (int wk = work0; wk < p.n_work && ok; wk += gridDim.x) {
                ok = ptx::mbar_wait(errw, acc_empty0 + 8u * acc, acc_ph ^ 1u);      // epilogue has drained this buffer
                ptx::tc_fence_after();
                // 3xTF32: the two small cross terms go to their own accumulator.  The tensor core adds into the
                // accumulator with round-toward-zero; adding 2^-11-sized terms to a full-size accumulator for 2/3 of
                // the K loop costs ~K/16 ulps of systematic shrink (measured 6e-5 at K = 4608), a separate
                // accumulator keeps that at the single-pass level.
                auto run_stages = [&](uint32_t d_tmem, uint32_t accum, int n_kblocks, int n_chunks, uint32_t hmask) {
                    int chunk = 0;
                    for (int it = 0; it < n_kblocks && ok; it += p.kbs) {
                        ok = ptx::mbar_wait(errw, full_bar(s), ph);
                        ptx::tc_fence_after();
                        const uint64_t md = desc0 + (uint64_t)(s * stage16), nd = md + n_off16;
                        for (int j = 0; j < p.kbs; ++j) {
                            const int nk = ((hmask >> chunk) & 1u) ? 2 : 4;
                            if (++chunk == n_chunks) chunk = 0;
#pragma unroll
                            for (int k = 0; k < 4; ++k) {   // 4 x (K = 8 tf32 / 16 fp16 = 32 bytes) inside the 128-byte swizzle atom
                                if (k >= nk) break;
                                const uint64_t mdk = md + (uint64_t)(j * m_step16 + 2 * k), ndk = nd + (uint64_t)(j * n_step16 + 2 * k);
                                if constexpr (kF16) {
                                    if constexpr (!kPair) ptx::mma_f16(d_tmem, mdk, ndk, idesc, accum);
                                    else ptx::mma_f16_2sm(d_tmem, mdk, ndk, idesc, accum);
                                } else {
                                    if constexpr (!kPair) ptx::mma_tf32(d_tmem, mdk, ndk, idesc, accum);
                                    else ptx::mma_tf32_2sm(d_tmem, mdk, ndk, idesc, accum);
                                }
                                accum = 1u;
                            }
                        }
                        // frees the smem slot when these MMAs retire -- in every CTA that multicasts into it
                        if constexpr (kPair) ptx::tc_commit_2sm(empty_bar(s), cmask);
                        else ptx::tc_commit(empty_bar(s));
                        if (++s == p.stages) { s = 0; ph ^= 1u; }
                    }
                };
                const uint32_t d_set = tmem_base + (uint32_t)(acc * p.acc_cols);
                int n_kb = iters_per_pass;
                if (p.posm) {                                   // taps inside the map at this tile's position (pair: the same for both tiles)
                    const int pos = (wk / p.n_split) / p.nblk_img, py = pos / p.L.W, px = pos - py * p.L.W;
                    const int ny = 1 + (py > 0) + (py < p.L.H - 1), nx = 1 + (px > 0) + (px < p.L.W - 1);
                    n_kb = ny * nx * nch;
                }
                // passes 1 and 2 of 3xTF32 share the correction accumulator
                for (int pass = 0; pass < p.npass && ok; ++pass)
                    run_stages(d_set + (pass ? (uint32_t)p.corr_col : 0u), pass == 2 ? 1u : 0u, n_kb, nch, p.half_mask);
                if (p.L.flags & CONV_RESACC) run_stages(d_set + (uint32_t)p.res_col, 0u, p.r_nch, p.r_nch, p.r_half_mask);
                if constexpr (kPair) ptx::tc_commit_2sm(acc_full0 + 8u * acc, cmask);   // accumulator complete, in both CTAs
                else ptx::tc_commit(acc_full0 + 8u * acc);
                if (++acc == p.acc_stages) { acc = 0; acc_ph ^= 1u; }
            }
        }
    } else {
        // ------------------------------------------------------------ epilogue (warps 2..5)
        // TMEM holds one output pixel per lane; warp w may only touch lane quarter w % 4.
        // Per warp a ring of 4 KB buffers [32 rows][32 columns], 128-byte swizzled: TMA loads the residual
        // chunk into a buffer, the warp adds its accumulator chunk in place (thread = row, conflict-free
        // thanks to the swizzle), TMA stores the buffer.  Bytes in flight do not depend on registers: the
        // first epilogue issued plain 16-byte loads/stores and was latency-bound at ~2 TB/s.
        // Optional fused tails (set by the forward plan in single-pass TF32 mode):
        //   CONV_RESX    residual = 1x1 conv of the raw C-channel input, recomputed per element
        //                (enc1.residual_conv, models.py:60) instead of a 128-channel tensor round trip
        //   CONV_POOL    also emit MaxPool2d(2) of the tile (models.py:191-201): a warp's 32 rows
        //                always hold 8 complete 2x2 windows when W <= 16
        //   CONV_FINAL   final 1x1 conv (models.py:224, evaluated at half resolution) on the rows while
        //                they are in registers; CONV_NOSTORE drops the main store when the full tensor
        //                has no other consumer
        // 3xTF32 (ACT_SPLIT) also writes the low plane y - trunc_tf32(y) through a second store.
        if constexpr (kF16) {
        // ---- fp16 feature maps (DTRAJ_PREC_F16): same chunking (32 columns per warp step), but a ring buffer is
        // [32 rows][32 channels] of HALFS: 64-byte rows, 64-byte swizzle (16-byte cell j of row r sits at
        // j ^ ((r >> 1) & 3): thread = row stores are conflict-free), and one 16-byte cell holds 8 channels.
        // Values are rounded to fp16 (rn) here, once; |v| > 65504 raises g_umma_error bit 1 instead of storing inf silently.
        const int q = warp & 3;
        const int h = (warp - 2) >> 2;
        const int ew = warp - 2;
        const int nchunk = ncols >> 5;
        const int fl = p.L.flags;
        const bool has_res = (fl & CONV_RESID) != 0;
        const bool do_store = !(fl & CONV_NOSTORE);
        const bool do_pool = (fl & CONV_POOL) != 0;
        const int epi_kind = (p.epi_kind == 1 && p.L.tb_rows) ? 0 : p.epi_kind;   // (per-row timesteps: the time-bias table stays in global memory)
        const uint32_t buf0 = ring_base + (uint32_t)ew * kEpiBufs * kEpiBufBytes;
        const uint32_t rbar = res_bar0 + 8u * (ew * kEpiBufsMax);
        const uint32_t swz = (uint32_t)((lane >> 1) & 3);
        __half* const pool_h = reinterpret_cast<__half*>(p.L.pool_out);
        uint32_t res_par = 0;
        int acc = 0;
        uint32_t acc_ph = 0;
        float amax = 0.f;
        for (int wk = work0; wk < p.n_work; wk += gridDim.x) {
            const int work = wk + crank;
            const int tile = work / p.n_split, n0 = (work % p.n_split) * ncols;
            const int64_t m_warp = (int64_t)tile * 128 + q * 32;
            const int row = (int)m_warp;
            // coordinates of this warp's 32-row box in the 4-d output / residual maps (halo modes; mode 2: the tile's first
            // column, its first row + 4q, its image)
            int hk1 = 0, hk2 = 2 * tile, hk3 = 2 * q;
            if (p.halo == 2) { halo2_tile(p, tile, hk3, hk2, hk1); hk2 += 4 * q; }
            int pm_pos = 0, pm_img0 = 0;
            if (p.posm) {                                           // box {32 ch, 1, 1, 32 images} at (x, y, first image of the warp)
                pm_pos = tile / p.nblk_img;
                pm_img0 = (tile - pm_pos * p.nblk_img) * 128 + 32 * q;
                hk2 = pm_pos / p.L.W; hk1 = pm_pos - hk2 * p.L.W; hk3 = pm_img0;
            }
            const bool st4 = p.halo != 0 || p.posm != 0;           // stores / residual loads through a 4-d map
#ifdef DTRAJ_PROBES
            const int tl_who = 1 + h;
            const bool tl_outer = tl_on;
            const bool tl_on = tl_outer && q == 2;       // (shadows the kernel-wide flag: warps 2 and 6 only)
#endif
            DTRAJ_TL(tl_who, 0);
            if (lane == 0) {
                ptx::bulk_wait_read<0>();
                if (has_res)
                    for (int k = 0; k < kEpiBufs && h + 2 * k < nchunk; ++k) {
                        ptx::mbar_expect_tx(rbar + 8u * k, 2048u);
                        if (st4) ptx::tma_load_4d(buf0 + kEpiBufBytes * k, &maps.res, rbar + 8u * k, n0 + 32 * (h + 2 * k), hk1, hk2, hk3);
                        else ptx::tma_load_2d(buf0 + kEpiBufBytes * k, &maps.res, rbar + 8u * k, n0 + 32 * (h + 2 * k), row);
                    }
            }
            __syncwarp();
            // halo mode: the tile's rows are ordered (y, image, x); `m` stays the row index of the standard [image][y][x] layout
            int64_t m = m_warp + lane;
            bool valid = m < p.L.M;
            int img = valid ? (int)(m >> p.log2_hw) : 0;
            if (p.halo == 1) {
                const int r = q * 32 + lane;
                img = 2 * tile + ((r >> 3) & 1);
                valid = (int64_t)img * 64 < p.L.M;
                m = (int64_t)img * 64 + (r >> 4) * 8 + (r & 7);
                if (!valid) img = 0;
            } else if (p.halo == 2) {                                // rows ordered (y, x): y = y0 + (r >> 3), x = x0 + (r & 7)
                const int r = q * 32 + lane;
                img = hk3;
                valid = ((int64_t)img << p.log2_hw) < p.L.M;
                m = ((int64_t)img << p.log2_hw) + (hk2 + (lane >> 3)) * p.L.W + hk1 + (r & 7);
                if (!valid) img = 0;
            } else if (p.posm) {                                     // rows = images at one position
                img = pm_img0 + lane;
                m = ((int64_t)img << p.log2_hw) + pm_pos;
                valid = m < p.L.M;
                if (!valid) img = 0;
            }
            const float* tb = nullptr;
            const float* tb_s = cst;                                 // (kind 1: the time-bias row in shared memory)
            if (fl & CONV_TBIAS) {
                const int var = p.L.row_variant ? p.L.row_variant[img] : 0;
                tb_s = cst + (2 + var) * coutp;
                tb = p.L.tb_rows ? p.L.tbias + (size_t)var * p.L.tb_var_stride : tb_s;   // per-row timesteps: the whole table stays in global memory
            }
            float xv[4] = {0.f, 0.f, 0.f, 0.f}, fe[4] = {0.f, 0.f, 0.f, 0.f};
            if ((fl & CONV_RESX) && valid) {
                const int HWm = (1 << p.log2_hw);
                const float* xs = p.L.xraw + (size_t)(p.L.row_sample ? p.L.row_sample[img] : img) * p.L.x_stride + (m & (HWm - 1));
#pragma unroll
                for (int ch = 0; ch < 4; ++ch) if (ch < p.L.xC) xv[ch] = xs[(size_t)ch * HWm];
            }
            ptx::mbar_wait(errw, acc_full0 + 8u * acc, acc_ph);
            ptx::tc_fence_after();
            DTRAJ_TL(tl_who, 1);
            const uint32_t t_acc = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(acc * p.acc_cols);
            const int c_last = nchunk - 1 - ((nchunk - 1 - h) & 1);
            if (c_last < h) {
                ptx::tc_fence_before();
                __syncwarp();
                if (lane == 0) arrive_acc_empty(acc);
            }
            // One 32-column chunk, first half: TMEM -> registers -> bias / ReLU / time bias / residuals -> 16 packed half2 words.
            // `b`: ring buffer holding the TMA-loaded residual chunk (CONV_RESID).
            // `kind_c` (std::integral_constant): 0 = every tail tested at run time; 1..4 = the forward plan's common flag sets with the
            // tests folded at compile time.  The run-time form splits the 32-value arithmetic into ~20 basic blocks the compiler cannot
            // schedule across (each LDS -> FADD -> FMNMX -> ... chain waits out its own latencies: 1400 cycles for ~250 instructions,
            // profiles/r02i_timeline.txt); as straight-line code the loads hoist and the chains interleave.
            auto compute_chunk = [&](auto kind_c, int c, int b, uint32_t (&pk)[16]) {
                constexpr int KIND = decltype(kind_c)::value;
                constexpr bool SPEC = KIND != 0;
                const bool f_relu = SPEC ? true : (fl & CONV_RELU) != 0;
                const bool f_tb = SPEC ? KIND == 1 : tb != nullptr;
                const bool f_resx = SPEC ? false : (fl & CONV_RESX) != 0;
                const bool f_resacc = SPEC ? (KIND == 2 || KIND == 4) : (fl & CONV_RESACC) != 0;
                const bool f_resid = SPEC ? KIND == 3 : has_res;
                const bool f_final = SPEC ? KIND == 4 : (fl & CONV_FINAL) != 0;
                const float* const tbp = SPEC ? tb_s : tb;
                uint32_t raw[32], rres[32];
                ptx::tmem_ld32(t_acc + (uint32_t)(32 * c), raw);
                if (f_resacc) ptx::tmem_ld32(t_acc + (uint32_t)(p.res_col + 32 * c), rres);
                ptx::tmem_ld_wait();
                DTRAJ_TL(tl_who, 2 + 3 * (((c - h) >> 1) & 3));
                if (c == c_last) {
                    ptx::tc_fence_before();
                    __syncwarp();
                    if (lane == 0) arrive_acc_empty(acc);
                }
                if (f_resid) { ptx::mbar_wait(errw, rbar + 8u * b, (res_par >> b) & 1u); res_par ^= 1u << b; }
                const uint8_t* rowp = smem_raw + (buf0 + kEpiBufBytes * b - ptx::smem_u32(smem_raw)) + lane * 64;
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const int col = n0 + 32 * c + 8 * j;
                    float v[8];
                    {
                        const float4 b0 = *reinterpret_cast<const float4*>(bias_s + col);
                        const float4 b1 = *reinterpret_cast<const float4*>(bias_s + col + 4);
                        v[0] = __uint_as_float(raw[8 * j]) + b0.x; v[1] = __uint_as_float(raw[8 * j + 1]) + b0.y;
                        v[2] = __uint_as_float(raw[8 * j + 2]) + b0.z; v[3] = __uint_as_float(raw[8 * j + 3]) + b0.w;
                        v[4] = __uint_as_float(raw[8 * j + 4]) + b1.x; v[5] = __uint_as_float(raw[8 * j + 5]) + b1.y;
                        v[6] = __uint_as_float(raw[8 * j + 6]) + b1.z; v[7] = __uint_as_float(raw[8 * j + 7]) + b1.w;
                    }
                    if (f_relu) {
#pragma unroll
                        for (int i = 0; i < 8; ++i) v[i] = fmaxf(v[i], 0.f);
                    }
                    if (f_tb) {
                        const float4 t0 = *reinterpret_cast<const float4*>(tbp + col);
                        const float4 t1 = *reinterpret_cast<const float4*>(tbp + col + 4);
                        v[0] += t0.x; v[1] += t0.y; v[2] += t0.z; v[3] += t0.w;
                        v[4] += t1.x; v[5] += t1.y; v[6] += t1.z; v[7] += t1.w;
                    }
                    if (f_resx) {
#pragma unroll
                        for (int hh = 0; hh < 2; ++hh) {
                            float4 r4 = __ldg(reinterpret_cast<const float4*>(p.L.rb1 + col + 4 * hh));
#pragma unroll
                            for (int ch = 0; ch < 4; ++ch) {
                                if (ch >= p.L.xC) break;
                                const float4 w4 = __ldg(reinterpret_cast<const float4*>(p.L.rw1 + (size_t)ch * coutp + col + 4 * hh));
                                r4.x = fmaf(xv[ch], w4.x, r4.x); r4.y = fmaf(xv[ch], w4.y, r4.y);
                                r4.z = fmaf(xv[ch], w4.z, r4.z); r4.w = fmaf(xv[ch], w4.w, r4.w);
                            }
                            v[4 * hh] += r4.x; v[4 * hh + 1] += r4.y; v[4 * hh + 2] += r4.z; v[4 * hh + 3] += r4.w;
                        }
                    }
                    if (f_resacc) {   // residual_conv(x) + its bias, accumulated by this kernel's extra MMAs
                        const float4 r0 = *reinterpret_cast<const float4*>(rbias_s + col);
                        const float4 r1 = *reinterpret_cast<const float4*>(rbias_s + col + 4);
                        v[0] += __uint_as_float(rres[8 * j]) + r0.x; v[1] += __uint_as_float(rres[8 * j + 1]) + r0.y;
                        v[2] += __uint_as_float(rres[8 * j + 2]) + r0.z; v[3] += __uint_as_float(rres[8 * j + 3]) + r0.w;
                        v[4] += __uint_as_float(rres[8 * j + 4]) + r1.x; v[5] += __uint_as_float(rres[8 * j + 5]) + r1.y;
                        v[6] += __uint_as_float(rres[8 * j + 6]) + r1.z; v[7] += __uint_as_float(rres[8 * j + 7]) + r1.w;
                    }
                    if (f_resid) {
                        const uint4 rr = *reinterpret_cast<const uint4*>(rowp + (((uint32_t)j ^ swz) << 4));
                        const __half2* rh = reinterpret_cast<const __half2*>(&rr);
#pragma unroll
                        for (int i = 0; i < 4; ++i) { const float2 f = __half22float2(rh[i]); v[2 * i] += f.x; v[2 * i + 1] += f.y; }
                    }
                    __half2 ph2[4];
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                        amax = fmaxf(amax, fmaxf(fabsf(v[2 * i]), fabsf(v[2 * i + 1])));
                        ph2[i] = __floats2half2_rn(v[2 * i], v[2 * i + 1]);
                        pk[4 * j + i] = *reinterpret_cast<const uint32_t*>(&ph2[i]);
                    }
                    if (f_final) {
                        float vr[8];
#pragma unroll
                        for (int i = 0; i < 4; ++i) { const float2 f = __half22float2(ph2[i]); vr[2 * i] = f.x; vr[2 * i + 1] = f.y; }
#pragma unroll
                        for (int o = 0; o < 4; ++o) {
                            if (o >= p.L.finC) break;
                            const float4 w0 = *reinterpret_cast<const float4*>(finw_s + (size_t)o * coutp + col);
                            const float4 w1 = *reinterpret_cast<const float4*>(finw_s + (size_t)o * coutp + col + 4);
                            fe[o] = fmaf(vr[0], w0.x, fmaf(vr[1], w0.y, fmaf(vr[2], w0.z, fmaf(vr[3], w0.w, fe[o]))));
                            fe[o] = fmaf(vr[4], w1.x, fmaf(vr[5], w1.y, fmaf(vr[6], w1.z, fmaf(vr[7], w1.w, fe[o]))));
                        }
                    }
                }
            };
            // ... second half: packed words -> swizzled ring buffer -> fused 2x2 max-pool -> TMA store (+ ring upkeep)
            auto emit_chunk = [&](int c, int k, int b, const uint32_t (&pk)[16]) {
                uint8_t* bufp = smem_raw + (buf0 + kEpiBufBytes * b - ptx::smem_u32(smem_raw));
                uint8_t* rowp = bufp + lane * 64;
                if (do_store || do_pool) {
#pragma unroll
                    for (int j = 0; j < 4; ++j)
                        *reinterpret_cast<uint4*>(rowp + (((uint32_t)j ^ swz) << 4)) = make_uint4(pk[4 * j], pk[4 * j + 1], pk[4 * j + 2], pk[4 * j + 3]);
                }
                if (do_store) ptx::fence_proxy_async();
                __syncwarp();
                if (do_pool) {
                    // 8 pooled rows x 4 cells (8 channels each) per chunk: one cell per lane
                    const int W = p.L.W, pr = lane >> 2, x2 = pr & ((W >> 1) - 1), t = pr >> p.log2_wh;
                    int r00 = 2 * t * W + 2 * x2, rdn = W;               // window rows r00, r00 + 1, r00 + rdn, r00 + rdn + 1 of the warp's buffer
                    int64_t prow = (m_warp >> 2) + pr;                   // pooled pixel (row of the [M/4, coutp] output)
                    bool pvalid = m_warp + r00 < p.L.M;
                    if (p.halo == 1) {                                   // warp rows = (y in {2q, 2q+1}, image, x): lane -> (image, window column)
                        const int im2 = pr >> 2, wx = pr & 3;
                        r00 = im2 * 8 + 2 * wx; rdn = 16;
                        prow = ((int64_t)(2 * tile + im2) * 4 + q) * 4 + wx;
                        pvalid = (int64_t)(2 * tile + im2) * 64 < p.L.M;
                    } else if (p.halo == 2) {                            // warp rows = (y in 4q .. 4q+3, x in x0 .. x0+7): 2 x 4 windows
                        const int wy = pr >> 2, wx = pr & 3;
                        r00 = wy * 16 + 2 * wx; rdn = 8;
                        prow = ((int64_t)hk3 * (W >> 1) + (hk2 >> 1) + wy) * (W >> 1) + (hk1 >> 1) + wx;
                        pvalid = ((int64_t)hk3 << p.log2_hw) < p.L.M;
                    }
                    if (pvalid) {
                        const uint32_t jj = (uint32_t)(lane & 3);
                        auto at = [&](int r) { return *reinterpret_cast<const uint4*>(bufp + r * 64 + ((jj ^ (((uint32_t)r >> 1) & 3u)) << 4)); };
                        const uint4 a = at(r00), bq = at(r00 + 1), cq = at(r00 + rdn), d = at(r00 + rdn + 1);
                        const __half2* ah = reinterpret_cast<const __half2*>(&a);
                        const __half2* bh = reinterpret_cast<const __half2*>(&bq);
                        const __half2* ch2 = reinterpret_cast<const __half2*>(&cq);
                        const __half2* dh = reinterpret_cast<const __half2*>(&d);
                        uint4 o4;
                        __half2* oh = reinterpret_cast<__half2*>(&o4);
#pragma unroll
                        for (int i = 0; i < 4; ++i) oh[i] = __hmax2(__hmax2(ah[i], bh[i]), __hmax2(ch2[i], dh[i]));
                        *reinterpret_cast<uint4*>(pool_h + prow * coutp + n0 + 32 * c + 8 * (int)jj) = o4;
                    }
                    __syncwarp();
                }
                if (lane == 0 && do_store) {
                    if (st4) ptx::tma_store_4d(&maps.out, buf0 + kEpiBufBytes * b, n0 + 32 * c, hk1, hk2, hk3);   // box {32 ch, 8 x, 2 images, 2 rows} / {32 ch, 8 x, 4 rows, 1 image}
                    else ptx::tma_store_2d(&maps.out, buf0 + kEpiBufBytes * b, n0 + 32 * c, row);
                    ptx::bulk_commit();
                }
                // ring upkeep (depth B = kEpiBufs): my next chunk reuses buffer (k + 1) % B, last read by the store of my chunk
                // k + 1 - B -- allow B - 1 younger stores to stay in flight, then refill (residual) / rewrite it
                if (c + 2 < nchunk && k + 1 >= kEpiBufs && (has_res || do_store)) {
                    if (lane == 0) {
                        if (do_store) { if (kEpiBufs == 2) ptx::bulk_wait_read<1>(); else ptx::bulk_wait_read<0>(); }
                        if (has_res) {
                            const int nb = (k + 1) & (kEpiBufs - 1);          // (depth 1 or 2)
                            ptx::mbar_expect_tx(rbar + 8u * nb, 2048u);
                            if (st4) ptx::tma_load_4d(buf0 + kEpiBufBytes * nb, &maps.res, rbar + 8u * nb, n0 + 32 * (c + 2), hk1, hk2, hk3);
                            else ptx::tma_load_2d(buf0 + kEpiBufBytes * nb, &maps.res, rbar + 8u * nb, n0 + 32 * (c + 2), row);
                        }
                    }
                    __syncwarp();
                }
            };
            auto run_chunks = [&](auto kind_c) {
                if constexpr (decltype(kind_c)::value == 2) {
                    // ONE accumulator set (main + residual accumulators of a 256-column tile fill TMEM): the issuer cannot start the next
                    // tile before the last tcgen05.ld of this one, so all chunks leave TMEM first -- as packed halfs, 16 registers per
                    // chunk -- and the ring buffer / pool / TMA-store halves (~950 cycles each) run under the next tile's K loop
                    if (p.acc_stages == 1 && nchunk <= 8) {
                        uint32_t pk4[4][16];
#pragma unroll
                        for (int k = 0; k < 4; ++k) {
                            if (h + 2 * k < nchunk) compute_chunk(kind_c, h + 2 * k, k & (kEpiBufs - 1), pk4[k]);
                            DTRAJ_TL(tl_who, 3 + 3 * k);
                        }
#pragma unroll
                        for (int k = 0; k < 4; ++k) {
                            if (h + 2 * k < nchunk) emit_chunk(h + 2 * k, k, k & (kEpiBufs - 1), pk4[k]);
                            DTRAJ_TL(tl_who, 4 + 3 * k);
                        }
                        return;
                    }
                }
                for (int c = h, k = 0; c < nchunk; c += 2, ++k) {
                    uint32_t pk[16];
                    compute_chunk(kind_c, c, k & (kEpiBufs - 1), pk);
                    DTRAJ_TL(tl_who, 3 + 3 * (k & 3));
                    emit_chunk(c, k, k & (kEpiBufs - 1), pk);
                    DTRAJ_TL(tl_who, 4 + 3 * (k & 3));
                }
            };
            switch (epi_kind) {
                case 1: run_chunks(std::integral_constant<int, 1>{}); break;
                case 2: run_chunks(std::integral_constant<int, 2>{}); break;
                case 3: run_chunks(std::integral_constant<int, 3>{}); break;
                case 4: run_chunks(std::integral_constant<int, 4>{}); break;
                default: run_chunks(std::integral_constant<int, 0>{}); break;
            }
#ifdef DTRAJ_PROBES
            ++tl_tile;
#endif
            if (fl & CONV_FINAL) {
                float4* part = reinterpret_cast<float4*>(smem_raw + (fin_base - ptx::smem_u32(smem_raw))) + q * 32 + lane;
                if (h == 1) *part = make_float4(fe[0], fe[1], fe[2], fe[3]);
                asm volatile("bar.sync %0, 64;" ::"r"(1 + q) : "memory");
                if (h == 0 && valid) {
                    const float4 o4 = *part;
                    const float other[4] = {o4.x, o4.y, o4.z, o4.w};
#pragma unroll
                    for (int o = 0; o < 4; ++o) if (o < p.L.finC) p.L.elow[m * p.L.finC + o] = (fe[o] + other[o]) + __ldg(p.L.finb + o);
                }
                asm volatile("bar.sync %0, 64;" ::"r"(1 + q) : "memory");
            }
            if (++acc == p.acc_stages) { acc = 0; acc_ph ^= 1u; }
        }
        if (!(amax <= 65504.f)) atomicOr(errw, 2u);              // also catches NaN
        if (lane == 0) ptx::bulk_wait_read<0>();
        __syncwarp();
        } else {
        const int q = warp & 3;
        const int h = (warp - 2) >> 2;          // which of the quarter's two warps: takes chunks h, h + 2, ...
        const int ew = warp - 2;
        const int nchunk = ncols >> 5;
        const int fl = p.L.flags;
        const bool has_res = (fl & CONV_RESID) != 0;
        const bool do_store = !(fl & CONV_NOSTORE);
        const bool do_pool = (fl & CONV_POOL) != 0;
        const bool split = p.L.act_mode == ACT_SPLIT;
        const uint32_t buf0 = ring_base + (uint32_t)ew * kEpiBufs * 4096u;
        const uint32_t rbar = res_bar0 + 8u * (ew * kEpiBufsMax);
        const uint32_t swz = (uint32_t)(lane & 7);
        uint32_t res_par = 0;                   // bit b = parity the next wait on residual barrier b uses
        int acc = 0;
        uint32_t acc_ph = 0;
        for (int wk = work0; wk < p.n_work; wk += gridDim.x) {
            const int work = wk + crank;
            const int tile = work / p.n_split, n0 = (work % p.n_split) * ncols;
            const int64_t m_warp = (int64_t)tile * 128 + q * 32;
            const int row = (int)m_warp;
            int pm_pos = 0, pm_img0 = 0, pk1 = 0, pk2 = 0;           // position-major tiles: box {32 ch, 1, 1, 32 images} at (x, y, first image of the warp)
            if (p.posm) {
                pm_pos = tile / p.nblk_img;
                pm_img0 = (tile - pm_pos * p.nblk_img) * 128 + 32 * q;
                pk2 = pm_pos / p.L.W; pk1 = pm_pos - pk2 * p.L.W;
            }        // TMA coordinates are 32-bit; M < 2^31 is checked on the host
            if (lane == 0) {
                ptx::bulk_wait_read<0>();       // the previous tile's stores have left the ring
                if (has_res)
                    for (int k = 0; k < kEpiBufs && h + 2 * k < nchunk; ++k) {
                        ptx::mbar_expect_tx(rbar + 8u * k, 4096u);
                        if (p.posm) ptx::tma_load_4d(buf0 + 4096u * k, &maps.res, rbar + 8u * k, n0 + 32 * (h + 2 * k), pk1, pk2, pm_img0);
                        else ptx::tma_load_2d(buf0 + 4096u * k, &maps.res, rbar + 8u * k, n0 + 32 * (h + 2 * k), row);
                    }
            }
            __syncwarp();
            int64_t m = m_warp + lane;
            bool valid = m < p.L.M;
            int img = valid ? (int)(m >> p.log2_hw) : 0;
            if (p.posm) {                                            // rows = images at one position (see the fp16 branch)
                img = pm_img0 + lane;
                m = ((int64_t)img << p.log2_hw) + pm_pos;
                valid = m < p.L.M;
                if (!valid) img = 0;
            }
            const float* tb = nullptr;
            if (fl & CONV_TBIAS) {
                const int var = p.L.row_variant ? p.L.row_variant[img] : 0;
                tb = p.L.tb_rows ? p.L.tbias + (size_t)var * p.L.tb_var_stride : cst + (2 + var) * coutp;   // per-row timesteps: the whole table stays in global memory
            }
            float xv[4] = {0.f, 0.f, 0.f, 0.f}, fe[4] = {0.f, 0.f, 0.f, 0.f};
            if ((fl & CONV_RESX) && valid) {
                const int HWm = (1 << p.log2_hw);
                const float* xs = p.L.xraw + (size_t)(p.L.row_sample ? p.L.row_sample[img] : img) * p.L.x_stride + (m & (HWm - 1));
#pragma unroll
                for (int ch = 0; ch < 4; ++ch) if (ch < p.L.xC) xv[ch] = xs[(size_t)ch * HWm];
            }
            ptx::mbar_wait(errw, acc_full0 + 8u * acc, acc_ph);
            ptx::tc_fence_after();
            const uint32_t t_acc = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(acc * p.acc_cols);
            const int c_last = nchunk - 1 - ((nchunk - 1 - h) & 1);   // this warp's last chunk (< h: it has none)
            if (c_last < h) {                   // a single-chunk item leaves the quarter's second warp idle
                ptx::tc_fence_before();
                __syncwarp();
                if (lane == 0) arrive_acc_empty(acc);
            }
            for (int c = h, k = 0; c < nchunk; c += 2, ++k) {
                const int b = k & (kEpiBufs - 1);
                uint32_t raw[32];
                ptx::tmem_ld32(t_acc + (uint32_t)(32 * c), raw);
                if (p.npass == 3) {
                    uint32_t raw2[32];
                    ptx::tmem_ld32(t_acc + (uint32_t)(p.corr_col + 32 * c), raw2);
                    ptx::tmem_ld_wait();
#pragma unroll
                    for (int j = 0; j < 32; ++j) raw[j] = __float_as_uint(__uint_as_float(raw[j]) + __uint_as_float(raw2[j]));
                } else {
                    ptx::tmem_ld_wait();
                }
                uint32_t rres[32];
                if (fl & CONV_RESACC) {
                    ptx::tmem_ld32(t_acc + (uint32_t)(p.res_col + 32 * c), rres);
                    ptx::tmem_ld_wait();
                }
                if (c == c_last) {
                    // every TMEM read of this warp for this tile is done: hand the accumulator back to the issuer
                    ptx::tc_fence_before();
                    __syncwarp();
                    if (lane == 0) arrive_acc_empty(acc);
                }
                if (has_res) { ptx::mbar_wait(errw, rbar + 8u * b, (res_par >> b) & 1u); res_par ^= 1u << b; }
                uint8_t* bufp = smem_raw + (buf0 + 4096u * b - ptx::smem_u32(smem_raw));
                uint8_t* rowp = bufp + lane * 128;
                float4 keep[8];                 // ACT_SPLIT: values for the low-plane store
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    const int col = n0 + 32 * c + 4 * j;
                    const float4 b4 = *reinterpret_cast<const float4*>(bias_s + col);
                    float4 v = make_float4(__uint_as_float(raw[4 * j]) + b4.x, __uint_as_float(raw[4 * j + 1]) + b4.y,
                                           __uint_as_float(raw[4 * j + 2]) + b4.z, __uint_as_float(raw[4 * j + 3]) + b4.w);
                    if (fl & CONV_RELU) {
                        v.x = fmaxf(v.x, 0.f); v.y = fmaxf(v.y, 0.f); v.z = fmaxf(v.z, 0.f); v.w = fmaxf(v.w, 0.f);
                    }
                    if (tb) {
                        const float4 t4 = *reinterpret_cast<const float4*>(tb + col);
                        v.x += t4.x; v.y += t4.y; v.z += t4.z; v.w += t4.w;
                    }
                    if (fl & CONV_RESX) {
                        float4 r4 = __ldg(reinterpret_cast<const float4*>(p.L.rb1 + col));
#pragma unroll
                        for (int ch = 0; ch < 4; ++ch) {
                            if (ch >= p.L.xC) break;
                            const float4 w4 = __ldg(reinterpret_cast<const float4*>(p.L.rw1 + (size_t)ch * coutp + col));
                            r4.x = fmaf(xv[ch], w4.x, r4.x); r4.y = fmaf(xv[ch], w4.y, r4.y);
                            r4.z = fmaf(xv[ch], w4.z, r4.z); r4.w = fmaf(xv[ch], w4.w, r4.w);
                        }
                        v.x += r4.x; v.y += r4.y; v.z += r4.z; v.w += r4.w;
                    }
                    if (fl & CONV_RESACC) {   // residual_conv(x) + its bias, accumulated by this kernel's extra MMAs
                        const float4 rb4 = *reinterpret_cast<const float4*>(rbias_s + col);
                        v.x += __uint_as_float(rres[4 * j]) + rb4.x; v.y += __uint_as_float(rres[4 * j + 1]) + rb4.y;
                        v.z += __uint_as_float(rres[4 * j + 2]) + rb4.z; v.w += __uint_as_float(rres[4 * j + 3]) + rb4.w;
                    }
                    float4* cell = reinterpret_cast<float4*>(rowp + (((uint32_t)j ^ swz) << 4));
                    if (has_res) {
                        const float4 r4 = *cell;
                        v.x += r4.x; v.y += r4.y; v.z += r4.z; v.w += r4.w;
                    }
                    v = act_round4(v, p.L.act_mode);
                    if (fl & CONV_FINAL) {
#pragma unroll
                        for (int o = 0; o < 4; ++o) {
                            if (o >= p.L.finC) break;
                            const float4 w4 = *reinterpret_cast<const float4*>(finw_s + (size_t)o * coutp + col);
                            fe[o] = fmaf(v.x, w4.x, fmaf(v.y, w4.y, fmaf(v.z, w4.z, fmaf(v.w, w4.w, fe[o]))));
                        }
                    }
                    if (do_store || do_pool) *cell = v;
                    if (split) keep[j] = v;
                }
                if (do_store) ptx::fence_proxy_async();
                __syncwarp();
                if (do_pool) {
                    // 8 pooled rows x 8 float4 per chunk: lane -> (pooled row, two float4 columns)
                    const int W = p.L.W, pr = lane >> 2, x2 = pr & ((W >> 1) - 1), t = pr >> p.log2_wh;
                    const int r00 = 2 * t * W + 2 * x2;
                    if (m_warp + r00 < p.L.M) {
                        float* dst = p.L.pool_out + ((m_warp >> 2) + pr) * coutp + n0 + 32 * c;
#pragma unroll
                        for (int jj = (lane & 3) * 2; jj < (lane & 3) * 2 + 2; ++jj) {
                            auto at = [&](int r) { return *reinterpret_cast<const float4*>(bufp + r * 128 + (((uint32_t)jj ^ (uint32_t)(r & 7)) << 4)); };
                            const float4 a = at(r00), bq = at(r00 + 1), cq = at(r00 + W), d = at(r00 + W + 1);
                            *reinterpret_cast<float4*>(dst + 4 * jj) =
                                make_float4(fmaxf(fmaxf(a.x, bq.x), fmaxf(cq.x, d.x)), fmaxf(fmaxf(a.y, bq.y), fmaxf(cq.y, d.y)),
                                            fmaxf(fmaxf(a.z, bq.z), fmaxf(cq.z, d.z)), fmaxf(fmaxf(a.w, bq.w), fmaxf(cq.w, d.w)));
                        }
                    }
                    __syncwarp();
                }
                if (lane == 0 && do_store) {
                    if (p.posm) ptx::tma_store_4d(&maps.out, buf0 + 4096u * b, n0 + 32 * c, pk1, pk2, pm_img0);
                    else ptx::tma_store_2d(&maps.out, buf0 + 4096u * b, n0 + 32 * c, row);
                    ptx::bulk_commit();
                }
                if (split && do_store) {
                    // low plane: reuse the same buffer once the high-plane store has read it
                    if (lane == 0) ptx::bulk_wait_read<0>();
                    __syncwarp();
#pragma unroll
                    for (int j = 0; j < 8; ++j) *reinterpret_cast<float4*>(rowp + (((uint32_t)j ^ swz) << 4)) = act_lo4(keep[j]);
                    ptx::fence_proxy_async();
                    __syncwarp();
                    if (lane == 0) {
                        if (p.posm) ptx::tma_store_4d(&maps.out_lo, buf0 + 4096u * b, n0 + 32 * c, pk1, pk2, pm_img0);
                        else ptx::tma_store_2d(&maps.out_lo, buf0 + 4096u * b, n0 + 32 * c, row);
                        ptx::bulk_commit();
                    }
                }
                // ring upkeep (depth B = kEpiBufs): my next chunk reuses buffer (k + 1) % B, last read by the store of
                // my chunk k + 1 - B -- allow B - 1 younger stores to stay in flight, then refill / rewrite it
                if (c + 2 < nchunk && k + 1 >= kEpiBufs && (has_res || do_store)) {
                    if (lane == 0) {
                        if (do_store) { if (kEpiBufs == 2) ptx::bulk_wait_read<1>(); else ptx::bulk_wait_read<0>(); }
                        if (has_res) {
                            const int nb = (k + 1) & (kEpiBufs - 1);          // (depth 1 or 2)
                            ptx::mbar_expect_tx(rbar + 8u * nb, 4096u);
                            if (p.posm) ptx::tma_load_4d(buf0 + 4096u * nb, &maps.res, rbar + 8u * nb, n0 + 32 * (c + 2), pk1, pk2, pm_img0);
                            else ptx::tma_load_2d(buf0 + 4096u * nb, &maps.res, rbar + 8u * nb, n0 + 32 * (c + 2), row);
                        }
                    }
                    __syncwarp();
                }
            }
            if (fl & CONV_FINAL) {
                // the quarter's two warps hold partial sums over alternate chunks of the same rows
                float4* part = reinterpret_cast<float4*>(smem_raw + (fin_base - ptx::smem_u32(smem_raw))) + q * 32 + lane;
                if (h == 1) *part = make_float4(fe[0], fe[1], fe[2], fe[3]);
                asm volatile("bar.sync %0, 64;" ::"r"(1 + q) : "memory");
                if (h == 0 && valid) {
                    const float4 o4 = *part;
                    const float other[4] = {o4.x, o4.y, o4.z, o4.w};
#pragma unroll
                    for (int o = 0; o < 4; ++o) if (o < p.L.finC) p.L.elow[m * p.L.finC + o] = (fe[o] + other[o]) + __ldg(p.L.finb + o);
                }
                asm volatile("bar.sync %0, 64;" ::"r"(1 + q) : "memory");
            }
            if (++acc == p.acc_stages) { acc = 0; acc_ph ^= 1u; }
        }
        if (lane == 0) ptx::bulk_wait_read<0>();    // smem must outlive the stores' reads
        __syncwarp();
        }
    }
    ptx::tc_fence_before();
    __syncthreads();
    if constexpr (kPair) ptx::cluster_sync_all(); // no CTA leaves while its peer can still write its smem / barriers
    if (warp == 0) {
        ptx::tc_fence_after();
        if constexpr (!kPair) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)p.tmem_cols) : "memory");
        else asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)p.tmem_cols) : "memory");
    }
}

// ---------------------------------------------------------------- host side: tensor maps
typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

inline PFN_encodeTiled get_encode_tiled() {
    static PFN_encodeTiled fn = nullptr;
    if (!fn) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            fn = (PFN_encodeTiled)p;
    }
    return fn;
}

// NHWC activation map {cp, W, H, n_img} with box {32, W, box_h, box_n}
// (f16: elements are halfs and a box carries 64 channels -- the same 128 bytes per pixel)
inline int make_act_map(CUtensorMap* m, const float* base, int cp, int W, int H, int64_t n_img, int box_h, int box_n, int f16 = 0) {
    PFN_encodeTiled enc = get_encode_tiled();
    if (!enc) return fail(DTRAJ_ECUDA, "cuTensorMapEncodeTiled not available");
    const cuuint64_t es_b = f16 ? 2 : 4;
    cuuint64_t dims[4] = {(cuuint64_t)cp, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)n_img};
    cuuint64_t strides[3] = {(cuuint64_t)cp * es_b, (cuuint64_t)W * cp * es_b, (cuuint64_t)H * W * cp * es_b};
    cuuint32_t box[4] = {f16 ? 64u : 32u, (cuuint32_t)W, (cuuint32_t)box_h, (cuuint32_t)box_n};
    cuuint32_t es[4] = {1, 1, 1, 1};
    CUresult r = enc(m, f16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, (void*)base, dims, strides, box, es,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(DTRAJ_ECUDA, "cuTensorMapEncodeTiled(act cp=%d W=%d H=%d n=%lld) -> %d", cp, W, H, (long long)n_img, (int)r);
    return 0;
}
// packed weights as a 2-d map {32, rows} with box {32, coutp}
inline int make_w_map(CUtensorMap* m, const float* base, int64_t rows, int coutp, int f16 = 0) {
    PFN_encodeTiled enc = get_encode_tiled();
    if (!enc) return fail(DTRAJ_ECUDA, "cuTensorMapEncodeTiled not available");
    cuuint64_t dims[2] = {f16 ? 64u : 32u, (cuuint64_t)rows};
    cuuint64_t strides[1] = {128};
    cuuint32_t box[2] = {f16 ? 64u : 32u, (cuuint32_t)coutp};
    cuuint32_t es[2] = {1, 1};
    CUresult r = enc(m, f16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, (void*)base, dims, strides, box, es,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(DTRAJ_ECUDA, "cuTensorMapEncodeTiled(weights rows=%lld) -> %d", (long long)rows, (int)r);
    return 0;
}

// row-major [M, coutp] activation as a 2-d map {coutp, M} with box {32, 32} (epilogue chunks)
// (f16: 64-byte rows of 32 halfs, 64-byte swizzle)
inline int make_rows_map(CUtensorMap* m, const float* base, int64_t M, int coutp, int f16 = 0) {
    PFN_encodeTiled enc = get_encode_tiled();
    if (!enc) return fail(DTRAJ_ECUDA, "cuTensorMapEncodeTiled not available");
    cuuint64_t dims[2] = {(cuuint64_t)coutp, (cuuint64_t)M};
    cuuint64_t strides[1] = {(cuuint64_t)coutp * (f16 ? 2 : 4)};
    cuuint32_t box[2] = {32, 32};
    cuuint32_t es[2] = {1, 1};
    CUresult r = enc(m, f16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, (void*)base, dims, strides, box, es,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, f16 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(DTRAJ_ECUDA, "cuTensorMapEncodeTiled(rows M=%lld cp=%d) -> %d", (long long)M, coutp, (int)r);
    return 0;
}

// fp16 NHWC map [n_img][8][8][cp] seen through the PERMUTED dimensions {c, x, image, y} (global strides not increasing;
// profiles/r01_tma_permuted_probe.txt): a box {box_c, box_x, 2, box_y} lands / leaves shared memory as [y][image][x] rows
inline int make_perm8_map(CUtensorMap* m, const float* base, int cp, int64_t n_img, int box_c, int box_x, int box_y, bool sw64) {
    PFN_encodeTiled enc = get_encode_tiled();
    if (!enc) return fail(DTRAJ_ECUDA, "cuTensorMapEncodeTiled not available");
    cuuint64_t dims[4] = {(cuuint64_t)cp, 8, (cuuint64_t)n_img, 8};
    cuuint64_t strides[3] = {(cuuint64_t)cp * 2, (cuuint64_t)64 * cp * 2, (cuuint64_t)8 * cp * 2};
    cuuint32_t box[4] = {(cuuint32_t)box_c, (cuuint32_t)box_x, 2, (cuuint32_t)box_y};
    cuuint32_t es[4] = {1, 1, 1, 1};
    CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 4, (void*)base, dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                     sw64 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(DTRAJ_ECUDA, "cuTensorMapEncodeTiled(permuted 8x8 map cp=%d n=%lld) -> %d", cp, (long long)n_img, (int)r);
    return 0;
}

inline cudaError_t umma_set_smem_attr() {
    cudaError_t e = cudaFuncSetAttribute(k_conv_umma_t<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(k_conv_umma_t<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(k_conv_umma_t<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(k_conv_umma_t<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
    return e;
}

// fp16 epilogue: the flag sets of the forward plan's layers that k_conv_umma_t compiles as straight-line code (CONV_POOL / CONV_NOSTORE
// only steer the stores and go with any of them)
inline int epi_kind_of(int flags) {
    switch (flags & ~(CONV_POOL | CONV_NOSTORE)) {
        case CONV_RELU | CONV_TBIAS: return 1;                 // conv1 of a block
        case CONV_RELU | CONV_RESACC: return 2;                // conv2 + fused 1x1 residual conv
        case CONV_RELU | CONV_RESID: return 3;                 // conv2 + identity residual
        case CONV_RELU | CONV_RESACC | CONV_FINAL: return 4;   // dec1.conv2 + residual conv + final 1x1
        default: return 0;
    }
}

struct UmmaLaunch {            // everything a launch needs, built once per (layer, batch)
    UmmaMaps maps;
    UmmaConv conv;
    unsigned grid;
    size_t smem;
};

// Position-major tiles (UmmaConv::posm) pay on 1x1 / 2x2 maps always (every tile skips the same taps) and on 4x4 maps only when the
// launch has more tiles than SMs: the four centre positions still run all nine taps, so a single wave is as long as before
// (measured at 128 rows in 3xTF32: enc3.conv1 58 -> 62 us with them, enc4.conv1 58 -> 35 us).  The forward plan asks the same
// question to decide where the 2x2 pool can stay fused into the producing conv.
inline bool umma_posm_applies(int H, int64_t n_img) {
    if (H > 4) return false;
    if (H <= 2) return true;
    return (int64_t)H * H * ((n_img + 127) / 128) > kNumSMs;
}

// `w_rows` = rows of the packed weight matrix (hi planes then, for 3 passes, lo planes)
// `form` (dtraj_bench_conv's A/B experiments; the forward plan passes 0): 0 = the form and shared-memory split chosen below;
// kUmmaGeneric = the generic [image][y][x] tiles even where a halo form exists; kUmmaSplit | n_hb << 4 | epi_bufs = the halo form
// with that many halo slots and epilogue buffers per warp, the rest of the shared memory as weight stages (at most 16)
constexpr int kUmmaGeneric = 1, kUmmaSplit = 0x100;
inline int build_umma_launch(UmmaLaunch* U, const ConvLayer& L, int npass, const float* wpk, int64_t w_rows,
                             const float* rwpk = nullptr, int64_t rw_rows = 0, int form = 0) {
    memset(U, 0, sizeof(*U));
    const int HW = L.H * L.W;
    // (a tile is 128 / W whole image rows: 2 at 64x64, the largest map of a supported model)
    if (L.W > 64 || L.H != L.W || (HW & (HW - 1)) != 0)
        return fail(DTRAJ_EINVAL, "umma conv: unsupported spatial size %dx%d", L.H, L.W);
    const int f16 = L.f16 ? 1 : 0, kch = f16 ? 64 : 32;     // channels per 128-byte K block
    // channel counts are padded to 32 in every mode; in fp16 mode a K block carries 64 channels, so a source padded to an odd
    // multiple of 32 ends in a half-filled block
    if (L.coutp % 32 || L.coutp > 256 || L.c0p % 32 || L.c1p % 32 || L.c0p > 512 || L.c1p > 512) return fail(DTRAJ_EINVAL, "umma conv: bad channel padding");
    if (f16 && (npass != 1 || L.act_mode == ACT_SPLIT)) return fail(DTRAJ_EINVAL, "umma conv: fp16 mode is single-pass");
    UmmaConv& c = U->conv;
    c.L = L;
    c.f16 = f16;
    c.npass = npass;
    auto chunks_of = [&](int cp) { return (cp + kch - 1) / kch; };
    auto halves_of = [&](int c0p, int c1p) {
        uint32_t m = 0;
        if (c0p % kch) m |= 1u << (chunks_of(c0p) - 1);
        if (c1p % kch) m |= 1u << (chunks_of(c0p) + chunks_of(c1p) - 1);
        return m;
    };
    c.nch0 = chunks_of(L.c0p);
    c.nch = c.nch0 + chunks_of(L.c1p);
    c.half_mask = halves_of(L.c0p, L.c1p);
    const int nkb_all = L.ntaps * c.nch;                       // K blocks (128 bytes of channels per row) of the whole K loop
    // a tile = 128 output pixels: box_h image rows of box_n images
    c.box_h = HW >= 128 ? 128 / L.W : L.H;
    c.box_n = HW >= 128 ? 1 : 128 / HW;
    c.tiles_per_img = HW >= 128 ? HW / 128 : 1;
    c.n_tiles = (int)((L.M + 127) / 128);
    // Maps of at most 4x4: POSITION-MAJOR tiles.  With [image][y][x] rows a 128-row tile mixes positions, so every one of the
    // nine taps is loaded and multiplied although most of them fall into the zero padding (2x2: 5 of 9, 4x4: 2.75 of 9 on average,
    // 1x1: 8 of 9) -- and these layers are bound by the weight tiles they pull through L2 (8.7 TB/s on enc4 of the teacher at 8880
    // rows).  A tile of 128 images at ONE position skips the taps outside the map for all its rows at once.  No fused pool there
    // (a 2x2 window spans four tiles): the forward plan keeps the stand-alone pool kernel at these levels.
    c.posm = (L.ntaps == 9 && umma_posm_applies(L.H, L.M / HW) && !(L.flags & (CONV_POOL | CONV_RESX | CONV_FINAL))) ? 1 : 0;
    const int64_t n_img_all = L.M / HW;
    if (c.posm) {
        c.nblk_img = (int)((n_img_all + 127) / 128);
        if (c.nblk_img >= 2 * kNumSMs / HW && (c.nblk_img & 1)) ++c.nblk_img;    // pairs: both tiles of a pair at the same position
        c.n_tiles = HW * c.nblk_img;
    }
    // fewer tiles than SMs (deep levels, small batches): split a tile's columns over up to 4 CTAs
    c.n_split = 1;
    if (!(L.flags & CONV_FINAL))
        while (c.n_tiles * c.n_split * 2 <= kNumSMs && (L.coutp / (c.n_split * 2)) % 32 == 0 && L.coutp / (c.n_split * 2) >= 64)
            c.n_split *= 2;
    c.ncols = L.coutp / c.n_split;
    c.n_work = c.n_tiles * c.n_split;
    const int n_rows = c.ncols;
    // CTA pairs (tcgen05.mma.cta_group::2): each CTA stages its own 128 pixels and HALF of the weight tile, so a K
    // block costs 16 + N/4 KB of its shared memory instead of 16 + N/2 KB -- more K blocks in flight in the
    // latency-bound operand ring.  Wide, long layers with at least two waves of tiles only (profiles/r01c_conv_layers.txt).
    c.pair = (c.n_split == 1 && L.coutp >= 64 && nkb_all >= 16 && c.n_work >= 2 * kNumSMs && (!c.posm || (c.nblk_img & 1) == 0)) ? 1 : 0;
    c.acc_cols = 32;
    while (c.acc_cols < n_rows) c.acc_cols *= 2;
    c.corr_col = 0;
    if (npass == 3) { c.corr_col = c.acc_cols; c.acc_cols *= 2; }
    c.res_col = 0;
    c.r_nch0 = chunks_of(L.rc0p);
    c.r_nch = c.r_nch0 + chunks_of(L.rc1p);
    c.r_half_mask = halves_of(L.rc0p, L.rc1p);
    if (L.flags & CONV_RESACC) {
        if (npass != 1 || !rwpk || L.rc0p % 32 || L.rc1p % 32 || !L.rsrc0 || (L.rc1p && !L.rsrc1))
            return fail(DTRAJ_EINVAL, "umma conv: fused residual conv needs a single-pass mode and packed residual weights");
        c.res_col = c.acc_cols;
        c.acc_cols *= 2;
    }
    c.acc_stages = 2 * c.acc_cols <= 512 ? 2 : 1;
    c.tmem_cols = c.acc_stages * c.acc_cols;
    c.b_lo_row = nkb_all * L.coutp;
    c.cb = 0;
    c.log2_hw = 0;
    while ((1 << c.log2_hw) < HW) ++c.log2_hw;
    if ((1 << c.log2_hw) != HW) return fail(DTRAJ_EINVAL, "umma conv: H*W=%d is not a power of two", HW);
    c.log2_wh = 0;
    while ((2 << c.log2_wh) < L.W) ++c.log2_wh;
    if ((L.flags & CONV_POOL) && (L.W < 2 || L.W > 16 || L.H != L.W)) return fail(DTRAJ_EINVAL, "umma conv: fused pool needs 2 <= W <= 16");
    if ((L.flags & (CONV_POOL | CONV_RESX | CONV_FINAL | CONV_NOSTORE)) && L.act_mode == ACT_SPLIT)
        return fail(DTRAJ_EINVAL, "umma conv: fused tails are not available in 3xTF32 mode");
    // one persistent CTA per SM: all shared memory that is not the epilogue ring goes to the operand ring.  The
    // ring is latency-bound (bytes in flight / ~1.3 us TMA latency): a deeper operand ring is worth more than a
    // deeper epilogue ring whenever halving the latter buys a whole stage and the K loop is long enough to hide a
    // single-buffered epilogue.
    // two K blocks per stage halve the single-thread loop overhead per MMA; worth it where an MMA is short
    // (N <= 128: <= 256 cycles per K block) and the stage stays small enough to keep >= 3 stages in flight
    const int n_stage_rows = c.pair ? n_rows / 2 : n_rows;
    c.kbs = (n_stage_rows <= (c.pair ? 64 : 128) && c.r_nch0 % 2 == 0 && (c.r_nch - c.r_nch0) % 2 == 0 && c.nch0 % 2 == 0 && (c.nch - c.nch0) % 2 == 0) ? 2 : 1;
    // halo mode (fp16, 8x8 / 16x16 / 32x32 maps, 3x3, no identity residual): pixels through the halo ring
    c.halo = (form != kUmmaGeneric && f16 && L.ntaps == 9 && !(L.flags & CONV_RESX) && c.n_split == 1 && L.act_mode != ACT_SPLIT)
                 ? (L.H == 8 && L.W == 8 ? 1 : ((L.H == 16 || L.H == 32) && L.W == L.H ? 2 : 0)) : 0;
    c.hlg_x = L.W == 32 ? 2 : 1;
    c.hlg_t = L.W == 32 ? 3 : 1;
    if (c.posm && (c.half_mask || c.r_half_mask || c.n_split > 1)) c.kbs = 1;   // (position-major tiles: two K blocks per stage where every chunk is a full one)
    c.n_hb = 0;
    // (halo mode: kbs = weight tiles (taps) per stage -- all nine where a tile is at most 4 KB, three where it is 8 KB, i.e. where four
    //  MMAs are shorter than the barrier round trip of the two single-thread loops)
    if (c.halo) { c.kbs = n_stage_rows * 128 <= 4096 ? 9 : n_stage_rows * 128 <= 8192 ? 3 : 1; c.n_hb = 3; }
    // Halo layers with a fused residual conv: its K blocks bring an un-shifted 16 KB pixel box EACH through the halo ring, so where they
    // outnumber the main chunks (dec1.conv2: 2 halo boxes + 8 residual boxes per tile at the teacher's widths) three slots make that
    // phase latency-bound (3 boxes per ~1.5 us TMA round trip): a fourth slot, paid for by a single-buffered epilogue ring
    // (profiles/r02q_ring_ab.txt: teacher dec1.conv2 259 -> 241 us, sf 0.5 115 -> 108 us; enc2.conv2 with the single-buffered
    // epilogue ring alone 550 -> 530 us).
    const bool halo_res = c.halo && (L.flags & CONV_RESACC);
    if (halo_res && c.r_nch > c.nch) c.n_hb = 4;
    // ... and a conv1 whose whole K loop is two halo boxes of 16 KB weight stages (enc2.conv1 at N = 256) does better with two halo
    // slots and a single-buffered epilogue ring, i.e. three more weight stages (teacher enc2.conv1 244 -> 227 us; the same
    // trade loses on the 8-chunk dec1.conv1 and on 8 KB stages, same file)
    const bool halo_short = c.halo && !(L.flags & CONV_RESACC) && c.nch <= 2 && n_stage_rows * 128 >= 16384;
    if (halo_short) c.n_hb = 2;
    const bool split_set = c.halo && (form & kUmmaSplit);
    if (split_set) c.n_hb = (form >> 4) & 15;
    if (c.n_hb > 4) return fail(DTRAJ_EINVAL, "umma conv: the kernel has four halo-ring barriers");
    const size_t stage = c.halo ? (size_t)c.kbs * n_stage_rows * 128 : (size_t)c.kbs * (kATileBytes + (size_t)n_stage_rows * 128);
    const size_t cst_bytes = (size_t)(5 + ((L.flags & CONV_FINAL) ? 4 : 0)) * L.coutp * 4;     // staged per-channel constants
    const size_t misc = 1024 + 512 + ((L.flags & CONV_FINAL) ? 2048 : 0) + cst_bytes + (size_t)c.n_hb * kHaloBytes;
    const size_t epi_buf_bytes = f16 ? 2048 : 4096;            // [32 rows][32 columns] of halfs / floats
    auto stages_for = [&](int bufs) { return (int)((227 * 1024 - misc - (size_t)kEpiWarps * bufs * epi_buf_bytes) / stage); };
    c.epi_bufs = 2;
    c.epi_kind = f16 ? epi_kind_of(L.flags) : 0;
    if (!c.halo && nkb_all >= 16 && stages_for(1) > stages_for(2) && stages_for(2) < 8) c.epi_bufs = 1;
    // (at 32x32 the short conv1 keeps its double-buffered epilogue ring: enc2.conv1 of 3x64x64 models at 7680 rows, teacher 2760 -> 2704 us,
    //  sf 0.5 1549 -> 1468 us with two halo slots; the other 32x32 layers are best with the 16x16 rules, profiles/r03b_halo_split_ab.txt)
    if ((halo_res || (halo_short && L.W != 32)) && stages_for(2) < 16) c.epi_bufs = 1;
    if (split_set) {
        c.epi_bufs = form & 15;
        if (c.n_hb < 1 || c.epi_bufs < 1 || c.epi_bufs > kEpiBufsMax) return fail(DTRAJ_EINVAL, "umma conv: bad shared-memory split 0x%x", form);
    }
    int stages = stages_for(c.epi_bufs);
    if (stages < 2) return fail(DTRAJ_EINVAL, "umma conv: operand ring does not fit");
    if (stages > 16) stages = 16;
    if (c.halo && !halo_res && !split_set && stages > 12) stages = 12;      // (dec1.conv1: 484 us with 10-12 weight stages, 495 with 14, 510 with 8, 550 with 6)
    c.stages = stages;
    U->smem = misc + (size_t)kEpiWarps * c.epi_bufs * epi_buf_bytes + stages * stage;
    U->grid = (unsigned)(c.n_work < kNumSMs ? c.n_work : kNumSMs);
    if (c.pair) U->grid = (U->grid + 1) / 2 * 2;
    const int64_t n_img = L.M / HW;
    DTRAJ_TRY(make_act_map(&U->maps.a[0], L.src0, L.c0p, L.W, L.H, n_img, c.box_h, c.box_n, f16));
    if (L.c1p) DTRAJ_TRY(make_act_map(&U->maps.a[1], L.src1, L.c1p, L.W, L.H, n_img, c.box_h, c.box_n, f16));
    if (npass == 3) {
        DTRAJ_TRY(make_act_map(&U->maps.a[2], L.src0_lo, L.c0p, L.W, L.H, n_img, c.box_h, c.box_n));
        if (L.c1p) DTRAJ_TRY(make_act_map(&U->maps.a[3], L.src1_lo, L.c1p, L.W, L.H, n_img, c.box_h, c.box_n));
    }
    DTRAJ_TRY(make_w_map(&U->maps.b, wpk, w_rows, c.ncols / (c.pair ? 2 : 1), f16));
    if (L.flags & CONV_RESACC) {
        DTRAJ_TRY(make_act_map(&U->maps.ra[0], L.rsrc0, L.rc0p, L.W, L.H, n_img, c.box_h, c.box_n, f16));
        if (L.rc1p) DTRAJ_TRY(make_act_map(&U->maps.ra[1], L.rsrc1, L.rc1p, L.W, L.H, n_img, c.box_h, c.box_n, f16));
        DTRAJ_TRY(make_w_map(&U->maps.rb, rwpk, rw_rows, c.ncols / (c.pair ? 2 : 1), f16));
    }
    if (L.M >= (int64_t)1 << 31) return fail(DTRAJ_EINVAL, "umma conv: M too large for 32-bit TMA coordinates");
    if (c.posm) {       // position-major tiles: dimensions {c, x, y, image}; operand box = one position of 128 images, output / residual box of 32
        const cuuint64_t esz = f16 ? 2 : 4;                    // operand box = 128 bytes of channels per pixel, epilogue box = 32 channels
        auto mapp = [&](CUtensorMap* m, const float* base, int cp, int bc, int bn, bool sw64) -> int {
            PFN_encodeTiled enc = get_encode_tiled();
            if (!enc) return fail(DTRAJ_ECUDA, "cuTensorMapEncodeTiled not available");
            cuuint64_t dims[4] = {(cuuint64_t)cp, (cuuint64_t)L.W, (cuuint64_t)L.H, (cuuint64_t)n_img};
            cuuint64_t strides[3] = {(cuuint64_t)cp * esz, (cuuint64_t)L.W * cp * esz, (cuuint64_t)HW * cp * esz};
            cuuint32_t box[4] = {(cuuint32_t)bc, 1, 1, (cuuint32_t)bn};
            cuuint32_t es[4] = {1, 1, 1, 1};
            CUresult r = enc(m, f16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, (void*)base, dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                             sw64 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                             CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
            if (r != CUDA_SUCCESS) return fail(DTRAJ_ECUDA, "cuTensorMapEncodeTiled(position-major map cp=%d n=%lld) -> %d", cp, (long long)n_img, (int)r);
            return 0;
        };
        DTRAJ_TRY(mapp(&U->maps.a[0], L.src0, L.c0p, kch, 128, false));
        if (L.c1p) DTRAJ_TRY(mapp(&U->maps.a[1], L.src1, L.c1p, kch, 128, false));
        if (npass == 3) {
            DTRAJ_TRY(mapp(&U->maps.a[2], L.src0_lo, L.c0p, kch, 128, false));
            if (L.c1p) DTRAJ_TRY(mapp(&U->maps.a[3], L.src1_lo, L.c1p, kch, 128, false));
        }
        if (L.flags & CONV_RESACC) {
            DTRAJ_TRY(mapp(&U->maps.ra[0], L.rsrc0, L.rc0p, kch, 128, false));
            if (L.rc1p) DTRAJ_TRY(mapp(&U->maps.ra[1], L.rsrc1, L.rc1p, kch, 128, false));
        }
        // (fp16 rows of 32 channels are 64 bytes: 64-byte swizzle; fp32 rows 128 bytes: 128-byte swizzle)
        if (!(L.flags & CONV_NOSTORE)) DTRAJ_TRY(mapp(&U->maps.out, L.out, L.coutp, 32, 32, f16 != 0));
        if (L.act_mode == ACT_SPLIT) DTRAJ_TRY(mapp(&U->maps.out_lo, L.out + L.lo_off, L.coutp, 32, 32, false));
        if (L.flags & CONV_RESID) DTRAJ_TRY(mapp(&U->maps.res, L.resid, L.coutp, 32, 32, f16 != 0));
        return 0;
    }
    if (c.halo == 2) {  // 16x16 / 32x32 maps: standard dimensions {c, x, y, image}; halo box 10 x 18, residual-conv box 8 x 16, output / residual box 8 x 4
        auto map4 = [&](CUtensorMap* m, const float* base, int cp, int bc, int bx, int by, bool sw64) -> int {
            PFN_encodeTiled enc = get_encode_tiled();
            if (!enc) return fail(DTRAJ_ECUDA, "cuTensorMapEncodeTiled not available");
            cuuint64_t dims[4] = {(cuuint64_t)cp, (cuuint64_t)L.W, (cuuint64_t)L.H, (cuuint64_t)n_img};
            cuuint64_t strides[3] = {(cuuint64_t)cp * 2, (cuuint64_t)L.W * cp * 2, (cuuint64_t)HW * cp * 2};
            cuuint32_t box[4] = {(cuuint32_t)bc, (cuuint32_t)bx, (cuuint32_t)by, 1};
            cuuint32_t es[4] = {1, 1, 1, 1};
            CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 4, (void*)base, dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                             sw64 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                             CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
            if (r != CUDA_SUCCESS) return fail(DTRAJ_ECUDA, "cuTensorMapEncodeTiled(%dx%d halo map cp=%d n=%lld) -> %d", L.H, L.W, cp, (long long)n_img, (int)r);
            return 0;
        };
        DTRAJ_TRY(map4(&U->maps.a[0], L.src0, L.c0p, 64, 10, 18, false));
        if (L.c1p) DTRAJ_TRY(map4(&U->maps.a[1], L.src1, L.c1p, 64, 10, 18, false));
        if (L.flags & CONV_RESACC) {
            DTRAJ_TRY(map4(&U->maps.ra[0], L.rsrc0, L.rc0p, 64, 8, 16, false));
            if (L.rc1p) DTRAJ_TRY(map4(&U->maps.ra[1], L.rsrc1, L.rc1p, 64, 8, 16, false));
        }
        if (!(L.flags & CONV_NOSTORE)) DTRAJ_TRY(map4(&U->maps.out, L.out, L.coutp, 32, 8, 4, true));
        if (L.flags & CONV_RESID) DTRAJ_TRY(map4(&U->maps.res, L.resid, L.coutp, 32, 8, 4, true));
        return 0;
    }
    if (c.halo) {      // every pixel-side map goes through the permuted dimensions {c, x, image, y}
        DTRAJ_TRY(make_perm8_map(&U->maps.a[0], L.src0, L.c0p, n_img, 64, 10, 10, false));
        if (L.c1p) DTRAJ_TRY(make_perm8_map(&U->maps.a[1], L.src1, L.c1p, n_img, 64, 10, 10, false));
        if (L.flags & CONV_RESACC) {
            DTRAJ_TRY(make_perm8_map(&U->maps.ra[0], L.rsrc0, L.rc0p, n_img, 64, 8, 8, false));
            if (L.rc1p) DTRAJ_TRY(make_perm8_map(&U->maps.ra[1], L.rsrc1, L.rc1p, n_img, 64, 8, 8, false));
        }
        if (!(L.flags & CONV_NOSTORE)) DTRAJ_TRY(make_perm8_map(&U->maps.out, L.out, L.coutp, n_img, 32, 8, 2, true));
        if (L.flags & CONV_RESID) DTRAJ_TRY(make_perm8_map(&U->maps.res, L.resid, L.coutp, n_img, 32, 8, 2, true));
        return 0;
    }
    if (!(L.flags & CONV_NOSTORE)) DTRAJ_TRY(make_rows_map(&U->maps.out, L.out, L.M, L.coutp, f16));
    if (L.act_mode == ACT_SPLIT) DTRAJ_TRY(make_rows_map(&U->maps.out_lo, L.out + L.lo_off, L.M, L.coutp));
    if (L.flags & CONV_RESID) DTRAJ_TRY(make_rows_map(&U->maps.res, L.resid, L.M, L.coutp, f16));
    return 0;
}

inline int launch_conv_umma(const UmmaLaunch& U, cudaStream_t st) {
    // (only the fp16 loop carries the PDL attribute: every kernel around it waits on its predecessor explicitly)
    if (U.conv.f16) {
        if (U.conv.pair) DTRAJ_CUDA(launch_ex(k_conv_umma_t<true, true>, U.grid, kUmmaThreads, U.smem, st, 2, true, U.maps, U.conv));
        else DTRAJ_CUDA(launch_ex(k_conv_umma_t<false, true>, U.grid, kUmmaThreads, U.smem, st, 1, true, U.maps, U.conv));
    } else {
        if (U.conv.pair) DTRAJ_CUDA(launch_ex(k_conv_umma_t<true, false>, U.grid, kUmmaThreads, U.smem, st, 2, false, U.maps, U.conv));
        else DTRAJ_CUDA(launch_ex(k_conv_umma_t<false, false>, U.grid, kUmmaThreads, U.smem, st, 1, false, U.maps, U.conv));
    }
    return 0;
}

}  // namespace dtraj
