// Fused enc1 block for sm_100a, fp16 mode (DTRAJ_PREC_F16): one kernel from the raw C-channel frame to the max-pooled
// enc1 output,
//     h  = relu(bn1(conv1_3x3(x))) + relu(time_mlp(temb))          (models.py:62-77, C = config.channels <= 4)
//     y  = relu(bn2(conv2_3x3(h))) + residual_conv_1x1(x)           (models.py:79-83)
//     p1 = MaxPool2d(2)(y)                                          (models.py:191)
// with BOTH convolutions on the tensor cores and nothing but x and p1 touching global memory inside the tile loop:
//   * conv2's packed weights ([tap][64-channel chunk][coutp][64] halfs) are RESIDENT in shared memory: 288 KB for the
//     teacher, 144 KB per CTA of a pair (each CTA holds its half of the output channels, tcgen05.mma.cta_group::2),
//     loaded once per CTA (the tf32 kernel re-read 295 KB of weights per 128-pixel tile);
//   * output tile = 16 image rows x 8 columns, halo = 18 x 10 = 180 pixels.  conv1 is a small GEMM
//     D1[halo pixel, cout] = A1[halo pixel, k] * W1[k, cout], k = tap * C + cin (9C <= 36 values, padded to K slices of
//     16): the MID warps gather A1 (one halo pixel per thread, prefetched a tile ahead) into shared memory as fp16,
//     the issuer runs it as one or two M = 256 MMAs per slice into a TMEM region of its own, and the mid warps read D1
//     back, add bias / ReLU / time bias, round to fp16 and write the 128-byte-swizzled K-major halo chunk buffers
//     (zero rows where the halo leaves the image: conv2's zero padding).  The first form of this kernel computed conv1
//     with CUDA-core FMAs in "generator" warps: 115 instructions per 8 outputs made it issue-bound (572 us against
//     ~170 us of conv2 MMAs for the teacher); the tensor-core form leaves ~25;
//   * the raw pixels conv1 needs -- a [C][20][12] fp32 patch per tile -- are copied by warp 0 with cp.async (zero-filled outside the
//     image = conv1's padding; a TMA box cannot be used: its innermost start x0 - 2 is not 16-byte aligned) into a small ring a few
//     tiles ahead, completion on an mbarrier, so the gather is 9C shared-memory loads without bounds checks
//     (round 1 gathered with 9C predicated global loads per halo pixel held in registers a tile ahead: at C = 3 that made the
//     mid warps the bottleneck, 64 ns per tile against 43 at C = 1, and spilled);
//   * each conv2 tap is a descriptor VIEW of the halo tile (start shifted by (dy*10 + dx) rows, 8-row groups 1280 bytes
//     apart; profiles/r01_umma_view_probe.txt): nothing is copied, no im2col re-reads;
//   * epilogue: bias, ReLU, 1x1 residual recomputed from x (fp32 FMAs), fp16 rounding, 2x2 max-pool, 16-byte stores.
// x enters conv1 rounded to fp16 like every other operand of this mode (11-bit significand; the range check of the
// mode covers it).
#pragma once
#include "enc1_umma.cuh"

namespace dtraj {

constexpr int kE1Mid = 8;                        // mid warps (two per TMEM lane quarter)
constexpr int kE1hThreads = 64 + 32 * kE1Epi + 32 * kE1Mid + 32;      // + the signal warp
constexpr int kE1SigBar = 11;                    // named barriers 11 .. 14: mid warps (bar.arrive) -> signal warp (bar.sync), one per halo buffer in flight
constexpr int kA1Rows = 192;                     // rows of an A1 operand slice kept in shared memory: 180 halo pixels, rounded up to 64.  The
                                                 // second M = 128 half of conv1's MMA reads rows 128..255 -- 64 rows past the slice, into
                                                 // whatever follows inside the CTA's allocation -- and D1 rows >= 180 are never looked at
constexpr int kA1SliceBytes = kA1Rows * 32;      // x 16 halfs
constexpr int kE1PatchH = 20, kE1PatchW = 12;    // conv1's receptive field of the 18 x 10 halo

struct Enc1hParams {
    int C, H, W, coutp;
    int n_chunks;                // coutp / 64: K chunks of conv2
    int n_tiles, tiles_x, tiles_per_img;
    int lg_tx, lg_tpi;           // log2(tiles_x), log2(tiles_per_img): both are powers of two (H = 16, 32 or 64)
    int n_hbuf;                  // halo chunk buffers in the ring (>= 1; 2 x n_chunks when they fit)
    int acc_cols;                // TMEM columns per accumulator; layout [acc0 | acc1 | n_d1 x (D1 rows 0-127 | D1 rows 128-255)]
    int n_d1;                    // D1 buffers: 2 when 6 x acc_cols <= 512 (conv1 of tile i+2 runs while tile i is converted), else 1
    int w_rows;                  // output channels this CTA holds: coutp, or coutp / 2 in pair mode
    int n_slices;                // K slices (16 values) of conv1's GEMM: ceil(9C / 16)
    const float* x; int64_t x_stride; const int32_t* row_sample; const int32_t* row_variant;
    int n_patch;                 // raw-input patch ring depth: 4, or 2 where 4 would cost a halo buffer
    const float* w3; const float* b3;          // conv1, BN folded, fp32: [9*C][coutp] (k = tap * C + cin); [coutp]
    const float* tbias; int tb_var_stride;     // relu(time_mlp(temb)) rows of enc1 for this t, 3 variants
    int tb_rows;                 // 1: row_variant indexes the whole [T][3] table (per-row timesteps): read the bias from global memory
    const float* bias2;                        // conv2 folded bias [coutp]
    const float* rw1; const float* rb1;        // residual 1x1: [C][coutp], [coutp]
    __half* pool_out;                          // [R, H/2, W/2, coutp]
    unsigned int* err;           // the owning handle's device error word (null: the library-wide word)
};

// byte offset of 16-byte K chunk kc (0/1) of row r inside a [rows][16 halfs] operand slice (32-byte rows, SWIZZLE_32B)
__device__ __forceinline__ uint32_t k16_off(int r, int kc) { return (uint32_t)(r * 32 + ((kc ^ ((r >> 2) & 1)) << 4)); }

template <bool kPair, int kC>
__global__ void __launch_bounds__(kE1hThreads, 1)
k_enc1_f16(const __grid_constant__ Enc1Maps maps, const Enc1hParams p) {
    constexpr int C = kC;                        // compile-time: the A1 gather is 9 * C loads, not 36 predicated ones
    constexpr int kBiasK = 9 * kC;               // K slots 9C and 9C + 1 carry conv1's folded bias (hi, lo) against A1 = 1
    extern __shared__ __align__(1024) uint8_t e1_smem[];
    const uint32_t base = (ptx::smem_u32(e1_smem) + 1023u) & ~1023u;
    uint8_t* gbase = e1_smem + (base - ptx::smem_u32(e1_smem));
    const int coutp = p.coutp;
    const uint32_t wblk_bytes = (uint32_t)p.w_rows * 128u;                 // one (tap, chunk) weight block in this CTA
    const uint32_t w_bytes = 9u * (uint32_t)p.n_chunks * wblk_bytes;
    const uint32_t b1_slice = (uint32_t)p.w_rows * 32u;
    // carve: [resident conv2 weights][halo ring][epilogue ring 4 x 2 KB][A1 slices][W1 slices][constants][barriers]
    const uint32_t wres0 = base;
    const uint32_t halo0 = wres0 + w_bytes;
    const uint32_t ring0 = halo0 + (uint32_t)p.n_hbuf * kE1HaloBytes;
    const uint32_t a1_0 = ring0 + kE1Epi * 2048u;
    const uint32_t a1_buf = (uint32_t)p.n_slices * kA1SliceBytes;         // one A1 buffer; there are n_d1 of them
    const uint32_t b1_0 = a1_0 + (uint32_t)p.n_d1 * a1_buf;
    const uint32_t cst0 = b1_0 + (((uint32_t)p.n_slices * b1_slice + 1023u) & ~1023u);
    // constants (floats): b3 | tbias [3][coutp] | bias2 | rb1 | rw1 [C][coutp]
    const int n_cst = (6 + C) * coutp;
    const uint32_t bar0 = (cst0 + (uint32_t)n_cst * 4u + 15u) & ~15u;
    auto hfull = [&](int b) { return bar0 + 8u * b; };
    auto hempty = [&](int b) { return bar0 + 64u + 8u * b; };
    const uint32_t acc_full0 = bar0 + 128u, acc_empty0 = bar0 + 144u, wbar = bar0 + 160u;
    const uint32_t a1_full0 = bar0 + 168u, d1_full0 = bar0 + 184u, d1_empty0 = bar0 + 200u;   // each [2]
    const uint32_t tmem_slot = bar0 + 216u;
    auto patch_full = [&](int b) { return bar0 + 232u + 8u * b; };
    auto patch_empty = [&](int b) { return bar0 + 264u + 8u * b; };
    const uint32_t patch_bytes = ((uint32_t)(C * kE1PatchH * kE1PatchW * 4) + 127u) & ~127u;
    const uint32_t patch0 = (bar0 + 296u + 127u) & ~127u;
    const uint32_t tmem_cols = (uint32_t)((2 + 2 * p.n_d1) * p.acc_cols) <= 256u ? 256u : 512u;
    volatile uint32_t* tmem_slot_ptr = reinterpret_cast<volatile uint32_t*>(gbase + (tmem_slot - base));
    float* cst = reinterpret_cast<float*>(gbase + (cst0 - base));
    const float* b3s = cst;
    const float* tbs = b3s + coutp;
    const float* bias2s = tbs + 3 * coutp;
    const float* rb1s = bias2s + coutp;
    const float* rw1s = rb1s + coutp;

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    unsigned int* const errw = p.err ? p.err : &g_umma_error;
    const int crank = kPair ? (int)ptx::cluster_ctarank() : 0;
    const uint16_t cmask = kPair ? 3 : 1;
    const int work0 = (int)blockIdx.x - crank;
    const uint32_t nrep = kPair ? 2u : 1u;                                 // CTAs reporting to the (leader's) barriers
#ifdef DTRAJ_PROBES
    // probe build (tools/timeline.py): slot 1 of g_timeline = this kernel's CTA 0: [tile][issuer | first mid warp | epilogue warp 2][event]
    const bool tl_on = blockIdx.x == 0 && (threadIdx.x & 31) == 0;
    const int tl_slot = 1;
    int tl_tile = 0;
#endif

    if (warp == 0) {
        if (ptx::elect_one()) {
            ptx::prefetch_tmap(&maps.w);
            // a role's warps meet at a named barrier and ONE thread arrives for the CTA: a cluster-scope release arrive
            // costs ~500 cycles of ERRBAR stall per arriving warp (ncu: a third of the mid warps' time when all eight arrived)
            for (int b = 0; b < p.n_hbuf; ++b) { ptx::mbar_init(hfull(b), nrep); ptx::mbar_init(hempty(b), 1); }
            for (int i = 0; i < 2; ++i) {
                ptx::mbar_init(acc_full0 + 8u * i, 1);
                ptx::mbar_init(acc_empty0 + 8u * i, kE1Epi * nrep);       // every epilogue warp reports its last accumulator load
            }
            ptx::mbar_init(wbar, 1);
            for (int i = 0; i < 2; ++i) {
                ptx::mbar_init(a1_full0 + 8u * i, nrep);
                ptx::mbar_init(d1_full0 + 8u * i, 1);
                ptx::mbar_init(d1_empty0 + 8u * i, kE1Mid * nrep);        // every mid warp reports its last D1 load
            }
            for (int i = 0; i < p.n_patch; ++i) { ptx::mbar_init(patch_full(i), 32); ptx::mbar_init(patch_empty(i), 1); }
            asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        }
        __syncwarp();
        if constexpr (!kPair) {
            asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "r"(tmem_cols) : "memory");
            asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
        } else {
            asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "r"(tmem_cols) : "memory");
            asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
        }
    }
    // constants, the conv1 weight operand W1 (fp16, this CTA's output channels) and zeroed A1 slices (all threads)
    for (int i = threadIdx.x; i < coutp; i += blockDim.x) {
        cst[i] = p.b3[i];
        for (int v = 0; v < 3; ++v) cst[(1 + v) * coutp + i] = p.tbias[(size_t)v * p.tb_var_stride + i];
        cst[4 * coutp + i] = p.bias2[i];
        cst[5 * coutp + i] = p.rb1[i];
    }
    for (int i = threadIdx.x; i < C * coutp; i += blockDim.x) cst[6 * coutp + i] = p.rw1[i];
    for (int i = threadIdx.x; i < p.n_d1 * p.n_slices * (kA1SliceBytes / 16); i += blockDim.x)
        reinterpret_cast<uint4*>(gbase + (a1_0 - base))[i] = make_uint4(0u, 0u, 0u, 0u);
    __syncthreads();
    for (int i = threadIdx.x; i < p.n_d1 * 2 * kA1Rows; i += blockDim.x) {    // the bias slots of every A1 row hold 1.0
        const int bb = i / (2 * kA1Rows), r = (i >> 1) % kA1Rows, k = kBiasK + (i & 1);
        *reinterpret_cast<__half*>(gbase + (a1_0 - base) + bb * a1_buf + (k >> 4) * kA1SliceBytes + k16_off(r, (k >> 3) & 1) + (k & 7) * 2) = __float2half_rn(1.f);
    }
    for (int i = threadIdx.x; i < p.n_slices * p.w_rows * 16; i += blockDim.x) {
        const int s = i / (p.w_rows * 16), rem = i - s * p.w_rows * 16, nl = rem >> 4, e = rem & 15, k = 16 * s + e;
        const int n = crank * p.w_rows + nl;
        float v = 0.f;
        if (k < 9 * C) v = p.w3[(size_t)k * coutp + n];
        else if (k == kBiasK) v = __half2float(__float2half_rn(p.b3[n]));
        else if (k == kBiasK + 1) v = p.b3[n] - __half2float(__float2half_rn(p.b3[n]));
        *reinterpret_cast<__half*>(gbase + (b1_0 - base) + s * b1_slice + k16_off(nl, e >> 3) + (e & 7) * 2) = __float2half_rn(v);
    }
    ptx::fence_proxy_async();
    ptx::tc_fence_before();
    __syncthreads();
    if constexpr (kPair) ptx::cluster_sync_all();
    ptx::tc_fence_after();
    const uint32_t tmem_base = *tmem_slot_ptr;
    pdl_launch_dependents();
    pdl_wait();                                // everything above read weights / tables only; x and pool_out belong to other kernels

    auto tile_geom = [&](int tile, int& img, int& y0, int& x0) {
        img = tile >> p.lg_tpi;
        const int r = tile & (p.tiles_per_img - 1);
        y0 = (r >> p.lg_tx) * 16;
        x0 = (r & (p.tiles_x - 1)) * 8;
    };

    if (warp == 0) {
        // ------------------------------------------------------------ one-time TMA load of the resident conv2 weights
        if (ptx::elect_one()) {
            uint32_t fb = wbar;
            if constexpr (kPair) fb = ptx::map_to_cta(fb, 0);              // both CTAs' bytes complete on the leader's barrier
            if (!kPair || crank == 0) ptx::mbar_expect_tx(wbar, w_bytes * nrep);
            for (int b = 0; b < 9 * p.n_chunks; ++b) {                     // block b = tap * n_chunks + chunk
                const int row = b * coutp + crank * p.w_rows;
                if constexpr (kPair) ptx::tma_load_2d_2sm(wres0 + b * wblk_bytes, &maps.w, fb, 0, row);
                else ptx::tma_load_2d(wres0 + b * wblk_bytes, &maps.w, fb, 0, row);
            }
        }
        __syncwarp();
        // ---- then (all 32 lanes) the raw-input patches of this CTA's tiles, a few tiles ahead of the mid warps: 4-byte cp.async
        // per element with zero fill outside the image, one cp.async.mbarrier.arrive per lane and patch
        {
            int pb = 0;
            uint32_t pph = 0;
            bool ok = true;
            // 8-byte copies: a patch row starts at x0 - 2 (even), so its 12 floats are 6 aligned pairs that lie inside or outside the image
            // together.  30 lanes = 5 rows x 6 pairs per trip, (channel, row) carried incrementally: 4 trips at C = 1, 12 at C = 3
            // (the first form -- 4-byte copies indexed by two divisions -- took ~4800 cycles per C = 3 patch in this one warp and
            // was the kernel's pace on 3-channel models, profiles/r02i_timeline.txt)
            const int HW = p.H * p.W, n_rows = C * kE1PatchH;
            const int l_row = lane / 6, l_pair = lane - 6 * l_row;           // lanes 30, 31 idle
            for (int wk = work0; wk < p.n_tiles && ok; wk += gridDim.x) {
                const int tile = wk + crank;
                int img, y0, x0;
                tile_geom(tile, img, y0, x0);
                const bool real = tile < p.n_tiles;                 // (a pair's padding tile gets an all-zero patch)
                const int smp = real ? (p.row_sample ? __ldg(p.row_sample + img) : img) : 0;
                const float* xs = p.x + (size_t)smp * p.x_stride;
                ok = ptx::mbar_wait(errw, patch_empty(pb), pph ^ 1u);
                const uint32_t dst0 = patch0 + (uint32_t)pb * patch_bytes;
                const int sx = x0 - 2 + 2 * l_pair;
                const bool in_x = real && lane < 30 && sx >= 0 && sx < p.W;
                int ci = 0, r = l_row;                              // this lane's (channel, patch row) of the current trip
                for (int rp = l_row; rp < n_rows; rp += 5) {
                    const int sy = y0 - 2 + r;
                    const bool in = in_x && sy >= 0 && sy < p.H;
                    const float* src = in ? xs + (size_t)ci * HW + sy * p.W + sx : p.x;
                    if (lane < 30)
                        asm volatile("cp.async.ca.shared.global [%0], [%1], 8, %2;" ::"r"(dst0 + 4u * (uint32_t)(rp * kE1PatchW + 2 * l_pair)), "l"(src), "r"(in ? 8u : 0u) : "memory");
                    r += 5;
                    if (r >= kE1PatchH) { r -= kE1PatchH; ++ci; }
                }
                asm volatile("cp.async.mbarrier.arrive.noinc.shared::cta.b64 [%0];" ::"r"(patch_full(pb)) : "memory");
                if (++pb == p.n_patch) { pb = 0; pph ^= 1u; }
            }
        }
    } else if (warp == 1) {
        // ------------------------------------------------------------ MMA issuer (pair: leader CTA only)
        if (ptx::elect_one() && (!kPair || crank == 0)) {
            const uint32_t idesc = umma_idesc_f16(coutp) + (kPair ? ((uint32_t)(128 >> 4) << 24) : 0u);
            // halo view: K-major SWIZZLE_128B, 8-row groups one halo row (10 pixels = 1280 B) apart
            const uint64_t hdesc0 = ((uint64_t)1 << 16) | ((uint64_t)(1280 >> 4) << 32) | ((uint64_t)1 << 46) | ((uint64_t)2 << 61);
            // 32-byte-row operands of conv1: 8-row groups 256 B apart, SWIZZLE_32B
            const uint64_t kdesc0 = ((uint64_t)1 << 16) | ((uint64_t)(256 >> 4) << 32) | ((uint64_t)1 << 46) | ((uint64_t)6 << 61);
            auto kdesc = [&](uint32_t addr) { return kdesc0 | (uint64_t)((addr >> 4) & 0x3fffu); };
            int hb = 0, acc = 0, it = 0;
            uint32_t hph = 0, acc_ph = 0;
            bool ok = ptx::mbar_wait(errw, wbar, 0u);
            const int n_my = work0 < p.n_tiles ? (p.n_tiles - work0 + (int)gridDim.x - 1) / (int)gridDim.x : 0;   // tile iterations of this CTA (pair)
            // conv1 of tile-iteration j into D1 buffer j % n_d1: D1[g] = A1[rows 128g ..] * W1^T, g = 0, 1
            auto issue_conv1 = [&](int j) {
                const int b = j & (p.n_d1 - 1);
                ok = ok && ptx::mbar_wait(errw, a1_full0 + 8u * b, (uint32_t)((j >> (p.n_d1 - 1)) & 1));
                ok = ok && ptx::mbar_wait(errw, d1_empty0 + 8u * b, (uint32_t)(((j >> (p.n_d1 - 1)) & 1) ^ 1));
                ptx::tc_fence_after();
                const uint32_t d1_tmem = tmem_base + (uint32_t)((2 + 2 * b) * p.acc_cols);
                for (int g = 0; g < 2; ++g)
                    for (int s = 0; s < p.n_slices; ++s) {
                        const uint64_t ad = kdesc(a1_0 + (uint32_t)b * a1_buf + (uint32_t)s * kA1SliceBytes + (uint32_t)g * 4096u);
                        const uint64_t bd = kdesc(b1_0 + (uint32_t)s * b1_slice);
                        if constexpr (!kPair) ptx::mma_f16(d1_tmem + (uint32_t)(g * p.acc_cols), ad, bd, idesc, s ? 1u : 0u);
                        else ptx::mma_f16_2sm(d1_tmem + (uint32_t)(g * p.acc_cols), ad, bd, idesc, s ? 1u : 0u);
                    }
                // (its completion also frees A1: the mid warps write the next tile's A1 after seeing d1_full)
                if constexpr (kPair) ptx::tc_commit_2sm(d1_full0 + 8u * b, cmask); else ptx::tc_commit(d1_full0 + 8u * b);
            };
            // A1 and D1 have n_d1 buffers each: the mid warps publish A1(j + n_d1) once they have seen conv1(j) complete
            if (n_my > 0) issue_conv1(0);
            if (p.n_d1 == 2 && n_my > 1) issue_conv1(1);
            for (int wk = work0; wk < p.n_tiles && ok; wk += gridDim.x, ++it) {
                DTRAJ_TL(0, 0);
                ok = ptx::mbar_wait(errw, acc_empty0 + 8u * acc, acc_ph ^ 1u);
                ptx::tc_fence_after();
                DTRAJ_TL(0, 1);
                const uint32_t d_tmem = tmem_base + (uint32_t)(acc * p.acc_cols);
                uint32_t accum = 0u;
                for (int c = 0; c < p.n_chunks && ok; ++c) {
                    ok = ok && ptx::mbar_wait(errw, hfull(hb), hph);      // this chunk's halo tile is in shared memory (both CTAs)
                    ptx::tc_fence_after();
                    // one D1 buffer: the next tile's conv1 goes in front of THIS tile's first chunk.  A1(it + 1) is published together
                    // with that chunk and the mid warps release D1(it) a few hundred cycles later (their last tcgen05.ld), so the issuer
                    // waits briefly here -- but D1(it + 1) is then ready one chunk of MMAs (~2500 cycles) earlier than behind chunk 0, and
                    // that wait was on the critical cycle D1 -> gather -> conversion -> chunk-0 MMAs -> conv1 (profiles/r02i_timeline.txt)
                    if (p.n_d1 == 1 && c == 0 && it + 1 < n_my) issue_conv1(it + 1);
                    DTRAJ_TL(0, 2 + 2 * (c & 1));
                    const uint32_t hbuf = halo0 + (uint32_t)hb * kE1HaloBytes;
                    int dy = 0, dx = 0;
                    for (int t = 0; t < 9; ++t) {
                        const uint32_t a_addr = hbuf + (uint32_t)(dy * 10 + dx) * 128u;
                        const uint64_t ad = hdesc0 | (uint64_t)((a_addr >> 4) & 0x3fffu);
                        const uint64_t bd = umma_desc_sw128(wres0 + (uint32_t)(t * p.n_chunks + c) * wblk_bytes);
#pragma unroll
                        for (int k = 0; k < 4; ++k) {
                            if constexpr (!kPair) ptx::mma_f16(d_tmem, ad + 2u * k, bd + 2u * k, idesc, accum);
                            else ptx::mma_f16_2sm(d_tmem, ad + 2u * k, bd + 2u * k, idesc, accum);
                            accum = 1u;
                        }
                        if (++dx == 3) { dx = 0; ++dy; }
                    }
                    if constexpr (kPair) ptx::tc_commit_2sm(hempty(hb), cmask); else ptx::tc_commit(hempty(hb));
                    DTRAJ_TL(0, 3 + 2 * (c & 1));
                    if (++hb == p.n_hbuf) { hb = 0; hph ^= 1u; }
                }
                if constexpr (kPair) ptx::tc_commit_2sm(acc_full0 + 8u * acc, cmask); else ptx::tc_commit(acc_full0 + 8u * acc);
                if (++acc == 2) { acc = 0; acc_ph ^= 1u; }
                // two D1 buffers: tile it's buffer is free once its conversion is done; refill it for tile it + 2
                if (p.n_d1 == 2 && it + 2 < n_my) issue_conv1(it + 2);
                DTRAJ_TL(0, 6);
#ifdef DTRAJ_PROBES
                ++tl_tile;
#endif
            }
        }
    } else if (warp == 2 + kE1Epi + kE1Mid) {
        // ------------------------------------------------------------ signal warp: publishes what the mid warps wrote
        // Round 1 published a halo chunk with fence.acq_rel.cluster + relaxed arrivals from a mid thread: MEMBAR.ALL.GPU + CCTL.IVALL,
        // 1500 - 2800 cycles, between every two chunks of all eight mid warps (they met at a barrier per chunk) -- the mid warps were
        // the kernel's bottleneck at 3000 cycles per chunk, 1350 of them work, the issuer waiting for halo tiles 60 % of the time
        // (profiles/r02i_timeline.txt).  Now the mid warps only bar.arrive and go on; this warp waits for all 256 of them and arrives
        // on the leader's barriers with CTA-scope release: every writer has already made its shared-memory stores visible to the
        // tensor core's proxy (fence.proxy.async) before the named barrier, so the arrival only has to follow that barrier.
        auto arrive_one = [&](uint32_t bar) {
            if constexpr (!kPair) ptx::mbar_arrive(bar);
            else ptx::mbar_arrive_cluster_cta(ptx::map_to_cta(bar, 0));
        };
        const int G = (int)gridDim.x, Ld = p.n_d1;
        int hb = 0, it = 0;
        unsigned cnt = 0;
        for (int wk = work0; wk < p.n_tiles; wk += G, ++it) {
            const int b = it & (Ld - 1);
            const bool next = wk + Ld * G < p.n_tiles;
            for (int c = 0; c < p.n_chunks; ++c, ++cnt) {
                asm volatile("bar.sync %0, %1;" ::"r"(kE1SigBar + (int)(cnt & 3u)), "r"(32 * kE1Mid + 32) : "memory");
                if (lane == 0) {
                    if (c == 0 && next) ptx::mbar_arrive(patch_empty((it + Ld) & (p.n_patch - 1)));   // every gatherer has arrived
                    if (c == 0 && next) arrive_one(a1_full0 + 8u * b);
                    arrive_one(hfull(hb));
                }
                __syncwarp();
                if (++hb == p.n_hbuf) hb = 0;
            }
        }
    } else if (warp >= 2 + kE1Epi) {
        // ------------------------------------------------------------ mid warps: A1 gather, D1 -> halo chunk buffers
        const int mt = threadIdx.x - 32 * (2 + kE1Epi);            // 0..255
        const int q = warp & 3;                                     // TMEM lane quarter of this warp
        const int h = (warp - (2 + kE1Epi)) >> 2;                   // the quarter's two warps split every 64-channel chunk: cells 4h..4h+3
        const int HW = p.H * p.W;
        // Work balance: quarters 0 and 1 convert two D1 rows per thread (regions 0 and 1), quarters 2 and 3 only one --
        // so the four warps of quarters 2 and 3 (128 threads) gather ALL of A1: rows tq and tq + 128 (< 180).
        constexpr bool bal = true;
        const bool a1_warp = q >= 2;
        const int tq = (2 * h + (q & 1)) * 32 + lane;               // 0..127 over the A1-gathering threads
        const int a_row[2] = {bal ? tq : mt, tq + 128};
        const bool a_has[2] = {bal ? a1_warp : mt < kE1HaloRows, bal && a1_warp && tq + 128 < kE1HaloRows};
        const int a_ry[2] = {a_row[0] / 10, a_row[1] / 10};
        const int a_rx[2] = {a_row[0] - a_ry[0] * 10, a_row[1] - a_ry[1] * 10};
        uint8_t* a1p = gbase + (a1_0 - base);
        // the two halo pixels whose D1 rows this thread converts: px0 = 32q + lane (region 0), px1 = 128 + 32q + lane (region 1)
        const int px0 = 32 * q + lane, px1 = 128 + 32 * q + lane;
        const bool has1 = 128 + 32 * q < kE1HaloRows;               // warp-uniform: quarters 0 and 1 own rows of region 1
        const int ry0 = px0 / 10, rx0 = px0 - ry0 * 10, ry1 = px1 / 10, rx1 = px1 - ry1 * 10;
        // the time-bias variant of a tile's image is fetched two tiles ahead, so that load is never waited for in the loop
        int var_n = 0;
        auto fetch_idx = [&](int wk) {
            const int tile = wk + crank;
            const int img = tile >> p.lg_tpi;
            var_n = (wk < p.n_tiles && tile < p.n_tiles && p.row_variant) ? __ldg(p.row_variant + img) : 0;
        };
        // this thread's A1 rows of tile-iteration `pit`, gathered from that tile's raw patch [C][20][12] (origin = two pixels up and
        // left of the tile; TMA zero-filled it outside the image): per K slice two 16-byte stores (taps, the two bias slots = 1.0,
        // zero padding).  The patch is released (patch_empty) by thread 0 after the named barrier that follows every call.
        auto gather_a1 = [&](int buf, int pit) {
            const int pbuf = pit & (p.n_patch - 1);
            ptx::mbar_wait(errw, patch_full(pbuf), (uint32_t)((pit / p.n_patch) & 1));
#ifdef DTRAJ_PROBES
            if (tl_on && mt == 0 && tl_tile < 16) g_timeline[1][tl_tile][1][12] = clock64();
#endif
            const float* patch = reinterpret_cast<const float*>(gbase + (patch0 - base) + (uint32_t)pbuf * patch_bytes);
            uint8_t* const a1b = a1p + (uint32_t)buf * a1_buf;
#pragma unroll
            for (int rr = 0; rr < 2; ++rr) {
                if (!a_has[rr]) continue;                           // (warp-uniform for rr = 0; the second row ends inside one warp)
                const float* pp = patch + a_ry[rr] * kE1PatchW + a_rx[rr];
                float xv[9 * kC];
#pragma unroll
                for (int k = 0; k < 9 * kC; ++k) xv[k] = pp[(k % kC) * (kE1PatchH * kE1PatchW) + ((k / kC) / 3) * kE1PatchW + (k / kC) % 3];
#pragma unroll
                for (int sl = 0; sl < (9 * kC + 2 + 15) / 16; ++sl)
#pragma unroll
                    for (int kc = 0; kc < 2; ++kc) {
                        float v[8];
#pragma unroll
                        for (int e = 0; e < 8; ++e) {
                            const int k = 16 * sl + 8 * kc + e;
                            v[e] = k < 9 * kC ? xv[k] : ((k == kBiasK || k == kBiasK + 1) ? 1.f : 0.f);
                        }
                        uint4 o;
                        __half2* oh = reinterpret_cast<__half2*>(&o);
#pragma unroll
                        for (int e = 0; e < 4; ++e) oh[e] = __floats2half2_rn(v[2 * e], v[2 * e + 1]);
                        *reinterpret_cast<uint4*>(a1b + sl * kA1SliceBytes + k16_off(a_row[rr], kc)) = o;
                    }
            }
        };
        // the CTA's single arrival on (the leader's) barrier `bar`, after the role's warps met at a named barrier
        auto arrive_one = [&](uint32_t bar) {
            if constexpr (!kPair) ptx::mbar_arrive(bar);
            else ptx::mbar_arrive_cluster_cta(ptx::map_to_cta(bar, 0));
        };
        // Software pipeline with lead Ld = n_d1 (buffers of A1 and of D1).  At the top of iteration `it`: A1(it .. it+Ld-1) are
        // published (their conv1 issued or done), the patch of tile it + Ld is loaded or in flight, vq[k] = variant of tile
        // it + k (k <= Ld), var_n = variant of tile it + Ld + 1.  With Ld = 2 the conv1 round trip (publish -> issue -> MMA ->
        // commit) of tile it + 2 runs under the conversion of tile it + 1, so the mid warps never wait for it.
        const int G = (int)gridDim.x, Ld = p.n_d1;
        int hb = 0, it = 0, vq[3] = {0, 0, 0};
        uint32_t hph = 0;
        unsigned cnt = 0;                                           // chunks handed to the signal warp
        if (work0 < p.n_tiles) {
            fetch_idx(work0);
            for (int j = 0; j < Ld; ++j) {                         // A1(0 .. Ld-1)
                const bool ex = work0 + j * G < p.n_tiles;          // (CTA-uniform)
                vq[j] = var_n;
                fetch_idx(work0 + (j + 1) * G);
                if (ex) {
                    gather_a1(j, j);
                    ptx::fence_proxy_async();
                    asm volatile("bar.sync 9, 256;" ::: "memory");
                    if (mt == 0) { ptx::mbar_arrive(patch_empty(j & (p.n_patch - 1))); arrive_one(a1_full0 + 8u * j); }
                }
            }
            vq[Ld] = var_n;
            fetch_idx(work0 + (Ld + 1) * G);
        }
        for (int wk = work0; wk < p.n_tiles; wk += G, ++it) {
            const int tile = wk + crank;
            int img, y0, x0;
            tile_geom(tile, img, y0, x0);
            const bool real = tile < p.n_tiles;
            const int b = it & (Ld - 1);
#ifdef DTRAJ_PROBES
            const bool tl_outer = tl_on;
            const bool tl_on = tl_outer && mt == 0;
#endif
            DTRAJ_TL(1, 0);
            ptx::mbar_wait(errw, d1_full0 + 8u * b, (uint32_t)((it >> (Ld - 1)) & 1));    // conv1(it) done: D1 readable, A1 buffer b free
            ptx::tc_fence_after();
            DTRAJ_TL(1, 1);
            const bool next = wk + Ld * G < p.n_tiles;
            if (next) gather_a1(b, it + Ld);
            DTRAJ_TL(1, 2);                        // A1(it + Ld); published together with the first halo chunk below
            const int var0 = vq[0];
            const float* tb = p.tb_rows ? p.tbias + (size_t)var0 * p.tb_var_stride : tbs + var0 * coutp;
            vq[0] = vq[1];
            if (Ld == 2) { vq[1] = vq[2]; vq[2] = var_n; } else vq[1] = var_n;
            fetch_idx(wk + (Ld + 2) * G);
            // ---- D1 -> halo chunk buffers
            const int yy0 = y0 - 1 + ry0, xx0 = x0 - 1 + rx0, yy1 = y0 - 1 + ry1, xx1 = x0 - 1 + rx1;
            const bool in0 = real && yy0 >= 0 && yy0 < p.H && xx0 >= 0 && xx0 < p.W;                       // else: conv2's zero padding
            const bool in1 = real && px1 < kE1HaloRows && yy1 >= 0 && yy1 < p.H && xx1 >= 0 && xx1 < p.W;
            const uint32_t t_d1 = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)((2 + 2 * b) * p.acc_cols);
            for (int c = 0; c < p.n_chunks; ++c) {
                const int col0 = 64 * c + 32 * h;                   // this warp's 32 channels of the chunk
                uint32_t r0[32], r1[32];
                ptx::tmem_ld32(t_d1 + (uint32_t)col0, r0);
                if (has1) ptx::tmem_ld32(t_d1 + (uint32_t)(p.acc_cols + col0), r1);
                ptx::tmem_ld_wait();
                ptx::tc_fence_before();
                // D1 is in registers: with the tile's last chunk this warp is done with the buffer.  Reported HERE, not with the chunk's
                // publication ~2000 cycles later: with one D1 buffer (coutp = 128) the next tile's conv1 -- and through it the whole next
                // tile of the mid warps -- hangs on this arrival (profiles/r02i_timeline.txt: they idled 2500 of 6600 cycles per tile)
                if (c == p.n_chunks - 1) {
                    __syncwarp();
                    if (lane == 0) arrive_one(d1_empty0 + 8u * b);
                }
                DTRAJ_TL(1, 3 + 4 * (c & 1));
                ptx::mbar_wait(errw, hempty(hb), hph ^ 1u);               // the conv2 MMAs that read this buffer have retired
                DTRAJ_TL(1, 4 + 4 * (c & 1));
                uint8_t* hbuf = gbase + (halo0 - base) + (size_t)hb * kE1HaloBytes;
                // h = relu(D1) + time bias (conv1's folded bias is inside D1), rounded to fp16; zero rows outside the image.
                // Both rows of a thread in ONE branch-free pass: they share the time-bias loads, and the two independent chains fill
                // each other's latencies (as two predicated passes the quarters that own two rows took 1800 cycles per chunk and set
                // the pace of all mid warps, profiles/r02i_timeline.txt)
                const bool st1 = has1 && px1 < kE1HaloRows;
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const float4 ta = *reinterpret_cast<const float4*>(tb + col0 + 8 * j), tc = *reinterpret_cast<const float4*>(tb + col0 + 8 * j + 4);
                    const float t8[8] = {ta.x, ta.y, ta.z, ta.w, tc.x, tc.y, tc.z, tc.w};
                    uint4 o0, o1;
                    __half2* h0 = reinterpret_cast<__half2*>(&o0);
                    __half2* h1 = reinterpret_cast<__half2*>(&o1);
#pragma unroll
                    for (int e = 0; e < 4; ++e) {
                        h0[e] = __floats2half2_rn(fmaxf(__uint_as_float(r0[8 * j + 2 * e]), 0.f) + t8[2 * e], fmaxf(__uint_as_float(r0[8 * j + 2 * e + 1]), 0.f) + t8[2 * e + 1]);
                        if (has1) h1[e] = __floats2half2_rn(fmaxf(__uint_as_float(r1[8 * j + 2 * e]), 0.f) + t8[2 * e], fmaxf(__uint_as_float(r1[8 * j + 2 * e + 1]), 0.f) + t8[2 * e + 1]);
                    }
                    if (!in0) o0 = make_uint4(0u, 0u, 0u, 0u);
                    *reinterpret_cast<uint4*>(hbuf + px0 * 128 + (((uint32_t)(4 * h + j) ^ (uint32_t)(px0 & 7)) << 4)) = o0;
                    if (has1) {
                        if (!in1) o1 = make_uint4(0u, 0u, 0u, 0u);
                        if (st1) *reinterpret_cast<uint4*>(hbuf + px1 * 128 + (((uint32_t)(4 * h + j) ^ (uint32_t)(px1 & 7)) << 4)) = o1;
                    }
                }
                DTRAJ_TL(1, 5 + 4 * (c & 1));
                ptx::fence_proxy_async();                           // generic-proxy writes -> visible to the tensor core
                // hand the chunk (with c == 0: also A1 of tile it + Ld and its consumed patch) to the signal warp and go on.  At most
                // n_hbuf <= 4 chunks are in flight (hempty above), one named barrier each
                asm volatile("bar.arrive %0, %1;" ::"r"(kE1SigBar + (int)(cnt & 3u)), "r"(32 * kE1Mid + 32) : "memory");
                ++cnt;
                DTRAJ_TL(1, 6 + 4 * (c & 1));
                if (++hb == p.n_hbuf) { hb = 0; hph ^= 1u; }
            }
            DTRAJ_TL(1, 11);
#ifdef DTRAJ_PROBES
            ++tl_tile;
#endif
        }
    } else {
        // ------------------------------------------------------------ epilogue (warps 2..5): thread = output pixel
        const int q = warp & 3, ew = warp - 2;
        const int nchunk = coutp >> 5;                              // 32-column steps
        uint8_t* bufp = gbase + (ring0 - base) + (size_t)ew * 2048; // [32 rows][32 halfs], 64-byte swizzle
        const uint32_t swz = (uint32_t)((lane >> 1) & 3);
        const int Wh = p.W >> 1, HW = p.H * p.W;
        const int r = 32 * q + lane, yl = r >> 3, xl = r & 7;      // row of the 16 x 8 tile
        int acc = 0;
        uint32_t acc_ph = 0;
        float amax = 0.f;
        auto arrive_acc_empty = [&]() {
            if constexpr (!kPair) ptx::mbar_arrive(acc_empty0 + 8u * acc);
            else ptx::mbar_arrive_cluster_relaxed(ptx::map_to_cta(acc_empty0 + 8u * acc, 0));
        };
        float xn[4] = {0.f, 0.f, 0.f, 0.f};                        // this thread's pixel of x for the NEXT tile
        int smp_n = 0;                                              // sample index of the next tile, fetched two tiles ahead
        auto fetch_idx = [&](int wk) {
            const int tile = wk + crank;
            const int img = tile >> p.lg_tpi;
            smp_n = (wk < p.n_tiles && tile < p.n_tiles) ? (p.row_sample ? __ldg(p.row_sample + img) : img) : 0;
        };
        auto prefetch = [&](int wk, int smp) {
            const int tile = wk + crank;
            int img, y0, x0;
            tile_geom(tile, img, y0, x0);
            if (tile < p.n_tiles) {
                const float* xs = p.x + (size_t)smp * p.x_stride + (size_t)(y0 + yl) * p.W + x0 + xl;
#pragma unroll
                for (int ci = 0; ci < kC; ++ci) xn[ci] = __ldg(xs + (size_t)ci * HW);
            }
        };
        fetch_idx(work0);
        prefetch(work0, smp_n);
        fetch_idx(work0 + (int)gridDim.x);
        for (int wk = work0; wk < p.n_tiles; wk += gridDim.x) {
            const int tile = wk + crank;
            int img, y0, x0;
            tile_geom(tile, img, y0, x0);
            const bool real = tile < p.n_tiles;
            float xv[4];
#pragma unroll
            for (int ci = 0; ci < 4; ++ci) xv[ci] = xn[ci];
            if (wk + (int)gridDim.x < p.n_tiles) {
                prefetch(wk + (int)gridDim.x, smp_n);
                fetch_idx(wk + 2 * (int)gridDim.x);
            }
#ifdef DTRAJ_PROBES
            const bool tl_outer = tl_on;
            const bool tl_on = tl_outer && ew == 0;
#endif
            DTRAJ_TL(2, 0);
            ptx::mbar_wait(errw, acc_full0 + 8u * acc, acc_ph);
            ptx::tc_fence_after();
            DTRAJ_TL(2, 1);
            const uint32_t t_acc = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(acc * p.acc_cols);
            // One warp per scheduler does all of this, and since the mid warps stopped being the kernel's pace the epilogue is (5600 of
            // 6200 cycles per tile, profiles/r02i_timeline.txt): the next chunk's TMEM load is issued before this chunk's pool + store,
            // the per-channel constants of the next 8 columns are loaded ahead of the math, and "accumulator drained" is a relaxed
            // arrival per warp instead of a named barrier + one arrival
            uint32_t raw[32];
            ptx::tmem_ld32(t_acc, raw);
            for (int c = 0; c < nchunk; ++c) {
                ptx::tmem_ld_wait();
                DTRAJ_TL(2, 2 + 3 * (c & 3));
                if (c == nchunk - 1) {
                    ptx::tc_fence_before();
                    __syncwarp();
                    if (lane == 0) arrive_acc_empty();
                }
                uint8_t* rowp = bufp + lane * 64;
                float4 cb[2][2], cr[2][2], cw[2][kC][2];            // [parity of j][...][half]: bias2 | rb1 | rw1 of 8 columns
                auto load_consts = [&](int j, int par) {
                    const int col = 32 * c + 8 * j;
#pragma unroll
                    for (int hh = 0; hh < 2; ++hh) {
                        cb[par][hh] = *reinterpret_cast<const float4*>(bias2s + col + 4 * hh);
                        cr[par][hh] = *reinterpret_cast<const float4*>(rb1s + col + 4 * hh);
#pragma unroll
                        for (int ci = 0; ci < kC; ++ci) cw[par][ci][hh] = *reinterpret_cast<const float4*>(rw1s + (size_t)ci * coutp + col + 4 * hh);
                    }
                };
                load_consts(0, 0);
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    if (j < 3) load_consts(j + 1, (j + 1) & 1);
                    float v[8];
#pragma unroll
                    for (int hh = 0; hh < 2; ++hh) {
                        const float4 b4 = cb[j & 1][hh];
                        float4 r4 = cr[j & 1][hh];
#pragma unroll
                        for (int ci = 0; ci < kC; ++ci) {
                            const float4 w4 = cw[j & 1][ci][hh];
                            r4.x = fmaf(xv[ci], w4.x, r4.x); r4.y = fmaf(xv[ci], w4.y, r4.y);
                            r4.z = fmaf(xv[ci], w4.z, r4.z); r4.w = fmaf(xv[ci], w4.w, r4.w);
                        }
                        v[4 * hh] = fmaxf(__uint_as_float(raw[8 * j + 4 * hh]) + b4.x, 0.f) + r4.x;
                        v[4 * hh + 1] = fmaxf(__uint_as_float(raw[8 * j + 4 * hh + 1]) + b4.y, 0.f) + r4.y;
                        v[4 * hh + 2] = fmaxf(__uint_as_float(raw[8 * j + 4 * hh + 2]) + b4.z, 0.f) + r4.z;
                        v[4 * hh + 3] = fmaxf(__uint_as_float(raw[8 * j + 4 * hh + 3]) + b4.w, 0.f) + r4.w;
                    }
                    uint4 pk;
                    __half2* ph2 = reinterpret_cast<__half2*>(&pk);
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                        amax = fmaxf(amax, fmaxf(fabsf(v[2 * i]), fabsf(v[2 * i + 1])));
                        ph2[i] = __floats2half2_rn(v[2 * i], v[2 * i + 1]);
                    }
                    *reinterpret_cast<uint4*>(rowp + (((uint32_t)j ^ swz) << 4)) = pk;
                }
                if (c + 1 < nchunk) ptx::tmem_ld32(t_acc + (uint32_t)(32 * (c + 1)), raw);     // in flight under the pool + store below
                DTRAJ_TL(2, 3 + 3 * (c & 3));
                __syncwarp();
                if (real) {
                    // the warp's 4 x 8 pixel patch holds 2 x 4 complete 2x2 windows: lane -> (window, 16-byte cell)
                    const int pr = lane >> 2, wy = pr >> 2, wx = pr & 3;
                    const int r00 = (2 * wy) * 8 + 2 * wx;
                    const int py = (y0 + 4 * q + 2 * wy) >> 1, pxx = (x0 + 2 * wx) >> 1;
                    const uint32_t jj = (uint32_t)(lane & 3);
                    auto at = [&](int rr) { return *reinterpret_cast<const uint4*>(bufp + rr * 64 + ((jj ^ (((uint32_t)rr >> 1) & 3u)) << 4)); };
                    const uint4 a = at(r00), b = at(r00 + 1), cq = at(r00 + 8), d = at(r00 + 9);
                    const __half2* ah = reinterpret_cast<const __half2*>(&a);
                    const __half2* bh = reinterpret_cast<const __half2*>(&b);
                    const __half2* ch2 = reinterpret_cast<const __half2*>(&cq);
                    const __half2* dh = reinterpret_cast<const __half2*>(&d);
                    uint4 o4;
                    __half2* oh = reinterpret_cast<__half2*>(&o4);
#pragma unroll
                    for (int i = 0; i < 4; ++i) oh[i] = __hmax2(__hmax2(ah[i], bh[i]), __hmax2(ch2[i], dh[i]));
                    *reinterpret_cast<uint4*>(p.pool_out + (((size_t)img * (p.H >> 1) + py) * Wh + pxx) * coutp + 32 * c + 8 * (int)jj) = o4;
                }
                __syncwarp();
                DTRAJ_TL(2, 4 + 3 * (c & 3));
            }
#ifdef DTRAJ_PROBES
            ++tl_tile;
#endif
            if (++acc == 2) { acc = 0; acc_ph ^= 1u; }
        }
        if (!(amax <= 65504.f)) atomicOr(errw, 2u);
    }
    ptx::tc_fence_before();
    __syncthreads();
    if constexpr (kPair) ptx::cluster_sync_all();
    if (warp == 0) {
        ptx::tc_fence_after();
        if constexpr (!kPair) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(tmem_cols) : "memory");
        else asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(tmem_cols) : "memory");
    }
}

struct Enc1hLaunch {
    Enc1Maps maps;
    Enc1hParams p;
    unsigned grid;
    size_t smem;
    int pair;
    double flops;                  // conv2's tensor-core flops (real channels)
};

// `w2` = conv2 weights packed by pack_conv in DTRAJ_PREC_F16 ([tap][chunk][coutp][64] halfs), `w2_rows` its 128-byte rows
inline int build_enc1h_launch(Enc1hLaunch* E, int C, int H, int coutp, int cout_real, int64_t R, const float* w2, int64_t w2_rows) {
    memset(E, 0, sizeof(*E));
    if (C < 1 || C > 4 || (H != 16 && H != 32 && H != 64) || coutp % 64 || coutp > 128) return fail(DTRAJ_EINVAL, "enc1(f16): unsupported geometry");
    Enc1hParams& p = E->p;
    p.C = C; p.H = H; p.W = H; p.coutp = coutp;
    p.n_chunks = coutp / 64;
    p.n_slices = (9 * C + 2 + 15) / 16;          // 9C taps + two bias slots
    p.tiles_x = H / 8;
    p.tiles_per_img = (H / 16) * p.tiles_x;
    p.lg_tx = 0;
    while ((1 << p.lg_tx) < p.tiles_x) ++p.lg_tx;
    p.lg_tpi = 0;
    while ((1 << p.lg_tpi) < p.tiles_per_img) ++p.lg_tpi;
    const int64_t nt = R * p.tiles_per_img;
    if (nt >= ((int64_t)1 << 30)) return fail(DTRAJ_EINVAL, "enc1(f16): batch too large");
    p.n_tiles = (int)nt;
    p.acc_cols = 32;
    while (p.acc_cols < coutp) p.acc_cols *= 2;
    p.n_d1 = 6 * p.acc_cols <= 512 ? 2 : 1;
    auto fixed_for = [&](int pair, int n_patch) {
        const size_t wr = (size_t)coutp / (pair ? 2 : 1);
        return (size_t)1024 + (size_t)9 * p.n_chunks * wr * 128 + kE1Epi * 2048 + (size_t)p.n_d1 * p.n_slices * kA1SliceBytes +
               (((size_t)p.n_slices * wr * 32 + 1023) & ~(size_t)1023) + (size_t)(6 + C) * coutp * 4 + 16 + 296 + 128 +
               (size_t)n_patch * (((size_t)C * kE1PatchH * kE1PatchW * 4 + 127) & ~(size_t)127);
    };
    // pairs halve the resident weights per CTA; without them the weights must still fit next to one halo buffer
    E->pair = p.n_tiles >= 2 * kNumSMs ? 1 : 0;
    if (!E->pair && fixed_for(0, 2) + kE1HaloBytes > 227 * 1024) E->pair = 1;     // n_tiles >= 2 always (two tiles per 16-row band)
    p.w_rows = coutp / (E->pair ? 2 : 1);
    auto halo_bufs = [&](int n_patch) {
        const size_t f = fixed_for(E->pair, n_patch);
        if (f + kE1HaloBytes > 227 * 1024) return 0;
        int nh = (int)((227 * 1024 - f) / kE1HaloBytes);
        if (nh > 2 * p.n_chunks) nh = 2 * p.n_chunks;
        return nh > 4 ? 4 : nh;                   // (one named barrier per buffer in flight: kE1SigBar .. kE1SigBar + 3)
    };
    p.n_patch = halo_bufs(4) == halo_bufs(2) ? 4 : 2;
    const size_t fixed = fixed_for(E->pair, p.n_patch);
    const int nh = halo_bufs(p.n_patch);
    if (nh < 1) return fail(DTRAJ_EINVAL, "enc1(f16): shared memory does not fit (coutp=%d C=%d)", coutp, C);
    p.n_hbuf = nh;
    E->smem = fixed + (size_t)nh * kE1HaloBytes;
    E->grid = (unsigned)(p.n_tiles < kNumSMs ? p.n_tiles : kNumSMs);
    if (E->pair) E->grid = (E->grid + 1) / 2 * 2;
    DTRAJ_TRY(make_w_map(&E->maps.w, w2, w2_rows, p.w_rows, 1));
    E->flops = 2.0 * (double)R * H * H * cout_real * (double)cout_real * 9.0;
    return 0;
}

typedef void (*Enc1hKernel)(const Enc1Maps, const Enc1hParams);
inline Enc1hKernel enc1h_kernel(int pair, int C) {
    static const Enc1hKernel tab[2][4] = {{k_enc1_f16<false, 1>, k_enc1_f16<false, 2>, k_enc1_f16<false, 3>, k_enc1_f16<false, 4>},
                                          {k_enc1_f16<true, 1>, k_enc1_f16<true, 2>, k_enc1_f16<true, 3>, k_enc1_f16<true, 4>}};
    return tab[pair ? 1 : 0][C - 1];
}

inline cudaError_t enc1h_set_smem_attr() {
    for (int pair = 0; pair < 2; ++pair)
        for (int C = 1; C <= 4; ++C) {
            cudaError_t e = cudaFuncSetAttribute(enc1h_kernel(pair, C), cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
            if (e != cudaSuccess) return e;
        }
    return cudaSuccess;
}

inline int launch_enc1h(const Enc1hLaunch& E, cudaStream_t st) {
    DTRAJ_CUDA(launch_ex(enc1h_kernel(E.pair, E.p.C), E.grid, kE1hThreads, E.smem, st, E.pair ? 2 : 1, true, E.maps, E.p));
    return 0;
}

}  // namespace dtraj
