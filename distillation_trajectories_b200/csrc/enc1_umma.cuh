// Fused enc1 block for sm_100a (single-pass TF32 mode): one kernel from the raw C-channel frame to the max-pooled
// enc1 output,
//     h  = relu(bn1(conv1_3x3(x))) + relu(time_mlp(temb))          (models.py:62-77, C = config.channels <= 4)
//     y  = relu(bn2(conv2_3x3(h))) + residual_conv_1x1(x)           (models.py:79-83)
//     p1 = MaxPool2d(2)(y)                                          (models.py:191; enc1's full-resolution output has
//                                                                    no other consumer, models.py:206-216)
// without h ever leaving the SM:
//   * an output tile is 16 image rows x 8 columns.  GENERATOR warps compute conv1 for the tile's 18 x 10 halo on the
//     CUDA cores (K = 9*C is far too small for the tensor cores) and write it, 32 channels at a time, straight into
//     shared memory in the 128-byte-swizzled K-major layout tcgen05.mma reads;
//   * each 3x3 tap of conv2 is then a VIEW of that halo tile -- a descriptor whose start is shifted by
//     ((dy+1)*10 + dx+1) pixel rows and whose stride between 8-row groups is one halo row (10 pixels = 1280 bytes).
//     The tensor core resolves the swizzle from the computed address (profiles/r01_umma_view_probe.txt), so nothing is
//     copied and the pixels are NOT re-read nine times through the SM's ingress port, which is what bounds the
//     TMA-im2col kernel on these full-resolution, narrow layers;
//   * only conv2's weights stream in by TMA (three taps per stage); CTA pairs (tcgen05.mma.cta_group::2) halve that
//     stream per SM;
//   * epilogue: bias, ReLU, the 1x1 residual recomputed from x, TF32 rounding, 2x2 max-pool, coalesced stores.
// Replaces k_conv_first + the enc1.conv2 launch of the generic kernel (and the h tensor round trip between them).
#pragma once
#include "conv_umma.cuh"

namespace dtraj {

// ncu on the first version (4 generator + 8 epilogue warps): the generators paced the kernel (311 cycles per
// pixel-iteration of one warp per scheduler, tensor pipe 43 % active) while the epilogue warps idled on the
// accumulator barrier -- hence 8 generator warps, two pixels per thread in flight, and 4 epilogue warps.
constexpr int kE1Gen = 8;                        // generator warps
constexpr int kE1Epi = 4;                        // epilogue warps (one per TMEM lane quarter); 8 + 8 warps measured slower (786 vs 690 us)
constexpr int kE1Threads = 64 + 32 * kE1Epi + 32 * kE1Gen;
constexpr int kE1HaloRows = 180;                 // 18 x 10 pixels
constexpr int kE1HaloBytes = 23552;              // 180 x 128 B rounded up to 1024

struct Enc1Params {
    int C, H, W, coutp;          // input channels, image size, padded enc1 width (conv2 is coutp -> coutp)
    int n_chunks;                // coutp / 32: K chunks of conv2
    int n_tiles, tiles_x, tiles_per_img;
    int stages;                  // weight stages
    int tps;                     // taps of one chunk per weight stage: 3, or 1 when three do not leave room for >= 3 stages
    int n_hbuf;                  // halo chunk buffers (one per 32-channel chunk)
    int acc_cols;                // TMEM columns per accumulator
    int w_rows;                  // weight rows this CTA stages per tap: coutp, or coutp / 2 in pair mode
    const float* x; int64_t x_stride; const int32_t* row_sample; const int32_t* row_variant;
    const float* w3; const float* b3;          // conv1, BN folded: [9*C][coutp] tap-major then cin; [coutp]
    const float* tbias; int tb_var_stride;     // relu(time_mlp(temb)) row of enc1 for this t: + variant * stride
    const float* bias2;                        // conv2 folded bias [coutp]
    const float* rw1; const float* rb1;        // residual 1x1: [C][coutp], [coutp]
    float* pool_out;                           // [R, H/2, W/2, coutp]
    int act_mode;
    unsigned int* err;           // the owning handle's device error word (null: the library-wide word)
};

struct Enc1Maps { CUtensorMap w; };            // conv2 packed weights, box {32, w_rows}

template <bool kPair>
__global__ void __launch_bounds__(kE1Threads, 1)
k_enc1_umma(const __grid_constant__ Enc1Maps maps, const Enc1Params p) {
    extern __shared__ __align__(1024) uint8_t e1_smem[];
    const uint32_t base = (ptx::smem_u32(e1_smem) + 1023u) & ~1023u;
    uint8_t* gbase = e1_smem + (base - ptx::smem_u32(e1_smem));
    const int coutp = p.coutp;
    const uint32_t wtap_bytes = (uint32_t)p.w_rows * 128u;                 // one tap's weight rows in this CTA
    const uint32_t stage_bytes = p.tps * wtap_bytes;
    // carve: [halo buffers][weight stages][epilogue ring 8 x 4 KB][x patches 2 x 4 ch x 240][conv1 weights][barriers]
    const uint32_t halo0 = base;
    const uint32_t wst0 = halo0 + (uint32_t)p.n_hbuf * kE1HaloBytes;
    const uint32_t ring0 = wst0 + (uint32_t)p.stages * stage_bytes;
    const uint32_t xp0 = ring0 + kE1Epi * 4096u;
    const uint32_t w3s0 = xp0 + 2u * 4u * 240u * 4u;
    const uint32_t bar0 = (w3s0 + (uint32_t)(9 * p.C + 2) * coutp * 4u + 15u) & ~15u;
    auto wfull = [&](int s) { return bar0 + 8u * s; };
    auto wempty = [&](int s) { return bar0 + 64u + 8u * s; };
    auto hfull = [&](int b) { return bar0 + 128u + 8u * b; };
    auto hempty = [&](int b) { return bar0 + 192u + 8u * b; };
    const uint32_t acc_full0 = bar0 + 256u, acc_empty0 = bar0 + 272u, tmem_slot = bar0 + 288u;
    volatile uint32_t* tmem_slot_ptr = reinterpret_cast<volatile uint32_t*>(gbase + (tmem_slot - base));
    float* xpatch = reinterpret_cast<float*>(gbase + (xp0 - base));       // [2][4][20][12]
    float* w3s = reinterpret_cast<float*>(gbase + (w3s0 - base));         // [9*C][coutp], then b3 [coutp], tb unused

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    unsigned int* const errw = p.err ? p.err : &g_umma_error;
    const int crank = kPair ? (int)ptx::cluster_ctarank() : 0;
    const uint16_t cmask = kPair ? 3 : 1;
    const int work0 = (int)blockIdx.x - crank;

    if (warp == 0) {
        if (ptx::elect_one()) {
            ptx::prefetch_tmap(&maps.w);
            for (int s = 0; s < p.stages; ++s) { ptx::mbar_init(wfull(s), 1); ptx::mbar_init(wempty(s), 1); }
            for (int b = 0; b < p.n_hbuf; ++b) { ptx::mbar_init(hfull(b), kE1Gen * (kPair ? 2 : 1)); ptx::mbar_init(hempty(b), 1); }
            for (int i = 0; i < 2; ++i) {
                ptx::mbar_init(acc_full0 + 8u * i, 1);
                ptx::mbar_init(acc_empty0 + 8u * i, kE1Epi * (kPair ? 2 : 1));
            }
            asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        }
        __syncwarp();
        if constexpr (!kPair) {
            asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "r"((uint32_t)(2 * p.acc_cols)) : "memory");
            asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
        } else {
            asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "r"((uint32_t)(2 * p.acc_cols)) : "memory");
            asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
        }
    }
    // conv1 weights + bias into shared memory (all threads)
    for (int i = threadIdx.x; i < 9 * p.C * coutp; i += blockDim.x) w3s[i] = p.w3[i];
    for (int i = threadIdx.x; i < coutp; i += blockDim.x) w3s[9 * p.C * coutp + i] = p.b3[i];
    ptx::tc_fence_before();
    __syncthreads();
    if constexpr (kPair) ptx::cluster_sync_all();
    ptx::tc_fence_after();
    const uint32_t tmem_base = *tmem_slot_ptr;

    auto tile_geom = [&](int tile, int& img, int& y0, int& x0) {
        img = tile / p.tiles_per_img;
        const int r = tile - img * p.tiles_per_img;
        y0 = (r / p.tiles_x) * 16;
        x0 = (r % p.tiles_x) * 8;
    };

    if (warp == 0) {
        // ------------------------------------------------------------ TMA producer: conv2 weights only
        if (ptx::elect_one()) {
            int s = 0;
            uint32_t ph = 0;
            bool ok = true;
            for (int wk = work0; wk < p.n_tiles && ok; wk += gridDim.x) {
                for (int c = 0; c < p.n_chunks && ok; ++c)
                    for (int t0 = 0; t0 < 9 && ok; t0 += p.tps) {
                        ok = ptx::mbar_wait(errw, wempty(s), ph ^ 1u);
                        uint32_t fb = wfull(s);
                        if constexpr (kPair) fb = ptx::map_to_cta(fb, 0);
                        if (!kPair || crank == 0) ptx::mbar_expect_tx(wfull(s), stage_bytes * (kPair ? 2u : 1u));
                        for (int j = 0; j < p.tps; ++j) {
                            const int row = ((t0 + j) * p.n_chunks + c) * coutp + crank * p.w_rows;
                            const uint32_t dst = wst0 + s * stage_bytes + j * wtap_bytes;
                            if constexpr (kPair) ptx::tma_load_2d_2sm(dst, &maps.w, fb, 0, row);
                            else ptx::tma_load_2d(dst, &maps.w, fb, 0, row);
                        }
                        if (++s == p.stages) { s = 0; ph ^= 1u; }
                    }
            }
        }
    } else if (warp == 1) {
        // ------------------------------------------------------------ MMA issuer (pair: leader CTA only)
        if (ptx::elect_one() && (!kPair || crank == 0)) {
            const uint32_t idesc = umma_idesc_tf32(coutp) + (kPair ? ((uint32_t)(128 >> 4) << 24) : 0u);
            // halo view: K-major SWIZZLE_128B, 8-row groups one halo row (10 pixels = 1280 B) apart
            const uint64_t hdesc0 = ((uint64_t)1 << 16) | ((uint64_t)(1280 >> 4) << 32) | ((uint64_t)1 << 46) | ((uint64_t)2 << 61);
            int s = 0, hb = 0, acc = 0;
            uint32_t ph = 0, hph = 0, acc_ph = 0;
            bool ok = true;
            for (int wk = work0; wk < p.n_tiles && ok; wk += gridDim.x) {
                ok = ptx::mbar_wait(errw, acc_empty0 + 8u * acc, acc_ph ^ 1u);
                ptx::tc_fence_after();
                const uint32_t d_tmem = tmem_base + (uint32_t)(acc * p.acc_cols);
                uint32_t accum = 0u;
                for (int c = 0; c < p.n_chunks && ok; ++c) {
                    ok = ptx::mbar_wait(errw, hfull(hb), hph);            // this chunk's halo tile is in shared memory (both CTAs)
                    ptx::tc_fence_after();
                    const uint32_t hbuf = halo0 + (uint32_t)hb * kE1HaloBytes;
                    int dy = 0, dx = 0;                              // tap (dy, dx) in 0..2
                    for (int t0 = 0; t0 < 9 && ok; t0 += p.tps) {
                        ok = ptx::mbar_wait(errw, wfull(s), ph);
                        ptx::tc_fence_after();
                        for (int j = 0; j < p.tps; ++j) {
                            const uint32_t a_addr = hbuf + (uint32_t)(dy * 10 + dx) * 128u;
                            const uint64_t ad = hdesc0 | (uint64_t)((a_addr >> 4) & 0x3fffu);
                            const uint64_t bd = umma_desc_sw128(wst0 + s * stage_bytes + j * wtap_bytes);
#pragma unroll
                            for (int k = 0; k < 4; ++k) {
                                if constexpr (!kPair) ptx::mma_tf32(d_tmem, ad + 2u * k, bd + 2u * k, idesc, accum);
                                else ptx::mma_tf32_2sm(d_tmem, ad + 2u * k, bd + 2u * k, idesc, accum);
                                accum = 1u;
                            }
                            if (++dx == 3) { dx = 0; ++dy; }
                        }
                        if constexpr (kPair) ptx::tc_commit_2sm(wempty(s), cmask); else ptx::tc_commit(wempty(s));
                        if (++s == p.stages) { s = 0; ph ^= 1u; }
                    }
                    if constexpr (kPair) ptx::tc_commit_2sm(hempty(hb), cmask); else ptx::tc_commit(hempty(hb));
                    if (++hb == p.n_hbuf) { hb = 0; hph ^= 1u; }
                }
                if constexpr (kPair) ptx::tc_commit_2sm(acc_full0 + 8u * acc, cmask); else ptx::tc_commit(acc_full0 + 8u * acc);
                if (++acc == 2) { acc = 0; acc_ph ^= 1u; }
            }
        }
    } else if (warp >= 2 + kE1Epi) {
        // ------------------------------------------------------------ generators: conv1 + BN + ReLU + time bias -> halo tiles
        const int gt = threadIdx.x - 32 * (2 + kE1Epi);            // 0..255
        const int g = gt & 7, pl = gt >> 3;                         // float4 group inside the 32-channel chunk, pixel lane (0..31)
        const int C = p.C;
        int hb = 0;
        uint32_t hph = 0;
        int it = 0;
        for (int wk = work0; wk < p.n_tiles; wk += gridDim.x, ++it) {
            const int tile = wk + crank;
            int img, y0, x0;
            tile_geom(tile, img, y0, x0);
            const bool real = tile < p.n_tiles;
            // x patch (zero outside the image): rows y0-2 .. y0+17, cols x0-2 .. x0+9, double-buffered across tiles
            float* xp = xpatch + (it & 1) * 4 * 240;
            const float* xs = p.x + (size_t)(real ? (p.row_sample ? p.row_sample[img] : img) : 0) * p.x_stride;
            for (int i = gt; i < C * 240; i += 32 * kE1Gen) {
                const int c = i / 240, r = i - c * 240, yy = y0 - 2 + r / 12, xx = x0 - 2 + r % 12;
                xp[i] = (real && yy >= 0 && yy < p.H && xx >= 0 && xx < p.W) ? __ldg(xs + ((size_t)c * p.H + yy) * p.W + xx) : 0.f;
            }
            asm volatile("bar.sync 9, 256;" ::: "memory");
            const int var = (real && p.row_variant) ? p.row_variant[img] : 0;
            const float* tb = p.tbias + (size_t)var * p.tb_var_stride;
            for (int c = 0; c < p.n_chunks; ++c) {
                const int ch = 32 * c + 4 * g;
                const float4 b3 = *reinterpret_cast<const float4*>(w3s + (size_t)9 * C * coutp + ch);
                const float4 t4 = __ldg(reinterpret_cast<const float4*>(tb + ch));
                float4 w[9];                                        // C == 1: the nine taps stay in registers
                if (C == 1) {
#pragma unroll
                    for (int t9 = 0; t9 < 9; ++t9) w[t9] = *reinterpret_cast<const float4*>(w3s + (size_t)t9 * coutp + ch);
                }
                ptx::mbar_wait(errw, hempty(hb), hph ^ 1u);               // the MMAs that read this buffer have retired
                uint8_t* hbuf = gbase + (halo0 - base) + (size_t)hb * kE1HaloBytes;
                // 32 pixel lanes x 6 rounds cover the 180 halo pixels; two pixels (px, px + 96) per trip keep eight
                // independent FMA chains in flight
                auto conv1_at = [&](int px) -> float4 {
                    const int ry = px / 10, rx = px - ry * 10;
                    const int yy = y0 - 1 + ry, xx = x0 - 1 + rx;
                    if (!(yy >= 0 && yy < p.H && xx >= 0 && xx < p.W)) return make_float4(0.f, 0.f, 0.f, 0.f);   // conv2's zero padding
                    float4 acc = b3;
                    if (C == 1) {
#pragma unroll
                        for (int ky = 0; ky < 3; ++ky)
#pragma unroll
                            for (int kx = 0; kx < 3; ++kx) {
                                const float v = xp[(ry + ky) * 12 + rx + kx];
                                const float4 ww = w[ky * 3 + kx];
                                acc.x = fmaf(v, ww.x, acc.x); acc.y = fmaf(v, ww.y, acc.y);
                                acc.z = fmaf(v, ww.z, acc.z); acc.w = fmaf(v, ww.w, acc.w);
                            }
                    } else {
                        for (int ci = 0; ci < C; ++ci)
#pragma unroll
                            for (int t9 = 0; t9 < 9; ++t9) {
                                const float v = xp[ci * 240 + (ry + t9 / 3) * 12 + rx + t9 % 3];
                                const float4 ww = *reinterpret_cast<const float4*>(w3s + (size_t)(t9 * C + ci) * coutp + ch);
                                acc.x = fmaf(v, ww.x, acc.x); acc.y = fmaf(v, ww.y, acc.y);
                                acc.z = fmaf(v, ww.z, acc.z); acc.w = fmaf(v, ww.w, acc.w);
                            }
                    }
                    float4 o = make_float4(fmaxf(acc.x, 0.f) + t4.x, fmaxf(acc.y, 0.f) + t4.y,
                                           fmaxf(acc.z, 0.f) + t4.z, fmaxf(acc.w, 0.f) + t4.w);
                    return act_round4(o, p.act_mode);
                };
                for (int px = pl; px < 96; px += 32) {
                    const int px1 = px + 96;
                    float4 o0 = conv1_at(px), o1 = make_float4(0.f, 0.f, 0.f, 0.f);
                    if (px1 < kE1HaloRows) o1 = conv1_at(px1);
                    *reinterpret_cast<float4*>(hbuf + px * 128 + (((uint32_t)g ^ (uint32_t)(px & 7)) << 4)) = o0;
                    if (px1 < kE1HaloRows) *reinterpret_cast<float4*>(hbuf + px1 * 128 + (((uint32_t)g ^ (uint32_t)(px1 & 7)) << 4)) = o1;
                }
                ptx::fence_proxy_async();                           // generic-proxy writes -> visible to the tensor core
                __syncwarp();
                if (lane == 0) {
                    if constexpr (!kPair) ptx::mbar_arrive(hfull(hb));
                    else ptx::mbar_arrive_cluster_cta(ptx::map_to_cta(hfull(hb), 0));
                }
                if (++hb == p.n_hbuf) { hb = 0; hph ^= 1u; }
            }
        }
    } else {
        // ------------------------------------------------------------ epilogue (warps 2..5): thread = output pixel
        const int q = warp & 3, ew = warp - 2;
        constexpr int h = 0;
        const int nchunk = coutp >> 5;
        uint8_t* bufp = gbase + (ring0 - base) + (size_t)ew * 4096;
        const uint32_t swz = (uint32_t)(lane & 7);
        const int Wh = p.W >> 1;
        int acc = 0;
        uint32_t acc_ph = 0;
        auto arrive_acc_empty = [&]() {
            if constexpr (!kPair) ptx::mbar_arrive(acc_empty0 + 8u * acc);
            else ptx::mbar_arrive_cluster_relaxed(ptx::map_to_cta(acc_empty0 + 8u * acc, 0));
        };
        for (int wk = work0; wk < p.n_tiles; wk += gridDim.x) {
            const int tile = wk + crank;
            int img, y0, x0;
            tile_geom(tile, img, y0, x0);
            const bool real = tile < p.n_tiles;
            const int r = 32 * q + lane, yl = r >> 3, xl = r & 7;          // row of the 16 x 8 tile
            float xv[4] = {0.f, 0.f, 0.f, 0.f};
            if (real) {
                const float* xs = p.x + (size_t)(p.row_sample ? p.row_sample[img] : img) * p.x_stride + (size_t)(y0 + yl) * p.W + x0 + xl;
#pragma unroll
                for (int ci = 0; ci < 4; ++ci) if (ci < p.C) xv[ci] = __ldg(xs + (size_t)ci * p.H * p.W);
            }
            ptx::mbar_wait(errw, acc_full0 + 8u * acc, acc_ph);
            ptx::tc_fence_after();
            const uint32_t t_acc = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(acc * p.acc_cols);
            const int c_last = nchunk - 1;
            for (int c = h; c < nchunk; c += kE1Epi / 4) {
                uint32_t raw[32];
                ptx::tmem_ld32(t_acc + (uint32_t)(32 * c), raw);
                ptx::tmem_ld_wait();
                if (c == c_last) { ptx::tc_fence_before(); __syncwarp(); if (lane == 0) arrive_acc_empty(); }
                uint8_t* rowp = bufp + lane * 128;
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    const int col = 32 * c + 4 * j;
                    const float4 b4 = __ldg(reinterpret_cast<const float4*>(p.bias2 + col));
                    float4 v = make_float4(fmaxf(__uint_as_float(raw[4 * j]) + b4.x, 0.f), fmaxf(__uint_as_float(raw[4 * j + 1]) + b4.y, 0.f),
                                           fmaxf(__uint_as_float(raw[4 * j + 2]) + b4.z, 0.f), fmaxf(__uint_as_float(raw[4 * j + 3]) + b4.w, 0.f));
                    float4 r4 = __ldg(reinterpret_cast<const float4*>(p.rb1 + col));
#pragma unroll
                    for (int ci = 0; ci < 4; ++ci) {
                        if (ci >= p.C) break;
                        const float4 w4 = __ldg(reinterpret_cast<const float4*>(p.rw1 + (size_t)ci * coutp + col));
                        r4.x = fmaf(xv[ci], w4.x, r4.x); r4.y = fmaf(xv[ci], w4.y, r4.y);
                        r4.z = fmaf(xv[ci], w4.z, r4.z); r4.w = fmaf(xv[ci], w4.w, r4.w);
                    }
                    v.x += r4.x; v.y += r4.y; v.z += r4.z; v.w += r4.w;
                    *reinterpret_cast<float4*>(rowp + (((uint32_t)j ^ swz) << 4)) = act_round4(v, p.act_mode);
                }
                __syncwarp();
                if (real) {
                    // the warp's 4 x 8 pixel patch holds 2 x 4 complete 2x2 windows: lane -> (window, two float4 columns)
                    const int pr = lane >> 2, wy = pr >> 2, wx = pr & 3;
                    const int r00 = (2 * wy) * 8 + 2 * wx;
                    const int py = (y0 + 4 * q + 2 * wy) >> 1, pxx = (x0 + 2 * wx) >> 1;
                    float* dst = p.pool_out + (((size_t)img * (p.H >> 1) + py) * Wh + pxx) * coutp + 32 * c;
#pragma unroll
                    for (int jj = (lane & 3) * 2; jj < (lane & 3) * 2 + 2; ++jj) {
                        auto at = [&](int rr) { return *reinterpret_cast<const float4*>(bufp + rr * 128 + (((uint32_t)jj ^ (uint32_t)(rr & 7)) << 4)); };
                        const float4 a = at(r00), b = at(r00 + 1), cq = at(r00 + 8), d = at(r00 + 9);
                        *reinterpret_cast<float4*>(dst + 4 * jj) =
                            make_float4(fmaxf(fmaxf(a.x, b.x), fmaxf(cq.x, d.x)), fmaxf(fmaxf(a.y, b.y), fmaxf(cq.y, d.y)),
                                        fmaxf(fmaxf(a.z, b.z), fmaxf(cq.z, d.z)), fmaxf(fmaxf(a.w, b.w), fmaxf(cq.w, d.w)));
                    }
                }
                __syncwarp();
            }
            if (++acc == 2) { acc = 0; acc_ph ^= 1u; }
        }
    }
    ptx::tc_fence_before();
    __syncthreads();
    if constexpr (kPair) ptx::cluster_sync_all();
    if (warp == 0) {
        ptx::tc_fence_after();
        if constexpr (!kPair) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)(2 * p.acc_cols)) : "memory");
        else asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)(2 * p.acc_cols)) : "memory");
    }
}

struct Enc1Launch {
    Enc1Maps maps;
    Enc1Params p;
    unsigned grid;
    size_t smem;
    int pair;
    double flops;                  // conv2's tensor-core flops (real channels)
};

// `w2` = conv2 weights packed by pack_conv ([tap][chunk][coutp][32], tf32-rounded), `w2_rows` its rows
inline int build_enc1_launch(Enc1Launch* E, int C, int H, int coutp, int cout_real, int64_t R, const float* w2, int64_t w2_rows) {
    memset(E, 0, sizeof(*E));
    if (C < 1 || C > 4 || (H != 16 && H != 32 && H != 64) || coutp % 32 || coutp > 256) return fail(DTRAJ_EINVAL, "enc1: unsupported geometry");
    Enc1Params& p = E->p;
    p.C = C; p.H = H; p.W = H; p.coutp = coutp;
    p.n_chunks = coutp / 32;
    p.tiles_x = H / 8;
    p.tiles_per_img = (H / 16) * p.tiles_x;
    const int64_t nt = R * p.tiles_per_img;
    if (nt >= ((int64_t)1 << 30)) return fail(DTRAJ_EINVAL, "enc1: batch too large");
    p.n_tiles = (int)nt;
    E->pair = (p.n_tiles >= 2 * kNumSMs && coutp >= 64) ? 1 : 0;
    p.w_rows = coutp / (E->pair ? 2 : 1);
    p.n_hbuf = p.n_chunks;       // chunk c of the next tile reuses chunk c's buffer as soon as its nine taps have retired
    if (p.n_hbuf > 8) return fail(DTRAJ_EINVAL, "enc1: too many halo buffers");
    p.acc_cols = 32;
    while (p.acc_cols < coutp) p.acc_cols *= 2;
    const size_t fixed = 1024 + (size_t)p.n_hbuf * kE1HaloBytes + kE1Epi * 4096 + 2 * 4 * 240 * 4 + (size_t)(9 * C + 2) * coutp * 4 + 16 + 512;
    p.tps = 3;
    if ((227 * 1024 - fixed) / ((size_t)3 * p.w_rows * 128) < 3) p.tps = 1;
    const size_t stage = (size_t)p.tps * p.w_rows * 128;
    int stages = (int)((227 * 1024 - fixed) / stage);
    if (stages < 2) return fail(DTRAJ_EINVAL, "enc1: weight ring does not fit (coutp=%d pair=%d w_rows=%d tps=%d fixed=%zu stage=%zu)", coutp, E->pair, p.w_rows, p.tps, fixed, stage);
    if (stages > 8) stages = 8;
    p.stages = stages;
    E->smem = fixed + stages * stage;
    E->grid = (unsigned)(p.n_tiles < kNumSMs ? p.n_tiles : kNumSMs);
    if (E->pair) E->grid = (E->grid + 1) / 2 * 2;
    DTRAJ_TRY(make_w_map(&E->maps.w, w2, w2_rows, p.w_rows));
    E->flops = 2.0 * (double)R * H * H * cout_real * (double)cout_real * 9.0;
    return 0;
}

inline cudaError_t enc1_set_smem_attr() {
    cudaError_t e = cudaFuncSetAttribute(k_enc1_umma<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
    if (e != cudaSuccess) return e;
    return cudaFuncSetAttribute(k_enc1_umma<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
}

inline int launch_enc1(const Enc1Launch& E, cudaStream_t st) {
    if (!E.pair) {
        k_enc1_umma<false><<<E.grid, kE1Threads, E.smem, st>>>(E.maps, E.p);
        DTRAJ_LAUNCH_CHECK();
        return 0;
    }
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = dim3(E.grid);
    cfg.blockDim = dim3(kE1Threads);
    cfg.dynamicSmemBytes = E.smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = 2;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    DTRAJ_CUDA(cudaLaunchKernelEx(&cfg, k_enc1_umma<true>, E.maps, E.p));
    return 0;
}

}  // namespace dtraj
