// Streaming trajectory-metric reductions (HBM-bound): every element of the teacher and the
// student trajectory tensors [N, L, D] is read exactly once with 128-bit loads.
//   reference per-frame reductions: analysis/metrics/trajectory_metrics.py:55-215
//                                   analysis/metrics/time_dependent.py:57,78
//   Wasserstein per frame:          analysis/metrics/trajectory_metrics.py:296-312
#pragma once
#include <cstdlib>
#include <type_traits>
#include "common.cuh"

namespace dtraj {

constexpr int kMetricQ = 6;   // floats per (pair, frame) in the output

// One group of G threads owns one trajectory pair and walks its L frames in order, keeping
// the previous frame (and frame 0) in registers: no element is loaded twice.  Per-warp
// partial sums of all frames are parked in shared memory, so there is a single barrier per
// pair instead of one per frame.
//   out[n][i][0] = sum (T_i - S_i)^2
//   out[n][i][1] = sum (T_{i+1} - T_i)^2, [2] same for S, [3] = sum dT_i * dS_i     (i < L-1)
//   out[n][0][4] = sum (T_{L-1} - T_0)^2, out[n][0][5] same for S
template <int K>   // float4 per thread per frame
__global__ void __launch_bounds__(256) k_metrics_pairs(const float* __restrict__ teacher,
                                                       const float* __restrict__ student,
                                                       int64_t N, int L, int D4, int G, float* __restrict__ out) {
    extern __shared__ float part[];          // [pairs_per_block][L][warps_per_group][4]
    const int ppb = 256 / G, wpg = G / 32 > 0 ? G / 32 : 1;
    const int g = threadIdx.x / G, tg = threadIdx.x % G;
    const int warp_in_group = tg >> 5, lane = threadIdx.x & 31;
    const int64_t n = (int64_t)blockIdx.x * ppb + g;
    const bool active = n < N;
    float* mypart = part + (size_t)g * L * wpg * 4;
    float4 firstT[K], firstS[K], prevT[K], prevS[K], nxtT[K], nxtS[K];
    const float4 zero4 = make_float4(0.f, 0.f, 0.f, 0.f);
    const float4* Tb = reinterpret_cast<const float4*>(teacher) + (active ? n : 0) * (int64_t)L * D4;
    const float4* Sb = reinterpret_cast<const float4*>(student) + (active ? n : 0) * (int64_t)L * D4;
    auto load_frame = [&](int i, float4* t, float4* s) {
#pragma unroll
        for (int k = 0; k < K; ++k) {
            const int e = tg + k * G;
            if (active && e < D4) {
                t[k] = ld_stream4(reinterpret_cast<const float*>(Tb + (int64_t)i * D4 + e));
                s[k] = ld_stream4(reinterpret_cast<const float*>(Sb + (int64_t)i * D4 + e));
            } else { t[k] = zero4; s[k] = zero4; }
        }
    };
    auto sq4 = [](float4 a) { return a.x * a.x + a.y * a.y + a.z * a.z + a.w * a.w; };
    auto sub4 = [](float4 a, float4 b) { return make_float4(a.x - b.x, a.y - b.y, a.z - b.z, a.w - b.w); };
    auto dot4 = [](float4 a, float4 b) { return a.x * b.x + a.y * b.y + a.z * b.z + a.w * b.w; };

    load_frame(0, nxtT, nxtS);
    float endT = 0.f, endS = 0.f;
    for (int i = 0; i < L; ++i) {
        float4 curT[K], curS[K];
#pragma unroll
        for (int k = 0; k < K; ++k) { curT[k] = nxtT[k]; curS[k] = nxtS[k]; }
        if (i + 1 < L) load_frame(i + 1, nxtT, nxtS);
        float d2 = 0.f, vt2 = 0.f, vs2 = 0.f, dot = 0.f;
#pragma unroll
        for (int k = 0; k < K; ++k) {
            d2 += sq4(sub4(curT[k], curS[k]));
            if (i > 0) {
                float4 dt = sub4(curT[k], prevT[k]), ds = sub4(curS[k], prevS[k]);
                vt2 += sq4(dt); vs2 += sq4(ds); dot += dot4(dt, ds);
            } else { firstT[k] = curT[k]; firstS[k] = curS[k]; }
            prevT[k] = curT[k]; prevS[k] = curS[k];
        }
        if (i == L - 1) {
#pragma unroll
            for (int k = 0; k < K; ++k) { endT += sq4(sub4(curT[k], firstT[k])); endS += sq4(sub4(curS[k], firstS[k])); }
        }
        d2 = warp_sum(d2); vt2 = warp_sum(vt2); vs2 = warp_sum(vs2); dot = warp_sum(dot);
        if (lane == 0) {
            // velocity-type sums of step (i-1 -> i) belong to frame index i-1
            mypart[(i * wpg + warp_in_group) * 4 + 0] = d2;
            if (i > 0) {
                float* q = mypart + ((i - 1) * wpg + warp_in_group) * 4;
                q[1] = vt2; q[2] = vs2; q[3] = dot;
            }
            if (i == L - 1) { float* q = mypart + (i * wpg + warp_in_group) * 4; q[1] = 0.f; q[2] = 0.f; q[3] = 0.f; }
        }
    }
    endT = warp_sum(endT); endS = warp_sum(endS);
    __shared__ float endpart[8][2];
    if (lane == 0) { endpart[threadIdx.x >> 5][0] = endT; endpart[threadIdx.x >> 5][1] = endS; }
    __syncthreads();
    if (!active) return;
    float* o = out + n * (int64_t)L * kMetricQ;
    for (int j = tg; j < L * 4; j += G) {
        const int i = j >> 2, q = j & 3;
        float s = 0.f;
        for (int w = 0; w < wpg; ++w) s += mypart[(i * wpg + w) * 4 + q];
        o[i * kMetricQ + q] = s;
    }
    for (int j = tg; j < L * 2; j += G) {
        const int i = j >> 1, q = j & 1;
        float s = 0.f;
        if (i == 0) for (int w = 0; w < wpg; ++w) s += endpart[g * wpg + w][q];
        o[i * kMetricQ + 4 + q] = s;
    }
}

inline int launch_metrics_pairs(const float* T, const float* S, int64_t N, int L, int D, float* out, cudaStream_t st) {
    if (D % 4 != 0 || D <= 0 || L < 1) return fail(DTRAJ_EINVAL, "metrics: D=%d must be a positive multiple of 4, L=%d >= 1", D, L);
    const int D4 = D / 4;
    int G = 32;
    while (G < 256 && (D4 + G - 1) / G > 3) G *= 2;
    const int K = (D4 + G - 1) / G;
    if (K > 4) return fail(DTRAJ_EINVAL, "metrics: D=%d too large (max 4096)", D);
    const int ppb = 256 / G, wpg = G / 32;
    const size_t smem = (size_t)ppb * L * wpg * 4 * sizeof(float);
    if (smem > 200 * 1024) return fail(DTRAJ_EINVAL, "metrics: L=%d too large", L);
    const unsigned grid = (unsigned)((N + ppb - 1) / ppb);
    if (N == 0) return 0;
#define DTRAJ_MP(KK)                                                                              \
    {                                                                                             \
        if (smem > 48 * 1024)                                                                     \
            DTRAJ_CUDA(cudaFuncSetAttribute(k_metrics_pairs<KK>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
        k_metrics_pairs<KK><<<grid, 256, smem, st>>>(T, S, N, L, D4, G, out);                     \
    }
    switch (K) {
        case 1: DTRAJ_MP(1); break;
        case 2: DTRAJ_MP(2); break;
        case 3: DTRAJ_MP(3); break;
        default: DTRAJ_MP(4); break;
    }
#undef DTRAJ_MP
    DTRAJ_LAUNCH_CHECK();
    return 0;
}

// Teacher and student of different lengths (analysis/metrics/trajectory_metrics.py:239-279: a student sampled with
// fewer steps than its teacher).  n = min(LT, LS); "long" is the teacher when LT >= LS, "short" the other one.
// Same walk as k_metrics_pairs over max(LT, LS) frames: frame i of each trajectory is loaded once while i < its length and
// the previous frame stays in registers.  The path-alignment term lerp(long[p_j], long[p_j + 1], f_j) is formed when the
// walk holds long frames p_j and p_j + 1; short frame j is read a second time for it.  Three single frames are read once
// more: T_0 and S_0 at each trajectory's last frame (holding them in registers for the whole walk would cost a second block
// per SM at D = 3072), and the short trajectory's last frame for the endpoint term.  Bytes requested per pair:
// 4 * D * (L_long + 2 * L_short + 3), against the algorithmic 4 * D * (LT + LS).
//   out[n][i][0] = sum (T_i - S_i)^2                               (i < n)
//   out[n][i][1] = sum (T_{i+1} - T_i)^2 (i < LT-1),  [2] = sum (S_{i+1} - S_i)^2 (i < LS-1)
//   out[n][i][3] = sum dT_i * dS_i                                 (i < n-1)
//   out[n][0][4] = sum (T_{LT-1} - T_0)^2,  [0][5] = sum (S_{LS-1} - S_0)^2,  [0][6] = sum (T_{LT-1} - S_{LS-1})^2
//   out[n][j][7] = sum ((1 - f_j) long_{p_j} + f_j long_{p_j+1} - short_j)^2   (j < n)
// every other entry of [N, max(LT, LS), 8] is 0.  Short frame j is taken once the walk has passed long frame p_j + 1
// (p non-decreasing, 0 <= p_j <= L_long - 2), and at the last long frame at the latest.
constexpr int kRaggedQ = 8;

// Frame source of k_metrics_pairs_ragged.  DirectFrames reads [N, LT, D] and [N, LS, D] in place through the pointers
// the kernel forms itself; ResampledFrames (below) reads a student of another frame size through the bilinear resize.
struct DirectFrames {
    static constexpr bool kInPlace = true;
};

template <int K, class Frames>
__global__ void __launch_bounds__(256) k_metrics_pairs_ragged(const float* __restrict__ teacher, const float* __restrict__ student,
                                                              int64_t N, int LT, int LS, int D4, int G,
                                                              const int32_t* __restrict__ rs_pos, const float* __restrict__ rs_frac,
                                                              float* __restrict__ out, Frames frames) {
    extern __shared__ float part[];          // [pairs_per_block][Lmax][warps_per_group][5]
    const int ppb = 256 / G, wpg = G / 32 > 0 ? G / 32 : 1;
    const int g = threadIdx.x / G, tg = threadIdx.x % G;
    const int warp_in_group = tg >> 5, lane = threadIdx.x & 31;
    const int64_t n = (int64_t)blockIdx.x * ppb + g;
    const bool active = n < N;
    const int Lmax = LT > LS ? LT : LS, Ln = LT < LS ? LT : LS;
    const bool t_long = LT >= LS;
    float* mypart = part + (size_t)g * Lmax * wpg * 5;
    float4 prevT[K], prevS[K], nxtT[K], nxtS[K], sh[K];
    const float4 zero4 = make_float4(0.f, 0.f, 0.f, 0.f);
    const float4* Tb = reinterpret_cast<const float4*>(teacher) + (active ? n : 0) * (int64_t)LT * D4;
    const float4* Sb = reinterpret_cast<const float4*>(student) + (active ? n : 0) * (int64_t)LS * D4;
    const float4* Shb = t_long ? Sb : Tb;
    // stu: base is the student's trajectory
    auto load = [&](const float4* base, bool stu, int i, bool ok, float4* v) {
#pragma unroll
        for (int k = 0; k < K; ++k) {
            const int e = tg + k * G;
            if constexpr (Frames::kInPlace)
                v[k] = (ok && active && e < D4) ? ld_stream4(reinterpret_cast<const float*>(base + (int64_t)i * D4 + e)) : zero4;
            else
                v[k] = (ok && active && e < D4) ? frames.load(teacher, student, stu, n, LT, LS, i, e, D4) : zero4;
        }
    };
    auto sq4 = [](float4 a) { return a.x * a.x + a.y * a.y + a.z * a.z + a.w * a.w; };
    auto sub4 = [](float4 a, float4 b) { return make_float4(a.x - b.x, a.y - b.y, a.z - b.z, a.w - b.w); };
    auto dot4 = [](float4 a, float4 b) { return a.x * b.x + a.y * b.y + a.z * b.z + a.w * b.w; };
    auto lerp4 = [](float4 a, float4 b, float f) {   // exact at f = 0 and f = 1
        const float e = 1.f - f;
        return make_float4(e * a.x + f * b.x, e * a.y + f * b.y, e * a.z + f * b.z, e * a.w + f * b.w);
    };

    load(Tb, false, 0, true, nxtT);
    load(Sb, true, 0, true, nxtS);
    float endT = 0.f, endS = 0.f, endTS = 0.f;
    int j = 0;                               // next short frame of the path-alignment term
    for (int i = 0; i < Lmax; ++i) {
        float4 curT[K], curS[K];
#pragma unroll
        for (int k = 0; k < K; ++k) { curT[k] = nxtT[k]; curS[k] = nxtS[k]; }
        load(Tb, false, i + 1, i + 1 < LT, nxtT);
        load(Sb, true, i + 1, i + 1 < LS, nxtS);
        const bool inT = i < LT, inS = i < LS;
        float d2 = 0.f, vt2 = 0.f, vs2 = 0.f, dot = 0.f;
#pragma unroll
        for (int k = 0; k < K; ++k) {
            d2 += sq4(sub4(curT[k], curS[k]));
            if (i > 0) {
                const float4 dt = sub4(curT[k], prevT[k]), ds = sub4(curS[k], prevS[k]);
                vt2 += sq4(dt); vs2 += sq4(ds); dot += dot4(dt, ds);
            }
        }
        if (i == LT - 1) {                   // frame 0 is re-read rather than held in registers for the whole walk
            load(Tb, false, 0, true, sh);
#pragma unroll
            for (int k = 0; k < K; ++k) endT += sq4(sub4(curT[k], sh[k]));
        }
        if (i == LS - 1) {
            load(Sb, true, 0, true, sh);
#pragma unroll
            for (int k = 0; k < K; ++k) endS += sq4(sub4(curS[k], sh[k]));
        }
        if (i == Lmax - 1) {                 // the long trajectory's last frame against the short one's (re-read)
            load(Shb, t_long, Ln - 1, true, sh);
#pragma unroll
            for (int k = 0; k < K; ++k) endTS += sq4(sub4(t_long ? curT[k] : curS[k], sh[k]));
        }
        // path alignment: every short frame j whose interval [p_j, p_j + 1] ends at this long frame
        while (i > 0 && j < Ln && (__ldg(rs_pos + j) <= i - 1 || i == Lmax - 1)) {
            const float f = __ldg(rs_frac + j);
            load(Shb, t_long, j, true, sh);
            float r2 = 0.f;
#pragma unroll
            for (int k = 0; k < K; ++k)
                r2 += t_long ? sq4(sub4(lerp4(prevT[k], curT[k], f), sh[k])) : sq4(sub4(lerp4(prevS[k], curS[k], f), sh[k]));
            r2 = warp_sum(r2);
            if (lane == 0) mypart[(j * wpg + warp_in_group) * 5 + 4] = r2;
            ++j;
        }
#pragma unroll
        for (int k = 0; k < K; ++k) {
            if (inT) prevT[k] = curT[k];
            if (inS) prevS[k] = curS[k];
        }
        d2 = warp_sum(d2); vt2 = warp_sum(vt2); vs2 = warp_sum(vs2); dot = warp_sum(dot);
        if (lane == 0) {
            mypart[(i * wpg + warp_in_group) * 5 + 0] = d2;
            if (i > 0) {                     // step (i-1 -> i) belongs to frame index i-1
                float* q = mypart + ((i - 1) * wpg + warp_in_group) * 5;
                q[1] = vt2; q[2] = vs2; q[3] = dot;
            }
        }
    }
    endT = warp_sum(endT); endS = warp_sum(endS); endTS = warp_sum(endTS);
    __shared__ float endpart[8][3];
    if (lane == 0) { endpart[threadIdx.x >> 5][0] = endT; endpart[threadIdx.x >> 5][1] = endS; endpart[threadIdx.x >> 5][2] = endTS; }
    __syncthreads();
    if (!active) return;
    float* o = out + n * (int64_t)Lmax * kRaggedQ;
    for (int e = tg; e < Lmax * kRaggedQ; e += G) {
        const int i = e / kRaggedQ, q = e % kRaggedQ;
        float s = 0.f;
        if (q >= 4 && q <= 6) {
            if (i == 0) for (int w = 0; w < wpg; ++w) s += endpart[g * wpg + w][q - 4];
        } else {
            const int c = q == 7 ? 4 : q;
            const bool valid = q == 0 ? i < Ln : q == 1 ? i < LT - 1 : q == 2 ? i < LS - 1 : q == 3 ? i < Ln - 1 : i < Ln;
            if (valid) for (int w = 0; w < wpg; ++w) s += mypart[(i * wpg + w) * 5 + c];
        }
        o[e] = s;
    }
}

// max(LT, LS) >= 2 and D4 <= 1024 float4 per group are checked by the callers.
template <class Frames>
inline int launch_ragged_walk(const float* T, const float* S, int64_t groups, int LT, int LS, int D4, const int32_t* rs_pos,
                              const float* rs_frac, float* out, Frames frames, const char* who, cudaStream_t st) {
    int G = 32;
    while (G < 256 && (D4 + G - 1) / G > 3) G *= 2;
    const int K = (D4 + G - 1) / G;
    const int ppb = 256 / G, wpg = G / 32, Lmax = LT > LS ? LT : LS;
    const size_t smem = (size_t)ppb * Lmax * wpg * 5 * sizeof(float);
    if (smem > 200 * 1024) return fail(DTRAJ_EINVAL, "%s: max(LT, LS)=%d too large", who, Lmax);
    if (groups == 0) return 0;
    const unsigned grid = (unsigned)((groups + ppb - 1) / ppb);
#define DTRAJ_MPR(KK)                                                                             \
    {                                                                                             \
        if (smem > 48 * 1024)                                                                     \
            DTRAJ_CUDA(cudaFuncSetAttribute(k_metrics_pairs_ragged<KK, Frames>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
        k_metrics_pairs_ragged<KK, Frames><<<grid, 256, smem, st>>>(T, S, groups, LT, LS, D4, G, rs_pos, rs_frac, out, frames); \
    }
    switch (K) {
        case 1: DTRAJ_MPR(1); break;
        case 2: DTRAJ_MPR(2); break;
        case 3: DTRAJ_MPR(3); break;
        default: DTRAJ_MPR(4); break;
    }
#undef DTRAJ_MPR
    DTRAJ_LAUNCH_CHECK();
    return 0;
}

inline int launch_metrics_pairs_ragged(const float* T, const float* S, int64_t N, int LT, int LS, int D,
                                       const int32_t* rs_pos, const float* rs_frac, float* out, cudaStream_t st) {
    if (D % 4 != 0 || D <= 0 || LT < 1 || LS < 1 || (LT < 2 && LS < 2))
        return fail(DTRAJ_EINVAL, "metrics_ragged: D=%d must be a positive multiple of 4, LT=%d, LS=%d >= 1 and one of them >= 2", D, LT, LS);
    if (D > 4096) return fail(DTRAJ_EINVAL, "metrics_ragged: D=%d too large (max 4096)", D);
    return launch_ragged_walk(T, S, N, LT, LS, D / 4, rs_pos, rs_frac, out, DirectFrames{}, "metrics_ragged", st);
}

// ---------------------------------------------------------------- student frames of another size
// compute_trajectory_metrics resizes every student frame to the teacher's H x W when the two differ
// (analysis/metrics/trajectory_metrics.py:40-52: F.interpolate(mode="bilinear", align_corners=True)).  The kernels below
// read the student at its own size and form the resized value of each teacher element on the fly, with torch's
// upsample_bilinear2d arithmetic in fp32: scale = (Hs - 1) / (Ht - 1) (0 when Ht == 1), src = scale * y, y0 = (int)src,
// y1 = y0 + (y0 < Hs - 1), ly = src - y0, the same along x, and four taps.  The resize has no antialiasing, so
// downsampling is the same four-tap formula.  No resized copy is ever written.
struct Bilinear {
    int Ht, Wt, Hs, Ws;
    float sh, sw;
    __host__ Bilinear(int ht, int wt, int hs, int ws)
        : Ht(ht), Wt(wt), Hs(hs), Ws(ws), sh(ht > 1 ? (float)(hs - 1) / (float)(ht - 1) : 0.f),
          sw(wt > 1 ? (float)(ws - 1) / (float)(wt - 1) : 0.f) {}
    // the resized value at teacher element (c, y, x) of the student frame s [C, Hs, Ws]
    __device__ __forceinline__ float at(const float* s, int c, int y, int x) const {
        const float fy = sh * (float)y, fx = sw * (float)x;
        const int y0 = (int)fy, x0 = (int)fx;
        const int y1 = y0 + (y0 < Hs - 1), x1 = x0 + (x0 < Ws - 1);
        const float ly = fy - (float)y0, lx = fx - (float)x0;
        const float* r0 = s + ((int64_t)c * Hs + y0) * Ws;
        const float* r1 = s + ((int64_t)c * Hs + y1) * Ws;
        return (1.f - ly) * ((1.f - lx) * __ldg(r0 + x0) + lx * __ldg(r0 + x1)) +
               ly * ((1.f - lx) * __ldg(r1 + x0) + lx * __ldg(r1 + x1));
    }
};

// Frame source of k_metrics_pairs_ragged for teacher [N, LT, C, Ht, Wt] and student [N, LS, C, Hs, Ws].  A teacher frame
// wider than one group's 4096 elements is cut into `parts` bands of whole teacher rows: group n covers band n % parts of
// pair n / parts and reads, through the resize, exactly the student rows its band needs.  Wt % 4 == 0, so the four
// elements of a teacher float4 lie on one row.  Teacher loads stream past L1 (ld.global.nc.L1::no_allocate); the
// student's taps, which neighbouring elements share, go through the read-only cache.
struct ResampledFrames {
    static constexpr bool kInPlace = false;
    Bilinear bl;
    int parts, HWt;
    int64_t Dt, Ds;                          // teacher and student frame sizes in floats
    // float4 e (of the band's D4) of frame i of group n's teacher or student
    __device__ __forceinline__ float4 load(const float* teacher, const float* student, bool stu, int64_t n, int LT, int LS, int i,
                                           int e, int D4) const {
        const int64_t pr = n / parts;
        const int d = (int)(n - pr * parts) * 4 * D4 + 4 * e;   // teacher element of the float4's first lane
        if (!stu) return ld_stream4(teacher + (pr * LT + i) * Dt + d);
        const float* f = student + (pr * LS + i) * Ds;
        const int c = d / HWt, r = d - c * HWt, y = r / bl.Wt, x = r - y * bl.Wt;
        return make_float4(bl.at(f, c, y, x), bl.at(f, c, y, x + 1), bl.at(f, c, y, x + 2), bl.at(f, c, y, x + 3));
    }
};

// out[n][m] = sum over the parts of part[n][p][m], added in f64 in part order
__global__ void __launch_bounds__(256) k_sum_parts(const float* __restrict__ part, int64_t N, int parts, int M, float* __restrict__ out) {
    for (int64_t o = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; o < N * M; o += (int64_t)gridDim.x * blockDim.x) {
        const int64_t n = o / M, m = o - n * M;
        double s = 0.0;
        for (int p = 0; p < parts; ++p) s += (double)part[(n * parts + p) * M + m];
        out[o] = (float)s;
    }
}

constexpr int kResampledMaxElems = 16384;    // C * Ht * Wt of a teacher frame for the reductions (4 x 64 x 64)

// teacher [.., C, Ht, Wt] against student [.., Cs, Hs, Ws]; frames of at most max_elems teacher elements
inline int check_resampled(const char* who, int LT, int LS, int C, int Ht, int Wt, int Cs, int Hs, int Ws, int64_t max_elems) {
    if (LT < 1 || LS < 1 || C < 1 || Ht < 1 || Wt < 1 || Cs < 1 || Hs < 1 || Ws < 1)
        return fail(DTRAJ_EINVAL, "%s: LT=%d, LS=%d and the sizes C=%d, Ht=%d, Wt=%d, Cs=%d, Hs=%d, Ws=%d must be positive", who, LT, LS,
                    C, Ht, Wt, Cs, Hs, Ws);
    if (Cs != C) return fail(DTRAJ_EINVAL, "%s: teacher has %d channels, student %d", who, C, Cs);
    if ((int64_t)C * Ht * Wt > max_elems)
        return fail(DTRAJ_EINVAL, "%s: teacher frame C*Ht*Wt=%lld too large (max %lld)", who, (long long)C * Ht * Wt, (long long)max_elems);
    if ((int64_t)C * Hs * Ws > 0x7fffffffLL) return fail(DTRAJ_EINVAL, "%s: student frame C*Hs*Ws too large", who);
    return 0;
}

inline int launch_metrics_pairs_resampled(const float* T, const float* S, int64_t N, int LT, int LS, int C, int Ht, int Wt, int Cs,
                                          int Hs, int Ws, const int32_t* rs_pos, const float* rs_frac, float* out, cudaStream_t st) {
    DTRAJ_TRY(check_resampled("metrics_resampled", LT, LS, C, Ht, Wt, Cs, Hs, Ws, kResampledMaxElems));
    if (LT < 2 && LS < 2) return fail(DTRAJ_EINVAL, "metrics_resampled: one of LT=%d, LS=%d must be >= 2", LT, LS);
    if (Wt % 4 != 0) return fail(DTRAJ_EINVAL, "metrics_resampled: Wt=%d must be a multiple of 4", Wt);
    const int rows = C * Ht;
    int parts = 1;                           // the fewest bands of whole rows of at most 4096 elements
    while (parts <= rows && (rows % parts || (rows / parts) * Wt > 4096)) ++parts;
    if (parts > rows) return fail(DTRAJ_EINVAL, "metrics_resampled: a teacher row of Wt=%d is wider than 4096", Wt);
    ResampledFrames fr{Bilinear(Ht, Wt, Hs, Ws), parts, Ht * Wt, (int64_t)C * Ht * Wt, (int64_t)C * Hs * Ws};
    const int D4 = rows / parts * Wt / 4, Lmax = LT > LS ? LT : LS;
    if (N == 0) return 0;
    if (parts == 1) return launch_ragged_walk(T, S, N, LT, LS, D4, rs_pos, rs_frac, out, fr, "metrics_resampled", st);
    float* part = nullptr;
    DTRAJ_CUDA(cudaMallocAsync(reinterpret_cast<void**>(&part), (size_t)N * parts * Lmax * kRaggedQ * sizeof(float), st));
    int rc = launch_ragged_walk(T, S, N * parts, LT, LS, D4, rs_pos, rs_frac, part, fr, "metrics_resampled", st);
    if (rc == 0) {
        const int64_t want = (N * Lmax * kRaggedQ + 255) / 256;
        k_sum_parts<<<(unsigned)(want < 8 * kNumSMs ? want : 8 * kNumSMs), 256, 0, st>>>(part, N, parts, Lmax * kRaggedQ, out);
        const cudaError_t e = cudaGetLastError();
        if (e != cudaSuccess) rc = fail(DTRAJ_ECUDA, "metrics_resampled: launch -> %s", cudaGetErrorString(e));
    }
    DTRAJ_CUDA(cudaFreeAsync(part, st));
    return rc;
}

// 1-d Wasserstein distance between K gathered elements of T_i and S_i: for equal-size
// samples W1 = mean |sort(u) - sort(v)| (scipy.stats.wasserstein_distance evaluates the
// same quantity through the two CDFs).  One CTA per (pair, frame): gather -> bitonic sort
// of both arrays in shared memory -> f64 sum of |a - b|.
__global__ void __launch_bounds__(256) k_wasserstein(const float* __restrict__ teacher, const float* __restrict__ student,
                                                     int L, int LT, int LS, int D, const int32_t* __restrict__ idx,
                                                     const int32_t* __restrict__ idx_set, int K, int P,
                                                     float* __restrict__ out) {
    extern __shared__ float sv[];   // [2][P]
    const int64_t pf = blockIdx.x;  // n*L + i
    const int64_t n = pf / L;
    const int i = (int)(pf % L);
    const float* t = teacher + (n * LT + i) * D;
    const float* s = student + (n * LS + i) * D;
    const int32_t* ix = idx ? idx + ((int64_t)(idx_set ? idx_set[n] : 0) * L + i) * K : nullptr;
    for (int k = threadIdx.x; k < P; k += blockDim.x) {
        float a = INFINITY, b = INFINITY;
        if (k < K) { const int e = ix ? ix[k] : k; a = t[e]; b = s[e]; }
        sv[k] = a; sv[P + k] = b;
    }
    __syncthreads();
    const int half = P >> 1;
    for (int size = 2; size <= P; size <<= 1) {
        for (int j = size >> 1; j > 0; j >>= 1) {
            for (int ce = threadIdx.x; ce < P; ce += blockDim.x) {   // P/2 exchanges per array, two arrays
                const int arr = ce / half, k = ce % half;
                const int lo = ((k / j) * 2 * j) + (k % j), hi = lo + j;
                float* v = sv + arr * P;
                const float a = v[lo], b = v[hi];
                const bool up = (lo & size) == 0;
                if ((a > b) == up) { v[lo] = b; v[hi] = a; }
            }
            __syncthreads();
        }
    }
    double acc = 0.0;
    for (int k = threadIdx.x; k < K; k += blockDim.x) acc += (double)fabsf(sv[k] - sv[P + k]);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    __shared__ double wsum[8];
    if ((threadIdx.x & 31) == 0) wsum[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
        double tot = 0.0;
        for (int w = 0; w < 8; ++w) tot += wsum[w];
        out[pf] = (float)(tot / (double)K);
    }
}

// Small-K form (P = 32 * E <= 1024 padded elements): ONE WARP per (pair, frame), both arrays sorted in registers by a
// bitonic network over element index = lane * E + e -- strides below E are register-register compare-exchanges,
// strides of E and more are __shfl_xor exchanges; no shared memory, no block barriers.  ncu on the block-per-frame
// kernel above at K = 256: 3166 instructions per warp x 8 warps per frame, issue-bound (3.3 ms for 120 k frames).
template <int E>
__device__ __forceinline__ void warp_bitonic_sort(float (&v)[E], int lane) {
#pragma unroll
    for (int k = 2; k <= 32 * E; k <<= 1) {
#pragma unroll
        for (int j = k >> 1; j > 0; j >>= 1) {
            if (j >= E) {
                const int lj = j / E;
                const bool lower = (lane & lj) == 0;
#pragma unroll
                for (int e = 0; e < E; ++e) {
                    const float o = __shfl_xor_sync(0xffffffffu, v[e], lj);
                    const bool up = ((lane * E + e) & k) == 0;
                    v[e] = (lower == up) ? fminf(v[e], o) : fmaxf(v[e], o);
                }
            } else {
#pragma unroll
                for (int e = 0; e < E; ++e) {
                    if ((e & j) == 0) {
                        const float a = v[e], b = v[e | j];
                        const bool up = ((lane * E + e) & k) == 0;
                        const float lo = fminf(a, b), hi = fmaxf(a, b);
                        v[e] = up ? lo : hi;
                        v[e | j] = up ? hi : lo;
                    }
                }
            }
        }
    }
}

// Student element source of k_wasserstein_warp: DirectSample reads element el of a student frame of the teacher's size,
// ResampledSample the resized value at teacher element el of a student [C, Hs, Ws] (the index sets are teacher-frame
// indices, as the reference draws them after resizing).
struct DirectSample {
    __device__ __forceinline__ const float* frame(const float* student, int64_t f, int D) const { return student + f * D; }
    __device__ __forceinline__ float at(const float* s, int el) const { return __ldg(s + el); }
};

struct ResampledSample {
    Bilinear bl;
    int64_t Ds;                              // student frame size in floats
    __device__ __forceinline__ const float* frame(const float* student, int64_t f, int /*D*/) const { return student + f * Ds; }
    __device__ __forceinline__ float at(const float* s, int el) const {
        const int hw = bl.Ht * bl.Wt, c = el / hw, r = el - c * hw, y = r / bl.Wt;
        return bl.at(s, c, y, r - y * bl.Wt);
    }
};

template <int E, class Student>
__global__ void __launch_bounds__(256) k_wasserstein_warp(const float* __restrict__ teacher, const float* __restrict__ student,
                                                          int64_t NL, int L, int LT, int LS, int D, const int32_t* __restrict__ idx,
                                                          const int32_t* __restrict__ idx_set, int K, float* __restrict__ out,
                                                          Student stu) {
    const int lane = threadIdx.x & 31;
    const int64_t pf = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);    // n*L + i
    if (pf >= NL) return;
    const int64_t n = pf / L;
    const int i = (int)(pf - n * L);
    const float* t = teacher + (n * LT + i) * D;
    const float* s = stu.frame(student, n * LS + i, D);
    const int32_t* ix = idx ? idx + ((int64_t)(idx_set ? idx_set[n] : 0) * L + i) * K : nullptr;
    float a[E], b[E];
#pragma unroll
    for (int e = 0; e < E; ++e) {
        const int k = lane * E + e;
        a[e] = INFINITY; b[e] = INFINITY;
        if (k < K) { const int el = ix ? __ldg(ix + k) : k; a[e] = __ldg(t + el); b[e] = stu.at(s, el); }
    }
    warp_bitonic_sort<E>(a, lane);
    warp_bitonic_sort<E>(b, lane);
    double acc = 0.0;
#pragma unroll
    for (int e = 0; e < E; ++e)
        if (lane * E + e < K) acc += (double)fabsf(a[e] - b[e]);        // the +inf padding sorts behind the K real elements
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if (lane == 0) out[pf] = (float)(acc / (double)K);
}

// Projection of trajectory frames onto K <= 8 principal directions (scripts/analysis/analyze_trajectories.py:66-80,100:
// process_trajectory -> [L, D] features, PCA(3).fit(reference).transform(features) for every trajectory of a sweep):
//   out[f][k] = sum_d x[f][d] * comps[k][d] - off[k],   off[k] = mean . comps[k]   (sklearn's transform order)
// HBM-bound: every element of the frames is read once (algorithmic bytes 4 * F * D); the K x D directions sit in shared
// memory, one warp per frame, 128-bit streaming loads, warp-shuffle reductions, persistent blocks.
__global__ void __launch_bounds__(256) k_project(const float* __restrict__ x, int64_t F, int D4, const float* __restrict__ comps,
                                                 const float* __restrict__ off, int K, float* __restrict__ out) {
    extern __shared__ float4 pc[];                   // [K][D4]
    for (int i = threadIdx.x; i < K * D4; i += blockDim.x) pc[i] = reinterpret_cast<const float4*>(comps)[i];
    __syncthreads();
    const int lane = threadIdx.x & 31, wpb = blockDim.x >> 5;
    for (int64_t f = (int64_t)blockIdx.x * wpb + (threadIdx.x >> 5); f < F; f += (int64_t)gridDim.x * wpb) {
        const float4* row = reinterpret_cast<const float4*>(x) + f * D4;
        float acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
        for (int d0 = lane; d0 < D4; d0 += 128) {          // four independent 16-byte loads per lane in flight
            float4 v[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int d = d0 + 32 * u;
                v[u] = d < D4 ? ld_stream4(reinterpret_cast<const float*>(row + d)) : make_float4(0.f, 0.f, 0.f, 0.f);
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int d = d0 + 32 * u;
                if (d < D4) {
#pragma unroll
                    for (int k = 0; k < 8; ++k)
                        if (k < K) {
                            const float4 c = pc[k * D4 + d];
                            acc[k] = fmaf(v[u].x, c.x, fmaf(v[u].y, c.y, fmaf(v[u].z, c.z, fmaf(v[u].w, c.w, acc[k]))));
                        }
                }
            }
        }
#pragma unroll
        for (int k = 0; k < 8; ++k)
            if (k < K) {
                const float s = warp_sum(acc[k]);
                if (lane == 0) out[f * K + k] = s - off[k];
            }
    }
}

inline int launch_project(const float* x, int64_t F, int D, const float* comps, const float* off, int K, float* out, cudaStream_t st) {
    if (D % 4 != 0 || D <= 0 || K < 1 || K > 8) return fail(DTRAJ_EINVAL, "project: D=%d must be a positive multiple of 4, K=%d in 1..8", D, K);
    const size_t smem = (size_t)K * D * sizeof(float);
    if (smem > 200 * 1024) return fail(DTRAJ_EINVAL, "project: K*D=%d too large for shared memory", K * D);
    if (F == 0) return 0;
    if (smem > 48 * 1024) DTRAJ_CUDA(cudaFuncSetAttribute(k_project, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const int64_t want = (F + 7) / 8;
    const unsigned grid = (unsigned)(want < 6 * kNumSMs ? want : 6 * kNumSMs);
    k_project<<<grid, 256, smem, st>>>(x, F, D / 4, comps, off, K, out);
    DTRAJ_LAUNCH_CHECK();
    return 0;
}

// Frames i < L = min(LT, LS) of pairs whose teacher holds LT frames and student LS frames ([N, LT, D] / [N, LS, D], read in
// place, or a student of another frame size through ResampledSample); idx is [n_sets, L, K] and out [N, L].  LT == LS is
// the equal-length form.  The block-per-frame form for K > 1024 reads students of the teacher's size only.
template <class Student = DirectSample>
inline int launch_wasserstein(const float* T, const float* S, int64_t N, int LT, int LS, int D, const int32_t* idx,
                              const int32_t* idx_set, int K, float* out, cudaStream_t st, Student stu = {}) {
    const int L = LT < LS ? LT : LS;
    if (L < 1) return fail(DTRAJ_EINVAL, "wasserstein: LT=%d and LS=%d must be >= 1", LT, LS);
    if (K < 1 || K > D || K > 4096) return fail(DTRAJ_EINVAL, "wasserstein: K=%d out of range (D=%d)", K, D);
    if (!idx && K != D) return fail(DTRAJ_EINVAL, "wasserstein: idx == NULL requires K == D");
    if (N * L > 0x7fffffffLL) return fail(DTRAJ_EINVAL, "wasserstein: N*L too large for one launch");
    if (N == 0) return 0;
    int P = 2;
    while (P < K) P *= 2;
    const int64_t NL = N * L;
    const unsigned wgrid = (unsigned)((NL + 7) / 8);
    if (P <= 256) {
        k_wasserstein_warp<8, Student><<<wgrid, 256, 0, st>>>(T, S, NL, L, LT, LS, D, idx, idx_set, K, out, stu);
        DTRAJ_LAUNCH_CHECK();
        return 0;
    }
    if (P <= 1024) {
        k_wasserstein_warp<32, Student><<<wgrid, 256, 0, st>>>(T, S, NL, L, LT, LS, D, idx, idx_set, K, out, stu);
        DTRAJ_LAUNCH_CHECK();
        return 0;
    }
    if (!std::is_same<Student, DirectSample>::value) return fail(DTRAJ_EINVAL, "wasserstein: K=%d > 1024 with a resampled student", K);
    k_wasserstein<<<(unsigned)(N * L), 256, 2 * P * sizeof(float), st>>>(T, S, L, LT, LS, D, idx, idx_set, K, P, out);
    DTRAJ_LAUNCH_CHECK();
    return 0;
}

// Frames of any size with int32 element indices: W1 gathers at most 1024 elements of a frame, so, unlike the reductions,
// it holds no frame in registers (C may count the images of a [B, C, H, W] frame times their channels).
inline int launch_wasserstein_resampled(const float* T, const float* S, int64_t N, int LT, int LS, int C, int Ht, int Wt, int Cs,
                                        int Hs, int Ws, const int32_t* idx, const int32_t* idx_set, int K, float* out, cudaStream_t st) {
    DTRAJ_TRY(check_resampled("wasserstein_resampled", LT, LS, C, Ht, Wt, Cs, Hs, Ws, 0x7fffffffLL));
    if (K > 1024) return fail(DTRAJ_EINVAL, "wasserstein_resampled: K=%d out of range (max 1024)", K);
    return launch_wasserstein(T, S, N, LT, LS, C * Ht * Wt, idx, idx_set, K, out, st,
                              ResampledSample{Bilinear(Ht, Wt, Hs, Ws), (int64_t)C * Hs * Ws});
}

// ---------------------------------------------------------------- Wasserstein subsample indices on the device
// compute_trajectory_metrics subsamples every frame larger than 1000 elements with
//     np.random.choice(D, 1000, replace=False)                        (analysis/metrics/trajectory_metrics.py:301-306)
// from the GLOBAL numpy RNG, which compare_trajectories' callers left seeded at seed + 1 (analysis/trajectory_engine.py:91-93).
// That is numpy's legacy RandomState (third-party, numpy==1.26.4 pinned by the reference; the legacy stream is frozen
// across versions): MT19937 seeded by init_genrand(seed); choice(replace=False) = permutation(D)[:K]; permutation =
// Fisher-Yates `for i = D-1 .. 1: j = random_interval(i); swap(x[i], x[j])` with random_interval(max) = draw 32-bit
// words, mask to the smallest 2^k - 1 >= max, reject values > max.  The kernel below reproduces that stream bit for bit
// (integer work: tests/test_gpu_metrics.py compares it with numpy itself): one thread per seed walks its L consecutive
// permutations; MT state and permutation live in shared memory, interleaved over the block's threads (bank = thread).
// kChoiceThreads seeds per block: 16 up to D = 4096; wider frames take 8 (D <= 12288: 216 KB) or 4 (D <= 16384: 138 KB) so that
// the interleaved uint16 permutations still fit the 227 KB of shared memory.
template <int kChoiceThreads>
__global__ void __launch_bounds__(kChoiceThreads) k_numpy_choice(const uint32_t* __restrict__ seeds, int n_seeds, int L, int D, int K,
                                                                 int32_t* __restrict__ out) {
    constexpr unsigned kMask = (1u << kChoiceThreads) - 1u;
    extern __shared__ __align__(16) uint8_t ch_smem[];
    uint32_t* mt = reinterpret_cast<uint32_t*>(ch_smem);                                   // [624][kChoiceThreads]
    uint16_t* perm = reinterpret_cast<uint16_t*>(ch_smem + 624 * kChoiceThreads * 4);      // [D][kChoiceThreads]
    const int t = threadIdx.x;
    const int sidx = blockIdx.x * kChoiceThreads + t;
    const bool live = sidx < n_seeds;
    uint32_t* my = mt + t;
    uint16_t* pm = perm + t;
    int pos = 624;
    if (live) {
        uint32_t sd = seeds[sidx];
        for (int i = 0; i < 624; ++i) { my[i * kChoiceThreads] = sd; sd = 1812433253u * (sd ^ (sd >> 30)) + (uint32_t)i + 1u; }
    }
    auto next32 = [&]() -> uint32_t {
        if (pos == 624) {
            int kk = 0;
            for (; kk < 624 - 397; ++kk) {
                const uint32_t y = (my[kk * kChoiceThreads] & 0x80000000u) | (my[(kk + 1) * kChoiceThreads] & 0x7fffffffu);
                my[kk * kChoiceThreads] = my[(kk + 397) * kChoiceThreads] ^ (y >> 1) ^ ((y & 1u) ? 0x9908b0dfu : 0u);
            }
            for (; kk < 623; ++kk) {
                const uint32_t y = (my[kk * kChoiceThreads] & 0x80000000u) | (my[(kk + 1) * kChoiceThreads] & 0x7fffffffu);
                my[kk * kChoiceThreads] = my[(kk - 227) * kChoiceThreads] ^ (y >> 1) ^ ((y & 1u) ? 0x9908b0dfu : 0u);
            }
            const uint32_t y = (my[623 * kChoiceThreads] & 0x80000000u) | (my[0] & 0x7fffffffu);
            my[623 * kChoiceThreads] = my[396 * kChoiceThreads] ^ (y >> 1) ^ ((y & 1u) ? 0x9908b0dfu : 0u);
            pos = 0;
        }
        uint32_t y = my[(pos++) * kChoiceThreads];
        y ^= y >> 11;
        y ^= (y << 7) & 0x9d2c5680u;
        y ^= (y << 15) & 0xefc60000u;
        y ^= y >> 18;
        return y;
    };
    for (int f = 0; f < L; ++f) {
        if (live) {
            for (int i = 0; i < D; ++i) pm[i * kChoiceThreads] = (uint16_t)i;
            for (int i = D - 1; i >= 1; --i) {
                const uint32_t mask = 0xffffffffu >> __clz((uint32_t)i);
                uint32_t j;
                do { j = next32() & mask; } while (j > (uint32_t)i);
                const uint16_t a = pm[i * kChoiceThreads], b = pm[j * kChoiceThreads];
                pm[i * kChoiceThreads] = b;
                pm[j * kChoiceThreads] = a;
            }
        }
        __syncwarp(kMask);
        // coalesced write-out: the block's threads share the rows of each seed
        for (int s = 0; s < kChoiceThreads; ++s) {
            const int so = blockIdx.x * kChoiceThreads + s;
            if (so >= n_seeds) break;
            int32_t* dst = out + ((size_t)so * L + f) * K;
            for (int k = t; k < K; k += kChoiceThreads) dst[k] = (int32_t)perm[k * kChoiceThreads + s];
        }
        __syncwarp(kMask);
    }
}

template <int kT>
inline int launch_numpy_choice_t(const uint32_t* seeds, int n_seeds, int L, int D, int K, int32_t* out, int d_max, cudaStream_t st) {
    const size_t smem = (size_t)624 * kT * 4 + (size_t)D * kT * 2;
    static bool attr_set = false;
    if (!attr_set) {
        DTRAJ_CUDA(cudaFuncSetAttribute(k_numpy_choice<kT>, cudaFuncAttributeMaxDynamicSharedMemorySize, 624 * kT * 4 + d_max * kT * 2));
        attr_set = true;
    }
    k_numpy_choice<kT><<<(unsigned)((n_seeds + kT - 1) / kT), kT, smem, st>>>(seeds, n_seeds, L, D, K, out);
    DTRAJ_LAUNCH_CHECK();
    return 0;
}

inline int launch_numpy_choice(const uint32_t* seeds, int n_seeds, int L, int D, int K, int32_t* out, cudaStream_t st) {
    if (n_seeds < 0 || L < 1 || D < 2 || D > 16384 || K < 1 || K > D) return fail(DTRAJ_EINVAL, "numpy_choice: bad argument (2 <= D <= 16384, 1 <= K <= D)");
    if (n_seeds == 0) return 0;
    if (D <= 4096) return launch_numpy_choice_t<16>(seeds, n_seeds, L, D, K, out, 4096, st);
    if (D <= 12288) return launch_numpy_choice_t<8>(seeds, n_seeds, L, D, K, out, 12288, st);
    return launch_numpy_choice_t<4>(seeds, n_seeds, L, D, K, out, 16384, st);
}

}  // namespace dtraj
