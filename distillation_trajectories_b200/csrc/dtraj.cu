// libdtraj.so -- C ABI (include/dtraj.h): model packing, forward plan, sampler loop with
// CUDA-graph capture, metric entry points.  sm_100a only; no torch types anywhere.
#include <map>
#include <string>
#include <vector>
#include <cmath>
#include <cstdlib>
#include <cuda_fp16.h>

#include "common.cuh"
#include "elem.cuh"
#include "conv_simt.cuh"
#include "conv_umma.cuh"
#include "metrics.cuh"
#include "enc1_umma.cuh"
#include "enc1_f16.cuh"
#ifdef DTRAJ_PROBES
#include "probe.cuh"        // hardware probes (tools/probe_*.py): built only with -DDTRAJ_PROBES, never part of the product library
#endif

using namespace dtraj;

// ======================================================================================
// model
// ======================================================================================
namespace {

const char* kBlockNames[8] = {"enc1", "enc2", "enc3", "enc4", "bottleneck", "dec3", "dec2", "dec1"};

struct PackedConv {          // one generic conv layer's parameters on the device
    const float* w = nullptr;   // [npl][nkb][coutp][32], plane 0 = hi (or the only one), plane 1 = lo
    const float* bias = nullptr;
    int64_t rows = 0;           // npl * nkb * coutp
    int c0p = 0, c1p = 0, coutp = 0, ntaps = 0;
    int c0 = 0, c1 = 0, cout = 0;   // real (unpadded) channels: algorithmic flop count
};

struct BlockW {
    int cin0 = 0, cin1 = 0, cout = 0, S = 0;   // real channels, spatial size
    bool has_res = false;
    PackedConv conv1, conv2, res;              // conv1/res unused for enc1 (first-conv kernel)
};

struct Arena {               // host staging of everything that goes to the device in one copy
    std::vector<float> h;
    size_t alloc(size_t n) {
        size_t off = (h.size() + 63) / 64 * 64;
        h.resize(off + n, 0.f);
        return off;
    }
};

}  // namespace

struct dtraj_unet {
    dtraj_unet_desc d;
    int dp[4];                  // padded dims
    int sizes[5];               // spatial size per level
    int act_mode;               // ACT_* for GEMM operands
    float* dev = nullptr;       // weight arena
    size_t dev_floats = 0;
    BlockW blk[8];
    // first conv (enc1.conv1 + enc1.residual_conv)
    const float *fw3 = nullptr, *fb3 = nullptr, *fw1 = nullptr, *fb1 = nullptr;
    // final 1x1
    const float *finw = nullptr, *finb = nullptr;
    // time table
    float* table = nullptr;     // [T][3][tb_stride]
    int tb_stride = 0;
    int tb_off[8];
    unsigned int* err = nullptr;   // this handle's device error word (inside the arena): bit 0 pipeline time-out, bit 1 fp16 overflow
    // cached forward plan for dtraj_unet_forward
    struct dtraj_plan* plan = nullptr;
};

namespace {

struct TensorDict {
    std::map<std::string, std::pair<const float*, int64_t>> m;
    const float* get(const std::string& k, int64_t expect, int* err) const {
        auto it = m.find(k);
        if (it == m.end()) { *err = fail(DTRAJ_EMISSING, "state_dict entry '%s' missing", k.c_str()); return nullptr; }
        if (expect >= 0 && it->second.second != expect) {
            *err = fail(DTRAJ_EINVAL, "state_dict entry '%s' has %lld elements, expected %lld", k.c_str(),
                        (long long)it->second.second, (long long)expect);
            return nullptr;
        }
        return it->second.first;
    }
    bool has(const std::string& k) const { return m.count(k) != 0; }
};

// eval-mode BatchNorm folded into the preceding conv (models.py:48-51, eps = 1e-5):
// y = (conv(x) + b - mean) * gamma / sqrt(var + eps) + beta
int bn_fold(const TensorDict& sd, const std::string& conv, const std::string& norm, int cout,
            std::vector<double>* scale, std::vector<double>* shift) {
    int err = 0;
    const float* b = sd.get(conv + ".bias", cout, &err);
    const float* g = sd.get(norm + ".weight", cout, &err);
    const float* be = sd.get(norm + ".bias", cout, &err);
    const float* mu = sd.get(norm + ".running_mean", cout, &err);
    const float* var = sd.get(norm + ".running_var", cout, &err);
    if (err) return err;
    scale->resize(cout); shift->resize(cout);
    for (int n = 0; n < cout; ++n) {
        double s = (double)g[n] / std::sqrt((double)var[n] + 1e-5);
        (*scale)[n] = s;
        (*shift)[n] = ((double)b[n] - (double)mu[n]) * s + (double)be[n];
    }
    return 0;
}

// Channel counts of feature maps and weights are padded to 32 in every mode.  A K block (128 bytes per pixel / per output
// channel) carries 32 fp32 / tf32 channels or 64 halfs (DTRAJ_PREC_F16): there a source padded to an odd multiple of 32 ends in
// a half-filled block (zero weights; the activation box is zero-filled by TMA beyond the map's channel dimension) of which only
// two of the four K = 16 MMAs are issued -- so fp16 models execute round_up(C, 32) channels, not round_up(C, 64).
inline int kblock_of(int precision) { return precision == DTRAJ_PREC_F16 ? 64 : 32; }
thread_local bool g_pack_overflow = false;   // a folded weight outside the fp16 range (DTRAJ_PREC_F16)

// Pack [cout][c0+c1][k][k] into K-major blocks of one 128-byte row per output channel: [tap][chunk][coutp][32] floats
// (+ low plane), or [tap][chunk][coutp][64] halfs in DTRAJ_PREC_F16.  c0p / c1p / coutp: the padded channel counts of the
// feature maps involved (multiples of 32; 0 = round the real count up to 32).
void pack_conv(Arena* A, size_t* w_off, size_t* b_off, PackedConv* pc, const float* w, int cout, int c0, int c1,
               int ksize, bool centre_only, const double* scale, const double* shift, int precision,
               int c0p = 0, int c1p = 0, int coutp = 0) {
    const int kch = kblock_of(precision);
    const bool f16 = precision == DTRAJ_PREC_F16;
    if (!c0p) c0p = round_up(c0, kCPad);
    if (!c1p) c1p = c1 ? round_up(c1, kCPad) : 0;
    if (!coutp) coutp = round_up(cout, kCPad);
    const int ntaps = (ksize == 3 && !centre_only) ? 9 : 1;
    const int nch0 = (c0p + kch - 1) / kch, nch = nch0 + (c1p + kch - 1) / kch, nkb = ntaps * nch;
    const int npl = precision == DTRAJ_PREC_TF32X3 ? 2 : 1;
    const size_t plane = (size_t)nkb * coutp * 32;          // floats: one 128-byte row per (K block, output channel)
    *w_off = A->alloc(plane * npl);
    *b_off = A->alloc(coutp);
    const int cin = c0 + c1;
    for (int tap = 0; tap < ntaps; ++tap) {
        int ky = 0, kx = 0;
        if (ksize == 3) { ky = centre_only ? 1 : tap / 3; kx = centre_only ? 1 : tap % 3; }
        for (int chunk = 0; chunk < nch; ++chunk)
            for (int n = 0; n < cout; ++n)
                for (int kk = 0; kk < kch; ++kk) {
                    int c, ci;
                    if (chunk < nch0) { c = chunk * kch + kk; ci = c < c0 ? c : -1; }
                    else { c = (chunk - nch0) * kch + kk; ci = c < c1 ? c0 + c : -1; }
                    if (ci < 0) continue;
                    double v = (double)w[(((size_t)n * cin + ci) * ksize + ky) * ksize + kx] * (scale ? scale[n] : 1.0);
                    float f = (float)v;
                    if (f16) {
                        if (!(std::fabs(f) <= 65504.f)) g_pack_overflow = true;
                        __half* hp = reinterpret_cast<__half*>(&A->h[*w_off]);
                        hp[((size_t)(tap * nch + chunk) * coutp + n) * 64 + kk] = __float2half_rn(f);
                        continue;
                    }
                    size_t o = *w_off + (((size_t)(tap * nch + chunk) * coutp + n) * 32 + kk);
                    if (precision == DTRAJ_PREC_FP32) A->h[o] = f;
                    else {
                        float hi = tf32_rna_host(f);
                        A->h[o] = hi;
                        if (npl == 2) A->h[o + plane] = f - hi;
                    }
                }
    }
    for (int n = 0; n < cout; ++n) A->h[*b_off + n] = (float)shift[n];
    pc->rows = (int64_t)npl * nkb * coutp;
    pc->c0p = c0p; pc->c1p = c1p; pc->coutp = coutp; pc->ntaps = ntaps;
    pc->c0 = c0; pc->c1 = c1; pc->cout = cout;
}

// dynamic shared memory of k_conv_first: the zero-padded C x (H+2) x (H+2) input, then 9C + C rows of coutp weights
inline size_t first_conv_smem(int C, int H, int coutp) {
    return (size_t)(round_up(C * (H + 2) * (H + 2), 4) + 10 * C * coutp) * sizeof(float);
}

}  // namespace

extern "C" const char* dtraj_last_error(void) { return err_buf(); }
extern "C" int dtraj_version(void) { return 100; }

extern "C" int dtraj_unet_destroy(dtraj_unet* u);

extern "C" int dtraj_unet_create(const dtraj_unet_desc* desc, const char* const* names, const float* const* tensors,
                                 const int64_t* numel, int32_t n_tensors, dtraj_unet** out) {
    if (!desc || !out || !names || !tensors || !numel) return fail(DTRAJ_EINVAL, "null argument");
    const int C = desc->channels, H = desc->image_size, temb = desc->temb_dim, T = desc->n_timesteps;
    if (C < 1 || C > 4) return fail(DTRAJ_EINVAL, "channels=%d unsupported (1..4)", C);
    if (H != 16 && H != 32 && H != 64) return fail(DTRAJ_EINVAL, "image_size=%d unsupported (16, 32 or 64)", H);
    if (temb < 2 || temb > 1024 || T < 1) return fail(DTRAJ_EINVAL, "bad temb_dim/n_timesteps");
    if (desc->precision < 0 || desc->precision > 3) return fail(DTRAJ_EINVAL, "bad precision");
    for (int i = 0; i < 4; ++i)
        if (desc->dims[i] < 1 || desc->dims[i] > 256) return fail(DTRAJ_EINVAL, "dims[%d]=%d unsupported (1..256)", i, desc->dims[i]);
    if (desc->dims[1] != desc->dims[2] || desc->dims[2] != desc->dims[3])
        return fail(DTRAJ_EINVAL, "dims must be [b, m, m, m] (models.py:107-110)");

    TensorDict sd;
    for (int i = 0; i < n_tensors; ++i) sd.m[names[i]] = {tensors[i], numel[i]};

    dtraj_unet* u = new dtraj_unet();
    u->d = *desc;
    const int cpad = kCPad;
    g_pack_overflow = false;
    for (int i = 0; i < 4; ++i) u->dp[i] = round_up(desc->dims[i], cpad);
    if (desc->precision == DTRAJ_PREC_F16) u->dp[0] = round_up(desc->dims[0], 64);   // the fused enc1 kernel works on whole 64-channel chunks
    for (int l = 0; l < 5; ++l) u->sizes[l] = H >> l;
    u->act_mode = desc->precision == DTRAJ_PREC_FP32 ? ACT_PLAIN : desc->precision == DTRAJ_PREC_TF32X3 ? ACT_SPLIT : ACT_ROUND;
    const int* d = desc->dims;
    // block geometry (models.py:137-154)
    const int cin0[8] = {C, d[0], d[1], d[2], d[3], d[3], d[2], d[1]};
    const int cin1[8] = {0, 0, 0, 0, 0, d[3], d[2], d[1]};
    const int cout[8] = {d[0], d[1], d[2], d[3], d[3], d[2], d[1], d[0]};
    const int lvl[8] = {0, 1, 2, 3, 4, 3, 2, 1};
    const int* dp = u->dp;
    const int cin0p[8] = {0, dp[0], dp[1], dp[2], dp[3], dp[3], dp[2], dp[1]};      // padded widths of the maps each block reads / writes
    const int cin1p[8] = {0, 0, 0, 0, 0, dp[3], dp[2], dp[1]};
    const int coutp[8] = {dp[0], dp[1], dp[2], dp[3], dp[3], dp[2], dp[1], dp[0]};

    Arena A;
    int err = 0;
    struct Off { size_t w1, b1, w2, b2, wr, br; } off[8] = {};
    size_t o_fw3 = 0, o_fb3 = 0, o_fw1 = 0, o_fb1 = 0, o_finw = 0, o_finb = 0;
    size_t o_tw1, o_tb1, o_cw0, o_cb0, o_cw2, o_cb2, o_bw[8], o_bb[8];

    for (int b = 0; b < 8 && !err; ++b) {
        BlockW& B = u->blk[b];
        const std::string nm = kBlockNames[b];
        B.cin0 = cin0[b]; B.cin1 = cin1[b]; B.cout = cout[b]; B.S = u->sizes[lvl[b]];
        const int cin = B.cin0 + B.cin1;
        B.has_res = sd.has(nm + ".residual_conv.weight");
        if (!B.has_res && cin != B.cout) { err = fail(DTRAJ_EMISSING, "%s.residual_conv missing but in_ch != out_ch", nm.c_str()); break; }
        const bool centre = B.S == 1;
        std::vector<double> sc, sh;
        // conv1
        const float* w = sd.get(nm + ".conv1.weight", (int64_t)B.cout * cin * 9, &err);
        if (err || (err = bn_fold(sd, nm + ".conv1", nm + ".norm1", B.cout, &sc, &sh))) break;
        if (b == 0) {
            // first conv: [9*C][coutp] tap-major (fp32 CUDA cores), residual [C][coutp]
            const int cp = u->dp[0];
            o_fw3 = A.alloc((size_t)9 * C * cp); o_fb3 = A.alloc(cp);
            for (int n = 0; n < B.cout; ++n) {
                for (int c = 0; c < C; ++c)
                    for (int t9 = 0; t9 < 9; ++t9)
                        A.h[o_fw3 + ((size_t)t9 * C + c) * cp + n] = (float)((double)w[((size_t)n * C + c) * 9 + t9] * sc[n]);
                A.h[o_fb3 + n] = (float)sh[n];
            }
            if (!B.has_res) { err = fail(DTRAJ_EINVAL, "enc1 without residual_conv is unsupported"); break; }
            const float* wr = sd.get(nm + ".residual_conv.weight", (int64_t)B.cout * C, &err);
            const float* br = sd.get(nm + ".residual_conv.bias", B.cout, &err);
            if (err) break;
            o_fw1 = A.alloc((size_t)C * cp); o_fb1 = A.alloc(cp);
            for (int n = 0; n < B.cout; ++n) {
                for (int c = 0; c < C; ++c) A.h[o_fw1 + (size_t)c * cp + n] = wr[(size_t)n * C + c];
                A.h[o_fb1 + n] = br[n];
            }
        } else {
            pack_conv(&A, &off[b].w1, &off[b].b1, &B.conv1, w, B.cout, B.cin0, B.cin1, 3, centre, sc.data(), sh.data(), desc->precision,
                      cin0p[b], cin1p[b], coutp[b]);
            if (B.has_res) {
                const float* wr = sd.get(nm + ".residual_conv.weight", (int64_t)B.cout * cin, &err);
                const float* br = sd.get(nm + ".residual_conv.bias", B.cout, &err);
                if (err) break;
                std::vector<double> rb(B.cout);
                for (int n = 0; n < B.cout; ++n) rb[n] = br[n];
                pack_conv(&A, &off[b].wr, &off[b].br, &B.res, wr, B.cout, B.cin0, B.cin1, 1, false, nullptr, rb.data(), desc->precision,
                          cin0p[b], cin1p[b], coutp[b]);
            }
        }
        // conv2
        const float* w2 = sd.get(nm + ".conv2.weight", (int64_t)B.cout * B.cout * 9, &err);
        if (err || (err = bn_fold(sd, nm + ".conv2", nm + ".norm2", B.cout, &sc, &sh))) break;
        pack_conv(&A, &off[b].w2, &off[b].b2, &B.conv2, w2, B.cout, B.cout, 0, 3, centre, sc.data(), sh.data(), desc->precision,
                  coutp[b], 0, coutp[b]);
        // block time MLP (raw)
        const float* tw = sd.get(nm + ".time_mlp.weight", (int64_t)B.cout * temb, &err);
        const float* tb = sd.get(nm + ".time_mlp.bias", B.cout, &err);
        if (err) break;
        o_bw[b] = A.alloc((size_t)B.cout * temb); memcpy(&A.h[o_bw[b]], tw, sizeof(float) * B.cout * temb);
        o_bb[b] = A.alloc(B.cout); memcpy(&A.h[o_bb[b]], tb, sizeof(float) * B.cout);
    }
    auto copy_in = [&](const char* key, int64_t n, size_t* o) {
        const float* p = sd.get(key, n, &err);
        if (!p) return;
        *o = A.alloc(n);
        memcpy(&A.h[*o], p, sizeof(float) * n);
    };
    if (!err) {
        copy_in("time_mlp.1.weight", (int64_t)temb * temb, &o_tw1); copy_in("time_mlp.1.bias", temb, &o_tb1);
        copy_in("cond_emb.0.weight", temb, &o_cw0); copy_in("cond_emb.0.bias", temb, &o_cb0);
        copy_in("cond_emb.2.weight", (int64_t)temb * temb, &o_cw2); copy_in("cond_emb.2.bias", temb, &o_cb2);
    }
    if (!err) {
        const float* fw = sd.get("final.weight", (int64_t)C * d[0], &err);
        const float* fb = sd.get("final.bias", C, &err);
        if (!err) {
            o_finw = A.alloc((size_t)C * u->dp[0]); o_finb = A.alloc(4);
            for (int c = 0; c < C; ++c) {
                for (int k = 0; k < d[0]; ++k) A.h[o_finw + (size_t)c * u->dp[0] + k] = fw[(size_t)c * d[0] + k];
                A.h[o_finb + c] = fb[c];
            }
        }
    }
    if (err) { delete u; return err; }
    if (g_pack_overflow) { delete u; return fail(DTRAJ_EINVAL, "a BatchNorm-folded conv weight exceeds the fp16 range: use precision tf32"); }

    // time table layout
    int tbs = 0;
    for (int b = 0; b < 8; ++b) { u->tb_off[b] = tbs; tbs += coutp[b]; }
    u->tb_stride = tbs;
    const size_t o_table = A.alloc((size_t)T * 3 * tbs);
    const size_t o_err = A.alloc(64);                 // (zero-initialised like the rest of the arena)

    u->dev_floats = A.h.size();
    cudaError_t ce = cudaMalloc(&u->dev, u->dev_floats * sizeof(float));
    if (ce != cudaSuccess) { delete u; return fail(DTRAJ_ECUDA, "cudaMalloc(weights %zu B) -> %s", u->dev_floats * 4, cudaGetErrorString(ce)); }
    ce = cudaMemcpy(u->dev, A.h.data(), u->dev_floats * sizeof(float), cudaMemcpyHostToDevice);
    if (ce != cudaSuccess) { dtraj_unet_destroy(u); return fail(DTRAJ_ECUDA, "weight upload -> %s", cudaGetErrorString(ce)); }
    float* D = u->dev;
    for (int b = 1; b < 8; ++b) {
        u->blk[b].conv1.w = D + off[b].w1; u->blk[b].conv1.bias = D + off[b].b1;
        if (u->blk[b].has_res) { u->blk[b].res.w = D + off[b].wr; u->blk[b].res.bias = D + off[b].br; }
    }
    for (int b = 0; b < 8; ++b) { u->blk[b].conv2.w = D + off[b].w2; u->blk[b].conv2.bias = D + off[b].b2; }
    u->fw3 = D + o_fw3; u->fb3 = D + o_fb3; u->fw1 = D + o_fw1; u->fb1 = D + o_fb1;
    u->finw = D + o_finw; u->finb = D + o_finb;
    u->table = D + o_table;
    u->err = reinterpret_cast<unsigned int*>(D + o_err);

    // time table on the device
    TimeTableParams tp;
    tp.temb = temb; tp.half = std::max(std::max(temb, 2) / 2, 1);
    tp.freq_scale = (float)(-(std::log(10000.0) / ((double)tp.half - 1.0 + 1e-8)));
    tp.w1 = D + o_tw1; tp.b1 = D + o_tb1; tp.cw0 = D + o_cw0; tp.cb0 = D + o_cb0; tp.cw2 = D + o_cw2; tp.cb2 = D + o_cb2;
    for (int b = 0; b < 8; ++b) { tp.bw[b] = D + o_bw[b]; tp.bb[b] = D + o_bb[b]; tp.bcout[b] = cout[b]; tp.boff[b] = u->tb_off[b]; }
    tp.tb_stride = tbs; tp.table = u->table;
    k_time_table<<<dim3(T, 3), 256, 3 * temb * sizeof(float)>>>(tp);
    ce = cudaGetLastError();
    if (ce == cudaSuccess) ce = cudaDeviceSynchronize();
    if (ce != cudaSuccess) { dtraj_unet_destroy(u); return fail(DTRAJ_ECUDA, "time table kernel -> %s", cudaGetErrorString(ce)); }
    // k_conv_first stages the padded C x (H+2)^2 input and its weights in shared memory.  The attribute belongs to the kernel, not to
    // this model, so it is set to what the largest supported model needs (4 x 64 x 64, 256 channels: 108 KB): a narrower model
    // packed later must not lower it below what an earlier, wider one launches with.
    ce = cudaFuncSetAttribute(k_conv_first, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)first_conv_smem(4, 64, 256));
    if (ce != cudaSuccess) { dtraj_unet_destroy(u); return fail(DTRAJ_ECUDA, "smem attribute (k_conv_first) -> %s", cudaGetErrorString(ce)); }
    if (desc->precision != DTRAJ_PREC_FP32) {
        ce = umma_set_smem_attr();
        if (ce == cudaSuccess) ce = enc1_set_smem_attr();
        if (ce == cudaSuccess) ce = enc1h_set_smem_attr();
        if (ce != cudaSuccess) { dtraj_unet_destroy(u); return fail(DTRAJ_ECUDA, "smem attribute -> %s", cudaGetErrorString(ce)); }
    }
    *out = u;
    return 0;
}

extern "C" int dtraj_unet_time_bias(const dtraj_unet* u, int32_t t, int32_t variant, int32_t block, float* out_host, int32_t n) {
    if (!u || t < 0 || t >= u->d.n_timesteps || variant < 0 || variant > 2 || block < 0 || block > 7 || n > u->blk[block].cout)
        return fail(DTRAJ_EINVAL, "time_bias: bad argument");
    DTRAJ_CUDA(cudaMemcpy(out_host, u->table + (size_t)(t * 3 + variant) * u->tb_stride + u->tb_off[block], sizeof(float) * n,
                          cudaMemcpyDeviceToHost));
    return 0;
}

// ======================================================================================
// forward plan: workspace carving + one launch record per kernel
// ======================================================================================
// Optional per-launch timing (dtraj_sampler_profile): one event pair per launch, summed per class.
enum KernelClass : int { KC_CONV = 0, KC_FIRST = 1, KC_RESAMPLE = 2, KC_STEP = 3, KC_ENC1 = 4, KC_COUNT = 5 };
struct Profiler {
    struct Rec { int cls; cudaEvent_t a, b; const char* name; int step; unsigned grid; double flops; float ms; };
    std::vector<Rec> recs;
    cudaStream_t st = nullptr;
    int step = 0;               // sampler step the launches belong to
    void begin(int cls, const char* name, unsigned grid, double flops) {
        Rec r; r.cls = cls; r.name = name; r.step = step; r.grid = grid; r.flops = flops;
        cudaEventCreate(&r.a); cudaEventCreate(&r.b);
        cudaEventRecord(r.a, st);
        recs.push_back(r);
    }
    void end() { cudaEventRecord(recs.back().b, st); }
};

// One kernel launch of a forward.  plan_build decides the kernel and builds its parameters once; plan_forward writes only
// the per-call inputs (frame, row tables, time-table row) into the fields the kind reads, and launches.
struct Launch {
    enum Kind : int { ENC1H, ENC1, FIRST, CONV_UMMA, CONV_SIMT, POOL, POOL_H, UP, UP_H, UP_H4, FINAL };
    Kind kind;
    KernelClass cls;
    char name[40];              // profiler name
    unsigned grid;              // CTAs (0 for CONV_SIMT: launch_conv_simt chooses its 2-d grid)
    double flops;               // executed tensor-core flops, real channels (KC_CONV, KC_ENC1)
    int tb_block = -1;          // block whose time-bias row this launch reads, -1: none
    Enc1hLaunch enc1h;          // ENC1H
    Enc1Launch enc1;            // ENC1
    FirstConvParams first; size_t first_smem;   // FIRST and its dynamic shared memory
    UmmaLaunch U;               // CONV_UMMA
    ConvLayer L;                // CONV_SIMT
    struct {                    // POOL*, UP*, FINAL: n = the kernel's element count, cv = channel vectors per pixel
        const float* in; float* out; int64_t n; int S, cv, lg_s, lg_cv; int64_t lo_off; int act_mode; Up2Coef cf;
    } rs;
};

// plan_build options (dtraj_test_plan_*; the product always builds with 0)
constexpr int kPlanNoEnc1 = 1;      // k_conv_first + the generic enc1.conv2 (RESX tails) instead of the fused enc1 kernel

struct dtraj_plan {
    const dtraj_unet* u = nullptr;
    int64_t R = 0;
    float* ws = nullptr;
    int options = 0;
    // buffers (float offsets into ws); lo planes follow at +size when act_mode == ACT_SPLIT
    struct Buf { float* p = nullptr; int64_t n = 0; int64_t lo = 0; };
    Buf tmp_h, tmp_r, tmp_x, p1, x2, p2, x3, p3, x4, p4, u3, u2, u1, y1, elow;
    std::vector<Launch> launches;   // one forward, in execution order
};

namespace {

int64_t plan_floats(const dtraj_unet* u, int64_t R, dtraj_plan* P) {
    const int* dp = u->dp;
    const int* S = u->sizes;
    const int C = u->d.channels;
    const bool split = u->act_mode == ACT_SPLIT;
    int64_t off = 0;
    const bool f16 = u->d.precision == DTRAJ_PREC_F16;
    // `act`: a feature map in the model's operand type (halfs in DTRAJ_PREC_F16: half the floats); else fp32
    auto take = [&](dtraj_plan::Buf* b, int64_t per_row, bool lo_plane, bool act = true) {
        int64_t n = round_up64(R * per_row, 256);
        if (P) { b->p = P->ws + off; b->n = n; b->lo = (split && lo_plane) ? n : 0; }
        off += (f16 && act) ? n / 2 : n * ((split && lo_plane) ? 2 : 1);
    };
    auto px = [&](int l) { return (int64_t)S[l] * S[l]; };
    dtraj_plan dummy;
    dtraj_plan* Q = P ? P : &dummy;
    int64_t mh = 0;
    for (int b = 0; b < 8; ++b) {
        const int lv[8] = {0, 1, 2, 3, 4, 3, 2, 1};
        const int co[8] = {dp[0], dp[1], dp[2], dp[3], dp[3], dp[2], dp[1], dp[0]};
        mh = std::max(mh, px(lv[b]) * co[b]);
    }
    take(&Q->tmp_h, mh, true);
    take(&Q->tmp_r, mh, false);
    take(&Q->tmp_x, mh, true);
    take(&Q->p1, px(1) * dp[0], true);
    take(&Q->x2, px(1) * dp[1], true);
    take(&Q->p2, px(2) * dp[1], true);
    take(&Q->x3, px(2) * dp[2], true);
    take(&Q->p3, px(3) * dp[2], true);
    take(&Q->x4, px(3) * dp[3], true);
    take(&Q->p4, px(4) * dp[3], true);
    take(&Q->u3, px(3) * dp[3], true);
    take(&Q->u2, px(2) * dp[2], true);
    take(&Q->u1, px(1) * dp[1], true);
    take(&Q->y1, px(1) * dp[0], false);
    take(&Q->elow, px(1) * C, false, false);
    return off;
}

struct Tail {                // optional fused epilogue tails of one conv
    float* pool_out = nullptr;
    bool resx = false, final1x1 = false, nostore = false;
    // fused residual conv (CONV_RESACC): the block's packed 1x1 weights and its input maps
    const PackedConv* res = nullptr;
    const dtraj_plan::Buf* rs0 = nullptr;
    const dtraj_plan::Buf* rs1 = nullptr;
};

inline unsigned blocks_for(int64_t n, int per) { return (unsigned)((n + per - 1) / per); }

// appends a zeroed launch record to the plan; the caller fills in the kind's parameters
Launch& add_launch(dtraj_plan* P, Launch::Kind kind, KernelClass cls, const char* name, unsigned grid = 0) {
    P->launches.emplace_back();
    Launch& l = P->launches.back();
    l.kind = kind; l.cls = cls; l.grid = grid;
    snprintf(l.name, sizeof(l.name), "%s", name);
    return l;
}

int add_conv(dtraj_plan* P, const char* name, const PackedConv& pc, const dtraj_plan::Buf& s0, const dtraj_plan::Buf* s1, int S,
             const dtraj_plan::Buf& out, const float* resid, int flags, int tb_block, bool is_residual_conv,
             const Tail& tail = Tail()) {
    const dtraj_unet* u = P->u;
    const bool umma = u->d.precision != DTRAJ_PREC_FP32;
    Launch& op = add_launch(P, umma ? Launch::CONV_UMMA : Launch::CONV_SIMT, KC_CONV, "");
    ConvLayer& L = op.L;
    L.src0 = s0.p; L.src0_lo = s0.p + s0.lo; L.c0p = pc.c0p;
    if (s1) { L.src1 = s1->p; L.src1_lo = s1->p + s1->lo; L.c1p = pc.c1p; }
    L.H = S; L.W = S; L.M = P->R * S * S; L.ntaps = pc.ntaps;
    L.wpk = pc.w; L.bias = pc.bias; L.coutp = pc.coutp;
    L.tb_var_stride = u->tb_stride;
    L.resid = resid; L.out = out.p;
    L.lo_off = out.lo;
    L.act_mode = is_residual_conv ? ACT_PLAIN : (u->act_mode == ACT_SPLIT && out.lo == 0 ? ACT_PLAIN : u->act_mode);
    L.flags = flags;
    L.f16 = u->d.precision == DTRAJ_PREC_F16 ? 1 : 0;
    L.err = u->err;
    snprintf(op.name, sizeof(op.name), "%s%s%s%s", name, tail.res ? " +res" : "", tail.pool_out ? " +pool" : "", tail.final1x1 ? " +final" : "");
    if (tail.pool_out) { L.flags |= CONV_POOL; L.pool_out = tail.pool_out; }
    if (tail.nostore) L.flags |= CONV_NOSTORE;
    if (tail.resx) {
        L.flags |= CONV_RESX;
        L.rw1 = u->fw1; L.rb1 = u->fb1; L.xC = u->d.channels;
    }
    if (tail.final1x1) {
        L.flags |= CONV_FINAL;
        L.finw = u->finw; L.finb = u->finb; L.finC = u->d.channels; L.elow = P->elow.p;
    }
    op.tb_block = tb_block;
    op.flops = 2.0 * (double)L.M * pc.cout * (double)(pc.c0 + pc.c1) * pc.ntaps;   // executed taps, real channels
    if (tail.res) {
        L.flags |= CONV_RESACC;
        L.rsrc0 = tail.rs0->p; L.rc0p = tail.res->c0p;
        if (tail.rs1) { L.rsrc1 = tail.rs1->p; L.rc1p = tail.res->c1p; }
        L.rbias = tail.res->bias;
        op.flops += 2.0 * (double)L.M * tail.res->cout * (double)(tail.res->c0 + tail.res->c1);
    }
    if (!umma) return 0;
    DTRAJ_TRY(build_umma_launch(&op.U, L, u->d.precision == DTRAJ_PREC_TF32X3 ? 3 : 1, pc.w, pc.rows,
                                tail.res ? tail.res->w : nullptr, tail.res ? tail.res->rows : 0));
    op.grid = op.U.grid;
    if (op.U.conv.posm) {    // position-major tiles skip the taps outside the map: ((3H - 2) / H)^2 of 9 are executed on average
        const double t_eff = ((3.0 * L.H - 2.0) / L.H) * ((3.0 * L.W - 2.0) / L.W);
        op.flops = 2.0 * (double)L.M * pc.cout * (double)(pc.c0 + pc.c1) * t_eff +
                   (tail.res ? 2.0 * (double)L.M * tail.res->cout * (double)(tail.res->c0 + tail.res->c1) : 0.0);
    }
    return 0;
}

int plan_build(const dtraj_unet* u, int64_t R, void* ws, int64_t ws_bytes, dtraj_plan** out, int options = 0) {
    if (R < 1) return fail(DTRAJ_EINVAL, "n_rows must be >= 1");
    const int64_t need = plan_floats(u, R, nullptr) * 4;
    if (ws_bytes < need) return fail(DTRAJ_ENOMEM, "workspace %lld B < required %lld B", (long long)ws_bytes, (long long)need);
    if (((uintptr_t)ws & 255) != 0) return fail(DTRAJ_EINVAL, "workspace must be 256-byte aligned");
    dtraj_plan* P = new dtraj_plan();
    P->u = u; P->R = R; P->ws = (float*)ws; P->options = options;
    plan_floats(u, R, P);
    const int* S = u->sizes;
    const int* dp = u->dp;
    const int C = u->d.channels;
    int rc = 0;
    const int RT = CONV_RELU | CONV_TBIAS, RR = CONV_RELU | CONV_RESID;
    auto blk = [&](int b) -> const BlockW& { return u->blk[b]; };
    auto conv = [&](auto&&... a) { if (!rc) rc = add_conv(P, a...); };
    // Fused epilogue tails exist in the tcgen05 kernel's bulk path only (single-pass TF32, the mode the
    // sweeps run in); the exact modes keep the stand-alone pool / final / residual kernels.
    const bool f16 = u->d.precision == DTRAJ_PREC_F16;
    const bool fused = f16 || u->d.precision == DTRAJ_PREC_TF32;
    const bool fuse_resx = fused, fuse_final = fused;
    // (maps of at most 4x4 run position-major tiles -- csrc/conv_umma.cuh -- whose rows are images, so a 2x2 pool window is not
    //  inside one tile: those levels keep the stand-alone pool kernel)
    bool fuse_pool[4];           // pool after enc1..enc4
    for (int l = 0; l < 4; ++l) fuse_pool[l] = fused && S[l] <= 16 && !umma_posm_applies(S[l], R);
    // Residual 1x1 convs as extra MMAs of the block's conv2 (CONV_RESACC): no r tensor, no extra launch.  (Measured in round 2
    // with the 1x1 convs of the 256-wide blocks as their own launches + the TMA residual path: conv2 alone gains -- enc2.conv2
    // 673 -> 454 us at 8880 rows, two accumulator stages instead of one -- but the stand-alone K = 128..512 GEMMs cost more than
    // that, 3579 vs 3499 us per teacher forward; profiles/r02b_resacc_ab.txt.)
    bool fuse_res[8] = {};
    for (int b = 1; b < 8; ++b) fuse_res[b] = fused && blk(b).has_res;
    auto with_res = [&](Tail t, int b, const dtraj_plan::Buf* s0, const dtraj_plan::Buf* s1) {
        if (fuse_res[b]) { t.res = &u->blk[b].res; t.rs0 = s0; t.rs1 = s1; }
        return t;
    };
    const dtraj_plan::Buf* pooled[4] = {&P->p1, &P->p2, &P->p3, &P->p4};
    auto tail_for = [&](int enc) {   // conv2 of encoder block `enc` (0..3)
        Tail t;
        if (fuse_pool[enc]) t.pool_out = pooled[enc]->p;
        return t;
    };
    // a stand-alone pool / upsample over n4 4-channel vectors (the fp16 kernels take 8-channel ones)
    auto resample = [&](Launch::Kind kind_h, Launch::Kind kind, const char* name, const dtraj_plan::Buf& in,
                        const dtraj_plan::Buf& o, int64_t n4, int S_in, int cp, int act_mode) {
        Launch& r = add_launch(P, f16 ? kind_h : kind, KC_RESAMPLE, name, blocks_for(f16 ? n4 / 2 : n4, 256));
        r.rs.in = in.p; r.rs.out = o.p; r.rs.n = f16 ? n4 / 2 : n4; r.rs.S = S_in; r.rs.cv = cp / (f16 ? 8 : 4);
        r.rs.lo_off = o.lo; r.rs.act_mode = act_mode;
    };
    // 2x2 max-pool after encoder level `lv`, unless the producing conv's epilogue emits it
    const dtraj_plan::Buf* pool_in[4] = {&P->tmp_x, &P->x2, &P->x3, &P->x4};
    auto pool = [&](int lv) {
        const int So = S[lv + 1];
        if (!fuse_pool[lv])
            resample(Launch::POOL_H, Launch::POOL, "maxpool 2x2", *pool_in[lv], *pooled[lv], R * So * So * (dp[lv] / 4), So, dp[lv],
                     pooled[lv]->lo ? ACT_SPLIT : ACT_PLAIN);
    };
    // bilinear x2 upsample of the map below decoder stage k (0..2) into its first input
    const dtraj_plan::Buf* up[3] = {&P->u3, &P->u2, &P->u1};
    auto upsample = [&](int k) -> int {
        const int Si = S[4 - k], cp = dp[3 - k], cp8 = cp / 8;
        const int64_t n4 = R * (2 * Si) * (2 * Si) * (cp / 4);
        if (n4 >= ((int64_t)1 << 31)) return fail(DTRAJ_EINVAL, "upsample: batch too large for 32-bit indexing");
        const std::string name = "upsample " + std::to_string(Si) + "->" + std::to_string(2 * Si);
        Up2Coef cf;
        if (!(f16 && (cp8 & (cp8 - 1)) == 0 && up2_static_ok(Si, &cf))) {
            resample(Launch::UP_H, Launch::UP, name.c_str(), P->tmp_x, *up[k], n4, Si, cp,
                     (u->act_mode == ACT_SPLIT && !up[k]->lo) ? ACT_PLAIN : u->act_mode);
            return 0;
        }
        const int64_t n_blk = R * Si * Si * cp8;
        Launch& r = add_launch(P, Launch::UP_H4, KC_RESAMPLE, name.c_str(), blocks_for(n_blk, 256));
        r.rs.in = P->tmp_x.p; r.rs.out = up[k]->p; r.rs.n = n_blk; r.rs.S = Si; r.rs.cv = cp8; r.rs.cf = cf;
        while ((1 << r.rs.lg_s) < Si) ++r.rs.lg_s;
        while ((1 << r.rs.lg_cv) < cp8) ++r.rs.lg_cv;
        return 0;
    };
    // enc1: conv1/res by k_conv_first; conv2 here.  x1 itself is never a skip input (models.py:206-216):
    // with the pool fused, only the pooled tile is written.
    bool fuse_enc1 = fused && S[0] % 16 == 0 && C <= 4;   // k_enc1_umma / k_enc1_f16 replace k_conv_first + the enc1.conv2 launch
    if (f16 && dp[0] > 128) fuse_enc1 = false;   // the fp16 fused kernel holds D1 + two accumulators in TMEM: widths up to 128;
                                                 // wider first blocks take k_conv_first + the generic conv2 (RESX + POOL tails)
    if (options & kPlanNoEnc1) fuse_enc1 = false;   // (that path for the narrower first blocks every supported model has)
    auto enc1_fused = [&](Launch& l, auto& E) {   // what the two fused enc1 launches (Enc1hLaunch, Enc1Launch) share
        auto& e = E.p;
        e.w3 = u->fw3; e.b3 = u->fb3; e.rw1 = u->fw1; e.rb1 = u->fb1; e.bias2 = blk(0).conv2.bias;
        e.tb_var_stride = u->tb_stride; e.pool_out = (decltype(e.pool_out))P->p1.p; e.err = u->err;
        l.grid = E.grid; l.flops = E.flops; l.tb_block = 0;
    };
    if (fuse_enc1 && f16) {      // conv2 weights resident in shared memory
        Launch& l = add_launch(P, Launch::ENC1H, KC_ENC1, "enc1 fused (k_enc1_f16)");
        rc = build_enc1h_launch(&l.enc1h, C, S[0], dp[0], blk(0).cout, R, blk(0).conv2.w, blk(0).conv2.rows);
        enc1_fused(l, l.enc1h);
    } else if (fuse_enc1) {      // whole enc1 block + pool in one kernel
        Launch& l = add_launch(P, Launch::ENC1, KC_ENC1, "enc1 fused (k_enc1_umma)");
        rc = build_enc1_launch(&l.enc1, C, S[0], dp[0], blk(0).cout, R, blk(0).conv2.w, blk(0).conv2.rows);
        enc1_fused(l, l.enc1);
        l.enc1.p.act_mode = u->act_mode;
    } else {                     // enc1.conv1 + residual
        Launch& l = add_launch(P, Launch::FIRST, KC_FIRST, "enc1.conv1 + res (k_conv_first)", (unsigned)R);
        FirstConvParams& f = l.first;
        f.C = C; f.H = S[0]; f.W = S[0]; f.coutp = dp[0];
        f.w3 = u->fw3; f.b3 = u->fb3; f.w1 = u->fw1; f.b1 = u->fb1; f.tb_var_stride = u->tb_stride;
        f.h = P->tmp_h.p; f.r = fuse_resx ? nullptr : P->tmp_r.p; f.lo_off = P->tmp_h.lo;
        f.f16 = f16 ? 1 : 0; f.act_mode = f16 ? ACT_PLAIN : u->act_mode;
        l.first_smem = first_conv_smem(C, S[0], dp[0]);
        l.tb_block = 0;
        Tail t = tail_for(0);
        t.resx = fuse_resx;
        t.nostore = fuse_pool[0];
        conv("enc1.conv2", blk(0).conv2, P->tmp_h, nullptr, S[0], P->tmp_x, t.resx ? nullptr : P->tmp_r.p, t.resx ? CONV_RELU : RR, -1, false, t);
        pool(0);
    }
    // enc2 @ level 1
    if (!blk(1).has_res) rc = fail(DTRAJ_EINVAL, "enc2 without residual_conv unsupported");
    {
        const bool fr = fuse_res[1];
        if (!fr) conv("enc2.res", blk(1).res, P->p1, nullptr, S[1], P->tmp_r, nullptr, 0, -1, true);
        conv("enc2.conv1", blk(1).conv1, P->p1, nullptr, S[1], P->tmp_h, nullptr, RT, 1, false);
        conv("enc2.conv2", blk(1).conv2, P->tmp_h, nullptr, S[1], P->x2, fr ? nullptr : P->tmp_r.p, fr ? CONV_RELU : RR, -1, false,
             with_res(tail_for(1), 1, &P->p1, nullptr));
        pool(1);
    }
    // enc3, enc4, bottleneck @ levels 2..4 (identity residual = the pooled input, unless the widths differ)
    const dtraj_plan::Buf* pin[3] = {&P->p2, &P->p3, &P->p4};
    const dtraj_plan::Buf* xo[3] = {&P->x3, &P->x4, &P->tmp_x};
    for (int k = 0; k < 3 && !rc; ++k) {
        const int b = 2 + k, lv = 2 + k;
        const float* resid = pin[k]->p;
        const bool fused_here = fuse_res[b];
        const std::string bn = kBlockNames[b];
        if (blk(b).has_res && !fused_here) { conv((bn + ".res").c_str(), blk(b).res, *pin[k], nullptr, S[lv], P->tmp_r, nullptr, 0, -1, true); resid = P->tmp_r.p; }
        conv((bn + ".conv1").c_str(), blk(b).conv1, *pin[k], nullptr, S[lv], P->tmp_h, nullptr, RT, b, false);
        conv((bn + ".conv2").c_str(), blk(b).conv2, P->tmp_h, nullptr, S[lv], *xo[k], fused_here ? nullptr : resid, fused_here ? CONV_RELU : RR, -1, false,
             with_res(k < 2 ? tail_for(2 + k) : Tail(), b, pin[k], nullptr));
        if (k < 2) pool(2 + k);
    }
    // decoders: [upsampled | skip]
    const dtraj_plan::Buf* skip[3] = {&P->x4, &P->x3, &P->x2};
    const dtraj_plan::Buf* yo[3] = {&P->tmp_x, &P->tmp_x, &P->y1};
    for (int k = 0; k < 3 && !rc; ++k) {
        const int b = 5 + k, lv = 3 - k;
        if (!blk(b).has_res) { rc = fail(DTRAJ_EINVAL, "%s without residual_conv unsupported", kBlockNames[b]); break; }
        const std::string bn = kBlockNames[b];
        const bool fr = fuse_res[b];
        rc = upsample(k);
        if (!fr) conv((bn + ".res").c_str(), blk(b).res, *up[k], skip[k], S[lv], P->tmp_r, nullptr, 0, -1, true);
        conv((bn + ".conv1").c_str(), blk(b).conv1, *up[k], skip[k], S[lv], P->tmp_h, nullptr, RT, b, false);
        Tail t;
        if (k == 2 && fuse_final) { t.final1x1 = true; t.nostore = true; }   // y1 only feeds the final 1x1
        conv((bn + ".conv2").c_str(), blk(b).conv2, P->tmp_h, nullptr, S[lv], *yo[k], fr ? nullptr : P->tmp_r.p, fr ? CONV_RELU : RR, -1, false,
             with_res(t, b, up[k], skip[k]));
    }
    if (!fuse_final) {   // final 1x1 at half resolution (else: dec1.conv2's epilogue)
        const int64_t npix = R * S[1] * S[1];
        Launch& r = add_launch(P, Launch::FINAL, KC_RESAMPLE, "final 1x1", blocks_for(npix * 32, 256));
        r.rs.in = P->y1.p; r.rs.out = P->elow.p; r.rs.n = npix; r.rs.cv = dp[0];
    }
    if (rc) { delete P; return rc; }
    *out = P;
    return 0;
}

// Writes the per-call inputs into the fields launch `l` reads and launches it.  `tbias`: the time-table row of this call's
// t at the record's block (null when it reads none).
int launch_record(Launch& l, const dtraj_unet* u, const float* x, int64_t x_stride, const int32_t* row_sample,
                  const int32_t* row_variant, const float* tbias, bool per_row, cudaStream_t st) {
    const auto& r = l.rs;
    auto enc1_inputs = [&](auto& p) {   // Enc1hParams, Enc1Params, FirstConvParams
        p.x = x; p.x_stride = x_stride; p.row_sample = row_sample; p.row_variant = row_variant; p.tbias = tbias;
    };
    switch (l.kind) {
    case Launch::ENC1H: enc1_inputs(l.enc1h.p); l.enc1h.p.tb_rows = per_row ? 1 : 0; return launch_enc1h(l.enc1h, st);
    case Launch::ENC1: enc1_inputs(l.enc1.p); return launch_enc1(l.enc1, st);
    case Launch::FIRST: enc1_inputs(l.first); k_conv_first<<<l.grid, 256, l.first_smem, st>>>(l.first); break;
    case Launch::CONV_UMMA: {
        ConvLayer& L = l.U.conv.L;
        L.tbias = tbias; L.row_variant = row_variant; L.tb_rows = per_row ? 1 : 0;
        if (L.flags & CONV_RESX) { L.xraw = x; L.x_stride = x_stride; L.row_sample = row_sample; }
        return launch_conv_umma(l.U, st);
    }
    case Launch::CONV_SIMT: l.L.tbias = tbias; l.L.row_variant = row_variant; return launch_conv_simt(l.L, st);
    case Launch::POOL: k_pool2<<<l.grid, 256, 0, st>>>(r.in, r.out, r.n, r.S, r.S, r.cv, r.lo_off, r.act_mode); break;
    case Launch::POOL_H: k_pool2_h<<<l.grid, 256, 0, st>>>((const __half*)r.in, (__half*)r.out, r.n, r.S, r.S, r.cv); break;
    case Launch::UP: k_upsample2<<<l.grid, 256, 0, st>>>(r.in, r.out, r.n, r.S, r.S, r.cv, r.lo_off, r.act_mode); break;
    case Launch::UP_H:
        DTRAJ_CUDA(launch_ex(k_upsample2_h, l.grid, 256, 0, st, 1, true, (const __half*)r.in, (__half*)r.out, r.n, r.S, r.S, r.cv));
        break;
    case Launch::UP_H4:
        DTRAJ_CUDA(launch_ex(k_upsample2_h4, l.grid, 256, 0, st, 1, true, (const __half*)r.in, (__half*)r.out, (uint32_t)r.n, r.S,
                             r.lg_s, r.cv, r.lg_cv, r.cf));
        break;
    case Launch::FINAL: k_final1x1<<<l.grid, 256, 0, st>>>(r.in, u->finw, u->finb, r.out, r.n, r.cv, u->d.channels); break;
    }
    DTRAJ_LAUNCH_CHECK();
    return 0;
}

// Enqueue one U-Net forward (models.py:159-224 up to the half-resolution eps map), or its launches [first, last) (test hook).
// `per_row`: row_variant holds t_i * 3 + variant_i (a row of the whole table) instead of the variant alone, `t` is 0.
int plan_forward(dtraj_plan* P, const float* x, int64_t x_stride, const int32_t* row_sample, const int32_t* row_variant, int t,
                 bool per_row, cudaStream_t st, Profiler* prof = nullptr, size_t first = 0, size_t last = SIZE_MAX) {
    const dtraj_unet* u = P->u;
    if (t < 0 || t >= u->d.n_timesteps) return fail(DTRAJ_EINVAL, "timestep %d outside the time table (0..%d)", t, u->d.n_timesteps - 1);
    const float* trow = u->table + (size_t)t * 3 * u->tb_stride;
    for (size_t i = first; i < std::min(last, P->launches.size()); ++i) {
        Launch& l = P->launches[i];
        const float* tb = l.tb_block >= 0 ? trow + u->tb_off[l.tb_block] : nullptr;
        if (prof) prof->begin(l.cls, l.name, l.grid, l.flops);
        const int rc = launch_record(l, u, x, x_stride, row_sample, row_variant, tb, per_row, st);
        if (prof) prof->end();
        DTRAJ_TRY(rc);
    }
    return 0;
}

// the handle's cached plan for this batch, workspace and option set, (re)built when one of them changes
int cached_plan(dtraj_unet* u, int64_t n_rows, void* workspace, int64_t workspace_bytes, int options) {
    if (!u->plan || u->plan->R != n_rows || u->plan->ws != (float*)workspace || u->plan->options != options) {
        if (u->plan) { delete u->plan; u->plan = nullptr; }
        DTRAJ_TRY(plan_build(u, n_rows, workspace, workspace_bytes, &u->plan, options));
    }
    return 0;
}

// dtraj_unet_forward*: (re)build the handle's cached plan for this batch and workspace, run it, expand eps to full resolution
int unet_forward(dtraj_unet* u, const float* x, int64_t n_rows, int t, const int32_t* row_variant, bool per_row, float* eps,
                 void* workspace, int64_t workspace_bytes, cudaStream_t st) {
    DTRAJ_TRY(cached_plan(u, n_rows, workspace, workspace_bytes, 0));
    const int C = u->d.channels, H = u->d.image_size;
    DTRAJ_TRY(plan_forward(u->plan, x, (int64_t)C * H * H, nullptr, row_variant, t, per_row, st));
    const int64_t n = n_rows * C * H * H;
    k_eps_out<<<blocks_for(n, 256), 256, 0, st>>>(u->plan->elow.p, eps, n, C, H, H);
    DTRAJ_LAUNCH_CHECK();
    return 0;
}

}  // namespace

extern "C" int64_t dtraj_unet_workspace_bytes(const dtraj_unet* u, int64_t n_rows) {
    if (!u || n_rows < 1) return -1;
    return plan_floats(u, n_rows, nullptr) * 4;
}

extern "C" int dtraj_unet_destroy(dtraj_unet* u) {
    if (!u) return 0;
    if (u->plan) delete u->plan;
    if (u->dev) cudaFree(u->dev);
    delete u;
    return 0;
}

extern "C" int dtraj_unet_forward(dtraj_unet* u, const float* x, int64_t n_rows, int32_t t, const int32_t* row_variant,
                                  float* eps, void* workspace, int64_t workspace_bytes, void* stream) {
    if (!u || !x || !eps || !workspace) return fail(DTRAJ_EINVAL, "null argument");
    return unet_forward(u, x, n_rows, t, row_variant, false, eps, workspace, workspace_bytes, (cudaStream_t)stream);
}

extern "C" int dtraj_unet_forward_rows(dtraj_unet* u, const float* x, int64_t n_rows, const int32_t* row_tv, float* eps,
                                       void* workspace, int64_t workspace_bytes, void* stream) {
    if (!u || !x || !eps || !workspace || !row_tv) return fail(DTRAJ_EINVAL, "null argument");
    return unet_forward(u, x, n_rows, 0, row_tv, true, eps, workspace, workspace_bytes, (cudaStream_t)stream);
}

extern "C" int dtraj_step_fused(int32_t rule, const float* k, const float* eps_u, const float* eps_c, const float* w,
                                const float* x, int64_t x_stride, const float* z, int64_t z_stride, float* x_out,
                                int64_t out_stride, int64_t n_samples, int64_t D, void* stream) {
    if (rule < 1 || rule > 3 || !k || !eps_u || !x || !x_out) return fail(DTRAJ_EINVAL, "step: bad argument");
    if (eps_c && !w) return fail(DTRAJ_EINVAL, "step: eps_c given without guidance weights");
    if (n_samples * D == 0) return 0;
    k_step_plain<<<blocks_for(n_samples * D, 256), 256, 0, (cudaStream_t)stream>>>(rule, k[0], k[1], k[2], eps_u, eps_c, w, x,
                                                                                    x_stride, z, z_stride, x_out, out_stride,
                                                                                    n_samples, D);
    DTRAJ_LAUNCH_CHECK();
    return 0;
}

// ======================================================================================
// sampler: n_updates x { forward, fused step } (+ duplicate frame), optionally one CUDA graph
// ======================================================================================
struct dtraj_sampler {
    dtraj_unet* u = nullptr;
    dtraj_sampler_desc d;
    std::vector<int32_t> ts;
    std::vector<float> coef;
    dtraj_plan* plan = nullptr;
    dtraj_plan* plan0 = nullptr;    // first step with shared rows (desc.n_rows0 > 0); same workspace
    cudaGraph_t graph = nullptr;
    cudaGraphExec_t exec = nullptr;
};

namespace {

// a per-forward quantity of the plans summed over the loop: step 0 runs the shared-row plan when there is one
template <class F> auto per_loop(const dtraj_sampler* s, F per_forward) -> decltype(per_forward(s->plan)) {
    const int nu = s->d.n_updates;
    return nu > 0 ? per_forward(s->plan0 ? s->plan0 : s->plan) + per_forward(s->plan) * (nu - 1) : 0;
}

int sampler_enqueue(dtraj_sampler* s, cudaStream_t st, Profiler* prof = nullptr) {
    const dtraj_sampler_desc& d = s->d;
    const int C = s->u->d.channels, H = s->u->d.image_size;
    const int64_t D = (int64_t)C * H * H, fs = (int64_t)d.n_frames * D;
    for (int k = 0; k < d.n_updates; ++k) {
        if (prof) prof->step = k;
        const float* xin = d.traj + (int64_t)k * D;
        const bool first = k == 0 && s->plan0 != nullptr;            // shared rows: every sample of a group still has x_T
        dtraj_plan* P = first ? s->plan0 : s->plan;
        DTRAJ_TRY(plan_forward(P, xin, fs, first ? d.row_sample0 : d.row_sample, first ? d.row_variant0 : d.row_variant,
                               s->ts[k], false, st, prof));
        StepParams p;
        p.rule = d.rule; p.k0 = s->coef[3 * k]; p.k1 = s->coef[3 * k + 1]; p.k2 = s->coef[3 * k + 2];
        p.elow = P->elow.p; p.sample_row_u = first ? d.sample_row_u0 : d.sample_row_u;
        p.sample_row_c = first ? d.sample_row_c0 : d.sample_row_c;
        p.guidance = d.guidance; p.z_bank = d.z_bank;
        p.z_index = d.z_index ? d.z_index + (int64_t)k * d.n_samples : nullptr;
        p.x_in = xin; p.x_out = d.traj + (int64_t)(k + 1) * D; p.frame_stride = fs;
        p.B = d.n_samples; p.C = C; p.H = H; p.W = H;
        const unsigned grid = blocks_for((int64_t)d.n_samples * C * H * (H / 4), 256);
        if (prof) prof->begin(KC_STEP, "k_step (CFG + update + store)", grid, 0.0);
        DTRAJ_CUDA(launch_ex(k_step, grid, 256, 0, st, 1, s->u->d.precision == DTRAJ_PREC_F16, p));
        if (prof) prof->end();
        DTRAJ_LAUNCH_CHECK();
    }
    if (d.copy_last) {
        const int64_t k = d.n_updates;
        const unsigned grid = blocks_for((int64_t)d.n_samples * (D / 4), 256);
        if (prof) prof->begin(KC_STEP, "k_copy_frame", grid, 0.0);
        DTRAJ_CUDA(launch_ex(k_copy_frame, grid, 256, 0, st, 1, s->u->d.precision == DTRAJ_PREC_F16, (const float*)(d.traj + k * D),
                             d.traj + (k + 1) * D, fs, d.n_samples, (int)(D / 4)));
        if (prof) prof->end();
        DTRAJ_LAUNCH_CHECK();
    }
    return 0;
}

}  // namespace

extern "C" int dtraj_sampler_destroy(dtraj_sampler* s) {
    if (!s) return 0;
    if (s->exec) cudaGraphExecDestroy(s->exec);
    if (s->graph) cudaGraphDestroy(s->graph);
    if (s->plan) delete s->plan;
    if (s->plan0) delete s->plan0;
    delete s;
    return 0;
}

extern "C" int dtraj_sampler_create(dtraj_unet* u, const dtraj_sampler_desc* d, dtraj_sampler** out) {
    if (!u || !d || !out) return fail(DTRAJ_EINVAL, "null argument");
    if (d->rule < 1 || d->rule > 3) return fail(DTRAJ_EINVAL, "bad rule %d", d->rule);
    if (d->n_samples < 1 || d->n_rows < d->n_samples || d->n_rows > 2 * d->n_samples) return fail(DTRAJ_EINVAL, "bad n_samples/n_rows");
    if (d->n_updates < 0 || d->n_frames != 1 + d->n_updates + (d->copy_last ? 1 : 0)) return fail(DTRAJ_EINVAL, "n_frames != 1 + n_updates + copy_last");
    if (!d->traj || !d->workspace || !d->row_sample || !d->row_variant || !d->sample_row_u) return fail(DTRAJ_EINVAL, "null device array");
    if (d->n_updates && (!d->step_timestep || !d->step_coef)) return fail(DTRAJ_EINVAL, "null step tables");
    if (d->sample_row_c && !d->guidance) return fail(DTRAJ_EINVAL, "sample_row_c given without guidance");
    if (d->z_index && !d->z_bank) return fail(DTRAJ_EINVAL, "z_index given without z_bank");
    dtraj_sampler* s = new dtraj_sampler();
    s->u = u; s->d = *d;
    s->ts.assign(d->step_timestep, d->step_timestep + d->n_updates);
    s->coef.assign(d->step_coef, d->step_coef + 3 * (size_t)d->n_updates);
    s->d.step_timestep = nullptr; s->d.step_coef = nullptr;
    for (int k = 0; k < d->n_updates; ++k)
        if (s->ts[k] < 0 || s->ts[k] >= u->d.n_timesteps) {
            int t = s->ts[k];
            delete s;
            return fail(DTRAJ_EINVAL, "step %d: timestep %d outside the time table", k, t);
        }
    int rc = plan_build(u, d->n_rows, d->workspace, d->workspace_bytes, &s->plan);
    if (rc) { delete s; return rc; }
    if (d->n_rows0 > 0) {
        if (d->n_rows0 > d->n_rows || !d->row_sample0 || !d->row_variant0 || !d->sample_row_u0 || (d->sample_row_c && !d->sample_row_c0)) {
            dtraj_sampler_destroy(s);
            return fail(DTRAJ_EINVAL, "bad first-step row layout");
        }
        rc = plan_build(u, d->n_rows0, d->workspace, d->workspace_bytes, &s->plan0);
        if (rc) { dtraj_sampler_destroy(s); return rc; }
    }
    if (d->use_graph) {
        cudaStream_t cs;
        cudaError_t ce = cudaStreamCreateWithFlags(&cs, cudaStreamNonBlocking);
        if (ce != cudaSuccess) { dtraj_sampler_destroy(s); return fail(DTRAJ_ECUDA, "stream create -> %s", cudaGetErrorString(ce)); }
        ce = cudaStreamBeginCapture(cs, cudaStreamCaptureModeThreadLocal);
        if (ce == cudaSuccess) {
            rc = sampler_enqueue(s, cs);
            cudaError_t ce2 = cudaStreamEndCapture(cs, &s->graph);
            if (rc == 0 && ce2 != cudaSuccess) rc = fail(DTRAJ_ECUDA, "graph capture -> %s", cudaGetErrorString(ce2));
            if (rc == 0) {
                ce2 = cudaGraphInstantiate(&s->exec, s->graph, 0);
                if (ce2 != cudaSuccess) rc = fail(DTRAJ_ECUDA, "graph instantiate -> %s", cudaGetErrorString(ce2));
            }
        } else rc = fail(DTRAJ_ECUDA, "begin capture -> %s", cudaGetErrorString(ce));
        cudaStreamDestroy(cs);
        if (rc) { dtraj_sampler_destroy(s); return rc; }
    }
    *out = s;
    return 0;
}

extern "C" int dtraj_sampler_run(dtraj_sampler* s, void* stream) {
    if (!s) return fail(DTRAJ_EINVAL, "null sampler");
    cudaStream_t st = (cudaStream_t)stream;
    if (s->exec) { DTRAJ_CUDA(cudaGraphLaunch(s->exec, st)); return 0; }
    return sampler_enqueue(s, st);
}

// per update one forward and one k_step, then the frame copy
extern "C" int64_t dtraj_sampler_launches(const dtraj_sampler* s) {
    if (!s) return -1;
    return per_loop(s, [](const dtraj_plan* P) { return (int64_t)P->launches.size(); }) + s->d.n_updates + (s->d.copy_last ? 1 : 0);
}

namespace {

// executed conv flops of a whole loop (real channels, evaluated taps): [0] generic convs, [1] the fused enc1 kernel's conv2
void sampler_flops(const dtraj_sampler* s, double* out2) {
    auto flops_of = [&](int cls) {
        return per_loop(s, [cls](const dtraj_plan* P) {
            double f = 0.0;
            for (const Launch& l : P->launches)
                if (l.cls == cls) f += l.flops;
            return f;
        });
    };
    out2[0] = flops_of(KC_CONV);
    out2[1] = flops_of(KC_ENC1);
}

// Runs the loop once, un-captured, with an event pair around every launch on `st`; appends the records of the launches
// that completed, with their device milliseconds, to `out`.  Synchronises the stream.
int profile_run(dtraj_sampler* s, cudaStream_t st, std::vector<Profiler::Rec>* out) {
    Profiler prof;
    prof.st = st;
    const int rc = sampler_enqueue(s, st, &prof);
    const cudaError_t ce = cudaStreamSynchronize(st);
    for (Profiler::Rec& r : prof.recs) {
        if (rc == 0 && ce == cudaSuccess && cudaEventElapsedTime(&r.ms, r.a, r.b) == cudaSuccess) out->push_back(r);
        cudaEventDestroy(r.a); cudaEventDestroy(r.b);
    }
    if (rc) return rc;
    if (ce != cudaSuccess) return fail(DTRAJ_ECUDA, "profile -> %s", cudaGetErrorString(ce));
    return 0;
}

}  // namespace

extern "C" int dtraj_sampler_flops(const dtraj_sampler* s, double* conv_flops2) {
    if (!s || !conv_flops2) return fail(DTRAJ_EINVAL, "sampler_flops: null argument");
    sampler_flops(s, conv_flops2);
    return 0;
}

extern "C" int dtraj_sampler_profile(dtraj_sampler* s, void* stream, double* class_ms, int64_t* class_launches, double* conv_flops) {
    if (!s || !class_ms || !class_launches || !conv_flops) return fail(DTRAJ_EINVAL, "profile: null argument");
    std::vector<Profiler::Rec> recs;
    const int rc = profile_run(s, (cudaStream_t)stream, &recs);
    for (int c = 0; c < KC_COUNT; ++c) { class_ms[c] = 0.0; class_launches[c] = 0; }
    for (const Profiler::Rec& r : recs) { class_ms[r.cls] += r.ms; class_launches[r.cls] += 1; }
    sampler_flops(s, conv_flops);
    return rc;
}

extern "C" int dtraj_sampler_profile_text(dtraj_sampler* s, void* stream, int32_t step, char* buf, int64_t buf_len) {
    if (!s || !buf || buf_len < 64) return fail(DTRAJ_EINVAL, "profile_text: bad argument");
    if (step < 0 || step >= s->d.n_updates) return fail(DTRAJ_EINVAL, "profile_text: step %d outside 0..%d", step, s->d.n_updates - 1);
    std::vector<Profiler::Rec> recs;
    const int rc = profile_run(s, (cudaStream_t)stream, &recs);
    int64_t off = 0;
    buf[0] = 0;
    for (const Profiler::Rec& r : recs)
        if (r.step == step && off + 128 < buf_len)
            off += snprintf(buf + off, (size_t)(buf_len - off), "%s\t%u\t%.2f\t%.6g\n", r.name, r.grid, r.ms * 1e3, r.flops);
    return rc;
}

// ======================================================================================
// metrics
// ======================================================================================
extern "C" int dtraj_metrics_pairs(const float* teacher, const float* student, int64_t N, int32_t L, int32_t D, float* out, void* stream) {
    if (N == 0) return 0;
    if (!teacher || !student || !out || N < 0) return fail(DTRAJ_EINVAL, "metrics: bad argument");
    return launch_metrics_pairs(teacher, student, N, L, D, out, (cudaStream_t)stream);
}

extern "C" int dtraj_wasserstein(const float* teacher, const float* student, int64_t N, int32_t L, int32_t D, const int32_t* idx,
                                 const int32_t* idx_set, int32_t K, float* out, void* stream) {
    if (N == 0) return 0;
    if (!teacher || !student || !out || N < 0 || L < 1) return fail(DTRAJ_EINVAL, "wasserstein: bad argument");
    return launch_wasserstein(teacher, student, N, L, L, D, idx, idx_set, K, out, (cudaStream_t)stream);
}

extern "C" int dtraj_metrics_pairs_ragged(const float* teacher, const float* student, int64_t N, int32_t LT, int32_t LS, int32_t D,
                                          const int32_t* rs_pos, const float* rs_frac, float* out, void* stream) {
    if (N == 0) return 0;
    if (!teacher || !student || !rs_pos || !rs_frac || !out || N < 0) return fail(DTRAJ_EINVAL, "metrics_ragged: bad argument");
    return launch_metrics_pairs_ragged(teacher, student, N, LT, LS, D, rs_pos, rs_frac, out, (cudaStream_t)stream);
}

extern "C" int dtraj_wasserstein_ragged(const float* teacher, const float* student, int64_t N, int32_t LT, int32_t LS, int32_t D,
                                        const int32_t* idx, const int32_t* idx_set, int32_t K, float* out, void* stream) {
    if (N == 0) return 0;
    if (!teacher || !student || !out || N < 0) return fail(DTRAJ_EINVAL, "wasserstein_ragged: bad argument");
    return launch_wasserstein(teacher, student, N, LT, LS, D, idx, idx_set, K, out, (cudaStream_t)stream);
}

extern "C" int dtraj_numpy_choice_sets(const uint32_t* seeds, int32_t n_seeds, int32_t L, int32_t D, int32_t K, int32_t* out, void* stream) {
    if (n_seeds == 0) return 0;
    if (!seeds || !out) return fail(DTRAJ_EINVAL, "numpy_choice_sets: null argument");
    return launch_numpy_choice(seeds, n_seeds, L, D, K, out, (cudaStream_t)stream);
}

extern "C" int dtraj_project(const float* frames, int64_t n_frames, int32_t D, const float* comps, const float* offset, int32_t K,
                             float* out, void* stream) {
    if (n_frames == 0) return 0;
    if (!frames || !comps || !offset || !out || n_frames < 0) return fail(DTRAJ_EINVAL, "project: bad argument");
    return launch_project(frames, n_frames, D, comps, offset, K, out, (cudaStream_t)stream);
}

// ======================================================================================
// test hooks
// ======================================================================================
namespace {
int report_error_word(unsigned int v) {
    if (!v) return 0;
    if (v & 1u) return fail(DTRAJ_ECUDA, "a tcgen05 pipeline role timed out on an mbarrier: results are invalid");
    return fail(DTRAJ_ERANGE, "fp16 mode: an activation left the fp16 range (|v| > 65504): rerun with precision 'tf32'");
}
}  // namespace

extern "C" int dtraj_check_errors(void) {
    unsigned int v = 0;
    DTRAJ_CUDA(cudaMemcpyFromSymbol(&v, g_umma_error, sizeof(v)));
    if (!v) return 0;
    const unsigned int z = 0;
    DTRAJ_CUDA(cudaMemcpyToSymbol(g_umma_error, &z, sizeof(z)));
    return report_error_word(v);
}

extern "C" int dtraj_unet_check_errors(dtraj_unet* u) {
    if (!u) return fail(DTRAJ_EINVAL, "unet_check_errors: null handle");
    unsigned int v = 0;
    DTRAJ_CUDA(cudaMemcpy(&v, u->err, sizeof(v), cudaMemcpyDeviceToHost));
    if (!v) return 0;
    DTRAJ_CUDA(cudaMemset(u->err, 0, sizeof(v)));
    return report_error_word(v);
}

extern "C" int dtraj_unet_error_flag_async(dtraj_unet* u, uint32_t* host_flag, void* stream) {
    if (!u || !host_flag) return fail(DTRAJ_EINVAL, "unet_error_flag_async: null argument");
    DTRAJ_CUDA(cudaMemcpyAsync(host_flag, u->err, sizeof(uint32_t), cudaMemcpyDeviceToHost, (cudaStream_t)stream));
    return 0;
}

extern "C" int dtraj_error_flag_async(uint32_t* host_flag, void* stream) {
    if (!host_flag) return fail(DTRAJ_EINVAL, "error_flag_async: null destination");
    void* sym = nullptr;
    DTRAJ_CUDA(cudaGetSymbolAddress(&sym, g_umma_error));
    DTRAJ_CUDA(cudaMemcpyAsync(host_flag, sym, sizeof(uint32_t), cudaMemcpyDeviceToHost, (cudaStream_t)stream));
    return 0;
}

#ifdef DTRAJ_PROBES
// hardware probe, see probe.cuh; out_host[128] = row id fetched for each of the 128 output rows
extern "C" int dtraj_probe_umma_view(int32_t rows, int32_t start_row, int32_t sbo_bytes, int32_t base_off_mode, float* out_host) {
    float* d = nullptr;
    DTRAJ_CUDA(cudaMalloc(&d, 128 * sizeof(float)));
    cudaFuncSetAttribute(k_probe_view, cudaFuncAttributeMaxDynamicSharedMemorySize, 40 * 1024);
    k_probe_view<<<1, 128, 36 * 1024>>>(rows, start_row, sbo_bytes, base_off_mode, d);
    cudaError_t ce = cudaDeviceSynchronize();
    if (ce == cudaSuccess) ce = cudaMemcpy(out_host, d, 128 * sizeof(float), cudaMemcpyDeviceToHost);
    cudaFree(d);
    if (ce != cudaSuccess) return fail(DTRAJ_ECUDA, "probe -> %s", cudaGetErrorString(ce));
    return 0;
}

// hardware probe, see probe.cuh: [n_img][8][8][64] fp16 map with element (n, y, x, c) = n*64 + y*8 + x + 1, loaded through a
// tensor map over {c, x, image, y}; out_host[200] = first channel of every shared-memory row of the box at image `img0`
extern "C" int dtraj_probe_tma_permuted(int32_t n_img, int32_t img0, float* out_host) {
    PFN_encodeTiled enc = get_encode_tiled();
    if (!enc) return fail(DTRAJ_ECUDA, "cuTensorMapEncodeTiled not available");
    std::vector<__half> h((size_t)n_img * 64 * 64);
    for (int n = 0; n < n_img; ++n)
        for (int p = 0; p < 64; ++p)
            for (int c = 0; c < 64; ++c) h[((size_t)n * 64 + p) * 64 + c] = __float2half_rn((float)(n * 64 + p + 1));
    __half* d = nullptr; float* o = nullptr;
    DTRAJ_CUDA(cudaMalloc(&d, h.size() * 2));
    DTRAJ_CUDA(cudaMalloc(&o, 200 * sizeof(float)));
    DTRAJ_CUDA(cudaMemcpy(d, h.data(), h.size() * 2, cudaMemcpyHostToDevice));
    CUtensorMap m;
    cuuint64_t dims[4] = {64, 8, (cuuint64_t)n_img, 8};                       // c, x, image, y
    cuuint64_t strides[3] = {64 * 2, 64 * 64 * 2, 8 * 64 * 2};                  // x, image, y  (bytes): NOT increasing
    cuuint32_t box[4] = {64, 10, 2, 10};
    cuuint32_t es[4] = {1, 1, 1, 1};
    CUresult r = enc(&m, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 4, (void*)d, dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                     CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { cudaFree(d); cudaFree(o); return fail(DTRAJ_ECUDA, "cuTensorMapEncodeTiled(permuted dims) -> %d", (int)r); }
    cudaFuncSetAttribute(k_probe_tma_perm, cudaFuncAttributeMaxDynamicSharedMemorySize, 32 * 1024);
    k_probe_tma_perm<<<1, 128, 28 * 1024>>>(m, img0, o);
    cudaError_t ce = cudaDeviceSynchronize();
    if (ce == cudaSuccess) ce = cudaMemcpy(out_host, o, 200 * sizeof(float), cudaMemcpyDeviceToHost);
    cudaFree(d); cudaFree(o);
    if (ce != cudaSuccess) return fail(DTRAJ_ECUDA, "tma permuted probe -> %s", cudaGetErrorString(ce));
    return 0;
}

// tools/timeline.py: which layer k_conv_umma_t records: (flags & mask) == value, coutp, W
extern "C" int dtraj_probe_timeline_select(int mask, int value, int coutp, int W) {
    const int sel[4] = {mask, value, coutp, W};
    DTRAJ_CUDA(cudaMemcpyToSymbol(g_tl_select, sel, sizeof(sel)));
    return 0;
}
// tools/timeline.py: copy out (and clear) the SM-clock stamps k_conv_umma_t leaves in a probe build
extern "C" int dtraj_probe_timeline(long long* host_out, int64_t n) {
    if (n != (int64_t)(sizeof(g_timeline) / sizeof(long long))) return fail(DTRAJ_EINVAL, "probe_timeline: expected %zu values", sizeof(g_timeline) / sizeof(long long));
    DTRAJ_CUDA(cudaDeviceSynchronize());
    DTRAJ_CUDA(cudaMemcpyFromSymbol(host_out, g_timeline, sizeof(g_timeline)));
    return 0;
}
#endif  // DTRAJ_PROBES

extern "C" unsigned int dtraj_debug_umma_error(void) {
    unsigned int v = 0;
    cudaMemcpyFromSymbol(&v, g_umma_error, sizeof(v));
    return v;
}

// Kernel-only timing of one conv layer shape (tools/conv_bench.py, tools/bench_image64.py): device buffers are allocated and
// zero-filled here, `iters` launches are timed with one event pair.  `debug`: 0 = the form and shared-memory split the forward plan
// uses, 2 = the generic [image][y][x] tiles where that form is a halo form, 0x100 | n_hb << 4 | epi_bufs = the halo form with that
// shared-memory split (A/B experiments); other values are refused.  flags & CONV_RESACC: x1 (c1 channels) feeds a fused 1x1
// residual conv instead of the main conv's K loop.
extern "C" int dtraj_bench_conv(int32_t precision, int32_t c0, int32_t c1, int32_t cout, int64_t n, int32_t H, int32_t ksize,
                                int32_t flags, int32_t iters, int32_t debug, float* ms_out) {
    if (debug != 0 && debug != 2 && !(debug & kUmmaSplit))
        return fail(DTRAJ_EINVAL, "bench_conv: the operand knock-out experiments (profiles/r01f_conv_knockout.txt) were removed from the kernels");
    const bool resacc = (flags & CONV_RESACC) != 0;
    const int cpad = kCPad;
    const int c0p = round_up(c0, cpad), c1p = c1 ? round_up(c1, cpad) : 0, coutp = round_up(cout, cpad);
    const int64_t M = n * H * H;
    const int cm1 = resacc ? 0 : c1;                  // second source of the main conv
    std::vector<float> w((size_t)cout * (c0 + cm1) * ksize * ksize, 0.01f), wr((size_t)cout * (c1 ? c1 : 1), 0.01f);
    std::vector<double> shift(cout, 0.0);
    Arena A;
    PackedConv pc, pr;
    size_t wo, bo, wro = 0, bro = 0;
    pack_conv(&A, &wo, &bo, &pc, w.data(), cout, c0, cm1, ksize, ksize == 3 && H == 1, nullptr, shift.data(), precision);
    if (resacc) pack_conv(&A, &wro, &bro, &pr, wr.data(), cout, c1, 0, 1, false, nullptr, shift.data(), precision);
    float *dev = nullptr, *x0 = nullptr, *x1 = nullptr, *res = nullptr, *out = nullptr;
    const int planes = precision == DTRAJ_PREC_TF32X3 ? 2 : 1;
    DTRAJ_CUDA(cudaMalloc(&dev, A.h.size() * sizeof(float)));
    DTRAJ_CUDA(cudaMemcpy(dev, A.h.data(), A.h.size() * sizeof(float), cudaMemcpyHostToDevice));
    DTRAJ_CUDA(cudaMalloc(&x0, (size_t)M * c0p * 4 * planes));
    DTRAJ_CUDA(cudaMemset(x0, 0, (size_t)M * c0p * 4 * planes));
    if (c1p) { DTRAJ_CUDA(cudaMalloc(&x1, (size_t)M * c1p * 4 * planes)); DTRAJ_CUDA(cudaMemset(x1, 0, (size_t)M * c1p * 4 * planes)); }
    DTRAJ_CUDA(cudaMalloc(&res, (size_t)M * coutp * 4));
    DTRAJ_CUDA(cudaMemset(res, 0, (size_t)M * coutp * 4));
    DTRAJ_CUDA(cudaMalloc(&out, (size_t)M * coutp * 4 * planes));
    ConvLayer L;
    memset(&L, 0, sizeof(L));
    L.src0 = x0; L.src0_lo = x0 + (size_t)M * c0p; L.c0p = c0p;
    if (resacc) { L.rsrc0 = x1; L.rc0p = pr.c0p; L.rbias = dev + bro; }
    else { L.src1 = x1; L.src1_lo = x1 ? x1 + (size_t)M * c1p : nullptr; L.c1p = c1p; }
    L.H = H; L.W = H; L.M = M; L.ntaps = pc.ntaps; L.wpk = dev + wo; L.bias = dev + bo; L.coutp = coutp;
    L.resid = (flags & 4) ? res : nullptr; L.out = out; L.lo_off = (int64_t)M * coutp;
    L.flags = (flags & 1 ? CONV_RELU : 0) | (flags & 4 ? CONV_RESID : 0) | (flags & (CONV_POOL | CONV_NOSTORE | CONV_RESX | CONV_FINAL | CONV_RESACC));
    L.act_mode = precision == DTRAJ_PREC_TF32 ? ACT_ROUND : precision == DTRAJ_PREC_TF32X3 ? ACT_SPLIT : ACT_PLAIN;
    L.f16 = precision == DTRAJ_PREC_F16 ? 1 : 0;      // (buffers stay sized for fp32: zeros either way)
    float* aux = nullptr;      // pooled output | raw input | 1x1 weights | final weights | eps, all zero
    DTRAJ_CUDA(cudaMalloc(&aux, ((size_t)M / 4 * coutp + (size_t)n * 4 * H * H + 16 * coutp + (size_t)M * 4) * 4));
    DTRAJ_CUDA(cudaMemset(aux, 0, ((size_t)M / 4 * coutp + (size_t)n * 4 * H * H + 16 * coutp + (size_t)M * 4) * 4));
    L.pool_out = aux;
    L.xraw = aux + (size_t)M / 4 * coutp; L.x_stride = 4 * H * H; L.xC = 1;
    L.rw1 = L.xraw + (size_t)n * 4 * H * H; L.rb1 = L.rw1 + 4 * coutp;
    L.finw = L.rb1 + 4 * coutp; L.finb = L.finw + 4 * coutp; L.finC = 1;
    L.elow = aux + (size_t)M / 4 * coutp + (size_t)n * 4 * H * H + 16 * coutp;
    int rc = 0;
    UmmaLaunch U;
    if (precision != DTRAJ_PREC_FP32) {
        umma_set_smem_attr();
        rc = build_umma_launch(&U, L, precision == DTRAJ_PREC_TF32X3 ? 3 : 1, dev + wo, pc.rows, resacc ? dev + wro : nullptr,
                               resacc ? pr.rows : 0, debug == 2 ? kUmmaGeneric : debug);
    }
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0); cudaEventCreate(&e1);
    for (int i = 0; i < iters + 2 && !rc; ++i) {
        if (i == 2) cudaEventRecord(e0, 0);
        rc = precision == DTRAJ_PREC_FP32 ? launch_conv_simt(L, 0) : launch_conv_umma(U, 0);
    }
    cudaEventRecord(e1, 0);
    cudaError_t ce = cudaDeviceSynchronize();
    float ms = 0.f;
    cudaEventElapsedTime(&ms, e0, e1);
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    cudaFree(dev); cudaFree(x0); if (x1) cudaFree(x1); cudaFree(res); cudaFree(out); cudaFree(aux);
    if (rc) return rc;
    if (ce != cudaSuccess) return fail(DTRAJ_ECUDA, "bench_conv -> %s", cudaGetErrorString(ce));
    *ms_out = ms / iters;
    return 0;
}

namespace {
const char* const kKindNames[] = {"ENC1H", "ENC1", "FIRST", "CONV_UMMA", "CONV_SIMT", "POOL", "POOL_H", "UP", "UP_H", "UP_H4", "FINAL"};

// Text form of a plan (dtraj_test_plan_describe).  Every tensor a launch reads or writes is named by the plan buffer its pointer
// points at, so the description is derived from the records themselves; a pointer into no buffer is an error.
struct PlanText {
    const dtraj_plan* P;
    std::string s;
    int rc = 0;
    void put(const char* fmt, ...) {
        char line[512];
        va_list ap;
        va_start(ap, fmt);
        vsnprintf(line, sizeof(line), fmt, ap);
        va_end(ap);
        s += line;
    }
    std::vector<std::pair<const char*, const dtraj_plan::Buf*>> bufs() const {
        return {{"tmp_h", &P->tmp_h}, {"tmp_r", &P->tmp_r}, {"tmp_x", &P->tmp_x}, {"p1", &P->p1}, {"x2", &P->x2}, {"p2", &P->p2},
                {"x3", &P->x3}, {"p3", &P->p3}, {"x4", &P->x4}, {"p4", &P->p4}, {"u3", &P->u3}, {"u2", &P->u2}, {"u1", &P->u1},
                {"y1", &P->y1}, {"elow", &P->elow}};
    }
    bool half_buf(const dtraj_plan::Buf* b) const { return P->u->d.precision == DTRAJ_PREC_F16 && b != &P->elow; }
    // one tensor of launch i: `role`, in / out, map size S, padded channels cp; p == nullptr names the raw frames x
    void tensor(int i, const char* role, const char* dir, const void* p, int S, int cp) {
        const char* name = "x";
        bool half = false;
        if (p) {
            name = nullptr;
            for (auto& b : bufs())
                if (b.second->p == p) { name = b.first; half = half_buf(b.second); }
            if (!name) { rc = fail(DTRAJ_EINVAL, "plan_describe: launch %d %s points into no plan buffer", i, role); return; }
        }
        put("tensor i=%d role=%s dir=%s buf=%s S=%d cp=%d type=%s\n", i, role, dir, name, S, cp, half ? "f16" : "f32");
    }
    void conv(int i, const ConvLayer& L) {
        tensor(i, "src0", "in", L.src0, L.H, L.c0p);
        if (L.src1) tensor(i, "src1", "in", L.src1, L.H, L.c1p);
        if (L.flags & CONV_RESID) tensor(i, "resid", "in", L.resid, L.H, L.coutp);
        if (L.flags & CONV_RESACC) {
            tensor(i, "rsrc0", "in", L.rsrc0, L.H, L.rc0p);
            if (L.rsrc1) tensor(i, "rsrc1", "in", L.rsrc1, L.H, L.rc1p);
        }
        if (L.flags & CONV_RESX) tensor(i, "x", "in", nullptr, L.H, L.xC);
        if (!(L.flags & CONV_NOSTORE)) tensor(i, "out", "out", L.out, L.H, L.coutp);
        if (L.flags & CONV_POOL) tensor(i, "pool", "out", L.pool_out, L.H / 2, L.coutp);
        if (L.flags & CONV_FINAL) tensor(i, "elow", "out", L.elow, L.H, L.finC);
    }
    void build() {
        const dtraj_unet* u = P->u;
        const bool f16 = u->d.precision == DTRAJ_PREC_F16;
        put("plan R=%lld options=%d precision=%d launches=%zu\n", (long long)P->R, P->options, u->d.precision, P->launches.size());
        for (auto& b : bufs()) {
            const int64_t esz = half_buf(b.second) ? 2 : 4;
            put("buf name=%s off=%lld bytes=%lld lo=%lld type=%s\n", b.first, (long long)((b.second->p - P->ws) * 4),
                (long long)(b.second->n * esz * (b.second->lo ? 2 : 1)), (long long)(b.second->lo * 4), esz == 2 ? "f16" : "f32");
        }
        for (size_t k = 0; k < P->launches.size() && !rc; ++k) {
            const Launch& l = P->launches[k];
            const int i = (int)k;
            const auto& r = l.rs;
            const char* form = "none";
            int flags = 0, act = 0, pair = 0, split = 1, nblk = 0, epi = 0;
            if (l.kind == Launch::CONV_UMMA) {
                const UmmaConv& c = l.U.conv;
                form = c.posm ? "posm" : c.halo == 1 ? "halo1" : c.halo == 2 ? "halo2" : "generic";
                flags = c.L.flags; act = c.L.act_mode; pair = c.pair; split = c.n_split; nblk = c.nblk_img; epi = epi_kind_of(c.L.flags);
            } else if (l.kind == Launch::CONV_SIMT) {
                flags = l.L.flags; act = l.L.act_mode;
            } else if (l.kind == Launch::ENC1H) {
                pair = l.enc1h.pair;
            } else if (l.kind == Launch::ENC1) {
                pair = l.enc1.pair; act = l.enc1.p.act_mode;
            } else if (l.kind == Launch::FIRST) {
                act = l.first.act_mode;
            } else if (l.kind != Launch::FINAL) {
                act = r.act_mode;
            }
            put("launch i=%d kind=%s grid=%u flags=%d act=%d tb=%d form=%s pair=%d split=%d nblk=%d epi=%d name=%s\n", i,
                kKindNames[l.kind], l.grid, flags, act, l.tb_block, form, pair, split, nblk, epi, l.name);
            const int S0 = u->sizes[0], C = u->d.channels, cv = f16 ? 8 : 4;
            switch (l.kind) {
            case Launch::ENC1H:
                tensor(i, "x", "in", nullptr, S0, C);
                tensor(i, "pool", "out", l.enc1h.p.pool_out, S0 / 2, l.enc1h.p.coutp);
                break;
            case Launch::ENC1:
                tensor(i, "x", "in", nullptr, S0, C);
                tensor(i, "pool", "out", l.enc1.p.pool_out, S0 / 2, l.enc1.p.coutp);
                break;
            case Launch::FIRST:
                tensor(i, "x", "in", nullptr, S0, C);
                tensor(i, "out", "out", l.first.h, S0, l.first.coutp);
                if (l.first.r) tensor(i, "res", "out", l.first.r, S0, l.first.coutp);
                break;
            case Launch::CONV_UMMA: conv(i, l.U.conv.L); break;
            case Launch::CONV_SIMT: conv(i, l.L); break;
            case Launch::POOL: case Launch::POOL_H:
                tensor(i, "src0", "in", r.in, 2 * r.S, r.cv * cv);
                tensor(i, "out", "out", r.out, r.S, r.cv * cv);
                break;
            case Launch::UP: case Launch::UP_H: case Launch::UP_H4:
                tensor(i, "src0", "in", r.in, r.S, r.cv * cv);
                tensor(i, "out", "out", r.out, 2 * r.S, r.cv * cv);
                break;
            case Launch::FINAL:
                tensor(i, "src0", "in", r.in, u->sizes[1], r.cv);
                tensor(i, "elow", "out", r.out, u->sizes[1], C);
                break;
            }
        }
    }
};
}  // namespace

extern "C" int dtraj_test_plan_describe(dtraj_unet* u, int64_t n_rows, void* workspace, int64_t workspace_bytes, int32_t options,
                                        char* buf, int64_t buf_len) {
    if (!u || !workspace || !buf || buf_len < 1) return fail(DTRAJ_EINVAL, "plan_describe: bad argument");
    DTRAJ_TRY(cached_plan(u, n_rows, workspace, workspace_bytes, options));
    PlanText T;
    T.P = u->plan;
    T.build();
    if (T.rc) return T.rc;
    if ((int64_t)T.s.size() + 1 > buf_len) return fail(DTRAJ_ENOMEM, "plan_describe: %zu bytes needed", T.s.size() + 1);
    memcpy(buf, T.s.c_str(), T.s.size() + 1);
    return 0;
}

extern "C" int dtraj_test_plan_run(dtraj_unet* u, const float* x, int64_t n_rows, int32_t t, const int32_t* row_variant,
                                   int32_t per_row, void* workspace, int64_t workspace_bytes, int32_t options, int32_t first,
                                   int32_t last, void* stream) {
    if (!u || !x || !workspace || (per_row && !row_variant)) return fail(DTRAJ_EINVAL, "plan_run: null argument");
    DTRAJ_TRY(cached_plan(u, n_rows, workspace, workspace_bytes, options));
    if (first < 0 || first > last || (size_t)last > u->plan->launches.size())
        return fail(DTRAJ_EINVAL, "plan_run: launches [%d, %d) outside the plan's %zu", first, last, u->plan->launches.size());
    const int C = u->d.channels, H = u->d.image_size;
    return plan_forward(u->plan, x, (int64_t)C * H * H, nullptr, row_variant, per_row ? 0 : t, per_row != 0, (cudaStream_t)stream,
                        nullptr, (size_t)first, (size_t)last);
}

extern "C" int dtraj_test_conv(int32_t precision, const float* x0, int32_t c0, const float* x1, int32_t c1, int64_t n, int32_t H,
                               int32_t W, const float* w_host, const float* bias_host, int32_t cout, int32_t ksize, int32_t flags,
                               const float* resid, float* out, void* stream) {
    if (H != W) return fail(DTRAJ_EINVAL, "test_conv: H must equal W");
    if (ksize != 1 && ksize != 3) return fail(DTRAJ_EINVAL, "test_conv: ksize must be 1 or 3");
    const bool resacc = (flags & 4) != 0;            // x1 feeds a fused 1x1 residual conv (CONV_RESACC), see include/dtraj.h
    if (resacc && (precision == DTRAJ_PREC_FP32 || precision == DTRAJ_PREC_TF32X3 || !x1 || c1 < 1))
        return fail(DTRAJ_EINVAL, "test_conv: a fused residual conv needs precision f16 or tf32 and a second input");
    cudaStream_t st = (cudaStream_t)stream;
    Arena A;
    PackedConv pc, pr;
    size_t wo, bo, wro = 0, bro = 0;
    std::vector<double> shift(cout), rshift(cout);
    for (int i = 0; i < cout; ++i) shift[i] = bias_host[i];
    pack_conv(&A, &wo, &bo, &pc, w_host, cout, c0, resacc ? 0 : c1, ksize, ksize == 3 && H == 1, nullptr, shift.data(), precision);
    if (resacc) {
        for (int i = 0; i < cout; ++i) rshift[i] = bias_host[cout + i];
        pack_conv(&A, &wro, &bro, &pr, w_host + (size_t)cout * c0 * ksize * ksize, cout, c1, 0, 1, false, nullptr, rshift.data(), precision);
    }
    float* dev = nullptr;
    DTRAJ_CUDA(cudaMalloc(&dev, A.h.size() * sizeof(float)));
    DTRAJ_CUDA(cudaMemcpy(dev, A.h.data(), A.h.size() * sizeof(float), cudaMemcpyHostToDevice));
    ConvLayer L;
    memset(&L, 0, sizeof(L));
    const int64_t M = n * H * W;
    L.src0 = x0; L.c0p = pc.c0p;
    if (resacc) { L.rsrc0 = x1; L.rc0p = pr.c0p; L.rbias = dev + bro; }
    else { L.src1 = x1; L.c1p = pc.c1p; }
    L.H = H; L.W = W; L.M = M; L.ntaps = pc.ntaps; L.wpk = dev + wo; L.bias = dev + bo; L.coutp = pc.coutp;
    L.resid = resid; L.out = out; L.flags = (flags & 1 ? CONV_RELU : 0) | (resid ? CONV_RESID : 0) | (resacc ? CONV_RESACC : 0);
    L.act_mode = (flags & 2) ? ACT_ROUND : ACT_PLAIN;
    L.f16 = precision == DTRAJ_PREC_F16 ? 1 : 0;
    int rc = 0;
    float* lo = nullptr;
    if (precision == DTRAJ_PREC_FP32) rc = launch_conv_simt(L, st);
    else {
        if (precision == DTRAJ_PREC_TF32X3) {
            // low planes of the inputs, computed here for the test
            const int64_t n0 = M * pc.c0p, n1 = M * pc.c1p;
            std::vector<float> h(n0 + n1);
            cudaMalloc(&lo, (n0 + n1) * sizeof(float));
            cudaMemcpy(h.data(), x0, n0 * sizeof(float), cudaMemcpyDeviceToHost);
            if (n1) cudaMemcpy(h.data() + n0, x1, n1 * sizeof(float), cudaMemcpyDeviceToHost);
            for (auto& v : h) v = v - tf32_trunc(v);
            cudaMemcpy(lo, h.data(), (n0 + n1) * sizeof(float), cudaMemcpyHostToDevice);
            L.src0_lo = lo; L.src1_lo = lo + n0;
        }
        umma_set_smem_attr();
        UmmaLaunch U;
        rc = build_umma_launch(&U, L, precision == DTRAJ_PREC_TF32X3 ? 3 : 1, dev + wo, pc.rows, resacc ? dev + wro : nullptr,
                               resacc ? pr.rows : 0);
        if (!rc) rc = launch_conv_umma(U, st);
    }
    cudaError_t ce = cudaStreamSynchronize(st);
    cudaFree(dev);
    if (lo) cudaFree(lo);
    if (rc) return rc;
    if (ce != cudaSuccess) return fail(DTRAJ_ECUDA, "test_conv -> %s", cudaGetErrorString(ce));
    return 0;
}
