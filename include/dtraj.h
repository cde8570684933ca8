/*
 * dtraj.h -- C ABI of libdtraj.so, the B200 (sm_100a) implementation of the trajectory
 * hot path of henriChevreux/distillation_trajectories.
 *
 * The reference has no FFI layer (it is pure Python/PyTorch); its boundary for this path
 * is a set of Python signatures (SURVEY.md 8b).  The Python package
 * `distillation_trajectories_b200` keeps those signatures and calls the entry points
 * below through ctypes.  Each entry point names the reference code it replaces.
 *
 * Conventions
 *   - every function returns 0 on success and a negative DTRAJ_E* code on failure;
 *     dtraj_last_error() returns a thread-local message.  Nothing throws.
 *   - pointers marked "dev" are CUDA device pointers owned by the caller (torch tensors'
 *     data_ptr()); "host" pointers are ordinary memory.  `stream` is a cudaStream_t
 *     passed as void* (0 = legacy default stream).
 *   - images, eps maps and trajectories are fp32 in the reference layout [N, C, H, W] /
 *     [N, L, C, H, W].  Internal feature maps live in the caller-owned workspace, NHWC:
 *     fp16 in DTRAJ_PREC_F16 (the default of the sweeps), fp32 in the other modes.
 *   - a handle is used by one host thread at a time; one process drives one GPU.
 */
#ifndef DTRAJ_H
#define DTRAJ_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DTRAJ_OK            0
#define DTRAJ_EINVAL      (-1)  /* bad argument / unsupported shape            */
#define DTRAJ_ECUDA       (-2)  /* CUDA runtime or driver error                */
#define DTRAJ_EMISSING    (-3)  /* a state_dict tensor the model needs is absent */
#define DTRAJ_ENOMEM      (-4)  /* workspace too small                         */
#define DTRAJ_ERANGE      (-5)  /* DTRAJ_PREC_F16: a value left the fp16 range  */

/* arithmetic used for the 3x3 / 1x1 convolutions of the U-Net */
#define DTRAJ_PREC_FP32     0   /* CUDA-core fp32 implicit GEMM (exact mode)                 */
#define DTRAJ_PREC_TF32     1   /* tcgen05.mma kind::tf32, one pass (fast mode)              */
#define DTRAJ_PREC_TF32X3   2   /* tcgen05.mma kind::tf32, hi/lo split, 3 passes (~fp32)     */
#define DTRAJ_PREC_F16      3   /* tcgen05.mma kind::f16: fp16 feature maps and weights (the  */
                                /* same 11-bit significand as tf32), fp32 accumulation; twice */
                                /* the MMA rate and half the operand bytes of DTRAJ_PREC_TF32. */
                                /* Range-checked: |activation| or |weight| > 65504 is an error */

/* conditioning variant of one forward row (reference models.py:181-185) */
#define DTRAJ_VAR_NONE      0   /* cond=None: time embedding only                            */
#define DTRAJ_VAR_COND0     1   /* cond=[[0.]] through cond_emb (trajectory_engine.py:72)    */
#define DTRAJ_VAR_COND1     2   /* cond=[[1.]] through cond_emb                              */

/* update rules of the three reference samplers (SURVEY.md 8a S1-S3) */
#define DTRAJ_RULE_S1       1   /* utils/diffusion.py:149-158        x' = k0*(x - k1*eps) + k2*z      */
#define DTRAJ_RULE_S2       2   /* analysis/trajectory_engine.py:98-110  x' = (k0*x - k1*eps) + k2*z  */
#define DTRAJ_RULE_S3       3   /* utils/trajectory_manager.py:194-203   x' = (x - k0*eps)/k1 + k2*z  */

const char* dtraj_last_error(void);
int dtraj_version(void);

/* ------------------------------------------------------------------ U-Net (models.py) */

typedef struct dtraj_unet dtraj_unet;

typedef struct {
    int32_t channels;      /* config.channels                       models.py:99           */
    int32_t image_size;    /* H == W; 16, 32 or 64 (any other size is refused)              */
    int32_t dims[4];       /* DiffusionUNet.dims                    models.py:110          */
    int32_t temb_dim;      /* DiffusionUNet.time_emb_dim            models.py:101          */
    int32_t n_timesteps;   /* time tables cover t = 0 .. n_timesteps-1                     */
    int32_t precision;     /* DTRAJ_PREC_*                                                 */
} dtraj_unet_desc;

/*
 * Replaces DiffusionUNet.__init__/load_state_dict + .eval()  (models.py:95-157).
 * `names[i]` are state_dict keys ("enc1.conv1.weight", "enc1.norm1.running_var", ...),
 * `tensors[i]` host fp32 arrays in the reference's layouts ([Cout,Cin,kh,kw], [out,in]),
 * `numel[i]` their element counts.  BatchNorm (eval, eps 1e-5) is folded into the conv
 * weights here; weights are padded and packed K-major for the kernels, uploaded, and the
 * per-(timestep, variant, block) time-embedding biases relu(time_mlp(temb)) are
 * precomputed on the device (models.py:15-39,66-67,175-185).
 */
int dtraj_unet_create(const dtraj_unet_desc* desc,
                      const char* const* names, const float* const* tensors,
                      const int64_t* numel, int32_t n_tensors,
                      dtraj_unet** out);
int dtraj_unet_destroy(dtraj_unet* unet);

/* bytes of workspace one forward over `n_rows` rows needs */
int64_t dtraj_unet_workspace_bytes(const dtraj_unet* unet, int64_t n_rows);

/* host copy of the time table row: relu(block.time_mlp(time_emb(t, variant))) for block
 * index `block` (0..7 = enc1..enc4, bottleneck, dec3, dec2, dec1); `out` host [dims]. */
int dtraj_unet_time_bias(const dtraj_unet* unet, int32_t t, int32_t variant, int32_t block,
                         float* out_host, int32_t n);

/*
 * Replaces DiffusionUNet.forward(x, t, cond)  (models.py:159-224) for a batch that shares
 * one timestep value `t` (every caller on the hot path does: utils/diffusion.py:204,
 * analysis/trajectory_engine.py:62).
 *   x            dev [n_rows, C, H, W]
 *   row_variant  dev int32 [n_rows], DTRAJ_VAR_* per row (NULL = all DTRAJ_VAR_NONE)
 *   eps          dev [n_rows, C, H, W]
 */
int dtraj_unet_forward(dtraj_unet* unet, const float* x, int64_t n_rows, int32_t t,
                       const int32_t* row_variant, float* eps,
                       void* workspace, int64_t workspace_bytes, void* stream);

/*
 * The same forward with a timestep PER ROW: what the training-side callers feed
 * (utils/diffusion.py:83-100 p_losses; the teacher half of the distillation step,
 * scripts/train_students.py:131-141, where t = randint(0, teacher_steps, (B,))).
 *   row_tv   dev int32 [n_rows]: t_i * 3 + DTRAJ_VAR_* of row i -- the row of the
 *            [n_timesteps][3] time-bias table its epilogues read; the caller guarantees
 *            0 <= t_i < n_timesteps.
 */
int dtraj_unet_forward_rows(dtraj_unet* unet, const float* x, int64_t n_rows,
                            const int32_t* row_tv, float* eps,
                            void* workspace, int64_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------ fused sampler step */

/*
 * One reverse-process step for `n_samples` samples: classifier-free-guidance combine
 * eps = eps_u + w*(eps_c - eps_u)  (utils/diffusion.py:126, trajectory_engine.py:80),
 * the update rule `rule` with coefficients k[3], and the store of x' (the next trajectory
 * frame).  All arrays dev fp32 [n_samples, D] with the given sample strides (in floats);
 * eps_c / w may be NULL (no guidance), z may be NULL (no noise, e.g. t == 0).
 * This is the stand-alone form; inside dtraj_sampler the same kernel also performs the
 * final bilinear x2 upsample of the half-resolution eps.
 */
int dtraj_step_fused(int32_t rule, const float* k_host3,
                     const float* eps_u, const float* eps_c, const float* w,
                     const float* x, int64_t x_stride,
                     const float* z, int64_t z_stride,
                     float* x_out, int64_t out_stride,
                     int64_t n_samples, int64_t D, void* stream);

/* ------------------------------------------------------------------ whole sampling loop */

typedef struct dtraj_sampler dtraj_sampler;

typedef struct {
    int32_t rule;              /* DTRAJ_RULE_*                                              */
    int32_t n_samples;         /* B trajectories generated together                         */
    int32_t n_rows;            /* forward rows per step (B, or up to 2B with guidance)       */
    int32_t n_updates;         /* model-driven steps                                         */
    int32_t copy_last;         /* 1: append a duplicate of the last frame (S2 at t == 0,
                                  trajectory_engine.py:86,113)                               */
    int32_t n_frames;          /* L = 1 + n_updates + copy_last                              */
    int32_t use_graph;         /* capture the whole loop in one CUDA graph                   */
    int32_t n_rows0;           /* > 0: the FIRST step uses its own, smaller row layout (below) */
    const int32_t* step_timestep;  /* host [n_updates]  timestep value fed to the model      */
    const float*   step_coef;      /* host [n_updates*3] k0,k1,k2 of the rule, per step      */
    const int32_t* row_sample;     /* dev [n_rows]   sample whose x this row evaluates       */
    const int32_t* row_variant;    /* dev [n_rows]   DTRAJ_VAR_*                             */
    const int32_t* sample_row_u;   /* dev [n_samples] row holding eps_u (or the only eps)    */
    const int32_t* sample_row_c;   /* dev [n_samples] row holding eps_c, -1 = no guidance    */
    const float*   guidance;       /* dev [n_samples] w                                      */
    const float*   z_bank;         /* dev [*, D] injected noise draws                        */
    const int32_t* z_index;        /* dev [n_updates, n_samples] draw index, -1 = z = 0      */
    float*         traj;           /* dev [n_samples, n_frames, C, H, W]; frame 0 = x_T in   */
    void*          workspace;      /* dev, >= dtraj_unet_workspace_bytes(unet, n_rows)       */
    int64_t        workspace_bytes;
    /* First-step row sharing (n_rows0 > 0): samples that start from the SAME x_T and differ only in their guidance
     * scale (compare_trajectories feeds one noise to every scale, analysis/trajectory_engine.py:147-156) need one
     * forward row per (x_T, variant) at the first step instead of one or two per sample.  Same meaning as the four
     * arrays above, for step 0 only; n_rows0 <= n_rows. */
    const int32_t* row_sample0;    /* dev [n_rows0]                                          */
    const int32_t* row_variant0;   /* dev [n_rows0]                                          */
    const int32_t* sample_row_u0;  /* dev [n_samples]                                        */
    const int32_t* sample_row_c0;  /* dev [n_samples], -1 = no guidance                      */
} dtraj_sampler_desc;

/*
 * Replaces the loops of p_sample_loop (utils/diffusion.py:199-208), generate_trajectory
 * (analysis/trajectory_engine.py:61-113) and TrajectoryManager.generate_trajectory
 * (utils/trajectory_manager.py:98-111): n_updates x { U-Net forward over n_rows rows,
 * fused step } writing every frame into `traj` on the device.  The device arrays named in
 * the descriptor are read at run time, so their CONTENTS (x_T in frame 0, noise bank,
 * guidance, indices) may change between runs; their addresses may not.
 */
int dtraj_sampler_create(dtraj_unet* unet, const dtraj_sampler_desc* desc, dtraj_sampler** out);
int dtraj_sampler_run(dtraj_sampler* s, void* stream);
int dtraj_sampler_destroy(dtraj_sampler* s);
/* number of kernel launches one dtraj_sampler_run performs (graph nodes) */
int64_t dtraj_sampler_launches(const dtraj_sampler* s);

/*
 * Measurement aid (bench.py roofline): runs the loop ONCE, un-captured, with a CUDA event pair around
 * every launch on `stream`, and returns the summed device time (ms) and launch count per kernel class
 *   [0] generic convolutions (tcgen05 implicit GEMM, or the CUDA-core kernel in DTRAJ_PREC_FP32)
 *   [1] first convolution (Cin <= 4)   [2] max-pool / upsample / final 1x1   [3] fused step / frame copy
 *   [4] fused enc1 block (conv1 into shared memory + conv2 by tap views + pool; conv1 runs on the tensor cores in
 *       DTRAJ_PREC_F16, on the CUDA cores in DTRAJ_PREC_TF32)
 * plus the algorithmic tensor-core flops of class 0 (conv_flops2[0]) and of class 4 (conv_flops2[1]): sum over
 * layers and steps of 2 * M * Cout * Cin * taps with REAL (unpadded) channel counts and the taps actually
 * evaluated.  Synchronises the stream.
 */
int dtraj_sampler_profile(dtraj_sampler* s, void* stream, double* class_ms5, int64_t* class_launches5,
                          double* conv_flops2);
/* the two flop counts of dtraj_sampler_profile without running anything */
int dtraj_sampler_flops(const dtraj_sampler* s, double* conv_flops2);
/* Per-launch form (tools/profile_layers.py): runs the loop once, un-captured, and writes one line
 * "name <TAB> grid <TAB> device microseconds <TAB> algorithmic flops" per launch of sampler step `step` into `buf`. */
int dtraj_sampler_profile_text(dtraj_sampler* s, void* stream, int32_t step, char* buf, int64_t buf_len);

/* ------------------------------------------------------------------ trajectory metrics */

/*
 * Streaming reductions behind compute_trajectory_metrics
 * (analysis/metrics/trajectory_metrics.py:55-215) and analyze_time_dependent_distances
 * (analysis/metrics/time_dependent.py:57,78) for N trajectory pairs at once.
 *   teacher, student  dev [N, L, D] fp32 (D = C*H*W)
 *   out               dev [N, L, 6] fp32:
 *        [i][0] = sum (T_i - S_i)^2                 position difference / mse numerators
 *        [i][1] = sum (T_{i+1} - T_i)^2   (i < L-1) teacher velocity^2
 *        [i][2] = sum (S_{i+1} - S_i)^2   (i < L-1) student velocity^2
 *        [i][3] = sum (T_{i+1}-T_i)(S_{i+1}-S_i)    direction dot product
 *        [0][4] = sum (T_{L-1} - T_0)^2,  [0][5] = sum (S_{L-1} - S_0)^2   (other [i][4..5] = 0)
 * Every element of both tensors is read exactly once.  The f64 scalar formulas
 * (log1p / exp / ratios) stay on the host as in the reference.
 */
int dtraj_metrics_pairs(const float* teacher, const float* student,
                        int64_t N, int32_t L, int32_t D, float* out, void* stream);

/*
 * 1-d Wasserstein distance per frame (trajectory_metrics.py:296-312; scipy's
 * wasserstein_distance on K = min(1000, D) subsampled elements).
 *   idx   dev int32 [n_idx_sets, L, K] element indices (np.random.choice on the host);
 *         pair n uses set idx_set[n] (dev int32 [N], NULL = set 0 for all);
 *         idx == NULL means K == D, all elements.
 *   out   dev [N, L] fp32
 */
int dtraj_wasserstein(const float* teacher, const float* student,
                      int64_t N, int32_t L, int32_t D,
                      const int32_t* idx, const int32_t* idx_set, int32_t K,
                      float* out, void* stream);

/*
 * Teacher and student trajectories of different lengths, N pairs in one launch: the branch of
 * compute_trajectory_metrics for len(teacher) != len(student) (trajectory_metrics.py:239-279; a
 * student sampled with fewer steps than its teacher).  n = min(LT, LS); "long" is the teacher when
 * LT >= LS and the student otherwise, "short" the other one.
 *   teacher  dev [N, LT, D] fp32,  student  dev [N, LS, D] fp32 (D = C*H*W, a multiple of 4, at most 4096)
 *   rs_pos   dev int32 [n], rs_frac dev fp32 [n]: the path-alignment resampling table, the same for
 *            every pair -- short frame j is compared with (1 - f_j) long[p_j] + f_j long[p_j + 1],
 *            np.interp's rule on linspace(0, 1, L) axes (p non-decreasing, 0 <= p_j <= L_long - 2)
 *   out      dev [N, max(LT, LS), 8] fp32:
 *        [i][0] = sum (T_i - S_i)^2                     (i < n)
 *        [i][1] = sum (T_{i+1} - T_i)^2  (i < LT-1),  [i][2] = sum (S_{i+1} - S_i)^2  (i < LS-1)
 *        [i][3] = sum (T_{i+1}-T_i)(S_{i+1}-S_i)        (i < n-1)
 *        [0][4] = sum (T_{LT-1} - T_0)^2,  [0][5] = sum (S_{LS-1} - S_0)^2
 *        [0][6] = sum (T_{LT-1} - S_{LS-1})^2           endpoint distance / mse numerator
 *        [j][7] = sum ((1 - f_j) long_{p_j} + f_j long_{p_j+1} - short_j)^2   (j < n) path alignment
 *        every other entry is 0.
 * The long trajectory is read once, the short one twice, and three single frames (T_0, S_0 and the
 * short one's last) once more: 4 * N * D * (L_long + 2 * L_short + 3) bytes requested, against the
 * algorithmic 4 * N * D * (LT + LS).
 * LT == LS is accepted (then the alignment term equals [j][0]); max(LT, LS) >= 2.
 */
int dtraj_metrics_pairs_ragged(const float* teacher, const float* student,
                               int64_t N, int32_t LT, int32_t LS, int32_t D,
                               const int32_t* rs_pos, const float* rs_frac, float* out, void* stream);

/*
 * dtraj_wasserstein for teacher [N, LT, D] and student [N, LS, D] of different lengths: the
 * distances of the first n = min(LT, LS) frames (trajectory_metrics.py:296-312 zips the two frame
 * lists), read in place.  idx dev int32 [n_idx_sets, n, K]; out dev [N, n] fp32.
 */
int dtraj_wasserstein_ragged(const float* teacher, const float* student,
                             int64_t N, int32_t LT, int32_t LS, int32_t D,
                             const int32_t* idx, const int32_t* idx_set, int32_t K,
                             float* out, void* stream);

/*
 * The subsample index sets compute_trajectory_metrics draws for frames larger than 1000 elements
 * (trajectory_metrics.py:301-306: np.random.choice(D, K, replace=False) per frame, from the global numpy RNG that
 * compare_trajectories' callers left at seed + 1, analysis/trajectory_engine.py:91-93), generated on the device: numpy's
 * legacy RandomState stream (MT19937 seeded by init_genrand, Fisher-Yates with masked rejection sampling) reproduced
 * bit for bit, L consecutive choice() calls per seed.
 *   seeds  dev uint32 [n_seeds]   (the value passed to np.random.seed)
 *   out    dev int32  [n_seeds, L, K]  -- directly usable as `idx` of dtraj_wasserstein
 * 2 <= D <= 16384, 1 <= K <= D.
 */
int dtraj_numpy_choice_sets(const uint32_t* seeds, int32_t n_seeds, int32_t L, int32_t D, int32_t K,
                            int32_t* out, void* stream);

/* ------------------------------------------------------------------ PCA projection
 * Replaces the per-trajectory `pca.transform(process_trajectory(traj))` of the visual analysis
 * (scripts/analysis/analyze_trajectories.py:66-80,100; same in :232-246): frames of any number
 * of trajectories are projected onto K <= 8 fitted directions in one streaming pass.
 *   frames  dev [n_frames, D] fp32 (a [N, L, C, H, W] trajectory tensor, n_frames = N*L)
 *   comps   dev [K, D] fp32 (sklearn PCA.components_), offset dev [K] = mean_ . components_[k]
 *   out     dev [n_frames, K] fp32 = frames @ comps^T - offset
 * Every element of `frames` is read exactly once (HBM-bound: 4 * n_frames * D bytes). */
int dtraj_project(const float* frames, int64_t n_frames, int32_t D, const float* comps,
                  const float* offset, int32_t K, float* out, void* stream);

/* ------------------------------------------------------------------ device-side error state
 * Kernels never trap: a tcgen05 pipeline role whose mbarrier wait times out (bit 0), or an
 * activation that leaves the fp16 range in DTRAJ_PREC_F16 (bit 1), sets a sticky device word.
 * Every dtraj_unet handle owns its own word, so two models running on two streams can tell whose
 * launch failed.  dtraj_unet_check_errors() reads and clears the handle's word (it synchronises
 * the device: call it where results leave the library).  Returns 0, DTRAJ_ECUDA (pipeline
 * time-out: results are invalid) or DTRAJ_ERANGE (fp16 overflow: rerun with DTRAJ_PREC_TF32). */
int dtraj_unet_check_errors(dtraj_unet* unet);
/* Non-blocking form for pipelined callers: enqueue a copy of the handle's word into `host_flag` (pinned host memory)
 * on `stream`; a non-zero word read after the stream has reached that point means "call dtraj_unet_check_errors()". */
int dtraj_unet_error_flag_async(dtraj_unet* unet, uint32_t* host_flag, void* stream);
/* The same pair for the library-wide word that launches WITHOUT a handle report to (dtraj_test_conv, dtraj_bench_conv). */
int dtraj_check_errors(void);
int dtraj_error_flag_async(uint32_t* host_flag, void* stream);

/* ------------------------------------------------------------------ test hooks
 * Single convolution layer through either implementation, for kernel-vs-kernel parity
 * tests (tests/test_gpu_conv.py).  x0/x1 NHWC dev [n, H, W, c0p]/[.., c1p] (x1 may be
 * NULL); w host [Cout, c0+c1, k, k] (k = 1 or 3), bias host [Cout]; out dev NHWC
 * [n, H, W, coutp] with coutp = round_up(Cout, 32).  flags: bit0 relu, bit1 round
 * outputs to tf32, bit2 (DTRAJ_PREC_F16 / DTRAJ_PREC_TF32 only) x1 is not a second source of the main conv but the input of
 * a fused 1x1 residual conv (CONV_RESACC, the decoder / enc2 conv2 form): w then holds [Cout, c0, k, k] followed by the
 * residual weights [Cout, c1], bias holds [Cout] followed by the residual bias [Cout], and out = act(conv(x0) + bias) +
 * conv1x1(x1) + residual bias (+ resid).  In DTRAJ_PREC_F16 x0/x1/resid/out are __half maps with channels
 * padded to 64. */
int dtraj_test_conv(int32_t precision, const float* x0, int32_t c0, const float* x1, int32_t c1,
                    int64_t n, int32_t H, int32_t W, const float* w_host, const float* bias_host,
                    int32_t cout, int32_t ksize, int32_t flags, const float* resid,
                    float* out, void* stream);

/* The forward plan one launch at a time (tests/test_gpu_layers.py).  Both build the plan dtraj_unet_forward would
 * use for (n_rows, workspace), or reuse the handle's cached one; `options` bit 0 builds it WITHOUT the fused enc1
 * kernel (k_conv_first, then the generic enc1.conv2 with the CONV_RESX tails), a plan the product never builds for the
 * supported models.  The cached plan is rebuilt whenever n_rows, the workspace or the options change.
 * dtraj_test_plan_describe writes NUL-terminated text into buf, one record per line:
 *   plan R=.. options=.. precision=.. launches=..
 *   buf name=.. off=.. bytes=.. lo=.. type=f16|f32             every workspace buffer: byte offset, bytes, lo-plane offset
 *   launch i=.. kind=.. grid=.. flags=.. act=.. tb=.. form=generic|halo1|halo2|posm|none pair=.. split=.. nblk=.. epi=.. name=..
 *   tensor i=.. role=.. dir=in|out buf=..|x S=.. cp=.. type=..  every map launch i reads or writes (x: the raw frames)
 * dtraj_test_plan_run enqueues launches [first, last) of that plan on `stream` exactly as the forward does; per_row = 1
 * is the dtraj_unet_forward_rows form (row_variant then holds t_i * 3 + variant_i and t is ignored). */
int dtraj_test_plan_describe(dtraj_unet* unet, int64_t n_rows, void* workspace, int64_t workspace_bytes,
                             int32_t options, char* buf, int64_t buf_len);
int dtraj_test_plan_run(dtraj_unet* unet, const float* x, int64_t n_rows, int32_t t, const int32_t* row_variant,
                        int32_t per_row, void* workspace, int64_t workspace_bytes, int32_t options,
                        int32_t first, int32_t last, void* stream);

/* ------------------------------------------------------------------ diagnostics (tools/, not used by the package's hot path)
 * Kernel-only timing of one conv layer shape on zero-filled buffers allocated inside (tools/conv_bench.py): `iters`
 * launches between one event pair, average milliseconds in *ms_out.  flags: bit0 relu, bit2 residual input, plus the
 * CONV_POOL / CONV_NOSTORE / CONV_RESX / CONV_FINAL / CONV_RESACC tail bits of csrc/conv_simt.cuh (CONV_RESACC: x1, c1
 * channels, feeds the fused 1x1 residual conv instead of the main conv).  `debug` (A/B experiments): 0 = the tile form and
 * shared-memory split the forward plan uses, 2 = the generic [image][y][x] tiles where that form is a halo form,
 * 0x100 | n_hb << 4 | epi_bufs = the halo form with n_hb halo slots and epi_bufs epilogue buffers per warp; other values
 * are refused. */
int dtraj_bench_conv(int32_t precision, int32_t c0, int32_t c1, int32_t cout, int64_t n, int32_t H, int32_t ksize,
                     int32_t flags, int32_t iters, int32_t debug, float* ms_out);
/* Peek at the library-wide error word without clearing it (tests assert it stays 0). */
unsigned int dtraj_debug_umma_error(void);
/* (csrc/probe.cuh -- the tcgen05 descriptor-view and permuted-TMA hardware probes behind profiles/r01_*_probe.txt -- is
 * compiled only with -DDTRAJ_PROBES and exports dtraj_probe_umma_view / dtraj_probe_tma_permuted; the same build flag
 * turns on the SM-clock stamps read by dtraj_probe_timeline / dtraj_probe_timeline_select (tools/timeline.py).  The product build has
 * none of them.) */

#ifdef __cplusplus
}
#endif
#endif /* DTRAJ_H */
