"""GPU: 64x64 models end to end -- conv layers at the 32x32 and 64x64 levels, DiffusionUNet.forward, the three samplers,
grid.sweep and the metric kernels at frame widths up to 16384 -- against an f64 convolution and the CPU oracle (which does
not depend on the image size).  Batches and step counts stay small: a CPU oracle forward of the 3x64x64 teacher is about
7 GFLOP per row."""
import functools

import numpy as np
import pytest
import torch

from oracle import metrics as om
from oracle import samplers as osmp
from oracle import unet as ounet
from distillation_trajectories_b200 import DtrajError, _lib, grid, sampling, set_precision, umma_error_flag
from distillation_trajectories_b200.analysis import trajectory_engine as te
from distillation_trajectories_b200.analysis.metrics import trajectory_metrics as tm
from distillation_trajectories_b200.engine import UNetEngine
from distillation_trajectories_b200.utils import diffusion
from distillation_trajectories_b200.utils.trajectory_manager import TrajectoryManager
from helpers import Cfg, assert_close, cpu_sd, make_model, oracle_fn
from test_gpu_conv import f16_round, reference, run_conv, tf32_rna, tf32_trunc
from test_gpu_forward import FWD_TOL

pytestmark = pytest.mark.gpu
RTOL, ATOL, RT_METRIC = 1e-3, 1e-4, 1e-4
PRECS = ["fp32", "tf32x3", "tf32", "f16"]


@pytest.fixture(autouse=True)
def cpu_noise():
    """draw noise with the CPU generator, as the oracle does"""
    sampling.set_noise_device("cpu")
    yield
    sampling.set_noise_device(None)


# ------------------------------------------------------------------ 1. conv layers at 32x32 and 64x64
SHAPES64 = [
    # n, c0, c1, cout, H, ksize
    (2, 128, 0, 128, 64, 3),     # enc1.conv2 of the teacher in the exact modes: 2-row im2col boxes
    (1, 38, 0, 38, 64, 3),       # ... of the sf 0.3 student (ragged channels)
    (2, 128, 0, 256, 32, 3),     # enc2.conv1 at the 32x32 level: halo form in fp16
    (2, 256, 0, 256, 32, 3),     # enc2.conv2
    (2, 256, 256, 128, 32, 3),   # dec1.conv1: two sources
    (3, 77, 77, 38, 32, 3),      # sf 0.3 dec1.conv1: two half-filled sources (96 + 96), N = 64
    (40, 128, 0, 128, 32, 3),    # 320 tiles of 16 x 8 pixels: CTA pairs, several tiles per pair
    (24, 256, 256, 128, 32, 3),  # 192 tiles, two sources: persistent single-CTA loop
    (3, 256, 0, 128, 32, 1),     # 1x1 residual conv of dec1
]


@pytest.mark.parametrize("prec", [_lib.PREC_FP32, _lib.PREC_TF32, _lib.PREC_TF32X3, _lib.PREC_F16],
                         ids=["fp32", "tf32", "tf32x3", "f16"])
@pytest.mark.parametrize("shape", SHAPES64, ids=lambda s: "n%d_c%d+%d_o%d_h%d_k%d" % s)
def test_conv_layer_64(prec, shape):
    n, c0, c1, cout, H, ksize = shape
    rng = np.random.RandomState(hash(shape) % (2 ** 31))
    x0 = rng.randn(n, c0, H, H).astype(np.float32)
    x1 = rng.randn(n, c1, H, H).astype(np.float32) if c1 else None
    w = (rng.randn(cout, c0 + c1, ksize, ksize) / np.sqrt((c0 + c1) * ksize * ksize)).astype(np.float32)
    b = rng.randn(cout).astype(np.float32) * 0.1
    resid = rng.randn(n, cout, H, H).astype(np.float32)
    if prec == _lib.PREC_TF32:
        x0 = tf32_trunc(x0)
        x1 = None if x1 is None else tf32_trunc(x1)
    if prec == _lib.PREC_F16:
        x0, resid, w = f16_round(x0), f16_round(resid), f16_round(w)
        x1 = None if x1 is None else f16_round(x1)
    K = (c0 + c1) * ksize * ksize
    for relu, rs in ((True, resid), (False, None)):
        got = run_conv(prec, x0, x1, w, b, ksize, relu, rs)
        want = reference(x0, x1, w, b, ksize, relu, rs, round_w=(prec == _lib.PREC_TF32))
        scale = np.abs(want).max()
        if prec == _lib.PREC_F16:
            bound = (4e-6 + 4e-9 * K) * scale + 2.0 ** -11 * np.abs(want) + 6e-8
            assert (np.abs(got - want) <= bound).all(), f"max excess {np.max(np.abs(got - want) - bound):.3e}"
            continue
        # (fp32: one FMA chain of K terms per output; at K = 4608 over 3 M outputs its largest error reaches ~3e-6 of max|ref|
        #  -- a sequential fp32 sum of the same terms on the CPU: 2.8e-6 over 4 of the 24 images -- so the bound grows with K)
        tol = 2e-6 + 1e-9 * K if prec == _lib.PREC_FP32 else 4e-6 + 4e-9 * K
        err = np.abs(got - want).max() / scale
        assert err < tol, f"max err / max|ref| = {err:.3e}"


RESACC_SHAPES = [
    # n, c0 (main conv), c_res (residual conv input), cout -- 32x32 maps
    (2, 256, 128, 256),          # enc2.conv2 of the teacher: 1x1 residual conv of the pooled enc1 output
    (2, 128, 512, 128),          # dec1.conv2: residual conv over [upsampled | skip] (8 residual K blocks, four halo slots)
    (40, 256, 128, 256),         # 320 tiles: CTA pairs, several tiles per pair
    (3, 38, 154, 38),            # sf 0.3 dec1.conv2: ragged widths, half-filled K blocks
]


def run_conv_resacc(prec, x0, xr, w, wr, b, br):
    """relu(conv3x3(x0) + b) + conv1x1(xr) + br through dtraj_test_conv with the fused residual conv (flags bit 2)"""
    import ctypes as Ct
    lib = _lib.load()
    n, c0, H, W = x0.shape
    cr, cout = xr.shape[1], w.shape[0]
    f16 = prec == _lib.PREC_F16
    dt = torch.float16 if f16 else torch.float32
    rup = lambda v: (v + 31) // 32 * 32

    def nhwc(a):
        t = torch.zeros(n, H, W, rup(a.shape[1]), dtype=dt)
        t[..., :a.shape[1]] = torch.from_numpy(a).permute(0, 2, 3, 1).to(dt)
        return t.cuda().contiguous()

    d0, dr = nhwc(x0), nhwc(xr)
    out = torch.full((n, H, W, rup(cout)), float("nan"), dtype=dt, device="cuda")
    wc = np.ascontiguousarray(np.concatenate([w.reshape(-1), wr.reshape(-1)]), np.float32)
    bc = np.ascontiguousarray(np.concatenate([b, br]), np.float32)
    _lib.check(lib.dtraj_test_conv(prec, _lib.ptr(d0), c0, _lib.ptr(dr), cr, n, H, W, wc.ctypes.data_as(Ct.c_void_p),
                                   bc.ctypes.data_as(Ct.c_void_p), cout, 3, 1 | 4, None, _lib.ptr(out), _lib.stream_ptr()))
    torch.cuda.synchronize()
    assert umma_error_flag() == 0
    o = out.float().cpu()
    assert torch.isfinite(o).all()
    return o[..., :cout].permute(0, 3, 1, 2).numpy()


@pytest.mark.parametrize("prec", [_lib.PREC_TF32, _lib.PREC_F16], ids=["tf32", "f16"])
@pytest.mark.parametrize("shape", RESACC_SHAPES, ids=lambda s: "n%d_c%d_r%d_o%d" % s)
def test_conv_fused_residual_conv_32x32(prec, shape):
    """conv2 of enc2 / dec1 at the 32x32 level with the block's 1x1 residual conv as extra MMAs (CONV_RESACC): in fp16 the
    halo form, whose residual K blocks bring the tile's un-shifted 16 x 8 pixels through the halo ring."""
    n, c0, cr, cout = shape
    H = 32
    rng = np.random.RandomState(sum(shape) + prec)
    x0 = rng.randn(n, c0, H, H).astype(np.float32)
    xr = rng.randn(n, cr, H, H).astype(np.float32)
    w = (rng.randn(cout, c0, 3, 3) / np.sqrt(c0 * 9)).astype(np.float32)
    wr = (rng.randn(cout, cr) / np.sqrt(cr)).astype(np.float32)
    b = rng.randn(cout).astype(np.float32) * 0.1
    br = rng.randn(cout).astype(np.float32) * 0.1
    if prec == _lib.PREC_TF32:
        x0, xr = tf32_trunc(x0), tf32_trunc(xr)
    else:
        x0, xr, w, wr = f16_round(x0), f16_round(xr), f16_round(w), f16_round(wr)
    got = run_conv_resacc(prec, x0, xr, w, wr, b, br)
    tw = (lambda a: a) if prec == _lib.PREC_F16 else tf32_rna          # (TF32 weights are rounded on the host, activations fed exact)
    y = torch.nn.functional.conv2d(torch.from_numpy(x0).double(), torch.from_numpy(tw(w)).double(), torch.from_numpy(b).double(),
                                   padding=1).relu()
    y = y + torch.nn.functional.conv2d(torch.from_numpy(xr).double(), torch.from_numpy(tw(wr)).double()[:, :, None, None],
                                       torch.from_numpy(br).double())
    want = y.numpy()
    scale = np.abs(want).max()
    K = c0 * 9 + cr
    if prec == _lib.PREC_F16:
        bound = (4e-6 + 4e-9 * K) * scale + 2.0 ** -11 * np.abs(want) + 6e-8
        assert (np.abs(got - want) <= bound).all(), f"max excess {np.max(np.abs(got - want) - bound):.3e}"
    else:
        err = np.abs(got - want).max() / scale
        assert err < 4e-6 + 4e-9 * K, f"max err / max|ref| = {err:.3e}"


# ------------------------------------------------------------------ 2. DiffusionUNet.forward at 64x64
@functools.lru_cache(maxsize=None)
def _fwd_case(C, sf):
    """model, input rows, conditioning variants and the oracle's eps for them (computed once per model)"""
    cfg = Cfg(C, 64, 50)
    model = make_model(cfg, sf, 64 + C + int(sf * 10), device="cuda")
    sd = cpu_sd(model)
    torch.manual_seed(C)
    x = torch.randn(4, C, 64, 64)
    variants = torch.tensor([0, 1, 2, 1], dtype=torch.int32)
    tt = torch.full((1,), 37, dtype=torch.long)
    want = []
    for r in range(4):
        cond = None if variants[r] == 0 else torch.full((1, 1), float(variants[r] - 1))
        want.append(ounet.unet_forward(sd, x[r:r + 1], tt, cond).numpy())
    return model, x, variants, np.concatenate(want)


@pytest.mark.parametrize("prec", PRECS)
@pytest.mark.parametrize("C,sf", [(1, 1.0), (1, 0.3), (3, 1.0), (3, 0.3)])
def test_forward_64_matches_oracle(C, sf, prec):
    model, x, variants, want = _fwd_case(C, sf)
    eng = UNetEngine.for_model(model, 64, 50, prec)
    got = eng.forward(x.cuda(), 37, variants.cuda()).cpu().numpy()
    for r in range(len(x)):
        assert_close(got[r:r + 1], want[r:r + 1], 0.0, FWD_TOL[prec], f"row {r} {C}x64 sf={sf} [{prec}]")
    assert umma_error_flag() == 0


@pytest.mark.parametrize("prec", ["fp32", "tf32x3"])
def test_wider_model_still_runs_after_a_narrower_one_was_packed(prec):
    """k_conv_first's shared-memory limit belongs to the kernel, not to a model: packing the sf 0.5 student (60 KB at 3x64x64)
    after the teacher (66 KB) must not leave the teacher's launches above the limit."""
    teacher, x, variants, want = _fwd_case(3, 1.0)
    student = make_model(Cfg(3, 64, 50), 0.5, 77, device="cuda")
    UNetEngine.invalidate(teacher)
    UNetEngine.invalidate(student)
    et = UNetEngine.for_model(teacher, 64, 50, prec)
    es = UNetEngine.for_model(student, 64, 50, prec)
    es.forward(x[:1].cuda(), 37, variants[:1].cuda())
    got = et.forward(x.cuda(), 37, variants.cuda()).cpu().numpy()
    assert_close(got, want, 0.0, FWD_TOL[prec], f"teacher after the student [{prec}]")
    assert umma_error_flag() == 0


@pytest.mark.parametrize("prec", ["tf32", "f16"])
def test_forward_64_large_batch(prec):
    """160 rows: 5120 enc1 tiles, 1280 halo tiles at the 32x32 level (CTA pairs, many tiles per CTA); sampled rows against
    the oracle, the whole batch against the same rows run in batches of 8 (other launch shapes of the same kernels)."""
    cfg = Cfg(1, 64, 50)
    model = make_model(cfg, 1.0, 65, device="cuda")
    sd = cpu_sd(model)
    torch.manual_seed(6)
    R = 160
    x = torch.randn(R, 1, 64, 64)
    variants = (torch.arange(R) % 3).to(torch.int32)
    eng = UNetEngine.for_model(model, 64, 50, prec)
    got = eng.forward(x.cuda(), 11, variants.cuda()).cpu().numpy()
    tt = torch.full((1,), 11, dtype=torch.long)
    for r in (0, 77, 159):
        cond = None if variants[r] == 0 else torch.full((1, 1), float(variants[r] - 1))
        want = ounet.unet_forward(sd, x[r:r + 1], tt, cond).numpy()
        assert_close(got[r:r + 1], want, 0.0, FWD_TOL[prec], f"row {r} [{prec}]")
    small = np.concatenate([eng.forward(x[i:i + 8].cuda(), 11, variants[i:i + 8].cuda()).cpu().numpy() for i in range(0, R, 8)])
    # (fp16: the CTA-pair and single-CTA forms of a layer sum in different orders; an output may round to the neighbouring
    # fp16 value)
    assert_close(got, small, 0.0, 1e-5 if prec == "tf32" else 1.5e-3, f"160-row batch vs 8-row batches [{prec}]")
    assert umma_error_flag() == 0


@pytest.mark.parametrize("prec", ["fp32", "tf32x3"])
def test_forward_64_four_channels_exact_modes(prec):
    """The exact modes run enc1.conv1 through k_conv_first, which stages the padded 4 x 66 x 66 input and its weights in
    shared memory (80 KB at this width, 90 KB at the teacher's), then enc1.conv2 as a generic conv over the 64x64 map
    (2-row boxes)."""
    cfg = Cfg(4, 64, 50)
    model = make_model(cfg, 0.3, 66, device="cuda")
    sd = cpu_sd(model)
    torch.manual_seed(7)
    x = torch.randn(2, 4, 64, 64)
    variants = torch.tensor([2, 0], dtype=torch.int32)
    eng = UNetEngine.for_model(model, 64, 50, prec)
    got = eng.forward(x.cuda(), 5, variants.cuda()).cpu().numpy()
    tt = torch.full((1,), 5, dtype=torch.long)
    for r in range(2):
        cond = None if variants[r] == 0 else torch.full((1, 1), float(variants[r] - 1))
        assert_close(got[r:r + 1], ounet.unet_forward(sd, x[r:r + 1], tt, cond).numpy(), 0.0, FWD_TOL[prec], f"row {r} [{prec}]")
    assert umma_error_flag() == 0


# ------------------------------------------------------------------ 3. samplers at 3x64x64
def _stack(traj):
    return torch.stack([t[0] if isinstance(t, tuple) else t for t in traj]).cpu().numpy()


def test_s1_p_sample_loop_64():
    """S1 in its default arithmetic (3xTF32), classifier-free guidance: both forwards per step."""
    T = 4
    cfg = Cfg(3, 64, T)
    model = make_model(cfg, 1.0, 67, stress=False, device="cuda")
    torch.manual_seed(21)
    _, want = osmp.s1_p_sample_loop(oracle_fn(model), (1, 3, 64, 64), T, osmp.diffusion_params(T), T, 3.0)
    torch.manual_seed(21)
    _, got = diffusion.p_sample_loop(model, (1, 3, 64, 64), T, diffusion.get_diffusion_params(T, cfg), device="cuda",
                                     config=cfg, track_trajectory=True, guidance_scale=3.0)
    assert_close(_stack(got), _stack(want), RTOL, ATOL, "S1 3x64x64")
    assert umma_error_flag() == 0


def _oracle_pair_metrics(t_frames, s_frames, seed):
    np.random.seed(seed + 1)
    return om.trajectory_metrics([torch.from_numpy(np.ascontiguousarray(f))[None] for f in t_frames],
                                 [torch.from_numpy(np.ascontiguousarray(f))[None] for f in s_frames])


def _check_scalars(got, want, what):
    for k in tm.SCALAR_KEYS:
        np.testing.assert_allclose(got[k], want[k], rtol=RT_METRIC, atol=1e-9, equal_nan=True, err_msg=f"{what}: {k}")


def _s2_oracle_frames(model, x, seeds, ws, T):
    f = oracle_fn(model)
    return np.stack([torch.stack(osmp.s2_generate_trajectory(f, x[p:p + 1], T, seed=seeds[p], guidance_scale=ws[p]))[:, 0].numpy()
                     for p in range(len(seeds))])


def test_s2_compare_trajectories_64():
    """S2 through the reference signature (default fp16 arithmetic): frames against the oracle sampler, the 18 scalars
    against the oracle's metrics of the CUDA frames (D = 12288: the device-drawn Wasserstein subsample sets)."""
    T = 4
    cfg = Cfg(3, 64, T)
    teacher = make_model(cfg, 0.5, 68, device="cuda")
    student = make_model(cfg, 0.3, 69, device="cuda")
    scales = [3.0]
    res = te.compare_trajectories(teacher, student, cfg, guidance_scales=scales, size_factor=0.3, num_samples=2)
    assert umma_error_flag() == 0
    x, seeds, ws = [], [], []
    for s in range(2):
        torch.manual_seed(42 + s)
        noise = torch.randn(1, 3, 64, 64)
        for gs in scales:
            x.append(noise); seeds.append(42 + s); ws.append(gs)
    x = torch.cat(x)
    groups = [0, 1]
    tg = te.generate_trajectories_batched(teacher, x, seeds, ws, T, "cuda", groups=groups).cpu().numpy().copy()
    sg = te.generate_trajectories_batched(student, x, seeds, ws, T, "cuda", groups=groups).cpu().numpy().copy()
    assert_close(tg, _s2_oracle_frames(teacher, x, seeds, ws, T), RTOL, ATOL, "S2 teacher frames")
    assert_close(sg, _s2_oracle_frames(student, x, seeds, ws, T), RTOL, ATOL, "S2 student frames")
    per = [_oracle_pair_metrics(tg[s], sg[s], 42 + s) for s in range(2)]
    _check_scalars(res["student_metrics"][3.0], om.average_scalar_metrics(per), "compare_trajectories 3x64x64")


@pytest.mark.parametrize("prec", ["tf32", "f16"])
def test_s3_trajectory_manager_pair_64(prec, tmp_path):
    T = 4
    cfg = Cfg(3, 64, T)
    cfg.trajectory_dir = str(tmp_path)
    cfg.student_steps = 2
    teacher = make_model(cfg, 0.5, 70, device="cuda")
    student = make_model(cfg, 0.3, 71, device="cuda")
    set_precision(prec, "S3")
    try:
        mgr = TrajectoryManager(teacher, student, cfg, size_factor=0.3)
        tt, st = mgr.generate_trajectory(seed=3)
    finally:
        set_precision("f16", "S3")
    ref_t, ref_s = osmp.s3_generate_pair(oracle_fn(teacher), oracle_fn(student), (1, 3, 64, 64), T, T, 2, seed=3)
    assert [t for _, t in tt] == [t for _, t in ref_t] and [t for _, t in st] == [t for _, t in ref_s]
    assert_close(_stack(tt), _stack(ref_t), RTOL, ATOL, f"S3 teacher [{prec}]")
    assert_close(_stack(st), _stack(ref_s), RTOL, ATOL, f"S3 student [{prec}]")
    assert umma_error_flag() == 0


# ------------------------------------------------------------------ 4. grid.sweep with two students
def test_sweep_two_students_64():
    T = 3
    cfg = Cfg(3, 64, T)
    teacher = make_model(cfg, 0.5, 72, device="cuda")
    students = {sf: make_model(cfg, sf, 1100 + int(sf * 100), device="cuda") for sf in (0.1, 0.3)}
    scales, n_seeds = [1.0, 7.5], 2
    res = grid.sweep(teacher, students, cfg, scales, n_seeds, reduce=False)
    assert umma_error_flag() == 0
    x, seeds, ws = [], [], []
    for s in range(n_seeds):
        torch.manual_seed(42 + s)
        noise = torch.randn(1, 3, 64, 64)
        for gs in scales:
            x.append(noise); seeds.append(42 + s); ws.append(gs)
    x = torch.cat(x)
    groups = [i // len(scales) for i in range(len(seeds))]
    t_gpu = te.generate_trajectories_batched(teacher, x, seeds, ws, T, "cuda", groups=groups).cpu().numpy().copy()
    assert_close(t_gpu, _s2_oracle_frames(teacher, x, seeds, ws, T), RTOL, ATOL, "teacher frames of the sweep")
    for sf, model in students.items():
        s_gpu = te.generate_trajectories_batched(model, x, seeds, ws, T, "cuda", groups=groups).cpu().numpy().copy()
        assert_close(s_gpu, _s2_oracle_frames(model, x, seeds, ws, T), RTOL, ATOL, f"student {sf} frames of the sweep")
        for g, gs in enumerate(scales):
            per = [_oracle_pair_metrics(t_gpu[s * len(scales) + g], s_gpu[s * len(scales) + g], 42 + s) for s in range(n_seeds)]
            _check_scalars(res[sf][gs], om.average_scalar_metrics(per), f"sf={sf} w={gs}")


# ------------------------------------------------------------------ 5. metric kernels at D up to 16384
@pytest.mark.parametrize("D", [4096, 12288, 16384])
def test_numpy_choice_sets_wide_frames(D):
    """dtraj_numpy_choice_sets == np.random.RandomState(seed).choice(D, K, replace=False), L calls per seed, bit for bit;
    seeds at both ends of the 32-bit range, and a seed count that leaves the last block partly empty."""
    K, L = 1000, 3
    seeds = [0, 1, 43, 2 ** 31 - 1, 2 ** 31, 2 ** 32 - 2, 2 ** 32 - 1, 12345, 999]
    sd = torch.tensor(seeds, dtype=torch.int64).to(torch.int32).cuda()
    out = torch.empty(len(seeds), L, K, dtype=torch.int32, device="cuda")
    _lib.check(_lib.load().dtraj_numpy_choice_sets(_lib.ptr(sd), len(seeds), L, D, K, _lib.ptr(out), _lib.stream_ptr()))
    got = out.cpu().numpy()
    for i, s in enumerate(seeds):
        rs = np.random.RandomState(s)
        want = np.stack([rs.choice(D, K, replace=False) for _ in range(L)])
        np.testing.assert_array_equal(got[i], want, err_msg=f"seed {s} D={D}")


def test_choice_sets_refuse_frames_beyond_16384():
    sd = torch.zeros(1, dtype=torch.int32, device="cuda")
    out = torch.empty(1, 1, 10, dtype=torch.int32, device="cuda")
    with pytest.raises(DtrajError, match="16384"):
        _lib.check(_lib.load().dtraj_numpy_choice_sets(_lib.ptr(sd), 1, 1, 16388, 10, _lib.ptr(out), _lib.stream_ptr()))


def test_metric_kernels_at_3x64x64():
    """pair_reductions (frames cut into parts of at most 4096 elements), Wasserstein on the K = 1000 subsample sets and on
    whole frames, and the PCA projection at D = 12288, against the oracle / f64 numpy."""
    D, N, L = 12288, 3, 5
    rng = np.random.RandomState(12288)
    T = np.cumsum(rng.randn(N, L, D).astype(np.float32) * 0.1, axis=1).astype(np.float32)
    S = (T + rng.randn(N, L, D).astype(np.float32) * 0.05).astype(np.float32)
    got = tm.pair_reductions(torch.from_numpy(T).cuda(), torch.from_numpy(S).cuda()).cpu().numpy()
    T64, S64 = T.astype(np.float64), S.astype(np.float64)
    want = np.zeros((N, L, 6))
    want[:, :, 0] = ((T64 - S64) ** 2).sum(-1)
    dT, dS = np.diff(T64, axis=1), np.diff(S64, axis=1)
    want[:, :-1, 1], want[:, :-1, 2], want[:, :-1, 3] = (dT ** 2).sum(-1), (dS ** 2).sum(-1), (dT * dS).sum(-1)
    want[:, 0, 4], want[:, 0, 5] = ((T64[:, -1] - T64[:, 0]) ** 2).sum(-1), ((S64[:, -1] - S64[:, 0]) ** 2).sum(-1)
    np.testing.assert_allclose(got, want, rtol=2e-5, atol=1e-6 * np.abs(want).max())

    idx = te.wasserstein_index_sets_device([42, 43], 50, L, D, "cuda")
    assert idx.shape == (2, L, 1000)
    idx_set = torch.tensor([0, 1, 1], dtype=torch.int32)
    w1 = tm.wasserstein_frames(torch.from_numpy(T).cuda(), torch.from_numpy(S).cuda(), idx, idx_set).cpu().numpy()
    sets = idx.cpu().numpy()
    for n in range(N):
        for i in range(L):
            sel = sets[[0, 1, 1][n], i]
            np.testing.assert_allclose(w1[n, i], om.wasserstein_1d(T[n, i, sel], S[n, i, sel]), rtol=1e-5, atol=1e-7)

    from distillation_trajectories_b200.analysis import trajectory_pca as tp

    class _PCA:                                      # the two attributes project_trajectories reads from a fitted PCA
        components_ = np.linalg.qr(rng.randn(D, 3))[0].T
        mean_ = rng.randn(D) * 0.1

    proj = tp.project_trajectories(torch.from_numpy(T).cuda(), _PCA).cpu().numpy()
    want_p = (T64.reshape(N * L, D) - _PCA.mean_) @ _PCA.components_.T
    np.testing.assert_allclose(proj.reshape(N * L, 3), want_p, rtol=1e-4, atol=1e-4 * np.abs(want_p).max())


# ------------------------------------------------------------------ 6. other sizes are refused
@pytest.mark.parametrize("H", [8, 48, 128])
def test_unsupported_sizes_are_refused(H):
    cfg = Cfg(1, H, 4)
    model = make_model(cfg, 0.1, 73, device="cuda")
    with pytest.raises(DtrajError, match=r"16, 32 or 64"):
        UNetEngine.for_model(model, H, 4, "f16")
