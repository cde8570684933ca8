"""GPU: the three samplers through the public drop-in entry points against the committed reference
trajectories (tests/golden) and, at BASELINE sizes, against the CPU oracle with identical noise.

Tolerance (north_star): rtol 1e-3 on trajectories.  Stated precisely: |got - ref| <= 1e-3 |ref| +
1e-4 max|ref| elementwise (the absolute term covers elements near zero).
"""
import contextlib
import io

import numpy as np
import pytest
import torch

from oracle import samplers as osmp
from distillation_trajectories_b200 import sampling, set_precision, umma_error_flag
from distillation_trajectories_b200.analysis import trajectory_engine as te
from distillation_trajectories_b200.utils import diffusion
from distillation_trajectories_b200.utils.trajectory_manager import TrajectoryManager
from helpers import Cfg, assert_close, golden_models, make_model, oracle_fn

pytestmark = pytest.mark.gpu
RTOL, ATOL = 1e-3, 1e-4


@pytest.fixture(autouse=True)
def cpu_noise():
    """draw noise with the CPU generator, as the reference run that made the fixtures did"""
    sampling.set_noise_device("cpu")
    yield
    sampling.set_noise_device(None)


@pytest.fixture(scope="module", params=["tiny16", "tiny32"])
def case(request):
    return golden_models(request.param, device="cuda")


def stack(traj):
    return torch.stack([t[0] if isinstance(t, tuple) else t for t in traj]).cpu().numpy()


@pytest.mark.parametrize("prec", ["fp32", "tf32x3"])
def test_s1_p_sample_loop_fixture(case, prec):
    g, cfg, teacher, _ = case
    C, H, T = cfg.channels, cfg.image_size, cfg.timesteps
    set_precision(prec, "S1")
    params = diffusion.get_diffusion_params(T, cfg)
    for w in (3.0, 1.0):
        torch.manual_seed(5)
        img, traj = diffusion.p_sample_loop(teacher, (2, C, H, H), T, params, device="cuda", config=cfg,
                                            track_trajectory=True, guidance_scale=w)
        assert len(traj) == T + 1 and all(f.device.type == "cpu" for f in traj) and img.device.type == "cuda"
        assert_close(stack(traj), g[f"s1_w{w}"], RTOL, ATOL, f"S1 w={w} [{prec}]")
        assert torch.equal(img.cpu(), traj[-1])
    torch.manual_seed(6)            # strided: sample_steps = 3T, config.timesteps = T
    _, traj = diffusion.p_sample_loop(teacher, (2, C, H, H), 3 * T, diffusion.get_diffusion_params(3 * T, cfg),
                                      device="cuda", config=cfg, track_trajectory=True, guidance_scale=2.0)
    assert_close(stack(traj), g["s1_strided"], RTOL, ATOL, f"S1 strided [{prec}]")
    set_precision("tf32x3", "S1")
    assert umma_error_flag() == 0


def test_s1_p_sample_single_step(case):
    g, cfg, teacher, _ = case
    C, H, T = cfg.channels, cfg.image_size, cfg.timesteps
    params = diffusion.get_diffusion_params(T, cfg)
    f = oracle_fn(teacher)
    torch.manual_seed(11)
    x = torch.randn(2, C, H, H)
    for tval in (T - 1, 0):
        t = torch.full((2,), tval, dtype=torch.long)
        torch.manual_seed(12)
        want = osmp.s1_p_sample(f, x, t, tval, osmp.diffusion_params(T), 2.5)
        torch.manual_seed(12)
        got = diffusion.p_sample(teacher, x.cuda(), t.cuda(), tval, params, 2.5)
        assert_close(got.cpu().numpy(), want.numpy(), RTOL, ATOL, f"p_sample t={tval}")


@pytest.mark.parametrize("prec", ["fp32", "tf32x3", "tf32", "f16"])
def test_s2_generate_trajectory_fixture(case, prec):
    g, cfg, teacher, student = case
    set_precision(prec, "S2")
    noise = torch.from_numpy(g["s2_noise"])
    for who, model in (("teacher", teacher), ("student", student)):
        for w in (None, 1.0, 3.0, 7.5):
            traj = te.generate_trajectory(model, noise, cfg.timesteps, "cuda", seed=42, guidance_scale=w)
            assert len(traj) == cfg.timesteps + 1 and all(f.device.type == "cpu" and f.shape == noise.shape for f in traj)
            assert torch.equal(traj[-1], traj[-2]) and torch.equal(traj[0], noise)
            assert_close(stack(traj), g[f"s2_{who}_w{w}"], RTOL, ATOL, f"S2 {who} w={w} [{prec}]")
    set_precision("f16", "S2")
    assert umma_error_flag() == 0


@pytest.mark.parametrize("prec", ["fp32", "tf32", "f16"])
def test_s3_trajectory_manager_fixture(case, prec, tmp_path):
    g, cfg, teacher, student = case
    T = cfg.timesteps
    set_precision(prec, "S3")
    cfg.trajectory_dir = str(tmp_path)
    for tag, ss in (("eq", T), ("uneq", max(2, T // 2))):
        cfg.sample_steps, cfg.teacher_steps, cfg.student_steps = T, T, ss
        mgr = TrajectoryManager(teacher, student, cfg, size_factor=0.5)
        tt, st = mgr.generate_trajectory(seed=3)
        assert [t for _, t in tt] == list(g[f"s3_{tag}_teacher_t"]) and [t for _, t in st] == list(g[f"s3_{tag}_student_t"])
        assert all(x.device.type == "cuda" for x, _ in tt)
        assert_close(stack(tt), g[f"s3_{tag}_teacher"], RTOL, ATOL, f"S3 {tag} teacher [{prec}]")
        assert_close(stack(st), g[f"s3_{tag}_student"], RTOL, ATOL, f"S3 {tag} student [{prec}]")
    cfg.sample_steps = cfg.teacher_steps = cfg.student_steps = T
    set_precision("f16", "S3")


# ------------------------------------------------------------------ BASELINE-size cases vs the oracle
def test_s1_config1_batch64_teacher():
    """BASELINE config 1: teacher 1x16x16, 50 steps, batch 64, w = 1.0 (both forwards still run)."""
    cfg = Cfg(1, 16, 50)
    model = make_model(cfg, 1.0, 0, stress=False, device="cuda")
    torch.manual_seed(123)
    tap = []
    _, want = osmp.s1_p_sample_loop(oracle_fn(model), (64, 1, 16, 16), 50, osmp.diffusion_params(50), 50, 1.0, noise_tap=tap)
    torch.manual_seed(123)
    _, got = diffusion.p_sample_loop(model, (64, 1, 16, 16), 50, diffusion.get_diffusion_params(50, cfg), device="cuda",
                                     config=cfg, track_trajectory=True, guidance_scale=1.0)
    assert_close(stack(got), stack(want), RTOL, ATOL, "S1 config 1")
    assert umma_error_flag() == 0


@pytest.mark.parametrize("prec", ["tf32", "f16"])
@pytest.mark.parametrize("C,H,sf,w", [(1, 16, 1.0, 7.5), (1, 16, 0.5, 20.0), (3, 32, 1.0, 7.5), (3, 32, 0.1, 7.5)])
def test_s2_full_length_vs_oracle(C, H, sf, w, prec):
    """BASELINE configs 2-3: 50 steps with CFG, in the two fast arithmetic modes (single-pass TF32, fp16)."""
    set_precision(prec, "S2")
    cfg = Cfg(C, H, 50)
    model = make_model(cfg, sf, 1000 + int(sf * 100), stress=False, device="cuda")
    torch.manual_seed(42)
    noise = torch.randn(1, C, H, H)
    want = osmp.s2_generate_trajectory(oracle_fn(model), noise, 50, seed=42, guidance_scale=w)
    got = te.generate_trajectory(model, noise, 50, "cuda", seed=42, guidance_scale=w)
    set_precision("f16", "S2")
    assert_close(stack(got), stack(want), RTOL, ATOL, f"S2 {C}x{H} sf={sf} w={w} [{prec}]")
    assert umma_error_flag() == 0


def test_s2_batched_equals_single():
    """the batched loop (per-sample guidance, shared noise bank) reproduces batch-1 calls"""
    cfg = Cfg(1, 16, 8)
    model = make_model(cfg, 0.2, 5, device="cuda")
    seeds, ws = [42, 42, 43, 44], [1.0, 7.5, 3.0, None]
    noises = []
    for s in seeds:
        torch.manual_seed(s)
        noises.append(torch.randn(1, 1, 16, 16))
    batched = te.generate_trajectories_batched(model, torch.cat(noises), seeds, ws, 8, "cuda").cpu().numpy()
    for b, (s, w) in enumerate(zip(seeds, ws)):
        single = stack(te.generate_trajectory(model, noises[b], 8, "cuda", seed=s, guidance_scale=w))[:, 0]
        np.testing.assert_array_equal(batched[b], single)


def test_graph_and_eager_loops_agree():
    """the captured and the eager loop give the same frames and report the same launch count, and that count is the
    number of launches an un-captured run performs.  Second case: at 16x16, the pool after enc3 (4x4 map) is fused into
    its conv at <= 1152 forward rows and a kernel of its own above that, so with first-step sharing (1280 rows, 160 at
    step 0) step 0 launches one kernel fewer than the other steps."""
    from distillation_trajectories_b200.engine import UNetEngine
    torch.manual_seed(1)
    seeds, scales = 80, [1.5, 2.0, 3.0, 4.0, 5.0, 6.0, 7.5, 10.0]
    cases = [  # (precision, T, x_T, guidance, groups, noise bank rows)
        ("tf32", 6, torch.randn(3, 1, 16, 16), [2.0, None, 7.5], None, 15),
        ("f16", 4, torch.randn(seeds, 1, 16, 16).repeat_interleave(len(scales), dim=0), scales * seeds,
         [i for i in range(seeds) for _ in scales], 64),
    ]
    for seed, (prec, T, x, guidance, groups, n_bank) in enumerate(cases):
        eng = UNetEngine.for_model(make_model(Cfg(1, 16, T), 0.1 if seed == 0 else 0.2, 9 + seed, device="cuda"), 16, T, prec)
        B = x.shape[0]
        bank = torch.randn(n_bank, 256)
        zi = np.random.RandomState(seed).randint(0, n_bank, size=(T - 1, B)).astype(np.int32)
        frames, samplers = [], []
        for use_graph in (True, False):
            frames.append(sampling.s2_sample(eng, x, T, guidance, bank, zi, use_graph=use_graph, groups=groups).cpu().numpy().copy())
            samplers.append(next(reversed(eng._samplers.values())))
        np.testing.assert_array_equal(frames[0], frames[1])
        graph, eager = samplers
        assert graph is not eager and graph.n_rows == eager.n_rows
        if groups is not None:
            assert eager.n_rows > 1152 >= len(eager.first[0]), (eager.n_rows, len(eager.first[0]))
        assert graph.launches == eager.launches, (prec, graph.launches, eager.launches)
        for s in samplers:
            assert s.launches == sum(s.profile()["launches"]), (prec, s.launches, s.profile()["launches"])
    assert umma_error_flag() == 0


def test_private_generators_reproduce_global_seeding():
    """the batched sweep draws with per-device private generators; the streams must equal what
    torch.manual_seed(k); torch.randn(...) gives on that device (analysis/trajectory_engine.py:88-95)"""
    for dev in ("cpu", "cuda"):
        g = te._generator(torch.device(dev))
        for k in (0, 43, 91, 12345):
            g.manual_seed(k)
            a = torch.randn(1, 3, 32, 32, device=dev, generator=g)
            torch.manual_seed(k)
            b = torch.randn(1, 3, 32, 32, device=dev)
            assert torch.equal(a, b), (dev, k)


def test_f16_overflow_is_reported_not_hidden():
    """fp16 mode: activations beyond 65504 must surface as DtrajError at the read-back, never as silent inf/NaN frames"""
    from distillation_trajectories_b200 import DtrajError
    cfg = Cfg(1, 16, 4)
    model = make_model(cfg, 0.2, 21, device="cuda")
    with torch.no_grad():
        model.enc2.conv1.weight.mul_(3e4)          # folded weights stay inside the fp16 range, the activations do not
    torch.manual_seed(1)
    noise = torch.randn(1, 1, 16, 16)
    set_precision("f16", "S2")
    with pytest.raises(DtrajError, match="fp16 range"):
        te.generate_trajectory(model, noise, 4, "cuda", seed=1, guidance_scale=2.0)
    assert umma_error_flag() == 0                  # the check clears the sticky flag
    traj = te.generate_trajectory(make_model(cfg, 0.2, 21, device="cuda"), noise, 4, "cuda", seed=1, guidance_scale=2.0)
    assert all(torch.isfinite(f).all() for f in traj)


@pytest.mark.parametrize("prec", ["tf32", "f16"])
def test_first_step_row_sharing_is_exact(prec):
    """samples of one group start from the same x_T: sharing their first-step forward rows (3 rows per group instead of
    up to 2 per sample) must reproduce the unshared loop bit for bit"""
    from distillation_trajectories_b200.engine import UNetEngine
    cfg = Cfg(1, 16, 7)
    model = make_model(cfg, 0.2, 23, device="cuda")
    eng = UNetEngine.for_model(model, 16, 7, prec)
    torch.manual_seed(2)
    ws = [1.0, 2.0, 7.5, None, 20.0]
    G, S = len(ws), 6
    x = torch.randn(S, 1, 16, 16).repeat_interleave(G, dim=0)
    guidance = ws * S
    groups = [i for i in range(S) for _ in range(G)]
    bank = torch.randn(6 * 4, 256)
    zi = np.random.RandomState(0).randint(0, 24, size=(6, S * G)).astype(np.int32)
    a = sampling.s2_sample(eng, x, 7, guidance, bank, zi, groups=groups).cpu().numpy().copy()
    b = sampling.s2_sample(eng, x, 7, guidance, bank, zi, groups=None).cpu().numpy()
    np.testing.assert_array_equal(a, b)
    assert umma_error_flag() == 0
