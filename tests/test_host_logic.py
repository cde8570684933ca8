"""CPU: host-side logic of the product package (schedules, coefficients, row layouts, f64 metric
formulas, sharding) checked against the oracle.  No CUDA call is made here."""
import re

import numpy as np
import pytest
import torch

from oracle import metrics as om
from oracle import samplers as osmp
from distillation_trajectories_b200 import sampling, grid
from distillation_trajectories_b200.analysis.metrics import trajectory_metrics as tm
from distillation_trajectories_b200.analysis import trajectory_engine as te
from distillation_trajectories_b200.utils import diffusion, metric_transformations
from distillation_trajectories_b200._lib import VAR_COND0, VAR_COND1, VAR_NONE
from helpers import Cfg, load_golden


@pytest.mark.parametrize("S,Tc", [(50, 50), (100, 50), (4000, 50), (10, 50), (7, 3), (1, 1)])
def test_s1_indices_bit_exact(S, Tc):
    assert sampling.s1_timestep_indices(S, Tc) == osmp.s1_timestep_indices(S, Tc)


@pytest.mark.parametrize("S,steps", [(50, 50), (100, 50), (100, 30), (6, 3), (20, 5)])
def test_s3_indices_bit_exact(S, steps):
    assert sampling.s3_timestep_indices(S, steps) == osmp.s3_timestep_indices(S, steps)


def test_schedule_tables_bit_exact():
    cfg = Cfg(force_cpu=True)
    for T in (1, 6, 50, 1000):
        a = diffusion.get_diffusion_params(T, cfg)
        b = osmp.diffusion_params(T)
        assert sorted(a) == sorted(b)
        for k in a:
            assert torch.equal(a[k].cpu(), b[k]), k


def test_s1_coefficients_bit_exact():
    p = osmp.diffusion_params(50)
    idx = [49, 7, 0, 75, -3]                       # includes out-of-range values: extract() clamps
    got = sampling.s1_coefficients(p, idx)
    for i, (k0, k1, k2) in zip(idx, got):
        t = torch.tensor([i])
        assert k0 == osmp.gather_coef(p["sqrt_recip_alphas"], t, 4).item()
        assert k1 == (1.0 - osmp.gather_coef(p["sqrt_one_minus_alphas_cumprod"], t, 4)).item()
        assert k2 == osmp.gather_coef(p["betas"], t, 4).item()


def test_s2_s3_coefficients_bit_exact():
    ours, ref = sampling.s2_coefficients(50), osmp.s2_coefficients(50)
    for t in range(1, 50):
        assert ours[t] == tuple(c.item() for c in ref[t])
    x, e, z = torch.randn(4), torch.randn(4), torch.randn(4)
    for t, (k0, k1, k2) in zip((49, 10, 1), sampling.s3_coefficients((49, 10, 1), 50)):
        want = osmp.s3_update(x, e, t, z, 50)
        got = (x - k0 * e) / k1 + k2 * z
        assert torch.equal(want, got)


def test_s2_layout():
    rs, rv, ru, rc = sampling.s2_layout([None, 1.0, 3.0, 0.5, 7.5])
    assert rs == [0, 1, 2, 3, 4, 2, 4]
    assert rv == [VAR_NONE, VAR_NONE, VAR_COND0, VAR_NONE, VAR_COND0, VAR_COND1, VAR_COND1]
    assert ru == [0, 1, 2, 3, 4] and rc == [-1, -1, 5, -1, 6]


def _cpu_reductions(T, S):
    """what dtraj_metrics_pairs computes, in numpy (test-side restatement of include/dtraj.h)."""
    T, S = T.astype(np.float64), S.astype(np.float64)
    N, L, D = T.shape
    red = np.zeros((N, L, 6))
    red[:, :, 0] = ((T - S) ** 2).sum(-1)
    dT, dS = np.diff(T, axis=1), np.diff(S, axis=1)
    red[:, :-1, 1], red[:, :-1, 2], red[:, :-1, 3] = (dT ** 2).sum(-1), (dS ** 2).sum(-1), (dT * dS).sum(-1)
    red[:, 0, 4], red[:, 0, 5] = ((T[:, -1] - T[:, 0]) ** 2).sum(-1), ((S[:, -1] - S[:, 0]) ** 2).sum(-1)
    return red.astype(np.float32)


@pytest.mark.parametrize("C,H,L", [(1, 16, 51), (3, 32, 11), (1, 16, 2)])
def test_scalar_metrics_match_oracle(C, H, L):
    rng = np.random.RandomState(1)
    N, D = 3, C * H * H
    T = np.cumsum(rng.randn(N, L, D).astype(np.float32) * 0.1, axis=1)
    S = T + rng.randn(N, L, D).astype(np.float32) * 0.01
    S[1] = T[1]                              # identical pair: zero distances
    T[2, 3:] = T[2, 2:3]                     # teacher stops moving: zero-norm steps are skipped
    S[2, 3:] = S[2, 2:3]
    w1 = np.zeros((N, L))
    want = []
    for n in range(N):
        np.random.seed(10 + n)
        m = om.trajectory_metrics([torch.from_numpy(T[n, i]).reshape(1, C, H, H) for i in range(L)],
                                  [torch.from_numpy(S[n, i]).reshape(1, C, H, H) for i in range(L)])
        want.append(m)
        w1[n] = m["wasserstein_distances"]
    got = tm.scalar_metrics_batched(_cpu_reductions(T, S), w1, H * H, D)
    for n in range(N):
        for k in tm.SCALAR_KEYS:
            np.testing.assert_allclose(got[k][n], want[n][k], rtol=1e-4, atol=1e-9, equal_nan=True, err_msg=f"{k}[{n}]")
        np.testing.assert_allclose(got["path_alignment"][n], want[n]["path_alignment"], rtol=1e-4, atol=1e-30)
        assert got["path_alignment"].dtype == np.float32
        dc = [c for c, ok in zip(got["_cos"][n], got["_cos_ok"][n]) if ok]
        np.testing.assert_allclose(dc, want[n]["directional_consistency"], rtol=1e-4, atol=1e-6)
    assert len(tm.SCALAR_KEYS) == 18 and set(tm.SCALAR_KEYS) == set(om.average_scalar_metrics(want))


def test_wasserstein_index_sets_follow_numpy_global_rng():
    idx = te.wasserstein_index_sets([42, 43], timesteps=5, n_frames=6, numel=3072)
    np.random.seed(44)                       # seed + 1 of the second sample
    for f in range(6):
        assert np.array_equal(idx[1, f], np.random.choice(3072, 1000, replace=False))
    assert te.wasserstein_index_sets([42], 5, 6, 256) is None     # all elements used, order irrelevant


def test_transform_metrics_golden():
    for r in load_golden("transform")["rows"]:
        out = metric_transformations.transform_metrics(*r[:4])
        got = [out["path_length_similarity"], out["trajectory_mse"], out["mean_directional_consistency"],
               out["distribution_similarity"]]
        np.testing.assert_allclose(got, r[4:], rtol=1e-15)
    assert list(out) == ["path_length_similarity", "trajectory_mse", "mean_directional_consistency",
                         "distribution_similarity"]


def test_shard_samples_partition():
    for n, w in ((10, 1), (10, 4), (3, 8), (65536, 8)):
        parts = [grid.shard_samples(n, r, w) for r in range(w)]
        assert sorted(sum(parts, [])) == list(range(n))


def test_cpu_device_is_refused_loudly():
    from distillation_trajectories_b200 import DtrajError
    from helpers import make_model
    cfg = Cfg()
    m = make_model(cfg, 0.05, 1)
    with pytest.raises(DtrajError):
        m(torch.zeros(1, 1, 16, 16), torch.tensor([0]))
    with pytest.raises(DtrajError):
        diffusion.p_sample_loop(m, (1, 1, 16, 16), 4, diffusion.get_diffusion_params(4, Cfg(force_cpu=True)), device="cpu")


def test_product_never_imports_oracle():
    import os
    root = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "distillation_trajectories_b200")
    for dp, _, files in os.walk(root):
        for f in files:
            if f.endswith(".py"):
                src = open(os.path.join(dp, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", src, re.M), os.path.join(dp, f)


def test_s2_first_step_layout_shares_rows_per_group_and_variant():
    """first-step row sharing (sampling.s2_first_step_layout): one row per (group, conditioning variant in use); every
    sample points at the rows of its own group; nothing is shared across groups"""
    from distillation_trajectories_b200 import sampling
    from distillation_trajectories_b200._lib import VAR_COND0, VAR_COND1, VAR_NONE
    ws = [1.0, 2.0, 7.5, None, 20.0]
    S = 4
    guidance = ws * S
    groups = [i for i in range(S) for _ in range(len(ws))]
    rs, rv, ru, rc = sampling.s2_first_step_layout(guidance, groups)
    assert len(rs) == 3 * S and sorted(set(rv)) == sorted({VAR_NONE, VAR_COND0, VAR_COND1})
    full = sampling.s2_layout(guidance)
    assert len(full[0]) == S * (2 + 2 * 3)                       # unshared: 1 row for w <= 1 / None, 2 rows for w > 1
    for b, w in enumerate(guidance):
        g = groups[b]
        assert groups[rs[ru[b]]] == g                             # the row evaluates a member of the same group (same x_T)
        if w is not None and w > 1.0:
            assert rv[ru[b]] == VAR_COND0 and rv[rc[b]] == VAR_COND1 and groups[rs[rc[b]]] == g
        else:
            assert rv[ru[b]] == VAR_NONE and rc[b] == -1
    # all guided samples of a group share the same two rows
    for g in range(S):
        guided = [b for b in range(len(guidance)) if groups[b] == g and guidance[b] is not None and guidance[b] > 1.0]
        assert len({ru[b] for b in guided}) == 1 and len({rc[b] for b in guided}) == 1


def test_shard_samples_blocks_are_contiguous_and_balanced():
    for n, w in ((10, 4), (7, 2), (65536, 8), (5, 8)):
        parts = [grid.shard_samples(n, r, w) for r in range(w)]
        sizes = [len(p) for p in parts]
        assert max(sizes) - min(sizes) <= 1
        for p in parts:
            assert p == list(range(p[0], p[0] + len(p))) if p else True


# ------------------------------------------------------------------ round-2 host logic
def test_weights_checksum_sees_data_writes_that_versions_miss():
    """ADVICE r1: in-place writes through ``.data`` (the EMA idiom) bump neither tensor versions nor data pointers;
    the content checksum of engine.for_model(verify=True) must change, the storage fingerprint must catch ``p.data = new``."""
    from distillation_trajectories_b200 import engine
    from helpers import make_model
    m = make_model(Cfg(1, 16, 4), 0.05, 3)
    fp0, cs0 = engine._weights_fingerprint(m), engine._weights_checksum(m)
    assert engine._weights_checksum(m) == cs0                       # deterministic
    p = m.enc2.conv1.weight
    p.data.mul_(0.999).add_(1e-3)                                    # EMA-style update: version stays 0
    assert engine._weights_fingerprint(m) == fp0 and engine._weights_checksum(m) != cs0
    cs1 = engine._weights_checksum(m)
    p.data = p.data.clone()                                          # same values, new storage
    assert engine._weights_fingerprint(m) != fp0 and engine._weights_checksum(m) == cs1
    m.dec1.norm2.running_var.data.add_(0.5)                          # buffers count too
    assert engine._weights_checksum(m) != cs1


def test_s3_repeated_zero_timesteps_are_frame_copies_not_errors(monkeypatch):
    """ADVICE r1: steps > sample_steps gives stride 0 and the index list [0, ..., 0, S-1] (utils/trajectory_manager.py:88-96);
    the reference stores one frame per entry and never updates at t == 0 -- the drop-in must not raise."""
    assert sampling.s3_timestep_indices(4, 6) == osmp.s3_timestep_indices(4, 6) == [0, 0, 0, 0, 0, 0, 3]
    calls = []

    def fake_sampler(engine, key, factory):
        calls.append(key)

        class S:
            n_updates = 1
            z_index = torch.zeros(1, 2, dtype=torch.int32)
            z_bank = torch.zeros(2, 256)
            traj = torch.arange(2 * 2 * 256, dtype=torch.float32).reshape(2, 2, 1, 16, 16)

            def run(self):
                return self.traj
        return S()

    class Eng:
        device = torch.device("cpu")
    monkeypatch.setattr(sampling, "cached_sampler", fake_sampler)
    out = sampling.s3_sample(Eng(), torch.zeros(2, 1, 16, 16), [3, 0, 0, 0, 0, 0, 0], 6, torch.zeros(1, 2, 1, 16, 16))
    assert out.shape == (2, 7, 1, 16, 16) and calls[0][2] == (3,)                    # one update, six copies of its result
    for k in range(2, 7):
        assert torch.equal(out[:, k], out[:, 1])
    with pytest.raises(ValueError):
        sampling.s3_sample(Eng(), torch.zeros(2, 1, 16, 16), [3, 0, 2, 0], 6, torch.zeros(2, 2, 1, 16, 16))


def test_oracle_matches_reference_batch_metrics_fixture():
    """E2 pin on the CPU side: the oracle's per-pair metrics reproduce every list the unmodified reference's
    compute_trajectory_metrics_batch returned (tests/golden/batch_metrics.npz, oracle/make_golden_batch.py)."""
    g = load_golden("batch_metrics")
    lists = {"wasserstein_distances": "mean_wasserstein", "endpoint_distances": "endpoint_distance",
             "teacher_path_lengths": "teacher_path_length", "student_path_lengths": "student_path_length",
             "teacher_efficiency": "teacher_efficiency", "student_efficiency": "student_efficiency"}
    same = ["path_length_similarity", "efficiency_similarity", "mean_velocity_similarity", "mean_directional_consistency",
            "mean_position_difference", "distribution_similarity"]
    for name in ("b16", "b32"):
        n = int(g[f"{name}/meta"][4])
        np.random.seed(7)
        per = []
        for i in range(n):
            t = [(torch.from_numpy(a), int(ts)) for a, ts in zip(g[f"{name}/teacher"][i], g[f"{name}/teacher_t"])]
            s = [(torch.from_numpy(a), int(ts)) for a, ts in zip(g[f"{name}/student"][i], g[f"{name}/student_t"])]
            per.append(om.trajectory_metrics(t, s))
        for dst, src in list(lists.items()) + [(k, k) for k in same]:
            np.testing.assert_allclose([m[src] for m in per], g[f"{name}/m/{dst}"], rtol=1e-6, atol=1e-9, err_msg=f"{name}/{dst}")
            np.testing.assert_allclose(np.mean([m[src] for m in per]), g[f"{name}/m/{dst}_avg"], rtol=1e-6, atol=1e-9)
        np.testing.assert_allclose([m["wasserstein_distances"] for m in per], g[f"{name}/m/wasserstein_distances_per_timestep"],
                                   rtol=1e-6, atol=1e-9)


def test_pack_reader_memory_maps_the_big_arrays(tmp_path):
    """ADVICE r1: np.load(mmap_mode=) is ignored for .npz archives; read_pack maps the stored members itself."""
    from distillation_trajectories_b200.utils import trajectory_store as store
    T = np.random.RandomState(0).randn(5, 4, 1, 16, 16).astype(np.float32)
    S = np.random.RandomState(1).randn(5, 3, 1, 16, 16).astype(np.float32)
    p = store.write_pack(str(tmp_path), 0.3, [2, 3, 4, 5, 6], T, S, [3, 2, 1, 0], [3, 1, 0])
    r = store.read_pack(p)
    assert isinstance(r["teacher"], np.memmap) and isinstance(r["student"], np.memmap)
    assert np.array_equal(r["teacher"], T) and np.array_equal(r["student"], S) and list(r["samples"]) == [2, 3, 4, 5, 6]
    assert np.array_equal(store.read_pack(p, mmap=False)["teacher"], T)
    assert store.stored_samples(str(tmp_path), 0.3) == {2, 3, 4, 5, 6}


def test_staged_reference_is_byte_identical_and_complete():
    """oracle/_ref (what bench.py --impl reference times on the GPU box) holds unmodified copies of the reference files."""
    import hashlib
    import os
    from oracle import sync_ref
    if not os.path.isfile(os.path.join(sync_ref.SRC, "models.py")):
        pytest.skip("reference tree not present")
    assert sync_ref.sync() == sync_ref.FILES and sync_ref.staged()
    for rel in sync_ref.FILES:
        a = hashlib.sha256(open(os.path.join(sync_ref.SRC, rel), "rb").read()).hexdigest()
        b = hashlib.sha256(open(os.path.join(sync_ref.DST, rel), "rb").read()).hexdigest()
        assert a == b, rel
    tracked = os.popen(f"git -C {os.path.dirname(sync_ref.DST)} ls-files _ref").read().strip()
    assert tracked == "", "oracle/_ref must stay out of the git history"


def test_model_aliases_match_the_reference_constructors():
    """M4 (models.py:227-242): SimpleUNet / StudentUNet create the same parameters as the reference's aliases: the names, shapes,
    per-tensor sums and widths stored in tests/golden/reference_checks.npz, and the reference's own parameters when present."""
    import contextlib
    import io
    from oracle import make_golden_reference_checks as mk
    from oracle import refload
    g = load_golden("reference_checks")
    cfg = refload.RefConfig(1, 16, 8)
    ref = refload.load() if refload.available() else None
    for which in ("simple", "student"):
        with contextlib.redirect_stdout(io.StringIO()):
            torch.manual_seed(4)
            b = mk.ours_alias(cfg, which)
            if ref is not None:
                torch.manual_seed(4)
                a = ref.models.SimpleUNet(cfg) if which == "simple" else ref.models.StudentUNet(cfg, 0.3, "tiny")
        if ref is not None:             # the reference's own constructors, in this process: exact
            sa, sb = a.state_dict(), b.state_dict()
            assert list(sa) == list(sb) and all(torch.equal(sa[k], sb[k]) for k in sa)
            assert a.dims == b.dims and a.time_emb_dim == b.time_emb_dim
        mk.check_weights(b, g, f"alias/{which}/weights/")
        assert list(b.dims) == list(g[f"alias/{which}/dims"]) and b.time_emb_dim == int(g[f"alias/{which}/time_emb_dim"]), which


def test_bench_flop_counts_match_the_survey_and_the_reference_layers():
    """bench.conv_flops_per_forward: the standard 2 x MACs of the eight blocks' convs (SURVEY.md 8d: 0.404 of 0.423 GFLOP per row at 16x16,
    1.62 of 1.69 at 32x32 for the 3x3 convs) -- checked against a count taken from the model's own Conv2d modules -- and the executed
    count of the position-major tiles (taps outside a <= 4x4 map skipped)."""
    import contextlib
    import io
    import bench
    from distillation_trajectories_b200 import models as ours
    for cfg, H, C in ((bench.Cfg, 16, 1), (bench.Cfg32, 32, 3)):
        with contextlib.redirect_stdout(io.StringIO()):
            m = ours.DiffusionUNet(cfg, 1.0)
        # every Conv2d of the eight blocks at its level's map size (models.py:138-157, 205-217)
        sizes = {"enc1": H, "enc2": H // 2, "enc3": H // 4, "enc4": H // 8, "bottleneck": H // 16, "dec3": H // 8, "dec2": H // 4, "dec1": H // 2}
        want = 0.0
        for name, mod in m.named_modules():
            if isinstance(mod, torch.nn.Conv2d) and name.split(".")[0] in sizes:
                h = sizes[name.split(".")[0]]
                want += 2.0 * h * h * mod.in_channels * mod.out_channels * mod.kernel_size[0] * mod.kernel_size[1]
        got = bench.conv_flops_per_forward(m.dims, C, H, False)
        assert abs(got - want) <= 1e-9 * want, (H, got, want)
        ex = bench.conv_flops_per_forward(m.dims, C, H, True)
        assert 0.85 * got < ex < got
    assert abs(bench.conv_flops_per_forward([128, 256, 256, 256], 1, 16, False) / 1e9 - 0.4219) < 1e-3
    # a 2x2 map meets 4 of the 9 taps, a 4x4 map 6.25 on average, a 1x1 map the centre tap only
    d = [8, 8, 8, 8]
    blocks_32 = bench.conv_flops_per_forward(d, 8, 32, True)
    assert blocks_32 < bench.conv_flops_per_forward(d, 8, 32, False)
