"""GPU: metrics of teacher / student trajectories whose frames differ in H x W (trajectory_metrics.py:40-52: every
student frame bilinearly resized to the teacher's size, align_corners=True).  The resampled kernels against f64
references of the resized student and against the ragged / equal-size kernels fed with F.interpolate's output; the
drop-in wrappers against the CPU oracle; batched pairs and pickles against the per-pair entry point, including the
global numpy RNG state they leave behind and the number of launches."""
import pickle

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import metrics as om
from distillation_trajectories_b200 import _lib
from distillation_trajectories_b200.analysis import trajectory_engine as te
from distillation_trajectories_b200.analysis.metrics import trajectory_metrics as tm
from distillation_trajectories_b200.utils.trajectory_manager import TrajectoryManager
from helpers import Cfg

pytestmark = pytest.mark.gpu
RT = 1e-4
EPS32 = 2.0 ** -23


@pytest.fixture(autouse=True)
def _error_word_stays_zero():
    yield
    torch.cuda.synchronize()
    assert _lib.load().dtraj_debug_umma_error() == 0


def _resize(x, C_, hw_from, hw_to, dtype=torch.float32):
    """[N, L, C*Hs*Ws] -> [N, L, C*Ht*Wt] through the reference's call."""
    N, L, _ = x.shape
    y = F.interpolate(x.reshape(N * L, C_, *hw_from).to(dtype), size=tuple(hw_to), mode="bilinear", align_corners=True)
    return y.reshape(N, L, -1)


def _want(T, S, delta):
    """f64 restatement of dtraj_metrics_pairs_resampled for T [N, LT, D] and the resized student S [N, LS, D], and for
    each entry a bound of what an error of at most delta[n] in every resized student value can change."""
    N, LT, _ = T.shape
    LS = S.shape[1]
    n, Lm = min(LT, LS), max(LT, LS)
    w = torch.zeros(N, Lm, 8, dtype=torch.float64, device=T.device)
    e = torch.zeros_like(w)
    d = delta.reshape(N, 1, 1)
    sq = lambda a: (a * a).sum(-1)
    err = lambda a, k: (k * d * (2 * a.abs() + k * d)).sum(-1)          # |sum a^2 - sum (a + k delta)^2| at most
    a = T[:, :n] - S[:, :n]
    w[:, :n, 0], e[:, :n, 0] = sq(a), err(a, 1)
    w[:, :LT - 1, 1] = sq(T.diff(dim=1))
    a = S.diff(dim=1)
    w[:, :LS - 1, 2], e[:, :LS - 1, 2] = sq(a), err(a, 2)
    dT = T[:, :n].diff(dim=1)
    w[:, :n - 1, 3] = (dT * S[:, :n].diff(dim=1)).sum(-1)
    e[:, :n - 1, 3] = 2 * d[:, :, 0] * dT.abs().sum(-1)
    w[:, 0, 4] = sq(T[:, -1] - T[:, 0])
    a = S[:, -1] - S[:, 0]
    w[:, 0, 5], e[:, 0, 5] = sq(a), err(a[:, None], 2)[:, 0]
    a = T[:, -1] - S[:, -1]
    w[:, 0, 6], e[:, 0, 6] = sq(a), err(a[:, None], 1)[:, 0]
    longer, shorter = (T, S) if LT >= LS else (S, T)
    lt, st = np.linspace(0, 1, Lm), np.linspace(0, 1, n)
    p = np.clip(np.searchsorted(lt, st, side="right") - 1, 0, Lm - 2)          # np.interp's rule, in f64
    f = torch.from_numpy((st - lt[p]) / (lt[p + 1] - lt[p])).to(T.device).reshape(1, n, 1)
    p = torch.from_numpy(p).to(T.device)
    a = (1 - f) * longer[:, p] + f * longer[:, p + 1] - shorter
    w[:, :n, 7], e[:, :n, 7] = sq(a), err(a, 2)
    return w, e


def _zero_mask(LT, LS):
    """Entries of the [max(LT, LS), 8] layout that include/dtraj.h defines as 0."""
    n, Lm = min(LT, LS), max(LT, LS)
    m = np.ones((Lm, 8), bool)
    m[:n, 0] = m[:LT - 1, 1] = m[:LS - 1, 2] = m[:n - 1, 3] = m[:n, 7] = False
    m[0, 4:7] = False
    return m


def _trajs(gen, N, L, D, dev):
    return (torch.randn(N, L, D, generator=gen, device=dev).cumsum(1) * 0.05
            + torch.randn(N, 1, D, generator=gen, device=dev)).contiguous()


@pytest.mark.parametrize("LT,LS", [(51, 51), (51, 26), (26, 51), (5, 4)])
@pytest.mark.parametrize("C_", [1, 3])
@pytest.mark.parametrize("Ht,Hs", [(32, 16), (16, 32), (64, 32), (32, 64), (16, 64)])
def test_resampled_reductions_vs_f64(Ht, Hs, C_, LT, LS):
    """300 pairs: 300 groups at 3x16x16 (8 pairs per block), 900 band groups at 3x64x64 (three bands of one channel)."""
    dev = torch.device("cuda")
    gen = torch.Generator(device=dev).manual_seed(Ht * 1000 + Hs * 10 + C_ + LT * 7 + LS)
    N = 300
    T = _trajs(gen, N, LT, C_ * Ht * Ht, dev)
    S = _trajs(gen, N, LS, C_ * Hs * Hs, dev)
    got = tm.pair_reductions_resampled(T, S, (Ht, Ht), (Hs, Hs)).double()
    # F.interpolate on fp32 frames, as the reference calls it: the same fp32 tap positions and weights as the kernel, whose
    # resized values may differ from it by the rounding of the weighted sum, a few ulp of max|S|
    delta = 8 * EPS32 * S.abs().amax(dim=(1, 2)).double()
    want, bound = _want(T.double(), _resize(S, C_, (Hs, Hs), (Ht, Ht)).double(), delta)
    assert got.shape == want.shape
    for q in range(8):
        g, w, b = got[:, :, q], want[:, :, q], bound[:, :, q]
        tol = 2e-5 * w.abs() + 2e-6 * w.abs().max() + b + 1e-30
        assert ((g - w).abs() <= tol).all(), (q, float(((g - w).abs() - tol).max()))
    zero = torch.from_numpy(_zero_mask(LT, LS)).to(dev)
    assert (got[:, zero] == 0).all()


@pytest.mark.parametrize("LT,LS", [(9, 9), (9, 5), (5, 9)])
@pytest.mark.parametrize("Hs", [32, 16])
def test_resampled_equals_ragged_of_interpolated(LT, LS, Hs):
    """3x64x64 teachers (12288 elements: three row bands) against 3x32x32 / 3x16x16 students: the same numbers as the
    ragged kernel (equal lengths: the equal-size kernel too) fed with F.interpolate's fp32 output."""
    dev = torch.device("cuda")
    gen = torch.Generator(device=dev).manual_seed(LT * 31 + LS + Hs)
    N = 64
    T = torch.randn(N, LT, 3 * 64 * 64, generator=gen, device=dev)
    S = torch.randn(N, LS, 3 * Hs * Hs, generator=gen, device=dev)
    got = tm.pair_reductions_resampled(T, S, (64, 64), (Hs, Hs))
    Sr = _resize(S, 3, (Hs, Hs), (64, 64)).contiguous()
    want = tm.pair_reductions_ragged(T, Sr)
    for q in range(8):
        torch.testing.assert_close(got[..., q], want[..., q], rtol=0, atol=1e-6 * float(want[..., q].abs().max()) + 1e-30)
    if LT == LS:
        eq = tm.pair_reductions(T, Sr)
        for q in range(6):
            torch.testing.assert_close(got[..., q], eq[..., q], rtol=0, atol=1e-6 * float(eq[..., q].abs().max()) + 1e-30)


@pytest.mark.parametrize("LT,LS", [(7, 7), (9, 4), (4, 9)])
@pytest.mark.parametrize("shape_t,shape_s", [((3, 32, 32), (3, 16, 16)), ((3, 16, 16), (3, 32, 32)),
                                             ((1, 16, 16), (1, 24, 20)), ((2 * 3, 64, 64), (2 * 3, 32, 32))])
def test_resampled_wasserstein(LT, LS, shape_t, shape_s):
    """Host index sets of draw_index_sets and device index sets of dtraj_numpy_choice_sets (teacher-frame indices), and
    all elements of a 256-element teacher; (6, 64, 64) is a frame of two 3x64x64 images."""
    dev = torch.device("cuda")
    gen = torch.Generator(device=dev).manual_seed(LT * 10 + LS + shape_t[1])
    N, n = 6, min(LT, LS)
    Dt, Ds = int(np.prod(shape_t)), int(np.prod(shape_s))
    T = torch.randn(N, LT, Dt, generator=gen, device=dev)
    S = torch.randn(N, LS, Ds, generator=gen, device=dev) * 1.3
    hw = (shape_t[1:], shape_s[1:])
    Sr = _resize(S, shape_s[0], shape_s[1:], shape_t[1:]).contiguous()
    np.random.seed(3)
    sets = [(None, None)]
    if Dt > 1000:
        host = torch.from_numpy(np.stack([tm.draw_index_sets(n, Dt) for _ in range(3)]))
        sets = [(host, torch.tensor([0, 2, 1, 1, 0, 2], dtype=torch.int32))]
        if Dt <= 16384:                                                    # dtraj_numpy_choice_sets' limit
            device = te.wasserstein_index_sets_device([11, 12], 1, n, Dt, dev)
            sets.append((device, torch.tensor([1, 0, 0, 1, 1, 0], dtype=torch.int32)))
    for idx, idx_set in sets:
        got = tm.wasserstein_frames(T, S, idx, idx_set, frame_hw=hw)
        want = tm.wasserstein_frames(T, Sr, idx, idx_set)
        assert got.shape == (N, n)
        torch.testing.assert_close(got, want, rtol=1e-6, atol=0)


def _frames(x, shape, tuples):
    fr = [torch.from_numpy(x[i].reshape(shape)).cuda() for i in range(x.shape[0])]
    return [(f, i) for i, f in enumerate(fr)] if tuples else fr


def _check_oracle(m, o):
    assert list(m.keys()) == list(o.keys())
    for k in o:
        assert type(m[k]) is type(o[k]), (k, type(m[k]), type(o[k]))
        np.testing.assert_allclose(np.asarray(m[k], np.float64), np.asarray(o[k], np.float64), rtol=RT, atol=1e-7,
                                   equal_nan=True, err_msg=k)


def _same_rng(a, b):
    return a[0] == b[0] and np.array_equal(a[1], b[1]) and a[2:] == b[2:]


def _smooth(rng, L, D, scale=0.01):
    return (np.cumsum(rng.randn(L, D), axis=0) * scale + rng.randn(1, D) * 0.1).astype(np.float32)


@pytest.mark.parametrize("tuples", [True, False])
@pytest.mark.parametrize("LT,LS", [(11, 11), (11, 6), (6, 11)])
@pytest.mark.parametrize("shape_t,shape_s", [((1, 3, 32, 32), (1, 3, 16, 16)), ((1, 3, 16, 16), (1, 3, 32, 32)),
                                             ((2, 1, 32, 32), (2, 1, 64, 64)), ((1, 3, 64, 64), (1, 3, 32, 32))])
def test_compute_trajectory_metrics_resized_vs_oracle(tuples, LT, LS, shape_t, shape_s):
    """All 25 keys, their value types and order, and the numpy RNG state afterwards."""
    rng = np.random.RandomState(LT + 3 * LS + shape_t[2] + shape_s[2])
    tt = _frames(_smooth(rng, LT, int(np.prod(shape_t))), shape_t, tuples)
    st = _frames(_smooth(rng, LS, int(np.prod(shape_s))), shape_s, tuples)
    np.random.seed(17)
    m = tm.compute_trajectory_metrics(tt, st)
    after = np.random.get_state()
    cpu = lambda tr: [(a.cpu(), t) for a, t in tr] if tuples else [a.cpu() for a in tr]
    np.random.seed(17)
    o = om.trajectory_metrics(cpu(tt), cpu(st))
    assert _same_rng(after, np.random.get_state())
    _check_oracle(m, o)


def _mixed_pairs(rng):
    """Interleaved pairs: equal size and length, unequal lengths, and two shape groups of resized students."""
    kinds = [((1, 3, 32, 32), 9, (1, 3, 32, 32), 9), ((1, 3, 32, 32), 9, (1, 3, 16, 16), 9),
             ((1, 3, 32, 32), 9, (1, 3, 32, 32), 5), ((1, 3, 32, 32), 9, (1, 3, 16, 16), 5),
             ((1, 3, 16, 16), 6, (1, 3, 32, 32), 6)]
    pairs, kind_of = [], []
    for i in range(15):
        k = [0, 1, 2, 1, 3, 4, 1][i % 7]
        st, LT, ss, LS = kinds[k]
        tt = _frames(_smooth(rng, LT, int(np.prod(st))), st, i % 2 == 0)
        sl = _frames(_smooth(rng, LS, int(np.prod(ss))), ss, i % 2 == 0)
        pairs.append((tt, sl))
        kind_of.append(k)
    return pairs, kind_of


def test_many_equals_per_pair_with_one_launch_per_shape_group(monkeypatch):
    rng = np.random.RandomState(9)
    pairs, kind_of = _mixed_pairs(rng)
    np.random.seed(23)
    want = [tm.compute_trajectory_metrics(t, s) for t, s in pairs]
    after_per_pair = np.random.get_state()

    lib = _lib.load()
    calls = {}
    for name in ("dtraj_metrics_pairs_resampled", "dtraj_wasserstein_resampled"):
        fn = getattr(lib, name)

        def counted(*a, _fn=fn, _name=name):
            calls[_name] = calls.get(_name, 0) + 1
            return _fn(*a)
        monkeypatch.setattr(lib, name, counted)
    np.random.seed(23)
    got = tm.compute_trajectory_metrics_many(pairs)
    assert _same_rng(after_per_pair, np.random.get_state())
    resized_groups = len({k for k in kind_of if k in (1, 3, 4)})
    assert calls == {"dtraj_metrics_pairs_resampled": resized_groups, "dtraj_wasserstein_resampled": resized_groups}
    assert len(got) == len(want)
    for g, w in zip(got, want):
        assert list(g.keys()) == list(w.keys())
        for k in w:
            assert type(g[k]) is type(w[k]) and np.array_equal(np.asarray(g[k]), np.asarray(w[k]), equal_nan=True), k


class _Model(torch.nn.Module):
    def __init__(self):
        super().__init__()
        self.w = torch.nn.Parameter(torch.zeros(1, device="cuda"))


def test_metrics_batch_of_pickles_with_resized_students(tmp_path):
    """compute_trajectory_metrics_batch over pickles (batch_size 4) whose students are 16x16 against 32x32 teachers,
    mixed with equal-size pairs: the per-pair values and the numpy RNG state afterwards."""
    cfg = Cfg(3, 32, 6)
    cfg.trajectory_dir = str(tmp_path)
    mgr = TrajectoryManager(_Model(), _Model(), cfg, size_factor=0.5)
    rng = np.random.RandomState(4)
    pairs = []
    for i in range(9):
        ss, LS = [((1, 3, 16, 16), 9), ((1, 3, 16, 16), 5), ((1, 3, 32, 32), 9)][i % 3]
        pair = ([(torch.from_numpy(f), k) for k, f in enumerate(_smooth(rng, 9, 3072).reshape(9, 1, 3, 32, 32))],
                [(torch.from_numpy(f), k) for k, f in enumerate(_smooth(rng, LS, int(np.prod(ss))).reshape(LS, *ss))])
        with open(mgr._path(i), "wb") as f:
            pickle.dump(pair, f)
        pairs.append(pair)
    np.random.seed(5)
    allm = mgr.compute_trajectory_metrics_batch(batch_size=4)
    after = np.random.get_state()
    np.random.seed(5)
    per_pair = [tm.compute_trajectory_metrics(t, s) for t, s in pairs]
    assert _same_rng(after, np.random.get_state())
    assert allm["endpoint_distances"] == [m["endpoint_distance"] for m in per_pair]
    assert allm["wasserstein_distances_per_timestep"] == [m["wasserstein_distances"] for m in per_pair]
    assert allm["mean_directional_consistency"] == [m["mean_directional_consistency"] for m in per_pair]
    assert allm["student_path_lengths"] == [m["student_path_length"] for m in per_pair]


def test_resampled_entry_points_refuse_bad_shapes():
    lib = _lib.load()
    t = torch.zeros(2, 3, 4 * 64 * 64, device="cuda")
    s = torch.zeros(2, 3, 4 * 32 * 32, device="cuda")
    pos, frac = (torch.from_numpy(a).cuda() for a in tm.resample_table(3, 3))
    out = torch.zeros(2, 3, 8, device="cuda")
    w = torch.zeros(2, 3, device="cuda")
    red = lambda C_, Ht, Cs, Hs: lib.dtraj_metrics_pairs_resampled(_lib.ptr(t), _lib.ptr(s), 2, 3, 3, C_, Ht, Ht, Cs, Hs, Hs,
                                                                   _lib.ptr(pos), _lib.ptr(frac), _lib.ptr(out),
                                                                   _lib.stream_ptr())
    was = lambda C_, Ht, Cs, Hs: lib.dtraj_wasserstein_resampled(_lib.ptr(t), _lib.ptr(s), 2, 3, 3, C_, Ht, Ht, Cs, Hs, Hs,
                                                                 None, None, C_ * Ht * Ht, _lib.ptr(w), _lib.stream_ptr())
    EINVAL = -1
    assert red(4, 64, 3, 32) == EINVAL and b"channels" in lib.dtraj_last_error()        # channel mismatch
    assert was(4, 16, 3, 16) == EINVAL and b"channels" in lib.dtraj_last_error()
    assert red(5, 64, 5, 32) == EINVAL and b"too large" in lib.dtraj_last_error()        # 5 * 64 * 64 > 16384
    assert red(4, 64, 4, 0) == EINVAL and was(4, 0, 4, 16) == EINVAL                   # non-positive sizes
    assert was(4, 64, 4, 32) == EINVAL and b"K=" in lib.dtraj_last_error()               # all 16384 elements: K > 1024
    assert red(4, 64, 4, 32) == 0                                                       # 4x64x64: the largest frame
    torch.cuda.synchronize()
