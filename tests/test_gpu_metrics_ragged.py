"""GPU: metrics of teacher / student trajectories of different lengths (trajectory_metrics.py:239-279), the ragged
kernels against f64 numpy and the drop-in wrappers against the CPU oracle; batched pickles and packs against the
per-pair entry point, including the global numpy RNG state they leave behind."""
import pickle

import numpy as np
import pytest
import torch

from oracle import metrics as om
from distillation_trajectories_b200.analysis.metrics import time_dependent as td
from distillation_trajectories_b200.analysis.metrics import trajectory_metrics as tm
from distillation_trajectories_b200.utils import trajectory_store as store
from distillation_trajectories_b200.utils.trajectory_manager import TrajectoryManager
from helpers import Cfg

pytestmark = pytest.mark.gpu
RT = 1e-4


def _paths(rng, N, LT, LS, D, scale=0.02):
    """N pairs sampled from one smooth path per pair at LT and LS points, plus noise."""
    base = np.cumsum(rng.randn(N, 8, D), axis=1) * scale
    grid = np.linspace(0, 7, 8)
    at = lambda L: np.stack([np.stack([np.interp(np.linspace(0, 7, L), grid, base[n, :, d]) for d in range(D)], axis=1)
                             for n in range(N)])
    T = at(LT) + rng.randn(N, LT, D) * scale * 0.1
    S = at(LS) + rng.randn(N, LS, D) * scale * 0.1
    return T.astype(np.float32), S.astype(np.float32)


def _want(T, S):
    """f64 restatement of dtraj_metrics_pairs_ragged (include/dtraj.h)."""
    T, S = T.astype(np.float64), S.astype(np.float64)
    N, LT, _ = T.shape
    LS = S.shape[1]
    n = min(LT, LS)
    w = np.zeros((N, max(LT, LS), 8))
    w[:, :n, 0] = ((T[:, :n] - S[:, :n]) ** 2).sum(-1)
    w[:, :LT - 1, 1] = (np.diff(T, axis=1) ** 2).sum(-1)
    w[:, :LS - 1, 2] = (np.diff(S, axis=1) ** 2).sum(-1)
    w[:, :n - 1, 3] = (np.diff(T[:, :n], axis=1) * np.diff(S[:, :n], axis=1)).sum(-1)
    w[:, 0, 4] = ((T[:, -1] - T[:, 0]) ** 2).sum(-1)
    w[:, 0, 5] = ((S[:, -1] - S[:, 0]) ** 2).sum(-1)
    w[:, 0, 6] = ((T[:, -1] - S[:, -1]) ** 2).sum(-1)
    longer, shorter = (T, S) if LT >= LS else (S, T)
    lt, st = np.linspace(0, 1, longer.shape[1]), np.linspace(0, 1, n)
    res = np.stack([np.stack([np.interp(st, lt, longer[p, :, d]) for d in range(T.shape[2])], axis=1) for p in range(N)])
    w[:, :n, 7] = ((res - shorter) ** 2).sum(-1)
    return w


@pytest.mark.parametrize("D", [256, 3072, 16384])
@pytest.mark.parametrize("LT,LS", [(51, 26), (26, 51), (50, 2), (5, 4), (7, 7)])
def test_ragged_reductions_vs_numpy(LT, LS, D):
    """13 pairs: 8 pairs share a block at D = 256, so the second block is partly empty; pair 0's teacher and student
    agree on their common frames."""
    rng = np.random.RandomState(LT * 100 + LS + D)
    N, n = 13, min(LT, LS)
    T, S = _paths(rng, N, LT, LS, D)
    S[0, :n] = T[0, :n]
    if LS > n:
        S[0, n:] = T[0, n - 1]
    got = tm.pair_reductions_ragged(torch.from_numpy(T).cuda(), torch.from_numpy(S).cuda()).cpu().numpy()
    want = _want(T, S)
    assert got.shape == want.shape
    for q in range(8):
        np.testing.assert_allclose(got[:, :, q], want[:, :, q], rtol=2e-5, atol=2e-6 * np.abs(want[:, :, q]).max() + 1e-30,
                                   err_msg=f"column {q}")
    assert (got[0, :n, 0] == 0).all() and (got[0, : n - 1, 3] == got[0, : n - 1, 1]).all()
    if LT == LS:
        np.testing.assert_array_equal(got[:, :, 7], got[:, :, 0])      # resampling onto the same axis is the identity
        eq = tm.pair_reductions(torch.from_numpy(T).cuda(), torch.from_numpy(S).cuda()).cpu().numpy()
        np.testing.assert_allclose(got[:, :, :6], eq, rtol=1e-6, atol=0)


@pytest.mark.parametrize("D,K", [(256, 256), (3072, 1000)])
def test_wasserstein_of_unequal_lengths_reads_the_common_frames(D, K):
    rng = np.random.RandomState(D)
    N, LT, LS = 5, 9, 4
    T = torch.from_numpy(rng.randn(N, LT, D).astype(np.float32)).cuda()
    S = torch.from_numpy((rng.randn(N, LS, D) * 1.2).astype(np.float32)).cuda()
    idx = idx_set = None
    if K < D:
        idx = torch.from_numpy(np.stack([tm.draw_index_sets(LS, D) for _ in range(2)]))
        idx_set = torch.tensor([0, 1, 1, 0, 1], dtype=torch.int32)
    got = tm.wasserstein_frames(T, S, idx, idx_set)
    assert torch.equal(got, tm.wasserstein_frames(T[:, :LS].contiguous(), S, idx, idx_set))
    assert torch.equal(tm.wasserstein_frames(S, T, idx, idx_set), tm.wasserstein_frames(S, T[:, :LS].contiguous(), idx, idx_set))


def _check_oracle(m, o):
    assert list(m.keys()) == list(o.keys())
    for k in o:
        np.testing.assert_allclose(np.asarray(m[k], np.float64), np.asarray(o[k], np.float64), rtol=RT, atol=1e-7,
                                   equal_nan=True, err_msg=k)
        assert type(m[k]) is type(o[k]), (k, type(m[k]), type(o[k]))


def _same_rng(a, b):
    return a[0] == b[0] and np.array_equal(a[1], b[1]) and a[2:] == b[2:]


@pytest.mark.parametrize("LT,LS,shape", [(51, 26, (1, 3, 32, 32)), (26, 51, (1, 3, 32, 32)), (50, 2, (1, 1, 16, 16)),
                                         (5, 4, (2, 3, 32, 32)), (9, 6, (1, 1, 80, 80))])
def test_compute_trajectory_metrics_unequal_vs_oracle(LT, LS, shape):
    """All 25 keys, value types and the numpy RNG state afterwards.  (2, 3, 32, 32): two images per frame;
    1x80x80 = 6400 elements per frame: reductions in parts."""
    rng = np.random.RandomState(LT + LS)
    D = int(np.prod(shape))
    T, S = _paths(rng, 1, LT, LS, D, scale=0.002)
    tt = [(torch.from_numpy(T[0, i].reshape(shape)).cuda(), i) for i in range(LT)]
    st = [(torch.from_numpy(S[0, i].reshape(shape)).cuda(), i) for i in range(LS)]
    np.random.seed(17)
    m = tm.compute_trajectory_metrics(tt, st)
    after = np.random.get_state()
    np.random.seed(17)
    o = om.trajectory_metrics([(a.cpu(), t) for a, t in tt], [(a.cpu(), t) for a, t in st])
    assert _same_rng(after, np.random.get_state())
    _check_oracle(m, o)


class _Model(torch.nn.Module):
    def __init__(self):
        super().__init__()
        self.w = torch.nn.Parameter(torch.zeros(1, device="cuda"))


def _manager(tmp_path, shape):
    cfg = Cfg(shape[1], shape[2], 6)
    cfg.trajectory_dir = str(tmp_path)
    return TrajectoryManager(_Model(), _Model(), cfg, size_factor=0.5)


def _reference_lists(allm_pairs):
    lists = {"wasserstein_distances": "mean_wasserstein", "wasserstein_distances_per_timestep": "wasserstein_distances",
             "endpoint_distances": "endpoint_distance", "teacher_path_lengths": "teacher_path_length",
             "student_path_lengths": "student_path_length", "teacher_efficiency": "teacher_efficiency",
             "student_efficiency": "student_efficiency"}
    new = ["path_length_similarity", "efficiency_similarity", "mean_velocity_similarity",
           "mean_directional_consistency", "mean_position_difference", "distribution_similarity"]
    out = {k: [] for k in list(lists) + new}
    for m in allm_pairs:
        for dst, src in lists.items():
            out[dst].append(m[src])
        for k in new:
            out[k].append(m[k])
    return out


@pytest.mark.parametrize("D", [256, 3072])
@pytest.mark.parametrize("LT,LS", [(6, 6), (9, 5)])
def test_metrics_batch_equals_per_pair(tmp_path, LT, LS, D):
    """compute_trajectory_metrics_batch over 7 pickles (batch_size 3; one pair of other lengths mixed in) and over a
    70-pair pack (two chunks at batch_size 1): every value equals the per-pair compute_trajectory_metrics result bit
    for bit, and the numpy RNG state afterwards is identical, also at D <= 1000 where the draws select every element."""
    shape = (1, 1, 16, 16) if D == 256 else (1, 3, 32, 32)
    rng = np.random.RandomState(D + LS)
    mgr = _manager(tmp_path, shape)
    pairs = []
    for i in range(7):
        ls = (LT if LS != LT else LT - 2) if i == 2 else LS
        T, S = _paths(rng, 1, LT, ls, D, scale=0.002)
        pair = ([(torch.from_numpy(T[0, k].reshape(shape)), k) for k in range(LT)],
                [(torch.from_numpy(S[0, k].reshape(shape)), k) for k in range(ls)])
        with open(mgr._path(i), "wb") as f:
            pickle.dump(pair, f)
        pairs.append(pair)
    T, S = _paths(rng, 70, LT, LS, D, scale=0.002)
    pack = store.write_pack(str(tmp_path), 0.5, list(range(100, 170)), T.reshape(70, LT, *shape[1:]),
                            S.reshape(70, LS, *shape[1:]), list(range(LT)), list(range(LS)))
    tl, sl = store.as_reference_lists(store.read_pack(pack), torch.from_numpy)
    pairs += list(zip(tl, sl))

    np.random.seed(5)
    allm = mgr.compute_trajectory_metrics_batch(batch_size=3)
    after_pickles_and_pack = np.random.get_state()
    np.random.seed(5)
    want = _reference_lists([tm.compute_trajectory_metrics(t, s) for t, s in pairs])
    assert _same_rng(after_pickles_and_pack, np.random.get_state())
    for k, v in want.items():
        assert len(allm[k]) == len(v) == 77, k
        assert allm[k] == v, k                                  # exact, lists of per-frame distances included

    np.random.seed(5)
    mgr.compute_trajectory_metrics_batch(batch_size=1)         # pack in 64-pair chunks
    a = np.random.get_state()
    np.random.seed(5)
    mgr.compute_trajectory_metrics_batch(batch_size=100)
    assert _same_rng(a, np.random.get_state()) and _same_rng(a, after_pickles_and_pack)


def test_time_dependent_distances_with_two_lengths():
    """Teacher and student lists whose trajectories have different lengths (one launch per length), a
    single-frame trajectory among them, against the oracle."""
    rng = np.random.RandomState(7)
    mk = lambda L, shape: [torch.from_numpy(x).cuda() for x in np.cumsum(rng.randn(L, *shape).astype(np.float32) * 0.1, axis=0)]
    teachers = [mk(L, (1, 3, 32, 32)) for L in (11, 6, 11, 1, 6)]
    students = [mk(L, (1, 3, 32, 32)) for L in (6, 11, 6)]
    r = td.analyze_time_dependent_distances(teachers, students, None, size_factor=0.5)
    o = om.time_dependent_distances([[f.cpu() for f in t] for t in teachers], [[f.cpu() for f in t] for t in students], 0.5)
    assert [len(d) for d in r["teacher_distances"]] == [10, 5, 10, 5] and [len(d) for d in r["student_distances"]] == [5, 10, 5]
    for k in o:
        if k.endswith("_distances"):
            assert len(r[k]) == len(o[k])
            for a, b in zip(r[k], o[k]):
                np.testing.assert_allclose(a, b, rtol=RT, err_msg=k)
        elif k != "size_factor":
            np.testing.assert_allclose(np.asarray(r[k], np.float64), np.asarray(o[k], np.float64), rtol=RT, err_msg=k)
    assert r["size_factor"] == 0.5
