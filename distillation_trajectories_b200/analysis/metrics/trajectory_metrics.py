"""Trajectory metrics on the GPU (drop-in for
/root/reference/analysis/metrics/trajectory_metrics.py:12-325, compute part only).

The per-frame reductions (||T_i - S_i||, consecutive-frame velocities, direction dot
products, start-to-end distances) and the per-frame Wasserstein distances come from two
streaming CUDA kernels (``dtraj_metrics_pairs`` / ``dtraj_wasserstein``); the f64 scalar
formulas (log1p / exp / ratios) are evaluated on the host exactly as the reference does, so
1e-4 parity does not depend on the device's libm.  Teacher and student trajectories of
different lengths (trajectory_metrics.py:239-279) take ``dtraj_metrics_pairs_ragged`` /
``dtraj_wasserstein_ragged``, which also compute the path alignment on the device.

Batched API (what the sweep drivers use): ``pair_reductions`` (``pair_reductions_ragged``) +
``wasserstein_frames`` + ``scalar_metrics_batched`` over [N, L, D] device tensors, or
``pair_metrics`` for all three.  ``compute_trajectory_metrics`` keeps the reference's
list-of-tensors signature and 25-key result; ``compute_trajectory_metrics_many`` returns the
same for a list of pairs with one launch per group of equally shaped pairs.
"""
import ctypes as C

import numpy as np
import torch

from ... import _lib

SCALAR_KEYS = (
    "endpoint_distance", "mse", "trajectory_mse", "point_by_point_similarity", "log_mse_similarity",
    "teacher_path_length", "student_path_length", "path_length_similarity", "teacher_efficiency",
    "student_efficiency", "efficiency_similarity", "mean_velocity_similarity", "mean_position_difference",
    "max_position_difference", "mean_directional_consistency", "weighted_directional_consistency",
    "mean_wasserstein", "distribution_similarity",
)   # the 18 keys compare_trajectories averages.  path_alignment is left out on purpose: the reference computes it as
#     np.exp(-10.0 * np.float32) -- an np.float32 under NumPy >= 2 promotion rules (NEP 50), which fails the
#     isinstance(v, (int, float)) filter of analysis/trajectory_engine.py:173, so it is dropped from the averages;
#     with the reference's pinned numpy==1.26.4 (value-based promotion) the same expression is an np.float64 and the
#     reference would average 19 keys.  The goldens (tests/golden) were made under NumPy 2.3 and pin the 18-key form;
#     compute_trajectory_metrics still returns path_alignment per pair (25 keys) for callers that want it.


MAX_GROUP_ELEMS = 4096      # elements of one frame a kernel group of dtraj_metrics_pairs holds in registers


# ----------------------------------------------------------------------------- kernels
def _dev(t):
    if t.device.type != "cuda":
        raise _lib.DtrajError("trajectory metrics run on CUDA only (no CPU fallback)")
    return t


def pair_reductions(teacher, student):
    """[N, L, D] x2 (CUDA fp32, contiguous) -> device tensor [N, L, 6] (see include/dtraj.h)."""
    lib = _lib.load()
    teacher, student = _dev(teacher).contiguous(), _dev(student).contiguous()
    if teacher.shape != student.shape or teacher.dim() != 3:
        raise ValueError("pair_reductions expects two [N, L, D] tensors of equal shape")
    N, L, D = teacher.shape
    if D > MAX_GROUP_ELEMS:
        return _reduce_in_parts(pair_reductions, teacher, student)
    out = torch.empty(N, L, _lib.METRIC_Q, dtype=torch.float32, device=teacher.device)
    with torch.cuda.device(teacher.device):
        _lib.check(lib.dtraj_metrics_pairs(_lib.ptr(teacher), _lib.ptr(student), N, L, D, _lib.ptr(out), _lib.stream_ptr()))
    return out


def _reduce_in_parts(reduce, teacher, student):
    """One kernel group owns at most 4096 elements of a frame (include/dtraj.h): wider frames (a batch axis folded
    into D, or images beyond 32x32x4) are cut into equal parts that are reduced separately and added in f64."""
    N, D = teacher.shape[0], teacher.shape[2]
    parts = 2
    while D // parts > MAX_GROUP_ELEMS or D % parts:
        parts += 1
    cut = lambda x: x.reshape(N, x.shape[1], parts, D // parts).permute(0, 2, 1, 3).reshape(N * parts, x.shape[1], D // parts).contiguous()
    r = reduce(cut(teacher), cut(student))
    return r.reshape(N, parts, *r.shape[1:]).double().sum(dim=1).float()


def resample_table(LT, LS):
    """Path-alignment resampling of the longer trajectory onto the shorter one's time axis (trajectory_metrics.py:239-279:
    interp1d on linspace(0, 1, L) axes, np.interp's rule), computed in f64: short frame j is compared with
    (1 - frac[j]) * long[pos[j]] + frac[j] * long[pos[j] + 1].  Returns (pos int32 [n], frac float32 [n]), n = min(LT, LS)."""
    n_long, n_short = max(LT, LS), min(LT, LS)
    lt, st = np.linspace(0, 1, n_long), np.linspace(0, 1, n_short)
    pos = np.clip(np.searchsorted(lt, st, side="right") - 1, 0, n_long - 2)
    frac = (st - lt[pos]) / (lt[pos + 1] - lt[pos])
    return pos.astype(np.int32), frac.astype(np.float32)


def pair_reductions_ragged(teacher, student):
    """teacher [N, LT, D], student [N, LS, D] (CUDA fp32, contiguous, max(LT, LS) >= 2) -> device tensor
    [N, max(LT, LS), 8] (dtraj_metrics_pairs_ragged in include/dtraj.h): the reductions of pair_reductions over the
    first min(LT, LS) frames, each trajectory's own velocities and start-to-end distance, the distance between the two
    last frames ([0][6]) and the squared path-alignment distances ([j][7])."""
    lib = _lib.load()
    teacher, student = _dev(teacher).contiguous(), _dev(student).contiguous()
    if teacher.dim() != 3 or student.dim() != 3 or teacher.shape[0] != student.shape[0] or teacher.shape[2] != student.shape[2]:
        raise ValueError("pair_reductions_ragged expects [N, LT, D] and [N, LS, D] tensors")
    N, LT, D = teacher.shape
    LS = student.shape[1]
    if D > MAX_GROUP_ELEMS:
        return _reduce_in_parts(pair_reductions_ragged, teacher, student)
    pos, frac = resample_table(LT, LS)
    pos, frac = torch.from_numpy(pos).to(teacher.device), torch.from_numpy(frac).to(teacher.device)
    out = torch.empty(N, max(LT, LS), _lib.METRIC_Q_RAGGED, dtype=torch.float32, device=teacher.device)
    with torch.cuda.device(teacher.device):
        _lib.check(lib.dtraj_metrics_pairs_ragged(_lib.ptr(teacher), _lib.ptr(student), N, LT, LS, D, _lib.ptr(pos),
                                                  _lib.ptr(frac), _lib.ptr(out), _lib.stream_ptr()))
    return out


def wasserstein_frames(teacher, student, idx=None, idx_set=None):
    """Per-frame W1 between gathered elements of teacher [N, LT, D] and student [N, LS, D], for the first
    L = min(LT, LS) frames.  ``idx``: int32 [n_sets, L, K] (CUDA) or None for all elements; ``idx_set``: int32 [N]
    choosing the set per pair.  Returns device [N, L] fp32."""
    lib = _lib.load()
    teacher, student = _dev(teacher).contiguous(), _dev(student).contiguous()
    N, LT, D = teacher.shape
    LS = student.shape[1]
    K = D if idx is None else int(idx.shape[-1])
    out = torch.empty(N, min(LT, LS), dtype=torch.float32, device=teacher.device)
    if idx is not None:
        idx = idx.to(teacher.device, torch.int32).contiguous()
    if idx_set is not None:
        idx_set = idx_set.to(teacher.device, torch.int32).contiguous()
    with torch.cuda.device(teacher.device):
        if LT == LS:
            rc = lib.dtraj_wasserstein(_lib.ptr(teacher), _lib.ptr(student), N, LT, D, _lib.ptr(idx), _lib.ptr(idx_set),
                                       K, _lib.ptr(out), _lib.stream_ptr())
        else:
            rc = lib.dtraj_wasserstein_ragged(_lib.ptr(teacher), _lib.ptr(student), N, LT, LS, D, _lib.ptr(idx),
                                              _lib.ptr(idx_set), K, _lib.ptr(out), _lib.stream_ptr())
        _lib.check(rc)
    return out


# ----------------------------------------------------------------------------- host formulas
def _ratio(a, b):
    hi = np.maximum(a, b)
    lo = np.minimum(a, b)
    with np.errstate(divide="ignore", invalid="ignore"):
        return np.where(hi > 0, lo / np.where(hi > 0, hi, 1.0), 1.0)


def scalar_metrics_batched(red, w1, pixels, numel, lengths=None):
    """Vectorised Q1 scalar formulas for N pairs of the same lengths.

    red     np.float32 [N, L, 6] from ``pair_reductions`` (equal lengths), or [N, max(LT, LS), 8] from
            ``pair_reductions_ragged`` with ``lengths`` = (LT, LS); summed over the batch axis of a frame if any
    w1      np.float64/32 [N, min(LT, LS)] per-frame Wasserstein distances
    pixels  H*W (the reference's path-length normaliser, trajectory_metrics.py:118-119)
    numel   elements per frame tensor (torch.mean's denominator)
    Returns dict key -> np.float64 [N] for the 18 scalar keys + 'path_alignment' (np.float32 [N] for equal
    lengths, np.float64 [N] otherwise, as the reference's f64 interpolation makes it) and the per-frame arrays
    behind the 7 list keys.  Unequal lengths (trajectory_metrics.py:55-59,140-164,239-279): the pairwise metrics
    cover the first min(LT, LS) frames, the endpoint distance and mse compare the two last frames, efficiencies
    and velocity lists use each trajectory's full length.
    """
    red = np.asarray(red, np.float32)
    N = red.shape[0]
    LT, LS = (red.shape[1], red.shape[1]) if lengths is None else lengths
    L = min(LT, LS)
    f32 = np.float32
    d = np.sqrt(red[:, :L, 0]).astype(f32)                      # torch.norm -> fp32
    m = (red[:, :L, 0] / f32(numel)).astype(f32)                # torch.mean -> fp32
    vt_all = np.sqrt(red[:, : LT - 1, 1]).astype(f32)
    vs_all = np.sqrt(red[:, : LS - 1, 2]).astype(f32)
    vt, vs = vt_all[:, : L - 1], vs_all[:, : L - 1]
    dot = red[:, : L - 1, 3]
    d64, m64, vt64, vs64 = d.astype(np.float64), m.astype(np.float64), vt.astype(np.float64), vs.astype(np.float64)
    out = {}
    if LT == LS:
        out["endpoint_distance"] = d64[:, -1]                                         # :55
        mse = m64[:, -1]                                                              # :59
    else:
        out["endpoint_distance"] = np.sqrt(red[:, 0, 6]).astype(f32).astype(np.float64)
        mse = (red[:, 0, 6] / f32(numel)).astype(f32).astype(np.float64)
    out["mse"] = mse
    with np.errstate(invalid="ignore", divide="ignore"):
        out["trajectory_mse"] = np.log1p(1.0 - m64.sum(axis=1) / L * 1000)            # :63-86
        out["point_by_point_similarity"] = np.exp(-5.0 * d64.mean(axis=1))            # :90-101
        out["log_mse_similarity"] = np.maximum(0, 1.0 - np.log1p(mse * 5000) / np.log1p(5000))   # :106-108
        if L > 1:
            tl = (vt64 / pixels).sum(axis=1) / (L - 1)                                # :111-131
            sl = (vs64 / pixels).sum(axis=1) / (L - 1)
        else:
            tl = sl = np.full(N, np.nan)
        out["teacher_path_length"], out["student_path_length"] = tl, sl
        out["path_length_similarity"] = np.log1p(_ratio(tl, sl))                      # :134-137
        te = np.sqrt(red[:, 0, 4]).astype(f32).astype(np.float64)                     # :140-153
        se = np.sqrt(red[:, 0, 5]).astype(f32).astype(np.float64)
        teff = np.where(tl > 0, te / np.where(tl > 0, tl, 1.0), 0.0)
        seff = np.where(sl > 0, se / np.where(sl > 0, sl, 1.0), 0.0)
        out["teacher_efficiency"], out["student_efficiency"] = teff, seff
        out["efficiency_similarity"] = np.log1p(_ratio(teff, seff))
        vsim = _ratio(vt64, vs64)                                                     # :156-177
        out["mean_velocity_similarity"] = vsim.mean(axis=1) if L > 1 else np.zeros(N)
        out["mean_position_difference"] = d64.mean(axis=1)                            # :180-187
        out["max_position_difference"] = d64.max(axis=1)
        ok = (vt > 0) & (vs > 0)                                                      # :190-231
        cos = np.where(ok, dot / np.where(ok, vt * vs, f32(1)), f32(0)).astype(f32).astype(np.float64)
        cnt = ok.sum(axis=1)
        out["mean_directional_consistency"] = np.where(cnt > 0, cos.sum(axis=1) / np.maximum(cnt, 1), 0.0)
        wgt = (vt64 + vs64) / 2
        tw = wgt.sum(axis=1)
        wm = np.where(tw > 0, (cos * wgt * ok).sum(axis=1) / np.where(tw > 0, tw, 1.0), 0.0)
        out["weighted_directional_consistency"] = np.where(cnt > 0, wm ** 2, 0.0)
        if LT == LS:                                                                  # :282-293 -- np.linalg.norm on
            area = d.sum(axis=1, dtype=f32)                                           # float32 rows, float32 sum and exp
            out["path_alignment"] = np.exp(f32(-10.0) * area / f32(L)).astype(f32)
        else:                                                                         # :239-279 -- f64 interpolation
            out["path_alignment"] = np.exp(-10.0 * np.sqrt(red[:, :L, 7].astype(np.float64)).sum(axis=1) / L)
        w1 = np.asarray(w1, np.float64)                                               # :296-323
        out["mean_wasserstein"] = w1.mean(axis=1)
        out["distribution_similarity"] = np.log1p(np.exp(-out["mean_wasserstein"]))
    out["_position_differences"] = d64
    out["_teacher_velocities"] = vt_all.astype(np.float64)
    out["_student_velocities"] = vs_all.astype(np.float64)
    out["_velocity_similarities"] = vsim
    out["_cos"], out["_cos_ok"] = cos, ok
    out["_wasserstein"] = w1
    return out


def _images(traj):
    # the third sampler stores (tensor, t) tuples (trajectory_metrics.py:29-37)
    return [it[0] for it in traj] if isinstance(traj[0], tuple) else list(traj)


def _stack_frames(images, device):
    """list of L tensors [B, C, H, W] -> device tensor [L, B*C*H*W]."""
    return torch.stack([im.detach().to(device, torch.float32).reshape(-1) for im in images])


def _pick_device(images):
    for im in images:
        if im.device.type == "cuda":
            return im.device
    if not torch.cuda.is_available():
        raise _lib.DtrajError("trajectory metrics need a CUDA device (no CPU fallback)")
    return torch.device("cuda", torch.cuda.current_device())


def draw_index_sets(n, numel):
    """The Wasserstein subsample draws of one pair: n np.random.choice(numel, min(1000, numel), replace=False) calls on
    the global numpy RNG, one per compared frame (trajectory_metrics.py:301-306), also where they select every element."""
    K = min(1000, numel)
    return np.stack([np.random.choice(numel, K, replace=False) for _ in range(n)]).astype(np.int32)


def pair_metrics(teacher, student, idx, pixels, samples=1):
    """Scalar formulas of ``scalar_metrics_batched`` for G pairs of the same lengths and frame shape.

    teacher  device fp32 [G, LT, numel], student [G, LS, numel]: whole frames, a frame's ``samples`` images one
             after another
    idx      np.int32 [G, min(LT, LS), K] from ``draw_index_sets``, pair by pair
    The reductions run per image and are added in f64 (torch.norm over a whole [B, C, H, W] frame).
    """
    G, LT, numel = teacher.shape
    LS = student.shape[1]
    per_image = lambda x: x.reshape(G, x.shape[1], samples, numel // samples).transpose(1, 2) \
        .reshape(G * samples, x.shape[1], numel // samples)
    reduce = pair_reductions if LT == LS else pair_reductions_ragged
    red = reduce(per_image(teacher), per_image(student)).cpu().numpy()
    red = red.reshape(G, samples, *red.shape[1:]).astype(np.float64).sum(axis=1).astype(np.float32)
    all_elements = idx.shape[-1] == numel
    w1 = wasserstein_frames(teacher, student, None if all_elements else torch.from_numpy(idx),
                            None if all_elements else torch.arange(G, dtype=torch.int32)).cpu().numpy()
    return scalar_metrics_batched(red, w1, pixels, numel, (LT, LS))


_KEY_ORDER = ["endpoint_distance", "mse", "trajectory_mse", "point_by_point_similarity", "log_mse_similarity",
              "teacher_path_length", "student_path_length", "path_length_similarity", "teacher_efficiency",
              "student_efficiency", "efficiency_similarity", "teacher_velocities", "student_velocities",
              "velocity_similarities", "mean_velocity_similarity", "position_differences", "mean_position_difference",
              "max_position_difference", "directional_consistency", "mean_directional_consistency",
              "weighted_directional_consistency", "path_alignment", "wasserstein_distances", "mean_wasserstein",
              "distribution_similarity"]


def _metrics_dict(sm, j):
    """Pair j of ``scalar_metrics_batched``'s result as the reference's 25-key dict, with its value types."""
    m = {}
    for k in SCALAR_KEYS:
        v = sm[k][j]
        m[k] = float(v) if k in ("endpoint_distance", "mse", "teacher_path_length", "student_path_length",
                                 "teacher_efficiency", "student_efficiency",
                                 "weighted_directional_consistency") else np.float64(v)
    m["path_alignment"] = sm["path_alignment"][j]
    m["teacher_velocities"] = [float(v) for v in sm["_teacher_velocities"][j]]
    m["student_velocities"] = [float(v) for v in sm["_student_velocities"][j]]
    m["velocity_similarities"] = [float(v) for v in sm["_velocity_similarities"][j]]
    m["position_differences"] = [float(v) for v in sm["_position_differences"][j]]
    m["directional_consistency"] = [float(c) for c, ok in zip(sm["_cos"][j], sm["_cos_ok"][j]) if ok]
    m["wasserstein_distances"] = [float(v) for v in sm["_wasserstein"][j]]
    return {k: m[k] for k in _KEY_ORDER}      # the reference's key order (dict order is observable through .keys())


def compute_trajectory_metrics(teacher_trajectory, student_trajectory, config=None):
    """Metrics between one teacher and one student trajectory (lists of [B, C, H, W] tensors or
    (tensor, t) tuples).  Same 25 keys, value types and numpy-global-RNG use as the reference."""
    T = _images(teacher_trajectory)
    S = _images(student_trajectory)
    if T[-1].shape != S[-1].shape and T[-1].shape[2:] != S[-1].shape[2:]:
        # trajectory_metrics.py:40-52: bilinear (align_corners) resize of every student frame
        dev = _pick_device(T + S)
        S = [torch.nn.functional.interpolate(s.to(dev), size=T[0].shape[2:], mode="bilinear", align_corners=True)
             for s in S]
    return compute_trajectory_metrics_many([(T, S)])[0]


def compute_trajectory_metrics_many(pairs):
    """``compute_trajectory_metrics`` of every (teacher, student) pair of ``pairs``, in order.  Pairs with the same
    lengths and frame shape share one launch of each kernel; the results, and the global numpy RNG's state afterwards,
    are those of calling ``compute_trajectory_metrics`` on each pair in turn."""
    out = [None] * len(pairs)
    groups = {}
    for k, (t, s) in enumerate(pairs):
        T, S = _images(t), _images(s)
        if T[-1].shape != S[-1].shape and T[-1].shape[2:] != S[-1].shape[2:]:
            out[k] = compute_trajectory_metrics(T, S)          # student frames resized on their own
            continue
        idx = draw_index_sets(min(len(T), len(S)), T[0].numel())
        groups.setdefault((len(T), len(S), tuple(T[0].shape)), []).append((k, T, S, idx))
    for (_, _, shape), items in groups.items():
        dev = _pick_device(items[0][1] + items[0][2])
        ft = torch.stack([_stack_frames(T, dev) for _, T, _, _ in items])
        fs = torch.stack([_stack_frames(S, dev) for _, _, S, _ in items])
        sm = pair_metrics(ft, fs, np.stack([it[3] for it in items]), shape[2] * shape[3], samples=shape[0])
        for j, it in enumerate(items):
            out[it[0]] = _metrics_dict(sm, j)
    return out
