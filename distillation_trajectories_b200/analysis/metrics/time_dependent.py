"""Time-dependent distances (drop-in for
/root/reference/analysis/metrics/time_dependent.py:10-152, compute part :42-120).

Consecutive-frame L2 distances per trajectory come from the same streaming reduction kernel
as the pair metrics (its velocity outputs); averaging over trajectories / steps is f64 host
arithmetic as in the reference.  The optional plot (:122-150) is out of scope; ``save_dir``
is accepted and ignored.
"""
import numpy as np
import torch

from .trajectory_metrics import _images, _pick_device, pair_reductions


def _stack(trajs, dev):
    """list of trajectories (lists of [B,C,H,W] frames) -> [n, L, B*C*H*W] if all lengths agree."""
    return torch.stack([torch.stack([f.detach().to(dev, torch.float32).reshape(-1) for f in _images(t)]) for t in trajs])


def _velocities(trajs_a, trajs_b, dev):
    """per-trajectory consecutive-frame distances for two lists; one kernel launch when shapes agree."""
    la = {len(t) for t in trajs_a}
    lb = {len(t) for t in trajs_b}
    if len(la) == 1 and la == lb and len(trajs_a) == len(trajs_b) and \
            _images(trajs_a[0])[0].shape == _images(trajs_b[0])[0].shape:
        red = _reduce(_stack(trajs_a, dev), _stack(trajs_b, dev))
        return _to_lists(red[:, :, 1]), _to_lists(red[:, :, 2])
    return _velocities_by_length(trajs_a, dev), _velocities_by_length(trajs_b, dev)


def _velocities_by_length(trajs, dev):
    """distances of one list of trajectories of different lengths: one launch per distinct (length, frame shape), each
    trajectory paired with itself; the lists come back in input order."""
    groups = {}
    for k, t in enumerate(trajs):
        im = _images(t)
        groups.setdefault((len(im), tuple(im[0].shape)), []).append(k)
    rows = [None] * len(trajs)
    for ks in groups.values():
        x = _stack([trajs[k] for k in ks], dev)
        for k, r in zip(ks, _reduce(x, x)[:, :, 1]):
            rows[k] = r
    return [d for r in rows for d in _to_lists(r[None])]


def _reduce(a, b):
    """[n, L, D] x2 -> host [n, L, 6]; frames wider than one kernel group are split inside pair_reductions."""
    return pair_reductions(a, b).cpu().numpy()


def _to_lists(sq):
    d = np.sqrt(sq[:, :-1].astype(np.float32)).astype(np.float32)
    return [[float(v) for v in row] for row in d if row.size]


def analyze_time_dependent_distances(teacher_trajectories, student_trajectories, config, size_factor=None, save_dir=None):
    """Distances between consecutive timesteps, per trajectory and averaged."""
    results = {"teacher_distances": [], "student_distances": [], "teacher_avg_distance": 0,
               "student_avg_distance": 0, "teacher_std_distance": 0, "student_std_distance": 0,
               "size_factor": size_factor}
    if not teacher_trajectories or not student_trajectories:
        return results
    dev = _pick_device(_images(teacher_trajectories[0]))
    td, sd = _velocities(teacher_trajectories, student_trajectories, dev)
    results["teacher_distances"], results["student_distances"] = td, sd
    avg = {"teacher": [], "student": []}
    if td and sd:
        for who, dd in (("teacher", td), ("student", sd)):
            for t in range(min(len(d) for d in dd)):
                avg[who].append(sum(d[t] for d in dd) / len(dd))
    for who, a in avg.items():
        results[who + "_avg_per_timestep"] = a
        results[who + "_avg_distance"] = sum(a) / len(a) if a else 0
        if a:
            mu = results[who + "_avg_distance"]
            results[who + "_std_distance"] = (sum((d - mu) ** 2 for d in a) / len(a)) ** 0.5
    return results
