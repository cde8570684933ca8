"""Teacher/student trajectory pairs with the placeholder sampler S3, pickle cache and batched metric
aggregation (drop-in for /root/reference/utils/trajectory_manager.py:9-581).

Each model's loop (store frame, forward, x <- (x - 0.1 eps)/sqrt(0.9) + 0.1 (t/teacher_steps) z) runs
as one captured CUDA loop; noise is drawn from torch's generators with the reference's calls in the
reference's order.  The default on-disk format stays ``pickle((teacher_list, student_list))`` of
``(tensor, t)`` tuples per (size factor, sample); ``packed=True`` writes one dense pack per call instead
(utils/trajectory_store.py: all pairs generated in ONE batched loop per model, metrics over the pack by the
batched kernels) and every reader accepts both formats.
"""
import os
import pickle

import numpy as np
import torch

from .. import sampling
from . import trajectory_store as store
from ..engine import UNetEngine, check_device_errors, get_precision
from ..analysis.metrics import trajectory_metrics as tm


class TrajectoryManager:
    def __init__(self, teacher_model, student_model, config, size_factor=1.0, fixed_samples=None):
        self.teacher_model = teacher_model
        self.student_model = student_model
        self.config = config
        self.size_factor = size_factor
        self.fixed_samples = fixed_samples
        os.makedirs(config.trajectory_dir, exist_ok=True)
        self.device = next(teacher_model.parameters()).device

    # ------------------------------------------------------------------ generation
    def _run_model(self, model, x, steps):
        """frames-before-update loop of one model (trajectory_manager.py:98-111) -> [(tensor, t), ...]"""
        cfg = self.config
        idx = sampling.s3_timestep_indices(cfg.sample_steps, steps)
        ts = list(reversed(idx))
        eng = UNetEngine.for_model(model, x.shape[2], max(ts) + 1, get_precision("S3"), self.device)
        n_upd = sum(1 for t in ts if t > 0)
        ndev = sampling.noise_device(self.device)
        noise = torch.stack([torch.randn(x.shape, device=ndev) for _ in range(n_upd)]) if n_upd else None
        traj = sampling.s3_sample(eng, x, ts, cfg.teacher_steps, noise)
        frames = [(traj[:, k].clone(), t) for k, t in enumerate(ts)]
        check_device_errors(self.device)         # frames leave the library here (pickled or handed to the caller)
        return frames

    def _pair(self, seed, sample):
        cfg = self.config
        self.teacher_model.eval()
        self.student_model.eval()
        shape = (1, cfg.channels, cfg.image_size, cfg.image_size)
        out = []
        for k, (model, steps) in enumerate(((self.teacher_model, cfg.teacher_steps),
                                            (self.student_model, cfg.student_steps))):
            if seed is not None and (sample is None or k == 0):
                torch.manual_seed(seed)
                np.random.seed(seed)
            x = (torch.randn(shape) if sample is None else sample.clone()).to(self.device)
            out.append(self._run_model(model, x, steps))
        return out[0], out[1]

    def generate_trajectory(self, seed=None):
        """One (teacher, student) pair from ``seed`` (trajectory_manager.py:65-165); both start from the
        same x_T and see the same noise sequence because the student re-seeds."""
        return self._pair(seed, None)

    def generate_trajectory_from_sample(self, sample, seed=None):
        """Pair starting from a fixed noise sample (trajectory_manager.py:265-387); errors are reported
        and yield empty lists, as in the reference."""
        try:
            return self._pair(seed, sample)
        except Exception as e:            # reference semantics: print and return empties
            print(f"Error generating trajectory from sample: {e}")
            return [], []

    def _path(self, i, size_factor=None):
        sf = self.size_factor if size_factor is None else size_factor
        return os.path.join(self.config.trajectory_dir, f"trajectory_size_{sf}_sample_{i}.pkl")

    def _draws(self, seed, shape, n_updates):
        """x_T and the per-step noise of sample ``seed`` exactly as ``generate_trajectory(seed)`` draws them
        (manual_seed(seed); randn on the CPU; randn_like on the model's device per update), from private
        generators (same streams, no global re-seeding)."""
        from ..analysis.trajectory_engine import _generator
        gc = _generator(torch.device("cpu"))
        gc.manual_seed(seed)
        x = torch.randn(shape, generator=gc)
        ndev = sampling.noise_device(self.device)
        gn = gc if ndev.type == "cpu" else _generator(ndev)
        if gn is not gc:
            gn.manual_seed(seed)
        z = [torch.randn(shape, device=ndev, generator=gn) for _ in range(n_updates)]
        return x, z

    def generate_packed(self, sample_ids):
        """All pairs of ``sample_ids`` (seeds) in one batched captured loop per model; returns the path of the
        pack written (utils/trajectory_store.py).  Frames are bit-identical to ``generate_trajectory(seed)``."""
        cfg = self.config
        self.teacher_model.eval()
        self.student_model.eval()
        shape = (1, cfg.channels, cfg.image_size, cfg.image_size)
        plans = []
        for model, steps in ((self.teacher_model, cfg.teacher_steps), (self.student_model, cfg.student_steps)):
            ts = list(reversed(sampling.s3_timestep_indices(cfg.sample_steps, steps)))
            plans.append((model, ts, sum(1 for t in ts if t > 0)))
        n_max = max(p[2] for p in plans)
        xs, zs = [], []
        for i in sample_ids:
            x, z = self._draws(int(i), shape, n_max)
            xs.append(x)
            zs.append(torch.cat(z) if z else None)
        x_T = torch.cat(xs).to(self.device)
        noise = torch.stack(zs, dim=1).to(self.device) if n_max else None        # [n_updates, B, C, H, W]
        out = []
        for model, ts, n_upd in plans:
            eng = UNetEngine.for_model(model, x_T.shape[2], max(ts) + 1, get_precision("S3"), self.device)
            traj = sampling.s3_sample(eng, x_T, ts, cfg.teacher_steps, None if noise is None else noise[:max(n_upd, 1)])
            out.append((traj.cpu().numpy(), ts))
            check_device_errors()
        return store.write_pack(cfg.trajectory_dir, self.size_factor, list(sample_ids), out[0][0], out[1][0],
                                out[0][1], out[1][1])

    def generate_and_save_trajectories(self, num_samples=10, packed=False):
        """trajectory_manager.py:207-263: one pickle per pair; a failing sample is reported and skipped.
        ``packed=True``: seeds 0..num_samples-1 in one batched loop, one pack file."""
        if packed and self.fixed_samples is None:
            return [self.generate_packed(range(num_samples))]
        paths = []
        fixed = self.fixed_samples is not None and num_samples <= len(self.fixed_samples)
        for i in range(num_samples):
            try:
                if fixed:
                    pair = self.generate_trajectory_from_sample(self.fixed_samples[i], i)
                else:
                    pair = self.generate_trajectory(seed=i)
            except Exception as e:
                print(f"Error generating trajectory {i}: {e}")
                continue
            with open(self._path(i), "wb") as f:
                pickle.dump(pair, f)
            paths.append(self._path(i))
        return paths

    # ------------------------------------------------------------------ cache
    def _files(self, size_factor):
        prefix = f"trajectory_size_{size_factor}_sample_"
        names = [f for f in os.listdir(self.config.trajectory_dir) if f.startswith(prefix) and f.endswith(".pkl")]
        names.sort(key=lambda s: int(s.split("_sample_")[1].split(".")[0]))
        return names

    def load_trajectories(self, size_factor=None, indices=None):
        """trajectory_manager.py:389-432."""
        sf = self.size_factor if size_factor is None else size_factor
        names = self._files(sf)
        if indices is not None:
            names = [n for n in names if int(n.split("_sample_")[1].split(".")[0]) in indices]
        teachers, students = [], []
        for n in names:
            with open(os.path.join(self.config.trajectory_dir, n), "rb") as f:
                t, s = pickle.load(f)
            teachers.append(t)
            students.append(s)
        for p in store.list_packs(self.config.trajectory_dir, sf):           # packed samples, same structure
            t, s = store.as_reference_lists(store.read_pack(p), lambda a: torch.from_numpy(a).to(self.device), indices)
            teachers.extend(t)
            students.extend(s)
        return teachers, students

    def compute_trajectory_metrics_batch(self, size_factor=None, batch_size=10):
        """trajectory_manager.py:434-548: per-pair metrics appended to 13 named lists, then ``*_avg`` means."""
        sf = self.size_factor if size_factor is None else size_factor
        names = self._files(sf)
        lists = {"wasserstein_distances": "mean_wasserstein", "wasserstein_distances_per_timestep": "wasserstein_distances",
                 "endpoint_distances": "endpoint_distance", "teacher_path_lengths": "teacher_path_length",
                 "student_path_lengths": "student_path_length", "teacher_efficiency": "teacher_efficiency",
                 "student_efficiency": "student_efficiency"}
        new = ["path_length_similarity", "efficiency_similarity", "mean_velocity_similarity",
               "mean_directional_consistency", "mean_position_difference", "distribution_similarity"]
        allm = {k: [] for k in list(lists) + new + ["architecture_type"]}
        for i in range(0, len(names), batch_size):
            pairs = []
            for n in names[i:i + batch_size]:
                with open(os.path.join(self.config.trajectory_dir, n), "rb") as f:
                    pairs.append(pickle.load(f))
            for m in tm.compute_trajectory_metrics_many(pairs):
                for dst, src in lists.items():
                    allm[dst].append(m[src])
                for k in new:
                    if k in m:
                        allm[k].append(m[k])
                if hasattr(self, "architecture_type"):
                    allm["architecture_type"].append(self.architecture_type)
        for p in store.list_packs(self.config.trajectory_dir, sf):
            self._pack_metrics(store.read_pack(p), allm, lists, new, batch_size)
        for k in ["endpoint_distances", "teacher_path_lengths", "student_path_lengths", "teacher_efficiency",
                  "student_efficiency", "wasserstein_distances"] + new:
            if allm.get(k):
                allm[k + "_avg"] = sum(allm[k]) / len(allm[k])
        return allm

    def _pack_metrics(self, pack, allm, lists, new, batch_size):
        """Metrics of every pair of a pack, equal or unequal teacher / student lengths, through the batched kernels
        (one launch per ``batch_size`` x 64 pairs) with the Wasserstein subsamples drawn from the global numpy RNG in
        the reference's order (pair by pair, frame by frame, trajectory_metrics.py:301-306)."""
        T, S = pack["teacher"], pack["student"]
        N, LT, LS = T.shape[0], T.shape[1], S.shape[1]
        D, pixels = int(np.prod(T.shape[2:])), T.shape[3] * T.shape[4]
        step = max(1, batch_size) * 64
        for n0 in range(0, N, step):
            n1 = min(N, n0 + step)
            t = torch.from_numpy(np.ascontiguousarray(T[n0:n1])).to(self.device).reshape(n1 - n0, LT, D)
            s_ = torch.from_numpy(np.ascontiguousarray(S[n0:n1])).to(self.device).reshape(n1 - n0, LS, D)
            idx = np.stack([tm.draw_index_sets(min(LT, LS), D) for _ in range(n1 - n0)])
            sm = tm.pair_metrics(t, s_, idx, pixels)
            for j in range(n1 - n0):
                for dst, src in lists.items():
                    allm[dst].append([float(v) for v in sm["_wasserstein"][j]] if src == "wasserstein_distances"
                                     else float(sm[src][j]))
                for k in new:
                    allm[k].append(float(sm[k][j]))


def generate_trajectories_with_disk_storage(teacher_model, student_model, config, size_factor=1.0, num_samples=10,
                                            fixed_samples=None, packed=False):
    """trajectory_manager.py:550-581: reuse cached trajectories (pickles or packs), generate the missing count."""
    manager = TrajectoryManager(teacher_model, student_model, config, size_factor, fixed_samples)
    existing = store.stored_samples(config.trajectory_dir, size_factor)
    if len(existing) < num_samples:
        print(f"Generating {num_samples - len(existing)} new trajectories...")
        manager.generate_and_save_trajectories(num_samples - len(existing), packed=packed)
    else:
        print(f"Using {num_samples} existing trajectories...")
    return manager
