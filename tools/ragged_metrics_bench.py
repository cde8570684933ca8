"""GPU: metrics of teacher / student trajectories of different lengths (a student sampled with fewer steps than its
teacher), one job:
  1. dtraj_metrics_pairs_ragged at 3x32x32, N = 4096, (LT, LS) = (51, 26): kernel time, GB/s over the algorithmic bytes
     4*N*D*(LT + LS) and over the bytes the kernel requests 4*N*D*(L_long + 2*L_short + 3); dtraj_metrics_pairs over
     [4096, 51, 3072] x2 in the same job for comparison.  Inputs (3.9 GB) exceed the 126 MB L2.
  2. TrajectoryManager.compute_trajectory_metrics_batch pairs/s over one 4096-pair unequal pack and over 1000 unequal
     pickles (3x32x32, (51, 26)), this tree against ``--parent-tree`` (a checkout of another commit with its library
     built), alternating, each run in its own process from the same seed; the two trees' results are compared.
    python tools/ragged_metrics_bench.py [--parent-tree DIR] [--rounds 2] [--out FILE]"""
import argparse
import json
import os
import pickle
import shutil
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LT, LS, C, H = 51, 26, 3, 32
D = C * H * H

# one timed run of compute_trajectory_metrics_batch, executed by `python -c` with the tree under test first on sys.path
RUN = r"""
import json, sys, time
import numpy as np, torch
from distillation_trajectories_b200.utils.trajectory_manager import TrajectoryManager
class Cfg: pass
class M(torch.nn.Module):
    def __init__(self):
        super().__init__(); self.w = torch.nn.Parameter(torch.zeros(1, device="cuda"))
def run(d):
    cfg = Cfg(); cfg.trajectory_dir = d
    np.random.seed(0)
    torch.cuda.synchronize(); t0 = time.perf_counter()
    allm = TrajectoryManager(M(), M(), cfg, size_factor=1.0).compute_trajectory_metrics_batch(batch_size=10)
    torch.cuda.synchronize()
    return time.perf_counter() - t0, allm
run(sys.argv[2])                                             # warm-up: module load, first launches
sec, allm = run(sys.argv[1])
keys = ["endpoint_distances", "teacher_path_lengths", "student_efficiency", "wasserstein_distances",
        "mean_directional_consistency", "distribution_similarity"]
print(json.dumps({"sec": sec, "pairs": len(allm["endpoint_distances"]), "rng": int(np.random.get_state()[1].sum()),
                  "values": {k: [float(v) for v in allm[k]] for k in keys}}))
"""


def make_paths(N, seed):
    """random walks from a shared start, generated 256 pairs at a time (host memory stays near the output's 4*N*D*77 B)"""
    import numpy as np
    rng = np.random.default_rng(seed)
    T, S = np.empty((N, LT, D), np.float32), np.empty((N, LS, D), np.float32)
    for n0 in range(0, N, 256):
        n1 = min(N, n0 + 256)
        x0 = rng.standard_normal((n1 - n0, 1, D), dtype=np.float32)
        for out, L in ((T, LT), (S, LS)):
            out[n0:n1] = x0 + np.cumsum(rng.standard_normal((n1 - n0, L, D), dtype=np.float32) * 0.02, axis=1)
    return T, S


def write_data(tmp, n_pack, n_pickles):
    import torch
    from distillation_trajectories_b200.utils import trajectory_store as store
    dirs = {k: os.path.join(tmp, k) for k in ("pack", "pickles", "warm")}
    for d in dirs.values():
        os.makedirs(d)
    T, S = make_paths(n_pack, 1)
    store.write_pack(dirs["pack"], 1.0, list(range(n_pack)), T.reshape(n_pack, LT, C, H, H), S.reshape(n_pack, LS, C, H, H),
                     list(range(LT)), list(range(LS)))
    del T, S
    for d, n, seed in ((dirs["pickles"], n_pickles, 2), (dirs["warm"], 4, 3)):
        T, S = make_paths(n, seed)
        for i in range(n):
            pair = ([(torch.from_numpy(T[i, k].reshape(1, C, H, H)).clone(), k) for k in range(LT)],
                    [(torch.from_numpy(S[i, k].reshape(1, C, H, H)).clone(), k) for k in range(LS)])
            with open(os.path.join(d, f"trajectory_size_1.0_sample_{i}.pkl"), "wb") as f:
                pickle.dump(pair, f)
    return dirs


def kernel_times(out):
    import numpy as np
    import torch
    from distillation_trajectories_b200 import _lib
    from distillation_trajectories_b200.analysis.metrics import trajectory_metrics as tm
    N = 4096
    g = torch.Generator(device="cuda").manual_seed(1234)
    T = torch.randn(N, 1, D, device="cuda", generator=g) + 0.02 * torch.cumsum(torch.randn(N, LT, D, device="cuda", generator=g), dim=1)
    S = T[:, :LS] + 0.01 * torch.randn(N, LS, D, device="cuda", generator=g)
    S = S.contiguous()
    lib = _lib.load()
    pos, frac = (torch.from_numpy(a).cuda() for a in tm.resample_table(LT, LS))
    red = torch.empty(N, LT, _lib.METRIC_Q_RAGGED, device="cuda")
    ragged = lambda: _lib.check(lib.dtraj_metrics_pairs_ragged(_lib.ptr(T), _lib.ptr(S), N, LT, LS, D, _lib.ptr(pos), _lib.ptr(frac),
                                                               _lib.ptr(red), _lib.stream_ptr()))
    S_eq = torch.cat([S, T[:, LS:]], dim=1).contiguous()
    red_eq = torch.empty(N, LT, _lib.METRIC_Q, device="cuda")
    equal = lambda: _lib.check(lib.dtraj_metrics_pairs(_lib.ptr(T), _lib.ptr(S_eq), N, LT, D, _lib.ptr(red_eq), _lib.stream_ptr()))

    def time_it(fn, iters=20):
        for _ in range(3):
            fn()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(iters):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / iters

    for rep in range(3):
        ms = time_it(ragged)
        alg, moved = 4 * N * D * (LT + LS) / 1e9, 4 * N * D * (max(LT, LS) + 2 * min(LT, LS) + 3) / 1e9
        out["kernel"].append({"kernel": "dtraj_metrics_pairs_ragged", "N": N, "LT": LT, "LS": LS, "D": D, "ms": ms,
                              "algorithmic_GB": alg, "algorithmic_GBps": alg / ms * 1e3,
                              "requested_GB": moved, "requested_GBps": moved / ms * 1e3})
        ms = time_it(equal)
        alg = 2 * 4 * N * D * LT / 1e9
        out["kernel"].append({"kernel": "dtraj_metrics_pairs", "N": N, "L": LT, "D": D, "ms": ms, "algorithmic_GB": alg,
                              "algorithmic_GBps": alg / ms * 1e3})
        print(json.dumps(out["kernel"][-2:]), flush=True)
    # the timed launches compute the f64 restatement's values (pair 0 and the last pair)
    r = red.cpu().numpy()
    for n in (0, N - 1):
        t, s = T[n].double().cpu().numpy(), S[n].double().cpu().numpy()
        np.testing.assert_allclose(r[n, :LS, 0], ((t[:LS] - s) ** 2).sum(-1), rtol=1e-4)
        np.testing.assert_allclose(r[n, 0, 6], ((t[-1] - s[-1]) ** 2).sum(), rtol=1e-4)
    del T, S, S_eq


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--parent-tree", default=None)
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--pack-pairs", type=int, default=4096)
    ap.add_argument("--pickles", type=int, default=1000)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    sys.path.insert(0, ROOT)
    import torch
    out = {"gpu": torch.cuda.get_device_name(0), "kernel": [], "batch": []}
    try:
        out["power_limit"] = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                                            capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        out["power_limit"] = f"unavailable: {e}"
    print(out["gpu"], out["power_limit"], flush=True)
    kernel_times(out)
    torch.cuda.empty_cache()

    tmp = tempfile.mkdtemp(prefix="ragged_bench_")
    try:
        dirs = write_data(tmp, a.pack_pairs, a.pickles)
        trees = [("this", ROOT)] + ([("parent", os.path.abspath(a.parent_tree))] if a.parent_tree else [])
        vals = {}
        for rnd in range(a.rounds):
            for what in ("pack", "pickles"):
                for name, tree in trees:
                    env = dict(os.environ, PYTHONPATH=tree)
                    res = subprocess.run([sys.executable, "-c", RUN, dirs[what], dirs["warm"]], capture_output=True, text=True,
                                         env=env, cwd=tree)
                    if res.returncode:
                        raise RuntimeError(f"{name}/{what}: {res.stderr[-3000:]}")
                    r = json.loads(res.stdout.strip().splitlines()[-1])
                    vals[(name, what)] = r.pop("values")
                    rec = {"round": rnd, "tree": name, "input": what, "pairs": r["pairs"], "sec": r["sec"],
                           "pairs_per_s": r["pairs"] / r["sec"], "rng_state_sum": r["rng"]}
                    out["batch"].append(rec)
                    print(json.dumps(rec), flush=True)
        if a.parent_tree:
            import numpy as np
            out["max_rel_diff_vs_parent"] = {}
            for what in ("pack", "pickles"):
                for k, v in vals[("this", what)].items():
                    x, y = np.asarray(v), np.asarray(vals[("parent", what)][k])
                    out["max_rel_diff_vs_parent"][f"{what}/{k}"] = float(np.max(np.abs(x - y) / np.maximum(np.abs(y), 1e-12)))
            print(json.dumps(out["max_rel_diff_vs_parent"]), flush=True)
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    t0 = time.time()
    main()
    print(f"total {time.time() - t0:.0f} s")
