"""GPU: metrics of teacher / student trajectories whose frames differ in size (a student sampled at half its teacher's
resolution: 3x32x32 teacher, 3x16x16 student), one job:
  1. dtraj_metrics_pairs_resampled, N = 4096 pairs, (LT, LS) = (51, 51) and (51, 26): kernel time, GB/s over the
     algorithmic bytes 4*N*(Dt*LT + Ds*LS) and over the bytes the kernel's loads request, 4 per teacher element and 16
     per resized student element (four taps, served by L1/L2 where neighbouring elements share them) for every frame
     the ragged walk reads.  Inputs (3.2 GB at (51, 51)) exceed the 126 MB L2.  dtraj_metrics_pairs_ragged of the
     teacher against the student resized beforehand, in the same job for comparison.
  2. compute_trajectory_metrics_many pairs/s over the same 4096 pairs (frames as host tensors, one [1, C, H, W] tensor
     per frame, as pickles hold them), this tree against ``--parent-tree`` (a checkout of another commit with its
     library built), alternating, each run in its own process from the same seed; the two trees' results and numpy RNG
     states are compared.
    python tools/resampled_metrics_bench.py [--parent-tree DIR] [--rounds 2] [--pairs 4096] [--out FILE]"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
C, HT, HS = 3, 32, 16
DT, DS = C * HT * HT, C * HS * HS
LENGTHS = [(51, 51), (51, 26)]

# one timed compute_trajectory_metrics_many call, executed by `python -c` with the tree under test first on sys.path
RUN = r"""
import json, sys, time
import numpy as np, torch
from distillation_trajectories_b200.analysis.metrics import trajectory_metrics as tm
N, LT, LS, C, HT, HS = (int(v) for v in sys.argv[1:7])
rng = np.random.default_rng(LT * 100 + LS)
T = rng.standard_normal((N, 1, C * HT * HT), dtype=np.float32) + np.cumsum(rng.standard_normal((N, LT, C * HT * HT), dtype=np.float32) * 0.02, axis=1)
S = rng.standard_normal((N, 1, C * HS * HS), dtype=np.float32) + np.cumsum(rng.standard_normal((N, LS, C * HS * HS), dtype=np.float32) * 0.02, axis=1)
tt = torch.from_numpy(T.reshape(N, LT, 1, C, HT, HT))
ss = torch.from_numpy(S.reshape(N, LS, 1, C, HS, HS))
pairs = [([tt[n, i] for i in range(LT)], [ss[n, i] for i in range(LS)]) for n in range(N)]
np.random.seed(0)
tm.compute_trajectory_metrics_many(pairs[:8])                 # warm-up: module load, first launches
np.random.seed(0)
torch.cuda.synchronize(); t0 = time.perf_counter()
res = tm.compute_trajectory_metrics_many(pairs)
torch.cuda.synchronize(); sec = time.perf_counter() - t0
keys = ["endpoint_distance", "mse", "student_path_length", "student_efficiency", "mean_directional_consistency",
        "path_alignment", "mean_wasserstein"]
print(json.dumps({"sec": sec, "pairs": len(res), "rng": int(np.random.get_state()[1].sum()),
                  "values": {k: [float(m[k]) for m in res] for k in keys}}))
"""


def reads(LT, LS):
    """frames of each trajectory the ragged walk loads: every frame once, frame 0 again, the shorter one's frames and
    last frame again (the teacher counts as the longer one at LT == LS)"""
    t_long = LT >= LS
    return LT + 1 + (0 if t_long else LT + 1), LS + 1 + (LS + 1 if t_long else 0)


def kernel_times(out, N):
    import torch
    import torch.nn.functional as F
    from distillation_trajectories_b200 import _lib
    from distillation_trajectories_b200.analysis.metrics import trajectory_metrics as tm
    lib = _lib.load()

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

    for LT, LS in LENGTHS:
        g = torch.Generator(device="cuda").manual_seed(LT + LS)
        T = torch.randn(N, 1, DT, device="cuda", generator=g) + 0.02 * torch.cumsum(torch.randn(N, LT, DT, device="cuda", generator=g), 1)
        S = torch.randn(N, 1, DS, device="cuda", generator=g) + 0.02 * torch.cumsum(torch.randn(N, LS, DS, device="cuda", generator=g), 1)
        T, S = T.contiguous(), S.contiguous()
        Sr = F.interpolate(S.reshape(N * LS, C, HS, HS), size=(HT, HT), mode="bilinear", align_corners=True).reshape(N, LS, DT)
        pos, frac = (torch.from_numpy(a).cuda() for a in tm.resample_table(LT, LS))
        red = torch.empty(N, max(LT, LS), _lib.METRIC_Q_RAGGED, device="cuda")
        red_r = torch.empty_like(red)
        resampled = lambda: _lib.check(lib.dtraj_metrics_pairs_resampled(
            _lib.ptr(T), _lib.ptr(S), N, LT, LS, C, HT, HT, C, HS, HS, _lib.ptr(pos), _lib.ptr(frac), _lib.ptr(red), _lib.stream_ptr()))
        ragged = lambda: _lib.check(lib.dtraj_metrics_pairs_ragged(
            _lib.ptr(T), _lib.ptr(Sr), N, LT, LS, DT, _lib.ptr(pos), _lib.ptr(frac), _lib.ptr(red_r), _lib.stream_ptr()))
        rt, rs = reads(LT, LS)
        alg = 4 * N * (DT * LT + DS * LS) / 1e9
        req = N * (4 * DT * rt + 16 * DT * rs) / 1e9
        alg_r, req_r = 4 * N * DT * (LT + LS) / 1e9, 4 * N * DT * (rt + rs) / 1e9
        for rep in range(3):
            ms = time_it(resampled)
            out["kernel"].append({"kernel": "dtraj_metrics_pairs_resampled", "N": N, "LT": LT, "LS": LS, "teacher": [C, HT, HT],
                                  "student": [C, HS, HS], "ms": ms, "algorithmic_GB": alg, "algorithmic_GBps": alg / ms * 1e3,
                                  "requested_GB": req, "requested_GBps": req / ms * 1e3})
            ms = time_it(ragged)
            out["kernel"].append({"kernel": "dtraj_metrics_pairs_ragged (student resized beforehand)", "N": N, "LT": LT, "LS": LS,
                                  "D": DT, "ms": ms, "algorithmic_GB": alg_r, "algorithmic_GBps": alg_r / ms * 1e3,
                                  "requested_GB": req_r, "requested_GBps": req_r / ms * 1e3})
            print(json.dumps(out["kernel"][-2:]), flush=True)
        # the timed launches agree with the ragged kernel on the interpolated student
        d = ((red.double() - red_r.double()).abs().amax(dim=(0, 1)) / red_r.double().abs().amax(dim=(0, 1)).clamp_min(1e-30))
        out["kernel_max_rel_diff_vs_ragged_of_interpolated"] = out.get("kernel_max_rel_diff_vs_ragged_of_interpolated", {})
        out["kernel_max_rel_diff_vs_ragged_of_interpolated"][f"{LT},{LS}"] = [float(v) for v in d]
        assert float(d.max()) < 1e-5, d
        del T, S, Sr, red, red_r
        torch.cuda.empty_cache()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--parent-tree", default=None)
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--pairs", type=int, default=4096)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    sys.path.insert(0, ROOT)
    import numpy as np
    import torch
    out = {"gpu": torch.cuda.get_device_name(0), "kernel": [], "many": []}
    try:
        out["power_limit"] = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                                            capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        out["power_limit"] = f"unavailable: {e}"
    print(out["gpu"], out["power_limit"], flush=True)
    kernel_times(out, a.pairs)

    trees = [("this", ROOT)] + ([("parent", os.path.abspath(a.parent_tree))] if a.parent_tree else [])
    vals = {}
    for rnd in range(a.rounds):
        for LT, LS in LENGTHS:
            for name, tree in trees:
                env = dict(os.environ, PYTHONPATH=tree)
                res = subprocess.run([sys.executable, "-c", RUN, str(a.pairs), str(LT), str(LS), str(C), str(HT), str(HS)],
                                     capture_output=True, text=True, env=env, cwd=tree)
                if res.returncode:
                    raise RuntimeError(f"{name}/{LT},{LS}: {res.stderr[-3000:]}")
                r = json.loads(res.stdout.strip().splitlines()[-1])
                vals[(name, LT, LS)] = (r.pop("values"), r["rng"])
                rec = {"round": rnd, "tree": name, "LT": LT, "LS": LS, "pairs": r["pairs"], "sec": r["sec"],
                       "pairs_per_s": r["pairs"] / r["sec"], "rng_state_sum": r["rng"]}
                out["many"].append(rec)
                print(json.dumps(rec), flush=True)
    if a.parent_tree:
        out["max_rel_diff_vs_parent"] = {}
        for LT, LS in LENGTHS:
            (v, rng), (pv, prng) = vals[("this", LT, LS)], vals[("parent", LT, LS)]
            assert rng == prng, "numpy RNG state differs from the parent's"
            for k in v:
                x, y = np.asarray(v[k]), np.asarray(pv[k])
                out["max_rel_diff_vs_parent"][f"{LT},{LS}/{k}"] = float(np.max(np.abs(x - y) / np.maximum(np.abs(y), 1e-12)))
        print(json.dumps(out["max_rel_diff_vs_parent"]), flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    t0 = time.time()
    main()
    print(f"total {time.time() - t0:.0f} s")
