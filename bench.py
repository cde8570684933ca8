#!/usr/bin/env python
"""Benchmark of the trajectory hot path (BASELINE.json metric: denoising trajectories/sec, 50 steps, CFG).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K ...  # the UNMODIFIED reference on the host CPUs (oracle/_ref)

Headline workload (BASELINE.json configs[1]): teacher U-Net (size_factor 1.0) vs student (0.5), 1x16x16, 50
timesteps, classifier-free-guidance sweep w in {1, 2, 3, 5, 7.5, 10, 15, 20}; one STEP = `--seeds` seeds
x 8 guidance scales on every GPU: teacher trajectories + student trajectories (sampler S2,
analysis/trajectory_engine.py:24-115) + the pair metrics of compute_trajectory_metrics.  A trajectory is
one (model, seed, w) run of 51 frames.  Seeds are sharded over ranks (weak scaling: `--seeds` per GPU),
the only collective is the final all-reduce of the metric sums.

value        device-resident: inputs already in HBM, K x (2 captured sampling loops + metric kernels), CUDA events.
e2e          through the public API (grid.sweep, the batched compare_trajectories): host RNG draws, pinned
             host -> device copies, device work, device -> host copy of the reductions, f64 scalar formulas.
parity       the oracle (CPU restatement of the reference, test infrastructure) on two seeds x 8 scales of a chunk run
             at the BENCH shape and precision: worst fraction of the trajectory tolerance used, worst metric error.
by_precision the same workload in the reference's own arithmetic classes (tf32 = what cuDNN runs on CUDA by default,
             tf32x3 ~ fp32), shorter runs.
by_config    BASELINE configs[0] (S1, batch 64), configs[2] (3x32x32, 11 students), a configs[3]-shaped
             strong-scaling slice (fixed total seeds over N GPUs) and the batch-1 latency of the reference-shaped call.
cpu_baseline the reference's own compare_trajectories timed on the host cores (a subprocess of --impl reference).
"""
import argparse
import contextlib
import functools
import io
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

GUIDANCE = [1.0, 2.0, 3.0, 5.0, 7.5, 10.0, 15.0, 20.0]
METRIC = "denoising trajectories/sec (50 steps, CFG)"
UNIT = "trajectories/s"
SF11 = [0.01, 0.1, 0.2, 0.3, 0.4, 0.5, 0.6, 0.7, 0.8, 0.9, 1.0]        # README.md:23, BASELINE configs[2]
TOLERANCE = {"trajectories": "|got - ref| <= 1e-3*|ref| + 1e-4*max|ref| elementwise (north_star states rtol 1e-3; the absolute "
                             "term, 1e-4 of the largest reference element, covers elements near zero)",
             "metric_scalars": "rtol 1e-4 given identical trajectories (north_star), NaN == NaN"}


class Cfg:                       # configs[0] / [1] / [3]: 1x16x16
    channels, image_size, timesteps, dropout = 1, 16, 50, 0.3
    sample_steps = teacher_steps = student_steps = 50
    beta_start, beta_end = 1e-4, 0.02


class Cfg32(Cfg):                # configs[2]: 3x32x32
    channels, image_size = 3, 32


def workload_config(seeds, world):
    return {"workload": "configs[1]: teacher(sf=1.0) vs student(sf=0.5), 1x16x16, 50 steps, CFG sweep "
                        "w in {1,2,3,5,7.5,10,15,20}, sampler S2 + pair metrics",
            "seeds_per_gpu_per_step": seeds, "guidance_scales": GUIDANCE,
            "trajectories_per_step": 2 * seeds * len(GUIDANCE) * world,
            "parallelism": f"seed-sharded x{world}, one all-reduce of metric sums",
            "dedup": "teacher trajectories computed once per (seed, w); at the first step the 8 scales of a seed still hold "
                     "the same x_T, so its forward rows are evaluated once per (seed, conditioning variant) -- bit-identical "
                     "frames (tests/test_gpu_samplers.py::test_first_step_row_sharing_is_exact)",
            "l2": f"per-step working set (2 x {seeds * 8 * 51 * 256 * 4 / 1e6:.0f} MB trajectory buffers + GBs of activations) "
                  "exceeds the 126 MB L2; no explicit flush"}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d["hbm_gbs"], d["bf16_tflops"], d["bf16_tflops_sustained"], "measured (MEASURED_PEAKS.json)"
    return 6650.0, 1590.0, 1400.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons while the timed region runs."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc, self.index = [], None, index

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def __exit__(self, *a):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except Exception:
                self.proc.kill()

    def summary(self):
        sm, mx, reasons = [], 0, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx = max(mx, float(r[1]))
            except Exception:
                continue
            for n, v in zip(names, r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": mx or None,
                "reasons": sorted(reasons), "samples": len(sm)}


def quiet():
    return contextlib.redirect_stdout(io.StringIO())


# --------------------------------------------------------------------------------------- CPU arm
def _port_state():
    """oracle port (used only when oracle/_ref is absent): forward closures of the two models"""
    import torch
    from oracle import unet as ounet
    from distillation_trajectories_b200.models import DiffusionUNet
    fns = []
    for sf, seed in ((1.0, 0), (0.5, 1050)):
        torch.manual_seed(seed)
        with quiet():
            m = DiffusionUNet(Cfg, sf).eval()
        sd = {k: v.detach().clone() for k, v in m.state_dict().items()}
        fns.append(functools.partial(ounet.unet_forward, sd))
    return fns


def _port_step(n_seeds, state):
    import numpy as np
    import torch
    from oracle import metrics as om
    from oracle import samplers as osmp
    ft, fs = state
    for s in range(n_seeds):
        seed = 42 + s
        torch.manual_seed(seed)
        np.random.seed(seed)
        noise = torch.randn(1, Cfg.channels, Cfg.image_size, Cfg.image_size)
        for gs in GUIDANCE:
            a = osmp.s2_generate_trajectory(ft, noise, Cfg.timesteps, seed=seed, guidance_scale=gs)
            b = osmp.s2_generate_trajectory(fs, noise, Cfg.timesteps, seed=seed, guidance_scale=gs)
            om.trajectory_metrics(a, b)


def cpu_arm(n_seeds, steps, warmup):
    """Time the reference's CPU implementation of the path on the host cores with every thread torch will use: the
    UNMODIFIED reference (oracle/_ref, staged by oracle/sync_ref.py; analysis/trajectory_engine.py:117 compare_trajectories
    driving its own models.DiffusionUNet) when present, else the oracle port.  One step = n_seeds seeds x 8 guidance scales x
    {teacher, student} trajectories + their metrics."""
    import torch
    from oracle import refload
    torch.set_num_threads(os.cpu_count() or 1)
    if refload.available():
        ref = refload.load()
        cfg = refload.RefConfig(Cfg.channels, Cfg.image_size, Cfg.timesteps)
        models = []
        for sf, seed in ((1.0, 0), (0.5, 1050)):
            torch.manual_seed(seed)
            with quiet():
                models.append(ref.models.DiffusionUNet(cfg, sf).eval())
        kind = "reference"

        def step():
            with quiet():           # the reference prints per trajectory
                return ref.trajectory_engine.compare_trajectories(models[0], models[1], cfg, guidance_scales=GUIDANCE,
                                                                  size_factor=0.5, num_samples=n_seeds)
    else:
        state = _port_state()
        kind = "port"

        def step():
            _port_step(n_seeds, state)
            return None
    res = None
    for _ in range(warmup):
        res = step()
    t0 = time.perf_counter()
    for _ in range(steps):
        res = step()
    dt = time.perf_counter() - t0
    n = 2 * n_seeds * len(GUIDANCE) * steps
    out = {"value": n / dt, "unit": UNIT, "cores": torch.get_num_threads(), "kind": kind,
           "sample": f"{steps} x ({n_seeds} seeds x {len(GUIDANCE)} guidance scales x (teacher, student) = {n // max(steps, 1)} trajectories + "
                     f"{n_seeds * len(GUIDANCE)} metric pairs), {dt:.1f} s; seeds 42.. as compare_trajectories draws them",
           "torch": torch.__version__, "seconds": dt,
           "what": ("unmodified reference: analysis/trajectory_engine.py:117 compare_trajectories (oracle/_ref), CPU fp32, "
                    "CUDA hidden the way scripts/run_on_cpu.py:26 does") if kind == "reference"
                   else "oracle port of compare_trajectories (oracle/_ref absent)"}
    if res is not None:
        out["check"] = {"trajectory_mse@w=7.5": res["student_metrics"][7.5]["trajectory_mse"],
                        "distribution_similarity@w=7.5": res["student_metrics"][7.5]["distribution_similarity"]}
    return out


def run_reference(args, emit=print):
    """--impl reference: rank 0 only; the other ranks exit without work."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    cb = cpu_arm(args.ref_seeds, args.steps, args.warmup)
    v = cb["value"]
    emit(json.dumps({
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": cb["seconds"] / max(args.steps, 1) * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic (random-init weights, seeded N(0,1) noise)",
        "config": dict(workload_config(args.ref_seeds, 1), note="CPU arm: rank 0 only, bounded sample per step"),
        "cpu_baseline": cb,
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0}))


def cpu_baseline_subprocess(n_seeds=2):
    """The cpu_baseline leg of the GPU arm: the reference needs CUDA hidden (it picks "cuda if available" for its schedule
    tables, utils/diffusion.py:52-56), so it runs as `bench.py --impl reference` in a child with CUDA_VISIBLE_DEVICES=''."""
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="", TQDM_DISABLE="1")
    for k in ("RANK", "LOCAL_RANK", "WORLD_SIZE"):
        env.pop(k, None)
    try:
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1",
                            "--ref-seeds", str(n_seeds)], capture_output=True, text=True, env=env, timeout=600)
        line = [ln for ln in r.stdout.splitlines() if ln.startswith("{")][-1]
        return json.loads(line)["cpu_baseline"]
    except Exception as e:        # a reported baseline, not the product: never take the GPU line down with it
        return {"value": None, "unit": UNIT, "kind": "unavailable", "error": repr(e)[:200]}


# --------------------------------------------------------------------------------------- GPU arm
def make_model(cfg, sf, seed, dev):
    import torch
    from distillation_trajectories_b200.models import DiffusionUNet
    torch.manual_seed(seed)
    with quiet():
        return DiffusionUNet(cfg, sf).eval().to(dev)


def samplers_of(models, cfg, precision, dev):
    from distillation_trajectories_b200.engine import UNetEngine
    return [next(reversed(UNetEngine.for_model(m, cfg.image_size, cfg.timesteps, precision, dev)._samplers.values())) for m in models]


def close_engines(models):
    from distillation_trajectories_b200.engine import UNetEngine
    for m in models:
        UNetEngine.invalidate(m)


def device_resident(teacher, students, cfg, scales, S, K, W, dev, precision, rank, world, barrier, max_over_ranks, clock=None,
                    last=None):
    """W untimed + K timed run_chunk calls on pre-staged chunks; returns (ms total, max over ranks).  ``last`` (dict): receives
    what the last timed call returned (red, w1) and its trajectories (the out_traj views, valid until the samplers run again)."""
    import torch
    from distillation_trajectories_b200 import grid
    chunks = [grid.stage_chunk([(i * world + rank) * S + j for j in range(S)], cfg, scales, dev) for i in range(W + K)]
    torch.cuda.synchronize()
    for i in range(W):
        grid.run_chunk(teacher, students, chunks[i], dev, precision)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with (clock if clock is not None else contextlib.nullcontext()):
        e0.record()
        for i in range(K):
            traj = []
            red, w1, _ = grid.run_chunk(teacher, students, chunks[W + i], dev, precision, out_traj=traj)
        e1.record()
        barrier()
    if last is not None:
        last.update(red=red, w1=w1, traj=traj)
    return max_over_ranks(e0.elapsed_time(e1))


DUMP_ROWS = 512         # 512 (seed, guidance) pairs of 1x16x16 frames: 54 MB of .npy files


def dump_outputs(out_dir, red, w1, traj):
    """--dump-outputs: what the last timed step returned, as float32 .npy files: the pair reductions red.npy [n_students, n, L, 6],
    the per-frame Wasserstein distances w1.npy [n_students, n, L] and the frames behind them, teacher_traj.npy and
    student<i>_traj.npy [n, L, D].  n = the same fixed sample (RandomState(0)) of at most DUMP_ROWS of the step's N pairs in every
    array, in ascending pair order; the whole step's trajectories are too large to keep."""
    import numpy as np
    import torch
    n_pairs = red.shape[1]
    rows = np.sort(np.random.RandomState(0).choice(n_pairs, min(n_pairs, DUMP_ROWS), replace=False))
    idx = torch.from_numpy(rows).to(red.device)
    arrays = {"red": red[:, idx], "w1": w1[:, idx], "teacher_traj": traj[0][0][idx]}
    arrays.update({f"student{i}_traj": s[idx] for i, (_, s) in enumerate(traj)})
    arrays = {k: v.float().cpu().numpy() for k, v in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    assert total <= 64 << 20, f"--dump-outputs would write {total / 2**20:.0f} MiB"
    os.makedirs(out_dir, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(out_dir, k + ".npy"), a)


def conv_flops_per_forward(dims, C, H, executed, skip_enc1=False):
    """2 x MACs of one forward row through the eight blocks (SURVEY.md 8d, models.py:59-83: conv1 3x3, conv2 3x3, 1x1 residual conv where
    the widths differ).  ``executed``: count a 3x3 tap only where it meets the map -- what this repo's kernels load and multiply on maps
    of at most 4x4 (position-major tiles: ((3h-2)/h)^2 of 9 taps on average, the centre tap at 1x1) in fp16 mode."""
    d0, d1, d2, d3 = dims
    blocks = [(C, d0, H), (d0, d1, H // 2), (d1, d2, H // 4), (d2, d3, H // 8), (d3, d3, H // 16),
              (d3 + d3, d2, H // 8), (d2 + d2, d1, H // 4), (d1 + d1, d0, H // 2)]
    total = 0.0
    for cin, cout, h in blocks[1 if skip_enc1 else 0:]:
        taps = ((3.0 * h - 2.0) / h) ** 2 if (executed and h <= 4) else 9.0
        total += 2.0 * h * h * (taps * cin * cout + taps * cout * cout + (cin * cout if cin != cout else 0))
    return total


def conv_roofline(samplers, precision, tc_sust, src):
    """K1's roofline from one un-captured pass of each loop with an event pair around every launch."""
    prof = [s.profile() for s in samplers]
    conv_ms = sum(p["ms"][0] for p in prof)
    conv_fl = sum(p["conv_flops"] for p in prof)
    conv_n = sum(p["launches"][0] for p in prof)
    all_ms = sum(sum(p["ms"]) for p in prof)
    ach = conv_fl / (conv_ms / 1e3) / 1e12
    kname = {"fp32": "k_conv_simt (CUDA-core fp32 implicit GEMM)",
             "f16": "k_conv_umma (tcgen05 kind::f16 implicit-GEMM conv, fp32 accumulate)",
             "tf32": "k_conv_umma (tcgen05 kind::tf32 implicit-GEMM conv)",
             "tf32x3": "k_conv_umma (tcgen05 kind::tf32, 3 passes hi/lo: algorithmic flops counted once)"}[precision]
    ceiling = {"f16": 1.0, "tf32": 0.5, "tf32x3": 1.0 / 6.0, "fp32": None}[precision]
    pnote = ": dense bf16 sustained; " + {"f16": "kind::f16 issues at the bf16 rate",
                                          "tf32": "kind::tf32 issues at half the bf16 rate (ceiling of frac: 0.5)",
                                          "tf32x3": "three kind::tf32 passes per algorithmic flop (ceiling of frac: 0.167)",
                                          "fp32": "CUDA cores: the tensor peak is not this mode's bound"}[precision]
    r = {"kernel": kname, "bound": "tensor", "achieved": ach, "peak": tc_sust, "unit": "TFLOP/s", "frac": ach / tc_sust,
         "frac_ceiling": ceiling, "traffic": None, "peak_source": src + pnote,
         "flops_accounting": "flops = 2 x MACs the kernels execute on REAL channels: a 3x3 tap is counted only where it meets the map "
                             "(fp16 mode skips the taps that fall into the zero padding of 1x1 / 2x2 / 4x4 maps for whole tiles), so "
                             "`achieved` never exceeds what the tensor pipe did; `achieved_algorithmic` / `frac_algorithmic` use the standard "
                             "2 x MACs count of the same launches (SURVEY.md 8d) = achieved / executed_over_standard",
         "launches_timed": conv_n, "avg_launch_us": conv_ms / max(conv_n, 1) * 1e3,
         "flops_per_launch": conv_fl / max(conv_n, 1), "share_of_loop_time": conv_ms / all_ms,
         "class_ms": {"conv": conv_ms, "first_conv": sum(p["ms"][1] for p in prof),
                      "pool_upsample_final": sum(p["ms"][2] for p in prof), "step": sum(p["ms"][3] for p in prof),
                      "enc1_fused": sum(p["ms"][4] for p in prof)}}
    e1_ms, e1_fl = sum(p["ms"][4] for p in prof), sum(p["enc1_flops"] for p in prof)
    if e1_ms > 0:
        e1name = ("k_enc1_f16 (fused enc1 block: conv1 AND conv2 on tcgen05, conv2 weights resident in smem, tap views, fused pool)"
                  if precision == "f16" else "k_enc1_umma (fused enc1 block, tf32: conv1 on CUDA cores, conv2 by tcgen05 tap views, fused pool)")
        r["enc1_kernel"] = {"kernel": e1name, "achieved": e1_fl / (e1_ms / 1e3) / 1e12, "unit": "TFLOP/s (conv2 flops only)",
                            "frac": e1_fl / (e1_ms / 1e3) / 1e12 / tc_sust}
    return r, prof


class ParityOracle:
    """CPU oracle (test infrastructure) results for two seeds x 8 scales of the bench workload, computed once and
    compared with chunks run at the bench shape in any arithmetic mode."""

    def __init__(self, teacher, student, S):
        self.S, self.seeds = S, [0, S - 1]
        self.t, self.s = teacher, student
        self.want = None

    def _oracle(self):
        import torch
        from oracle import samplers as osmp
        from oracle import unet as ounet
        fns = [functools.partial(ounet.unet_forward, {k: v.detach().cpu() for k, v in m.state_dict().items()}) for m in (self.t, self.s)]
        want = []
        for s in self.seeds:
            torch.manual_seed(42 + s)
            noise = torch.randn(1, Cfg.channels, Cfg.image_size, Cfg.image_size)
            for gs in GUIDANCE:
                want.append([torch.stack(osmp.s2_generate_trajectory(f, noise, Cfg.timesteps, seed=42 + s, guidance_scale=gs))[:, 0].numpy()
                             for f in fns])
        self.want = want

    def check(self, dev, precision):
        import numpy as np
        import torch
        from oracle import metrics as om
        from distillation_trajectories_b200 import grid, sampling
        from distillation_trajectories_b200.analysis.metrics import trajectory_metrics as tm
        t0 = time.perf_counter()
        if self.want is None:
            self._oracle()
        G, L = len(GUIDANCE), Cfg.timesteps + 1
        C, H = Cfg.channels, Cfg.image_size
        sampling.set_noise_device("cpu")             # the oracle draws with torch's CPU generator
        try:
            ck = grid.stage_chunk(list(range(self.S)), Cfg, GUIDANCE, dev)
            keep = []
            red, w1, _ = grid.run_chunk(self.t, [self.s], ck, dev, precision, out_traj=keep)
            torch.cuda.synchronize()
        finally:
            sampling.set_noise_device(None)
        rows = [s * G + g for s in self.seeds for g in range(G)]
        got = [k[rows].cpu().numpy().reshape(len(rows), L, C, H, H) for k in keep[0]]
        sm = tm.scalar_metrics_batched(red[0][rows].cpu().numpy(), w1[0][rows].cpu().numpy(), H * H, C * H * H)
        tol_frac, metric_err, metric_err_e2e = 0.0, 0.0, 0.0
        for i, (s, gs) in enumerate((s, gs) for s in self.seeds for gs in GUIDANCE):
            for m in range(2):
                ref = self.want[i][m].astype(np.float64)
                tol = 1e-3 * np.abs(ref) + 1e-4 * np.abs(ref).max()
                tol_frac = max(tol_frac, float((np.abs(got[m][i] - ref) / tol).max()))
            frames = lambda a: [torch.from_numpy(np.ascontiguousarray(f))[None] for f in a]
            for which, (a, b) in (("same", (got[0][i], got[1][i])), ("e2e", (self.want[i][0], self.want[i][1]))):
                np.random.seed(42 + s + 1)
                mo = om.trajectory_metrics(frames(a), frames(b))
                for k in tm.SCALAR_KEYS:
                    x, y = float(sm[k][i]), float(mo[k])
                    if np.isnan(x) and np.isnan(y):
                        continue
                    err = abs(x - y) / max(abs(y), 1e-12)
                    if which == "same":
                        metric_err = max(metric_err, err)
                    else:
                        metric_err_e2e = max(metric_err_e2e, err)
        return {"max_tol_frac": tol_frac, "n_traj": 2 * len(rows), "metric_rel_err": metric_err,
                "metric_rel_err_vs_reference_frames": metric_err_e2e,
                "shape": f"chunk of {self.S} seeds x {G} scales run as in the timed region ({2 * self.S * G - self.S} forward rows per model "
                         f"and step); seeds {self.seeds} x all scales x (teacher, student) compared with the oracle",
                "precision": precision, "seconds": time.perf_counter() - t0,
                "note": "max_tol_frac < 1 <=> every element of every compared frame inside the trajectory tolerance; metric_rel_err: "
                        "the 18 scalars of the CUDA metric path vs the oracle's metrics of the SAME frames (north_star: 1e-4); "
                        "..._vs_reference_frames: the same scalars vs the oracle's metrics of ITS OWN frames (carries the trajectory error)"}


def run_ours(args, emit=print):
    import numpy as np
    import torch
    import torch.distributed as dist

    from distillation_trajectories_b200 import grid

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product path has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
        # one process per GPU on one host: do not let every rank's tiny host-side torch ops spawn a full-size thread pool
        torch.set_num_threads(max(1, (os.cpu_count() or world) // world))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    teacher, student = make_model(Cfg, 1.0, 0, dev), make_model(Cfg, 0.5, 1050, dev)
    models = [teacher, student]
    S, K, W, G = args.seeds, args.steps, args.warmup, len(GUIDANCE)
    hbm, tc_burst, tc_sust, src = peaks()
    traj_per_step = 2 * S * G * world

    def e2e_sweep(precision, steps, warm):
        stats = {}
        for _ in range(warm):
            grid.sweep(teacher, {"student": student}, Cfg, GUIDANCE, S * world, dev, rank, world, max_pairs=S * G, precision=precision)
        barrier()
        # ONE sweep call over `steps` steps' worth of seeds, chunked at a step (S seeds x G scales per rank): the API's own
        # software pipeline (stage chunk i+1 / run chunk i / finish chunk i-1) is what a sweep larger than one batch gets.
        # Every chunk's host draws, pinned H2D copies, D2H read-back and f64 host formulas are inside the timed region.
        t0 = time.perf_counter()
        res = grid.sweep(teacher, {"student": student}, Cfg, GUIDANCE, steps * S * world, dev, rank, world, max_pairs=S * G,
                         precision=precision, stats=stats)
        barrier()
        secs = max_over_ranks(time.perf_counter() - t0)
        return {"value": traj_per_step * steps / secs, "unit": UNIT, "h2d_bytes_per_step": stats["h2d_bytes"] // steps,
                "d2h_bytes_per_step": stats["d2h_bytes"] // steps, "ms_per_step": secs / steps * 1e3,
                "check": {"trajectory_mse@w=7.5": res["student"][7.5]["trajectory_mse"],
                          "distribution_similarity@w=7.5": res["student"][7.5]["distribution_similarity"]}}, stats

    # ---- headline: device-resident leg, then the end-to-end leg (public sweep API, host-side inputs)
    clk = ClockSampler(local)
    last = {}
    ms = device_resident(teacher, [student], Cfg, GUIDANCE, S, K, W, dev, args.precision, rank, world, barrier, max_over_ranks, clk,
                         last)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, **last)
    value = traj_per_step * K / (ms / 1e3)
    samplers = samplers_of(models, Cfg, args.precision, dev)
    launches = K * (sum(s.launches for s in samplers) + 2)
    e2e, stats = e2e_sweep(args.precision, K, max(1, W // 2))
    e2e["api"] = ("distillation_trajectories_b200.grid.sweep (batched compare_trajectories): one call over steps x seeds, "
                  "one chunk per step, chunks software-pipelined by the API")
    if os.environ.get("DTRAJ_SWEEP_TIMING"):
        print(f"[rank {rank}] e2e {e2e['ms_per_step'] * K:.0f} ms; host ms per phase: " +
              ", ".join(f"{k[7:]} {v * 1e3:.0f}" for k, v in stats.items() if k.startswith("host_s_")), file=sys.stderr)

    # ---- BASELINE configs[3]-shaped strong-scaling slice: a FIXED total number of seeds over however many GPUs there are
    by_config = {}
    n4 = args.config4_seeds
    if n4 > 0:
        st4 = {}
        barrier()
        t0 = time.perf_counter()
        grid.sweep(teacher, {"student": student}, Cfg, GUIDANCE, n4, dev, rank, world, max_pairs=S * G, precision=args.precision, stats=st4)
        barrier()
        secs = max_over_ranks(time.perf_counter() - t0)
        by_config["configs[3] slice"] = {
            "workload": f"{n4} seeds x 8 guidance scales x (teacher, student), 1x16x16, sharded over {world} GPU(s), "
                        f"metric sums all-reduced (BASELINE configs[3] is 65,536 seeds: this is a {n4}/65536 slice)",
            "scaling": "strong", "value": 2 * n4 * G / secs, "unit": UNIT + " (end to end through grid.sweep)", "seconds": secs,
            "n_gpus": world, "precision": args.precision}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant kernel: per-launch CUDA events over one un-captured pass of each loop
    roofline, prof = conv_roofline(samplers, args.precision, tc_sust, src)
    if args.precision == "f16":     # teacher + student rows weigh equally in a step: ratio of the two counts for one row through both models
        # (the conv class of `achieved` = blocks 2..8; the fused enc1 kernel, reported next to it, skips nothing)
        ex = sum(conv_flops_per_forward(m.dims, Cfg.channels, Cfg.image_size, True, True) for m in (teacher, student))
        st = sum(conv_flops_per_forward(m.dims, Cfg.channels, Cfg.image_size, False, True) for m in (teacher, student))
        roofline["executed_over_standard"] = ex / st
        roofline["achieved_algorithmic"] = roofline["achieved"] * st / ex     # the standard 2 x MACs of the same launches / the same time
        roofline["frac_algorithmic"] = roofline["frac"] * st / ex
    else:
        roofline["executed_over_standard"] = None   # (tf32 modes run every tap except on 1x1 maps)
    tp = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tp) and args.precision == "f16":
        tj = json.load(open(tp))
        roofline["traffic"] = tj.get("k_conv_umma_dram_bytes_per_launch")
        roofline["traffic_source"] = tj.get("source")
    all_ms = sum(sum(p["ms"]) for p in prof)
    # HBM-bound side kernels (algorithmic bytes: SURVEY.md 8d)
    D, L, N = Cfg.channels * Cfg.image_size ** 2, Cfg.timesteps + 1, S * G
    step_ms = sum(p["ms"][3] for p in prof)
    step_bytes = sum(((16 if w <= 1.0 else 20) * D) for w in GUIDANCE) * S * (Cfg.timesteps - 1) * 2 + 2 * N * D * 8
    from distillation_trajectories_b200.analysis.metrics import trajectory_metrics as tm

    def time_pairs(ta, sa, reps=10):
        for _ in range(3):
            tm.pair_reductions(ta, sa)
        m0, m1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        m0.record()
        for _ in range(reps):
            tm.pair_reductions(ta, sa)
        m1.record()
        torch.cuda.synchronize()
        return m0.elapsed_time(m1) / reps

    met_ms = time_pairs(samplers[0].traj.reshape(N, L, D), samplers[1].traj.reshape(N, L, D))
    met_bytes = 2 * N * L * D * 4
    # BASELINE configs[4] ("metric-kernel bandwidth test"): a chunk of the synthetic [262144, 50, 3, 32, 32] pair
    # (the full tensors are 2 x 150 GiB and are processed in chunks of N on one GPU, SURVEY.md 8d)
    N5, L5, D5 = 8192, 50, 3 * 32 * 32
    gen = torch.Generator(device=dev).manual_seed(1234)
    t5 = torch.randn(N5, 1, D5, device=dev, generator=gen) + 0.1 * torch.cumsum(torch.randn(N5, L5, D5, device=dev, generator=gen), dim=1)
    s5 = t5 + 0.05 * torch.randn(N5, L5, D5, device=dev, generator=gen)
    m5_ms = time_pairs(t5, s5)
    m5_bytes = 2 * N5 * L5 * D5 * 4
    del t5, s5
    torch.cuda.empty_cache()
    side = [{"kernel": "k_step (+ k_copy_frame)", "bound": "hbm", "achieved": step_bytes / (step_ms / 1e3) / 1e9, "peak": hbm,
             "unit": "GB/s", "frac": step_bytes / (step_ms / 1e3) / 1e9 / hbm, "traffic": None,
             "note": f"{step_bytes / (2 * (Cfg.timesteps - 1)) / 1e6:.0f} MB per launch: launch-latency bound at this batch, "
                     f"{step_ms / all_ms * 100:.1f} % of the loop time"},
            {"kernel": f"k_metrics_pairs (this workload: [{N}, {L}, {D}] x 2)", "bound": "hbm",
             "achieved": met_bytes / (met_ms / 1e3) / 1e9, "peak": hbm, "unit": "GB/s",
             "frac": met_bytes / (met_ms / 1e3) / 1e9 / hbm, "traffic": None,
             "note": f"{met_bytes / 1e6:.0f} MB per launch"},
            {"kernel": "k_metrics_pairs (BASELINE configs[4] chunk: [8192, 50, 3, 32, 32] x 2, path length + directional "
                       "consistency + MSE reductions)", "bound": "hbm", "achieved": m5_bytes / (m5_ms / 1e3) / 1e9, "peak": hbm,
             "unit": "GB/s", "frac": m5_bytes / (m5_ms / 1e3) / 1e9 / hbm, "traffic": None,
             "note": f"{m5_bytes / 1e9:.1f} GB per launch, every element read once; metric-kernel GB/s of BASELINE.json's metric"}]
    if os.path.exists(tp):          # per-launch DRAM bytes of the side kernels from the committed ncu passes (profiles/traffic.json)
        tj = json.load(open(tp))
        side[0]["traffic"] = tj.get("k_step_dram_bytes_per_launch")
        if args.seeds == 592:
            side[1]["traffic"] = tj.get("k_metrics_pairs_workload_dram_bytes_per_launch")
        side[2]["traffic"] = tj.get("k_metrics_pairs_config4_chunk_dram_bytes_per_launch")
        for sd in side:
            sd["traffic_source"] = tj.get("side_kernels_source")
    by_config["configs[4] chunk"] = {"workload": "metric-kernel bandwidth on a [8192, 50, 3, 32, 32] x 2 chunk of the synthetic pair",
                                     "value": side[2]["achieved"], "unit": "GB/s", "frac_of_hbm_peak": side[2]["frac"]}

    out = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
           "ms_per_step": ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
           "dtype": {"tf32": "tf32", "tf32x3": "tf32x3", "fp32": "f32", "f16": "f16 (fp32 accumulate)"}[args.precision],
           "data": "synthetic (random-init weights, seeded N(0,1) noise)",
           "config": workload_config(S, world), "e2e": e2e, "gpu_launches": launches,
           "clocks": clk.summary(), "roofline": roofline, "roofline_other": side, "tolerance": TOLERANCE}

    if world == 1 and not args.quick:
        flops_step = sum(sum(s.flops()) for s in samplers)
        out["whole_step_tflops"] = {"value": flops_step / (ms / K / 1e3) / 1e12, "frac_of_peak": flops_step / (ms / K / 1e3) / 1e12 / tc_sust,
                                    "note": "algorithmic conv flops of both loops / device-resident step time (metric kernels, step kernels, "
                                            "resampling included in the time)"}
        # ---- parity at the benchmarked shape and precision (oracle = checker)
        oracle = ParityOracle(teacher, student, S)
        out["parity"] = oracle.check(dev, args.precision)
        # ---- the reference's own arithmetic classes on the same workload
        by_prec = {}
        for prec in ("tf32", "tf32x3"):
            if prec == args.precision:
                continue
            Kp, Wp = min(K, 5), 3
            msp = device_resident(teacher, [student], Cfg, GUIDANCE, S, Kp, Wp, dev, prec, 0, 1, barrier, max_over_ranks)
            sp = samplers_of(models, Cfg, prec, dev)
            rl, _ = conv_roofline(sp, prec, tc_sust, src)
            e2p, _ = e2e_sweep(prec, Kp, 1)
            par = oracle.check(dev, prec)
            by_prec[prec] = {"value": traj_per_step * Kp / (msp / 1e3), "unit": UNIT, "steps": Kp, "warmup": Wp, "ms_per_step": msp / Kp,
                             "e2e": {k: e2p[k] for k in ("value", "ms_per_step", "h2d_bytes_per_step", "d2h_bytes_per_step")},
                             "roofline": {k: rl[k] for k in ("kernel", "achieved", "peak", "frac", "frac_ceiling", "share_of_loop_time")},
                             "parity": {k: par[k] for k in ("max_tol_frac", "metric_rel_err", "n_traj")}}
            from distillation_trajectories_b200.engine import UNetEngine
            for m in models:                       # free this mode's workspaces before the next one
                ent = m.__dict__.get("_dtraj_engines", {})
                for key in [k for k in ent if k[0] != {"f16": 3, "tf32": 1, "tf32x3": 2, "fp32": 0}[args.precision]]:
                    ent.pop(key)[1].close()
            torch.cuda.empty_cache()
        out["by_precision"] = by_prec
        by_config.update(config_legs(dev, tc_sust, teacher, args))
    out["by_config"] = by_config

    if world == 1 and not args.no_cpu_baseline:
        out["cpu_baseline"] = cpu_baseline_subprocess(2)
        if out["cpu_baseline"].get("check") and "check" in e2e:
            out["cpu_baseline"]["note"] = ("check = the reference's own averages over ITS seeds 42, 43 (CPU fp32); e2e.check = this repo's "
                                           f"averages over {K * S * world} seeds -- different sample sets, same order of magnitude expected")
    emit(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


def config_legs(dev, tc_sust, teacher16, args):
    """BASELINE configs[0], configs[2] and the batch-1 latency of the reference-shaped call (single GPU)."""
    import torch
    from distillation_trajectories_b200 import grid
    from distillation_trajectories_b200.analysis import trajectory_engine as te
    from distillation_trajectories_b200.engine import UNetEngine, get_precision
    from distillation_trajectories_b200.utils import diffusion
    out = {}

    def timed(fn, reps, warm=2):
        for _ in range(warm):
            fn()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
        return (time.perf_counter() - t0) / reps

    # configs[0]: S1 (utils/diffusion.py:160-212), teacher, batch 64, 50 steps, "no CFG" (w = 1: both forwards still run), through
    # the public p_sample_loop with trajectory capture: noise draws, captured loop, D2H of the 51 frames
    params = diffusion.get_diffusion_params(Cfg.timesteps, Cfg)
    p1 = get_precision("S1")
    run = lambda: diffusion.p_sample_loop(teacher16, (64, 1, 16, 16), Cfg.timesteps, params, device=dev, config=Cfg,
                                          track_trajectory=True, guidance_scale=1.0)
    sec = timed(run, 10)
    eng = UNetEngine.for_model(teacher16, 16, Cfg.timesteps, p1, dev)
    fl = sum(next(reversed(eng._samplers.values())).flops())
    out["configs[0]"] = {"workload": "teacher 1x16x16, p_sample_loop(shape=(64,1,16,16), 50 steps, track_trajectory=True, w=1.0): S1, "
                                     "128 forward rows per step", "precision": p1, "value": 64 / sec, "unit": UNIT + " (end to end, public API)",
                         "ms_per_loop": sec * 1e3, "tflops": fl / sec / 1e12, "frac_of_peak": fl / sec / 1e12 / tc_sust,
                         "frac_ceiling": {"tf32x3": 1.0 / 6.0, "tf32": 0.5, "f16": 1.0}.get(p1)}
    # batch-1 latency: analysis/trajectory_engine.generate_trajectory (the reference's own call shape), CFG w = 7.5
    torch.manual_seed(42)
    noise = torch.randn(1, 1, 16, 16)
    sec1 = timed(lambda: te.generate_trajectory(teacher16, noise, Cfg.timesteps, dev, seed=42, guidance_scale=7.5), 20)
    out["batch-1 latency"] = {"workload": "generate_trajectory(teacher, noise[1,1,16,16], 50, device, seed, guidance_scale=7.5): one trajectory, "
                                          "2 forward rows per step, noise draws + captured loop + D2H", "precision": get_precision("S2"),
                              "ms_per_trajectory": sec1 * 1e3, "value": 1.0 / sec1, "unit": UNIT}
    # configs[2]: all 11 student size factors vs the teacher at 3x32x32, 50 steps, w = 7.5, through grid.sweep (teacher once)
    S2 = args.config3_seeds
    if S2 > 0:
        t32 = make_model(Cfg32, 1.0, 0, dev)
        students = {f"sf{sf}": make_model(Cfg32, sf, 1000 + int(sf * 100), dev) for sf in SF11}
        prec = get_precision("S2")
        grid.sweep(t32, students, Cfg32, [7.5], S2, dev, max_pairs=S2)                       # builds + captures (untimed)
        torch.cuda.synchronize()
        st = {}
        t0 = time.perf_counter()
        res = grid.sweep(t32, students, Cfg32, [7.5], 2 * S2, dev, max_pairs=S2, stats=st)
        torch.cuda.synchronize()
        sec = time.perf_counter() - t0
        fl = 0.0
        for m in [t32] + list(students.values()):
            eng = UNetEngine.for_model(m, 32, Cfg32.timesteps, prec, dev)
            fl += sum(next(reversed(eng._samplers.values())).flops())            # one chunk: all 12 loops
        # device-resident: the same chunks pre-staged, CUDA events around 2 x run_chunk
        chunks = [grid.stage_chunk(list(range(i * S2, (i + 1) * S2)), Cfg32, [7.5], dev) for i in range(3)]
        studs = list(students.values())
        grid.run_chunk(t32, studs, chunks[0], dev, prec)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in (1, 2):
            grid.run_chunk(t32, studs, chunks[i], dev, prec)
        e1.record()
        torch.cuda.synchronize()
        dsec = e0.elapsed_time(e1) / 1e3
        n_traj = 12 * S2
        out["configs[2]"] = {"workload": f"teacher + 11 students {SF11} at 3x32x32, 50 steps, w=7.5, S2 + pair metrics (teacher trajectories "
                                         f"computed once); chunks of {S2} seeds = {n_traj} trajectories", "precision": prec,
                             "value": 2 * n_traj / dsec, "unit": UNIT + " (device-resident, 2 chunks, CUDA events)",
                             "tflops": 2 * fl / dsec / 1e12, "frac_of_peak": 2 * fl / dsec / 1e12 / tc_sust, "ms_per_chunk": dsec / 2 * 1e3,
                             "e2e": {"value": st["trajectories"] / sec, "unit": UNIT + " (grid.sweep: host draws, H2D, device, D2H, f64 formulas)",
                                     "seconds": sec, "tflops": 2 * fl / sec / 1e12, "frac_of_peak": 2 * fl / sec / 1e12 / tc_sust,
                                     "host_seconds": {k[7:]: round(v, 3) for k, v in st.items() if k.startswith("host_s_")}},
                             "check": {"trajectory_mse@sf0.5": res["sf0.5"][7.5]["trajectory_mse"]},
                             "note": "tflops = algorithmic conv flops (real channels, evaluated taps) of all 12 loops / time"}
        del chunks
        close_engines([t32] + list(students.values()))
        torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--seeds", type=int, default=592, help="seeds per GPU per step (x 8 guidance scales x 2 models); "
                    "a multiple of 148 keeps every conv grid a whole number of waves")
    ap.add_argument("--precision", default="f16", choices=["tf32", "tf32x3", "fp32", "f16"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--quick", action="store_true", help="headline line only: no parity / by_precision / by_config legs")
    ap.add_argument("--ref-seeds", type=int, default=1, help="--impl reference: seeds per step (x 8 scales x 2 models)")
    ap.add_argument("--config3-seeds", type=int, default=1024, help="seeds per chunk of the configs[2] leg (0 = skip)")
    ap.add_argument("--config4-seeds", type=int, default=9472, help="TOTAL seeds of the configs[3]-shaped strong-scaling slice (0 = skip)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's outputs to DIR/<name>.npy (rank 0; see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the CUDA path's outputs: it cannot be combined with --impl reference")
    if args.quick:
        args.config4_seeds = 0
    if args.impl == "reference":
        # the reference picks "cuda if available" for its schedule tables (utils/diffusion.py:52-56): hide CUDA the way its own
        # scripts/run_on_cpu.py:26 does, before torch is imported
        os.environ["CUDA_VISIBLE_DEVICES"] = ""
        os.environ.setdefault("TQDM_DISABLE", "1")
    # stdout carries exactly one JSON line: anything libraries print there meanwhile (NCCL's version banner,
    # model constructors) is sent to stderr
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    lines = []
    emit = lines.append
    try:
        if args.impl == "reference":
            run_reference(args, emit)
        else:
            run_ours(args, emit)
    finally:
        sys.stdout.flush()
        os.dup2(real_stdout, 1)
        os.close(real_stdout)
    for ln in lines:
        print(ln, flush=True)


if __name__ == "__main__":
    main()
