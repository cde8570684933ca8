"""(seed x guidance scale x student) sweep: the batched, sharded form of the reference's CFG analysis
(scripts/analysis/analyze_trajectory_metrics.py:476-511 calling compare_trajectories per student).

* every (seed, guidance) of a model is one row group of a captured sampling loop (large batch);
* the teacher trajectory of a (seed, guidance) is generated ONCE and compared with every student
  (the reference regenerates it per student although it only depends on seed and guidance);
* seeds are sharded round-robin over ranks -- the grid is embarrassingly parallel -- and the only
  communication is one all-reduce (sum, f64) of the per-(student, guidance) metric sums and counts
  at the end (NCCL over NVLink when the process group is NCCL; gloo in the CPU tests).

A chunk of the sweep goes through three stages so that the device part can be timed on its own:
``stage_chunk`` (host RNG draws exactly as the reference makes them + host-to-device copies),
``run_chunk`` (device only: sampling loops + metric kernels) and ``finish_chunk`` (device-to-host copy
of the per-frame reductions + the f64 scalar formulas).
"""
import os
import time

import numpy as np
import torch

from . import _lib, sampling
from .analysis import trajectory_engine as te
from .analysis.metrics import trajectory_metrics as tm


def shard_samples(num_samples, rank, world_size):
    """Contiguous block ownership (sizes differ by at most one).  Contiguous, not round-robin, because the noise of
    step t of sample s is the stream seeded 42 + s + t (analysis/trajectory_engine.py:88-95): a rank's noise bank holds
    one entry per DISTINCT seed + t, i.e. n + T entries for n consecutive samples but up to n * T for samples spread
    world_size apart (measured at 8 GPUs: 300 ms of host draws per 592-sample chunk, more than the chunk's device time)."""
    base, extra = divmod(num_samples, world_size)
    lo = rank * base + min(rank, extra)
    return list(range(lo, lo + base + (1 if rank < extra else 0)))


def reduce_sums(sums, group=None):
    """All-reduce (sum) of the f64 partial sums [n_students, n_gs, n_keys + 1] (last slot = count)."""
    import torch.distributed as dist
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
        return sums
    backend = dist.get_backend(group)
    dev = torch.device("cuda", torch.cuda.current_device()) if backend == "nccl" else torch.device("cpu")
    t = torch.from_numpy(np.ascontiguousarray(sums)).to(dev)
    dist.all_reduce(t, op=dist.ReduceOp.SUM, group=group)
    return t.cpu().numpy()


def averages_from_sums(sums, student_keys, guidance_scales):
    """{student: {gs: {metric: mean over all seeds}}} (analysis/trajectory_engine.py:171-175)."""
    out = {}
    for i, sk in enumerate(student_keys):
        out[sk] = {}
        for g, gs in enumerate(guidance_scales):
            cnt = sums[i, g, -1]
            out[sk][gs] = {k: (float(sums[i, g, j] / cnt) if cnt > 0 else float("nan"))
                           for j, k in enumerate(tm.SCALAR_KEYS)}
    return out


class Chunk:
    """Device-resident inputs of one batch of (seed, guidance) pairs; pair p = seed-major, guidance-minor."""
    __slots__ = ("samples", "G", "x", "seeds", "groups", "ws", "ws_dev", "bank", "z_index", "idx", "idx_set", "T", "h2d_bytes")


def stage_chunk(samples, config, guidance_scales, device):
    """Host side of a chunk: x_T per sample from the CPU generator seeded 42 + s
    (analysis/trajectory_engine.py:144-149), the per-step noise bank (every distinct seed + t drawn once
    with the reference's calls), the noise index table and the Wasserstein subsample indices; everything
    is copied to ``device`` from pinned host memory."""
    device = torch.device(device)
    C, H, T = config.channels, config.image_size, config.timesteps
    G = len(guidance_scales)
    ck = Chunk()
    ck.samples, ck.G, ck.T = list(samples), G, T
    noises = []
    gen = te._generator(torch.device("cpu"))       # same stream as torch.manual_seed(42 + s); torch.randn(...)
    for s in ck.samples:
        gen.manual_seed(42 + s)
        noises.append(torch.randn(1, C, H, H, generator=gen))
    x = torch.cat(noises).repeat_interleave(G, dim=0)
    ck.seeds = [42 + s for s in ck.samples for _ in range(G)]
    ck.groups = [i for i in range(len(ck.samples)) for _ in range(G)]      # pairs of one sample share x_T: first-step rows are shared
    ck.ws = [gs for _ in ck.samples for gs in guidance_scales]
    ndev = sampling.noise_device(device)
    bank, first = te._noise_bank(ck.seeds, (1, C, H, H), ndev, T)
    ts = np.arange(T - 1, 0, -1)
    zi = (np.asarray(ck.seeds)[None, :] + ts[:, None] - first).astype(np.int32) if len(ts) else np.zeros((1, len(ck.seeds)), np.int32)
    L, D = T + 1, C * H * H
    idx = te.wasserstein_index_sets_device([42 + s for s in ck.samples], T, L, D, device) if device.type == "cuda" else \
        te.wasserstein_index_sets([42 + s for s in ck.samples], T, L, D)
    nbytes = 0

    def up(t):
        nonlocal nbytes
        if t.device == device:
            return t
        nbytes += t.numel() * t.element_size()
        return t.pin_memory().to(device, non_blocking=True)

    ck.x = up(x)
    ck.ws_dev = up(torch.tensor([float(w) if w is not None else 0.0 for w in ck.ws], dtype=torch.float32))
    ck.bank = up(bank)
    ck.z_index = up(torch.from_numpy(zi))
    ck.idx = None if idx is None else (idx if torch.is_tensor(idx) else up(torch.from_numpy(idx)))
    ck.idx_set = None if idx is None else torch.arange(len(ck.samples), dtype=torch.int32, device=device).repeat_interleave(G)
    ck.h2d_bytes = nbytes
    return ck


def run_chunk(teacher_model, student_models, ck, device, precision=None, out_traj=None, verify_weights=False):
    """Device side of a chunk: one captured S2 loop per model over all pairs, then the streaming metric
    kernels for every (teacher, student).  Returns device tensors (red [n_students, N, L, 6],
    w1 [n_students, N, L]) and the number of trajectories generated.  ``out_traj`` (list): receives one
    (teacher [N, L, D], student [N, L, D]) pair of views of the samplers' trajectory buffers per student -- valid
    until the owning sampler runs again (parity checks read the frames behind the reductions through it).
    ``verify_weights``: content-check the cached packed weights against the live modules first (one synchronisation per
    model, engine.UNetEngine.for_model); ``sweep`` does it for its first chunk only, so later chunks stay asynchronous."""
    device = torch.device(device)
    prec = precision or te.get_precision("S2")

    def gen(model):
        model.eval()
        eng = te.UNetEngine.for_model(model, ck.x.shape[2], ck.T, prec, device, verify=verify_weights)
        return sampling.s2_sample(eng, ck.x, ck.T, ck.ws, ck.bank, ck.z_index, guidance_dev=ck.ws_dev,
                                  groups=getattr(ck, "groups", None))

    # The teacher's and the students' loops are independent until the metrics: the students run on side streams, so that
    # their CTAs fill the tails of the teacher's persistent kernels and vice versa (+2.3 % trajectories/s on the bench
    # workload, identical results).  DTRAJ_MODEL_STREAMS = number of side streams the students are dealt over (default 3:
    # the narrow students of an 11-student sweep leave most SMs idle on their own); 0 serialises everything.
    cur = torch.cuda.current_stream(device)
    n_side = int(os.environ.get("DTRAJ_MODEL_STREAMS", "3"))
    if os.environ.get("DTRAJ_OVERLAP_MODELS", "1") == "0":
        n_side = 0
    distinct = [m for m in student_models if m is not teacher_model]
    sides = [_copy_stream(device, f"models{i}") for i in range(min(n_side, len(distinct)))]
    for sd in sides:
        sd.wait_stream(cur)                           # the chunk's uploads were queued on the current stream
    tt = gen(teacher_model)
    t_flat = tt.reshape(tt.shape[0], tt.shape[1], -1)
    n_traj = tt.shape[0]
    flats, k = [], 0
    for sm_model in student_models:                   # queue every student loop first ...
        if sm_model is teacher_model:
            flats.append((t_flat, None))
            continue
        sd = sides[k % len(sides)] if sides else None
        k += 1
        if sd is not None:
            with torch.cuda.stream(sd):
                st = gen(sm_model)
        else:
            st = gen(sm_model)
        flats.append((st.reshape(st.shape[0], st.shape[1], -1), sd))
        n_traj += st.shape[0]
    for sd in sides:
        cur.wait_stream(sd)
    reds, w1s = [], []
    for s_flat, sd in flats:                          # ... then the pair metrics behind all of them
        reds.append(tm.pair_reductions(t_flat, s_flat))
        w1s.append(tm.wasserstein_frames(t_flat, s_flat, ck.idx, ck.idx_set))
        if out_traj is not None:
            out_traj.append((t_flat, s_flat))
    for sd in sides:
        sd.wait_stream(cur)                           # the next chunk's student loops must not overtake these metric kernels
    return torch.stack(reds), torch.stack(w1s), n_traj


class _Readback:
    """Device-to-host copy of a chunk's reductions on a side stream, so that waiting for chunk i's numbers
    does not wait for chunk i+1's kernels (already queued on the compute stream)."""

    def __init__(self, red, w1, device, engines=()):
        self.stream = _copy_stream(device)
        ready = torch.cuda.Event()
        ready.record(torch.cuda.current_stream(device))
        self.red_h = torch.empty(red.shape, dtype=red.dtype, pin_memory=True)
        self.w1_h = torch.empty(w1.shape, dtype=w1.dtype, pin_memory=True)
        self.engines = list(engines)
        self.flag_h = torch.zeros(1 + len(self.engines), dtype=torch.int32, pin_memory=True)   # device error words (library-wide, then
                                                                                                 # one per engine), read without a device-wide sync
        self.keep = (red, w1)                       # keep the device tensors alive until the copy is done
        with torch.cuda.stream(self.stream):
            self.stream.wait_event(ready)
            self.red_h.copy_(red, non_blocking=True)
            self.w1_h.copy_(w1, non_blocking=True)
            _lib.check(_lib.load().dtraj_error_flag_async(self.flag_h.data_ptr(), self.stream.cuda_stream))
            for i, eng in enumerate(self.engines):
                eng.error_flag_async(self.flag_h.data_ptr() + 4 * (i + 1), self.stream.cuda_stream)
            self.done = torch.cuda.Event()
            self.done.record(self.stream)

    def wait(self):
        self.done.synchronize()
        self.keep = None
        for i, eng in enumerate(self.engines):        # the engine (model) whose kernels flagged the error is named in the message
            if int(self.flag_h[i + 1]) != 0:
                eng.check_errors()
        if int(self.flag_h[0]) != 0:
            te.check_device_errors()                  # raises (pipeline time-out / fp16 overflow) and clears the flag
        return self.red_h.numpy(), self.w1_h.numpy()


_copy_streams = {}


def _copy_stream(device, tag="copy"):
    key = (str(device), tag)
    if key not in _copy_streams:
        _copy_streams[key] = torch.cuda.Stream(device)
    return _copy_streams[key]


def finish_chunk(red, w1, ck, config, sums):
    """Device-to-host copy of the reductions and the f64 scalar formulas; accumulates into ``sums``.
    ``red`` / ``w1`` are device tensors or the numpy arrays of a finished ``_Readback``.  Returns the bytes copied."""
    H, D = config.image_size, config.channels * config.image_size ** 2
    if not isinstance(red, np.ndarray):               # (a finished _Readback has checked the device error word already)
        red, w1 = red.cpu().numpy(), w1.cpu().numpy()
        te.check_device_errors()                      # pipeline time-out / fp16 overflow flagged by a kernel of this chunk
    red_h, w1_h = red, w1
    for i in range(red_h.shape[0]):
        sm = tm.scalar_metrics_batched(red_h[i], w1_h[i], H * H, D)
        for j, k in enumerate(tm.SCALAR_KEYS):
            sums[i, :, j] += sm[k].reshape(len(ck.samples), ck.G).sum(axis=0)
        sums[i, :, -1] += len(ck.samples)
    return red_h.nbytes + w1_h.nbytes


def seeds_per_chunk_64(teacher_model, student_models, config, n_scales, precision, device, mem_fraction=0.6):
    """64x64 sweeps only: the most seeds per chunk whose buffers fit in ``mem_fraction`` of the device's memory.  Per (seed, guidance)
    pair and model: the forward workspace of up to two rows (CFG; dtraj_unet_workspace_bytes: about 5 MB per row of the 3x64x64
    teacher in fp16, twice that in the TF32 modes) and the trajectory buffer of the model's captured loop; per student also the
    contiguous copies of both trajectories that ``pair_reductions`` reduces when a frame is wider than MAX_GROUP_ELEMS.  (Measured
    on a B200 with the teacher and the sf 0.5 student: 101.8 GB peak against about 106 GB estimated for a 512-seed fp16 chunk,
    profiles/r03a_image64_bench.json.)  At 16x16 and 32x32 the chunk is ``max_pairs`` alone."""
    prec = precision or te.get_precision("S2")
    H, T = int(config.image_size), int(config.timesteps)
    D = int(config.channels) * H * H
    frames = (T + 2) * D * 4                          # one trajectory (x_T, T - 1 updates, the repeated last frame) + slack
    models = {id(m): m for m in [teacher_model] + list(student_models)}
    per_pair = 0.0
    for m in models.values():
        eng = te.UNetEngine.for_model(m.eval(), H, T, prec, device, verify=False)
        per_pair += eng.workspace_bytes(2 * 1024) / 1024 + frames
    n_students = sum(1 for m in student_models if m is not teacher_model)
    if D > tm.MAX_GROUP_ELEMS:
        per_pair += n_students * 2 * frames
    budget = mem_fraction * torch.cuda.get_device_properties(device).total_memory
    return max(1, int(budget // (per_pair * n_scales)))


def _drop_samplers(models, device):
    """Release the captured loops (workspaces, trajectory buffers) cached on the engines of ``models`` once the device has
    finished with them."""
    torch.cuda.synchronize(device)
    for m in models:
        for ent in m.__dict__.get("_dtraj_engines", {}).values():
            ent[1].drop_samplers()


@torch.no_grad()
def sweep(teacher_model, students, config, guidance_scales, num_samples, device=None, rank=0, world_size=1,
          max_pairs=4096, precision=None, reduce=True, stats=None):
    """Run the sweep for ``students`` (dict name -> model) against ``teacher_model``.

    Returns {name: {gs: {18 scalar metrics averaged over all ``num_samples`` seeds}}}; with
    ``reduce=True`` every rank returns the global averages.  ``stats`` (dict) receives counters:
    trajectories generated, pairs measured, bytes moved each way.

    Chunks are software-pipelined: while the GPU runs chunk i (kernel launches are asynchronous), the
    host draws and uploads chunk i+1's noise and evaluates chunk i-1's scalar formulas from a side-stream
    read-back, so host work hides behind device work whenever a sweep has more than one chunk.
    """
    if device is None:
        device = next(teacher_model.parameters()).device
    device = torch.device(device)
    guidance_scales = list(guidance_scales)
    G = len(guidance_scales)
    names = list(students)
    models = [students[n] for n in names]
    sums = np.zeros((len(names), G, len(tm.SCALAR_KEYS) + 1), np.float64)
    mine = shard_samples(num_samples, rank, world_size)
    per_chunk = max(1, max_pairs // G)
    big = int(config.image_size) == 64 and device.type == "cuda"
    if big:
        per_chunk = min(per_chunk, seeds_per_chunk_64(teacher_model, models, config, G, precision, device))
    pieces = [mine[c0:c0 + per_chunk] for c0 in range(0, len(mine), per_chunk)]
    n_traj = n_pairs = h2d = d2h = 0
    pending = None                                  # (readback, chunk) of the previous chunk
    nxt = stage_chunk(pieces[0], config, guidance_scales, device) if pieces else None
    tm_ = {"run": 0.0, "stage": 0.0, "wait": 0.0, "finish": 0.0}
    for i in range(len(pieces)):
        ck = nxt
        if big and i > 0 and len(pieces[i]) != len(pieces[i - 1]):
            _drop_samplers([teacher_model] + models, device)   # (64x64: the loops of the full chunks would stay cached beside the last one's)
        t0 = time.perf_counter()
        red, w1, nt = run_chunk(teacher_model, models, ck, device, precision, verify_weights=(i == 0))   # queued, not waited for
        engines = [ent[1] for m in [teacher_model] + models for ent in m.__dict__.get("_dtraj_engines", {}).values()
                   if getattr(ent[1], "handle", None)]
        rb = _Readback(red, w1, device, engines)
        t1 = time.perf_counter()
        nxt = stage_chunk(pieces[i + 1], config, guidance_scales, device) if i + 1 < len(pieces) else None
        t2 = time.perf_counter()
        tm_["run"] += t1 - t0
        tm_["stage"] += t2 - t1
        if pending is not None:
            arrs = pending[0].wait()
            t3 = time.perf_counter()
            d2h += finish_chunk(*arrs, pending[1], config, sums)
            tm_["wait"] += t3 - t2
            tm_["finish"] += time.perf_counter() - t3
        pending = (rb, ck)
        h2d += ck.h2d_bytes
        n_traj += nt
        n_pairs += len(ck.seeds) * len(names)
    if pending is not None:
        d2h += finish_chunk(*pending[0].wait(), pending[1], config, sums)
    if stats is not None:
        for k, v in (("trajectories", n_traj), ("pairs", n_pairs), ("h2d_bytes", h2d), ("d2h_bytes", d2h)):
            stats[k] = stats.get(k, 0) + v
        for k, v in tm_.items():                      # host seconds per phase (wait = blocked on the previous chunk's read-back)
            stats["host_s_" + k] = stats.get("host_s_" + k, 0.0) + v
    if reduce:
        sums = reduce_sums(sums)
    return averages_from_sums(sums, names, guidance_scales)
