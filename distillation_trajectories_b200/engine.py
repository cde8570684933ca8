"""Host-side owners of the libdtraj handles: a packed U-Net and a captured sampling loop.

PyTorch is used here only for device memory, streams and the RNG draws that must match
the reference's noise; all arithmetic of the hot path runs inside libdtraj.so.
"""
import ctypes as C
import os
import weakref

import numpy as np
import torch

from . import _lib
from ._lib import (PREC_FP32, PREC_TF32, PREC_TF32X3, RULE_S1, RULE_S2, RULE_S3, VAR_COND0, VAR_COND1,
                   VAR_NONE, DtrajError)

_default_precision = {"S1": os.environ.get("DTRAJ_PRECISION_S1", os.environ.get("DTRAJ_PRECISION", "tf32x3")),
                      "S2": os.environ.get("DTRAJ_PRECISION_S2", os.environ.get("DTRAJ_PRECISION", "f16")),
                      "S3": os.environ.get("DTRAJ_PRECISION_S3", os.environ.get("DTRAJ_PRECISION", "f16")),
                      "forward": os.environ.get("DTRAJ_PRECISION", "tf32x3")}


def set_precision(mode, path=None):
    """Choose the conv arithmetic: 'fp32' (CUDA cores), 'tf32' (tcgen05 kind::tf32, one pass), 'tf32x3'
    (tcgen05, error-compensated) or 'f16' (tcgen05 kind::f16: fp16 feature maps and weights -- the same 11-bit
    significand as tf32 -- with fp32 accumulation; a value outside the fp16 range raises DtrajError instead of
    overflowing silently).  ``path`` in {'S1','S2','S3','forward'} or None for all."""
    if mode not in _lib.PRECISIONS:
        raise ValueError(f"precision must be one of {sorted(_lib.PRECISIONS)}")
    for k in ([path] if path else list(_default_precision)):
        _default_precision[k] = mode


def get_precision(path):
    return _default_precision[path]


def _require_cuda(device):
    device = torch.device(device)
    if device.type != "cuda":
        raise DtrajError(f"distillation_trajectories_b200 runs on CUDA (sm_100a) only; got device '{device}'. "
                         "There is no CPU fallback.")
    return device


def _model_geometry(model):
    """Duck-typed read of a reference DiffusionUNet (models.py:95-110)."""
    return dict(channels=int(model.channels), dims=[int(d) for d in model.dims],
                temb_dim=int(model.time_emb_dim))


def _weights_fingerprint(model):
    """Identity of the weight STORAGE: tensor ids, autograd versions and data pointers.  Catches ``load_state_dict``,
    optimizer steps, ``p.data = new`` and re-allocations; an in-place write through ``p.data`` (the EMA idiom
    ``p.data.mul_(d).add_(...)``) bumps none of them -- that is what ``_weights_checksum`` is for."""
    return tuple((id(t), t._version, t.data_ptr()) for t in list(model.parameters()) + list(model.buffers()))


def _weights_checksum(model):
    """Content check of every floating-point parameter / buffer: position-weighted sums of the per-tensor L1 and L2
    norms, two multi-tensor kernels and one scalar read-back (synchronises the current stream, so it runs where an
    entry point hands results to the host anyway -- not between the chunks of a sweep, see ``for_model(verify=)``)."""
    ts = [t.detach() for t in list(model.parameters()) + list(model.buffers()) if torch.is_floating_point(t)]
    if not ts:
        return 0.0
    v = torch.stack(torch._foreach_norm(ts, 1) + torch._foreach_norm(ts, 2)).double()
    w = torch.arange(1, v.numel() + 1, dtype=torch.float64, device=v.device)
    return float((v * w).sum())


_live_engines = weakref.WeakSet()      # every UNetEngine with an open handle: check_device_errors() polls their error words


class UNetEngine:
    """BN-folded, packed copy of one U-Net on one GPU + its time-embedding tables."""

    def __init__(self, state_dict, channels, image_size, dims, temb_dim, n_timesteps, precision, device):
        self.lib = _lib.load()
        self.device = _require_cuda(device)
        self.channels, self.image_size, self.dims, self.temb_dim = channels, image_size, list(dims), temb_dim
        self.n_timesteps = int(n_timesteps)
        self.precision = precision if isinstance(precision, int) else _lib.PRECISIONS[precision]
        self.D = channels * image_size * image_size
        desc = _lib.UNetDesc(channels, image_size, (C.c_int32 * 4)(*dims), temb_dim, self.n_timesteps, self.precision)
        keep, names, ptrs, numel = [], [], [], []
        for k, v in state_dict.items():
            if not torch.is_floating_point(v):
                continue                       # num_batches_tracked
            a = v.detach().to("cpu", torch.float32).contiguous()
            keep.append(a)
            names.append(k.encode())
            ptrs.append(a.data_ptr())
            numel.append(a.numel())
        n = len(names)
        handle = C.c_void_p()
        with torch.cuda.device(self.device):
            _lib.check(self.lib.dtraj_unet_create(C.byref(desc), (C.c_char_p * n)(*names), (C.c_void_p * n)(*ptrs),
                                                  (C.c_int64 * n)(*numel), n, C.byref(handle)))
        self.handle = handle
        self._ws = None
        self._samplers = {}
        self.label = f"U-Net dims={list(dims)} {channels}x{image_size}x{image_size} [{ {v: k for k, v in _lib.PRECISIONS.items()}[self.precision] }]"
        _live_engines.add(self)

    @classmethod
    def for_model(cls, model, image_size, n_timesteps, precision, device=None, verify=True):
        """Engine cached on the module; rebuilt when weights, precision or table size change.
        ``verify=True`` also compares a content checksum of the weights with the one taken when the cached engine was
        packed, so that in-place ``.data`` updates (which leave tensor versions untouched) are noticed; it costs one
        host-device synchronisation.  Loops that must stay asynchronous (the chunks of ``grid.sweep``) verify once up
        front and pass ``verify=False`` afterwards; ``invalidate(model)`` drops the cache explicitly."""
        if getattr(model, "training", False):
            raise DtrajError("model is in training mode; the hot path needs model.eval() "
                             "(eval-mode BatchNorm/Dropout, as every reference caller does)")
        if device is None:
            device = next(model.parameters()).device
        device = _require_cuda(device)
        prec = precision if isinstance(precision, int) else _lib.PRECISIONS[precision]
        cache = model.__dict__.setdefault("_dtraj_engines", {})
        key = (prec, int(image_size), str(device))
        fp = _weights_fingerprint(model)
        ent = cache.get(key)
        if ent is not None and ent[0] == fp and ent[1].n_timesteps >= n_timesteps:
            if not verify or _weights_checksum(model) == ent[2]:
                return ent[1]
        if ent is not None:
            n_timesteps = max(n_timesteps, ent[1].n_timesteps)
            ent[1].close()
        g = _model_geometry(model)
        eng = cls(model.state_dict(), g["channels"], int(image_size), g["dims"], g["temb_dim"], n_timesteps, prec, device)
        cache[key] = (fp, eng, _weights_checksum(model))
        return eng

    @staticmethod
    def invalidate(model):
        """Drop every cached engine of ``model`` (and the CUDA graphs captured on them)."""
        for ent in model.__dict__.pop("_dtraj_engines", {}).values():
            ent[1].close()

    def drop_samplers(self):
        """Destroy the cached sampling loops (captured graphs) and release their workspaces and trajectory buffers.  The caller
        makes sure the device has finished with them."""
        for s in self._samplers.values():
            s.close()
        self._samplers = {}

    def close(self):
        self.drop_samplers()
        _live_engines.discard(self)
        if getattr(self, "handle", None):
            self.lib.dtraj_unet_destroy(self.handle)
            self.handle = None

    def check_errors(self):
        """Read and clear THIS engine's device error word (pipeline time-out / fp16 overflow flagged by one of its
        kernels); raises DtrajError naming the model.  Synchronises the device."""
        if not getattr(self, "handle", None):
            return
        with torch.cuda.device(self.device):
            rc = self.lib.dtraj_unet_check_errors(self.handle)
        if rc != 0:
            msg = self.lib.dtraj_last_error()
            raise DtrajError(f"libdtraj error {rc} in {self.label}: {msg.decode() if msg else '?'}")

    def error_flag_async(self, host_flag_ptr, stream_ptr):
        """Enqueue a copy of this engine's error word into pinned host memory (non-blocking form of check_errors)."""
        _lib.check(self.lib.dtraj_unet_error_flag_async(self.handle, C.c_void_p(host_flag_ptr), C.c_void_p(stream_ptr)))

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def workspace_bytes(self, n_rows):
        b = self.lib.dtraj_unet_workspace_bytes(self.handle, n_rows)
        if b < 0:
            raise DtrajError("workspace query failed")
        return b

    def workspace(self, n_rows):
        need = self.workspace_bytes(n_rows)
        if self._ws is None or self._ws.numel() < need:
            self._ws = torch.empty(need, dtype=torch.uint8, device=self.device)
        return self._ws

    def time_bias(self, t, variant, block):
        n = [self.dims[0], self.dims[1], self.dims[2], self.dims[3], self.dims[3], self.dims[2], self.dims[1], self.dims[0]][block]
        out = np.empty(n, dtype=np.float32)
        _lib.check(self.lib.dtraj_unet_time_bias(self.handle, t, variant, block, out.ctypes.data_as(C.c_void_p), n))
        return out

    def forward(self, x, t, variants=None):
        """eps = U-Net(x, t, cond).  ``t``: one int for the whole batch (the sampling loops), or an int tensor [R]
        with a timestep per row (p_losses, the distillation step).  ``variants``: int32 [R] of VAR_*."""
        x = x.to(self.device, torch.float32).contiguous()
        R = x.shape[0]
        if tuple(x.shape[1:]) != (self.channels, self.image_size, self.image_size):
            raise DtrajError(f"input shape {tuple(x.shape)} does not match engine "
                             f"({self.channels},{self.image_size},{self.image_size})")
        if variants is not None:
            variants = variants.to(self.device, torch.int32).contiguous()
        eps = torch.empty_like(x)
        ws = self.workspace(R)
        if torch.is_tensor(t):
            tv = t.reshape(R, -1)[:, 0].to(self.device, torch.int64)
            if int(tv.min()) < 0 or int(tv.max()) >= self.n_timesteps:
                raise DtrajError(f"timesteps outside the engine's table (0..{self.n_timesteps - 1})")
            row_tv = (tv * 3 + (variants.to(torch.int64) if variants is not None else 0)).to(torch.int32).contiguous()
            with torch.cuda.device(self.device):
                _lib.check(self.lib.dtraj_unet_forward_rows(self.handle, _lib.ptr(x), R, _lib.ptr(row_tv), _lib.ptr(eps),
                                                            _lib.ptr(ws), ws.numel(), _lib.stream_ptr()))
            return eps
        with torch.cuda.device(self.device):
            _lib.check(self.lib.dtraj_unet_forward(self.handle, _lib.ptr(x), R, int(t), _lib.ptr(variants), _lib.ptr(eps),
                                                   _lib.ptr(ws), ws.numel(), _lib.stream_ptr()))
        return eps


class TrajectorySampler:
    """One captured sampling loop: fixed (rule, batch layout, timestep list, coefficients).

    Inputs are written into the device buffers it owns (``traj[:, 0]`` = x_T, ``z_bank``,
    ``guidance``, ``z_index``) and ``run()`` replays the loop (one CUDA graph launch).
    """

    def __init__(self, engine, rule, n_samples, row_sample, row_variant, sample_row_u, sample_row_c,
                 timesteps, coefs, copy_last, n_noise, use_graph=True, first_layout=None):
        self.engine = engine
        self.lib = engine.lib
        dev = engine.device
        self.rule, self.B = rule, int(n_samples)
        self.n_updates = len(timesteps)
        self.n_frames = 1 + self.n_updates + (1 if copy_last else 0)
        self.n_rows = len(row_sample)
        i32 = dict(dtype=torch.int32, device=dev)
        self.row_sample = torch.as_tensor(np.asarray(row_sample, np.int32), **i32)
        self.row_variant = torch.as_tensor(np.asarray(row_variant, np.int32), **i32)
        self.sample_row_u = torch.as_tensor(np.asarray(sample_row_u, np.int32), **i32)
        self.sample_row_c = None if sample_row_c is None else torch.as_tensor(np.asarray(sample_row_c, np.int32), **i32)
        self.guidance = torch.zeros(self.B, dtype=torch.float32, device=dev)
        self.n_noise = int(n_noise)
        self.z_bank = torch.zeros(max(self.n_noise, 1), engine.D, dtype=torch.float32, device=dev)
        self.z_index = torch.full((max(self.n_updates, 1), self.B), -1, **i32)
        self.traj = torch.zeros(self.B, self.n_frames, engine.channels, engine.image_size, engine.image_size,
                                dtype=torch.float32, device=dev)
        self.ws = torch.empty(engine.workspace_bytes(self.n_rows), dtype=torch.uint8, device=dev)
        ts = np.asarray(timesteps, np.int32)
        cf = np.ascontiguousarray(np.asarray(coefs, np.float32).reshape(-1))
        if cf.size != 3 * self.n_updates:
            raise ValueError("coefs must be [n_updates, 3]")
        d = _lib.SamplerDesc()
        d.rule, d.n_samples, d.n_rows, d.n_updates = rule, self.B, self.n_rows, self.n_updates
        d.copy_last, d.n_frames, d.use_graph = int(bool(copy_last)), self.n_frames, int(bool(use_graph))
        d.step_timestep = ts.ctypes.data if ts.size else None
        d.step_coef = cf.ctypes.data if cf.size else None
        d.row_sample, d.row_variant = self.row_sample.data_ptr(), self.row_variant.data_ptr()
        d.sample_row_u = self.sample_row_u.data_ptr()
        d.sample_row_c = None if self.sample_row_c is None else self.sample_row_c.data_ptr()
        d.guidance = self.guidance.data_ptr()
        d.z_bank, d.z_index = self.z_bank.data_ptr(), self.z_index.data_ptr()
        d.traj, d.workspace, d.workspace_bytes = self.traj.data_ptr(), self.ws.data_ptr(), self.ws.numel()
        if first_layout is not None:          # (row_sample0, row_variant0, sample_row_u0, sample_row_c0): shared rows at step 0
            self.first = [torch.as_tensor(np.asarray(a, np.int32), **i32) for a in first_layout]
            d.n_rows0 = len(first_layout[0])
            d.row_sample0, d.row_variant0 = self.first[0].data_ptr(), self.first[1].data_ptr()
            d.sample_row_u0, d.sample_row_c0 = self.first[2].data_ptr(), self.first[3].data_ptr()
        h = C.c_void_p()
        with torch.cuda.device(dev):
            torch.cuda.synchronize(dev)
            _lib.check(self.lib.dtraj_sampler_create(engine.handle, C.byref(d), C.byref(h)))
        self.handle = h
        self.launches = int(self.lib.dtraj_sampler_launches(h))

    def run(self):
        with torch.cuda.device(self.engine.device):
            _lib.check(self.lib.dtraj_sampler_run(self.handle, _lib.stream_ptr()))
        return self.traj

    def profile(self):
        """One un-captured run with an event pair around every launch (see include/dtraj.h).
        Returns dict(ms=[5], launches=[5], conv_flops=float, enc1_flops=float)."""
        ms, nl, fl = (C.c_double * 5)(), (C.c_int64 * 5)(), (C.c_double * 2)()
        with torch.cuda.device(self.engine.device):
            _lib.check(self.lib.dtraj_sampler_profile(self.handle, _lib.stream_ptr(), ms, nl, fl))
        return dict(ms=list(ms), launches=list(nl), conv_flops=fl[0], enc1_flops=fl[1])

    def flops(self):
        """Algorithmic conv flops of one run() (real channels, evaluated taps): (generic convs, fused enc1 kernel)."""
        fl = (C.c_double * 2)()
        _lib.check(self.lib.dtraj_sampler_flops(self.handle, fl))
        return float(fl[0]), float(fl[1])

    def profile_layers(self, step=1):
        """One un-captured run with an event pair around every launch; returns [(name, grid, microseconds, flops)] for the
        launches of sampler step ``step`` (diagnostics, tools/profile_layers.py)."""
        buf = C.create_string_buffer(1 << 16)
        with torch.cuda.device(self.engine.device):
            _lib.check(self.lib.dtraj_sampler_profile_text(self.handle, _lib.stream_ptr(), int(min(step, self.n_updates - 1)), buf, len(buf)))
        rows = []
        for ln in buf.value.decode().splitlines():
            name, grid, us, fl = ln.split("\t")
            rows.append((name, int(grid), float(us), float(fl)))
        return rows

    def close(self):
        if getattr(self, "handle", None):
            self.lib.dtraj_sampler_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def cached_sampler(engine, key, factory):
    s = engine._samplers.get(key)
    if s is None:
        if len(engine._samplers) >= 8:            # bound the device memory held by old layouts
            old = next(iter(engine._samplers))
            engine._samplers.pop(old).close()
        s = factory()
        engine._samplers[key] = s
    return s


def check_device_errors(device=None):
    """Raise DtrajError if a kernel flagged a pipeline time-out or an fp16 overflow since the last check.
    Synchronises the device: called where results leave the library.  ``device``: the engine's device (the error
    word lives in that device's copy of the library's globals); default = the current device."""
    dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
    if dev.index is None:
        dev = torch.device("cuda", torch.cuda.current_device())
    first = None
    for eng in list(_live_engines):          # every word is read (and cleared) before the first failure is raised
        if eng.device.index in (None, dev.index):
            try:
                eng.check_errors()
            except DtrajError as e:
                first = first or e
    with torch.cuda.device(dev):
        rc = _lib.load().dtraj_check_errors()     # launches without a handle (test hooks)
    if first is not None:
        raise first
    _lib.check(rc)


def umma_error_flag():
    """Non-zero if a kernel flagged a pipeline time-out or an fp16 overflow that nobody has collected yet: the
    library-wide word OR-ed with the word of every live engine (peeked, not cleared)."""
    v = int(_lib.load().dtraj_debug_umma_error())
    for eng in list(_live_engines):
        if getattr(eng, "handle", None):
            flag = torch.zeros(1, dtype=torch.int32).pin_memory()
            with torch.cuda.device(eng.device):
                eng.error_flag_async(flag.data_ptr(), torch.cuda.current_stream().cuda_stream)
                torch.cuda.current_stream().synchronize()
            v |= int(flag[0])
    return v
