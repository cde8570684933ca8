"""Generate tests/golden/reference_checks.npz: the stored side of tests/test_oracle_vs_reference.py and of
tests/test_host_logic.py::test_model_aliases_match_the_reference_constructors.

TEST INFRASTRUCTURE (see oracle/__init__.py).

    python -m oracle.make_golden_reference_checks

Those tests used to compare the oracle only live against the unmodified reference, so they checked nothing where the
reference tree is absent.  This file holds, for exactly their seeded inputs, the values they compared: forwards of three
(channels, size, size_factor) models under three conditionings, one S1 and one S2 trajectory, the Q1 metrics dict (key
order, values, value types), and the parameter names, shapes, per-tensor sums and widths of the SimpleUNet / StudentUNet
aliases.  Seeded weights are pinned by those per-tensor sums, not by their bytes: torch.randn's vectorised CPU kernels
differ in the last bit between CPU capability levels.

Provenance: the reference tree was not available when this file was made, so the values come from the oracle
(``oracle/unet.py``, ``oracle/samplers.py``, ``oracle/metrics.py``) and the package's model constructors, at a commit where
the live tests had last passed against the reference with the same oracle code: bit-exact forwards and samplers, metrics
within 1e-10, equal alias parameters.  Whenever the reference is present the tests also compare the oracle with it live.
"""
import contextlib
import functools
import io
import os

import numpy as np
import torch

from . import metrics as om
from . import samplers as osmp
from . import unet

OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden", "reference_checks.npz")

FORWARD_CASES = [(1, 16, 1.0), (3, 32, 0.3), (1, 16, 0.6)]
CONDS = {"none": None, "cond1": torch.ones(2, 1), "cond0": torch.zeros(2, 1)}


class Config:
    """The attributes the model constructors read (oracle/refload.py::RefConfig without the reference import)."""

    def __init__(self, channels, image_size, timesteps):
        self.channels, self.image_size, self.timesteps, self.dropout = channels, image_size, timesteps, 0.3


def weights(model, prefix):
    """Fingerprint of a state_dict: its keys in order, each tensor's shape, sum and sum of magnitudes (float64)."""
    sd = model.state_dict()
    return {prefix + "keys": np.array(list(sd)), prefix + "shapes": np.array(["x".join(map(str, v.shape)) for v in sd.values()]),
            prefix + "sums": np.array([[v.double().sum().item(), v.double().abs().sum().item()] for v in sd.values()])}


def check_weights(model, g, prefix):
    """``model``'s parameters are the ones ``g`` fingerprints under ``prefix``: same keys and shapes, sums within 1e-6 of
    the sum of magnitudes."""
    got = weights(model, prefix)
    assert list(got[prefix + "keys"]) == list(g[prefix + "keys"]), prefix
    assert list(got[prefix + "shapes"]) == list(g[prefix + "shapes"]), prefix
    a, b = got[prefix + "sums"], g[prefix + "sums"]
    assert (np.abs(a - b) <= 1e-6 * b[:, 1:2]).all(), f"{prefix}: seeded weights differ from the ones the vectors were made with"


def forward_case_key(C, H, sf):
    return f"fwd/{C}x{H}_sf{sf}"


def metric_inputs():
    rng = np.random.RandomState(0)
    T = [torch.from_numpy(rng.randn(1, 3, 32, 32).astype(np.float32)) for _ in range(9)]
    S = [t + 0.05 * torch.from_numpy(rng.randn(1, 3, 32, 32).astype(np.float32)) for t in T]
    return T, S


def build(make_model, make_alias):
    """``make_model(cfg, sf, seed)`` -> a seeded DiffusionUNet; ``make_alias(cfg, which)`` -> SimpleUNet / StudentUNet(cfg, 0.3, "tiny")."""
    g = {}
    for C, H, sf in FORWARD_CASES:
        key = forward_case_key(C, H, sf)
        m = make_model(Config(C, H, 50), sf, 0)
        x, t = torch.randn(2, C, H, H), torch.tensor([17, 17])
        g[key + "/x"] = x.numpy()
        g.update(weights(m, key + "/weights/"))
        for name, cond in CONDS.items():
            g[f"{key}/{name}"] = unet.unet_forward(m.state_dict(), x, t, cond).numpy()

    m = make_model(Config(1, 16, 4), 1.0, 0)
    f = functools.partial(unet.unet_forward, m.state_dict())
    g.update(weights(m, "samplers/weights/"))
    torch.manual_seed(9)
    _, traj = osmp.s1_p_sample_loop(f, (2, 1, 16, 16), 4, osmp.diffusion_params(4), 4, 7.5)
    g["samplers/s1"] = torch.stack(traj).numpy()
    noise = torch.randn(1, 1, 16, 16)
    g["samplers/s2_noise"] = noise.numpy()
    g["samplers/s2"] = torch.stack(osmp.s2_generate_trajectory(f, noise, 4, seed=1, guidance_scale=20.0)).numpy()

    T, S = metric_inputs()
    np.random.seed(4)
    mt = om.trajectory_metrics(T, S)
    g["metrics/keys"] = np.array(list(mt))
    g["metrics/types"] = np.array([type(v).__name__ for v in mt.values()])
    for k, v in mt.items():
        g["metrics/value/" + k] = np.asarray(v, np.float64)

    cfg = Config(1, 16, 8)
    for which in ("simple", "student"):
        with contextlib.redirect_stdout(io.StringIO()):
            torch.manual_seed(4)
            a = make_alias(cfg, which)
        g.update(weights(a, f"alias/{which}/weights/"))
        g[f"alias/{which}/dims"] = np.array(a.dims, np.int64)
        g[f"alias/{which}/time_emb_dim"] = np.array(a.time_emb_dim, np.int64)
    return g


def ours_model(cfg, sf, seed):
    from distillation_trajectories_b200.models import DiffusionUNet
    torch.manual_seed(seed)
    with contextlib.redirect_stdout(io.StringIO()):
        return DiffusionUNet(cfg, sf).eval()


def ours_alias(cfg, which):
    from distillation_trajectories_b200 import models
    return models.SimpleUNet(cfg) if which == "simple" else models.StudentUNet(cfg, 0.3, "tiny")


def main():
    with torch.no_grad():
        g = build(ours_model, ours_alias)
    np.savez_compressed(OUT, **g)
    print(OUT, os.path.getsize(OUT) // 1024, "KiB")


if __name__ == "__main__":
    main()
