"""CPU: the oracle restatement against what the unmodified reference computes on the same seeded inputs.

The compared values are stored in tests/golden/reference_checks.npz (oracle/make_golden_reference_checks.py says where
they come from), so these tests run everywhere.  Where the reference tree is present (oracle/refload.py) each test also
compares the oracle with the reference live, bit for bit in one process (metrics within 1e-10).

Stored forwards and trajectories are compared within 1e-5 of their largest element, not bit for bit: the CPU convolutions
sum in an order that depends on the thread count and the CPU's vector width (1 thread instead of 8, or AVX2 instead of
AVX-512, moves these values by up to 1.9e-6 of their largest element)."""
import contextlib
import functools
import io

import numpy as np
import pytest
import torch

from helpers import assert_close, load_golden
from oracle import make_golden_reference_checks as mk
from oracle import metrics as om
from oracle import refload, samplers as osmp, unet

TOL = dict(rtol=1e-5, atol_frac=1e-5)


@pytest.fixture(scope="module")
def stored():
    return load_golden("reference_checks")


@pytest.fixture(scope="module")
def ref():
    """The unmodified reference, or None where its tree is absent."""
    return refload.load() if refload.available() else None


def _ref_model(ref, cfg, sf, seed):
    torch.manual_seed(seed)
    with contextlib.redirect_stdout(io.StringIO()):
        return ref.models.DiffusionUNet(refload.RefConfig(cfg.channels, cfg.image_size, cfg.timesteps), sf).eval()


@pytest.mark.parametrize("C,H,sf", mk.FORWARD_CASES)
def test_forward_bit_exact(stored, ref, C, H, sf):
    key = mk.forward_case_key(C, H, sf)
    m = mk.ours_model(mk.Config(C, H, 50), sf, 0)
    mk.check_weights(m, stored, key + "/weights/")
    x, t = torch.from_numpy(stored[key + "/x"]), torch.tensor([17, 17])
    rm = None if ref is None else _ref_model(ref, mk.Config(C, H, 50), sf, 0)
    if rm is not None:
        mk.check_weights(rm, stored, key + "/weights/")
    for name, cond in mk.CONDS.items():
        with torch.no_grad():
            got = unet.unet_forward(m.state_dict(), x, t, cond)
            if rm is not None:
                assert torch.equal(rm(x, t, cond), unet.unet_forward(rm.state_dict(), x, t, cond)), name
        assert_close(got, stored[f"{key}/{name}"], what=f"{key}/{name}", **TOL)


def test_samplers_bit_exact_teacher(stored, ref):
    m = mk.ours_model(mk.Config(1, 16, 4), 1.0, 0)
    mk.check_weights(m, stored, "samplers/weights/")
    f = functools.partial(unet.unet_forward, m.state_dict())
    torch.manual_seed(9)
    _, a = osmp.s1_p_sample_loop(f, (2, 1, 16, 16), 4, osmp.diffusion_params(4), 4, 7.5)
    assert_close(torch.stack(a), stored["samplers/s1"], what="S1", **TOL)
    noise = torch.from_numpy(stored["samplers/s2_noise"])
    b = osmp.s2_generate_trajectory(f, noise, 4, seed=1, guidance_scale=20.0)
    assert_close(torch.stack(b), stored["samplers/s2"], what="S2", **TOL)
    if ref is None:
        return
    cfg = refload.RefConfig(channels=1, image_size=16, timesteps=4)
    rm = _ref_model(ref, cfg, 1.0, 0)
    mk.check_weights(rm, stored, "samplers/weights/")
    f = functools.partial(unet.unet_forward, rm.state_dict())
    torch.manual_seed(9)
    with contextlib.redirect_stderr(io.StringIO()):
        _, a = ref.diffusion.p_sample_loop(rm, (2, 1, 16, 16), 4, ref.diffusion.get_diffusion_params(4, cfg), device="cpu",
                                           config=cfg, track_trajectory=True, guidance_scale=7.5)
    torch.manual_seed(9)
    _, b = osmp.s1_p_sample_loop(f, (2, 1, 16, 16), 4, osmp.diffusion_params(4), 4, 7.5)
    assert all(torch.equal(x, y) for x, y in zip(a, b))
    with contextlib.redirect_stdout(io.StringIO()), contextlib.redirect_stderr(io.StringIO()):
        a = ref.trajectory_engine.generate_trajectory(rm, noise, 4, "cpu", seed=1, guidance_scale=20.0)
    b = osmp.s2_generate_trajectory(f, noise, 4, seed=1, guidance_scale=20.0)
    assert all(torch.equal(x, y) for x, y in zip(a, b))


def test_metrics_match_reference(stored, ref):
    T, S = mk.metric_inputs()
    np.random.seed(4)
    b = om.trajectory_metrics(T, S)
    assert list(b) == list(stored["metrics/keys"])
    for k, tname in zip(stored["metrics/keys"], stored["metrics/types"]):
        np.testing.assert_allclose(np.asarray(b[k], np.float64), stored["metrics/value/" + k], rtol=1e-10, atol=1e-12,
                                   equal_nan=True, err_msg=k)
        assert type(b[k]).__name__ == tname, k
    if ref is None:
        return
    np.random.seed(4)
    a = ref.trajectory_metrics.compute_trajectory_metrics(T, S)
    assert list(a) == list(b)
    for k in a:
        np.testing.assert_allclose(np.asarray(a[k], np.float64), np.asarray(b[k], np.float64), rtol=1e-10, atol=1e-12,
                                   equal_nan=True, err_msg=k)
        assert type(a[k]) is type(b[k]), k
