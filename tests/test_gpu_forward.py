"""GPU: DiffusionUNet.forward through libdtraj against the committed reference outputs
(tests/golden, made by the unmodified reference on CPU) and against the CPU oracle."""
import numpy as np
import pytest
import torch

from oracle import unet as ounet
from distillation_trajectories_b200 import set_precision, umma_error_flag, _lib
from distillation_trajectories_b200.engine import UNetEngine
from helpers import Cfg, assert_close, cpu_sd, golden_models, make_model

pytestmark = pytest.mark.gpu

# max |err| / max |ref| allowed for one forward.  fp32 / 3xTF32 differ from the reference only by
# summation order and BatchNorm folding (3xTF32 also by the tensor core's round-toward-zero
# accumulation, ~1e-5 per deep layer); single-pass TF32 carries 10-bit-mantissa operand rounding.
# fp16 operands ("f16") have the same 11-bit significand as tf32, hence the same bound.
FWD_TOL = {"fp32": 2e-5, "tf32x3": 6e-5, "tf32": 4e-3, "f16": 4e-3}


@pytest.fixture(scope="module", params=["tiny16", "tiny32"])
def case(request):
    return golden_models(request.param, device="cuda")


@pytest.mark.parametrize("prec", ["fp32", "tf32x3", "tf32", "f16"])
def test_forward_matches_reference_fixture(case, prec):
    g, cfg, teacher, student = case
    set_precision(prec, "forward")
    try:
        x = torch.from_numpy(g["fwd_x"]).cuda()
        for tval in (0, cfg.timesteps - 1):
            t = torch.full((3,), tval, dtype=torch.long, device="cuda")
            for name, model, cond in ((f"fwd_t{tval}_none", teacher, None),
                                      (f"fwd_t{tval}_cond1", teacher, torch.ones(3, 1, device="cuda")),
                                      (f"fwd_t{tval}_cond0", teacher, torch.zeros(3, 1, device="cuda")),
                                      (f"fwd_student_t{tval}_cond1", student, torch.ones(3, 1, device="cuda"))):
                out = model(x, t, cond)
                assert out.shape == x.shape and out.device.type == "cuda"
                assert_close(out.cpu().numpy(), g[name], 0.0, FWD_TOL[prec], f"{name} [{prec}]")
        assert umma_error_flag() == 0
    finally:
        set_precision("tf32x3", "forward")


def test_time_bias_table_matches_oracle(case):
    """per-(t, variant, block) relu(time_mlp(temb)) table (models.py:15-39,66-67,175-185)."""
    g, cfg, teacher, _ = case
    sd = cpu_sd(teacher)
    eng = UNetEngine.for_model(teacher, cfg.image_size, cfg.timesteps, "fp32")
    for t in (0, 1, cfg.timesteps - 1):
        tt = torch.tensor([t])
        for variant, cond in ((_lib.VAR_NONE, None), (_lib.VAR_COND0, torch.zeros(1, 1)), (_lib.VAR_COND1, torch.ones(1, 1))):
            temb = ounet.time_embedding(sd, tt, cond)
            for b, name in enumerate(ounet.BLOCKS):
                want = ounet.block_time_bias(sd, name, temb)[0].numpy()
                got = eng.time_bias(t, variant, b)
                np.testing.assert_allclose(got, want, rtol=2e-5, atol=2e-6, err_msg=f"t={t} v={variant} {name}")


@pytest.mark.parametrize("sf,C,H", [(1.0, 1, 16), (0.5, 1, 16), (0.3, 3, 32), (1.0, 3, 32)])
@pytest.mark.parametrize("prec", ["fp32", "tf32x3", "tf32", "f16"])
def test_forward_matches_oracle_real_widths(sf, C, H, prec):
    """teacher / student widths of the BASELINE configs, mixed conditioning variants in one batch."""
    cfg = Cfg(C, H, 50)
    model = make_model(cfg, sf, 7, device="cuda")
    sd = cpu_sd(model)
    torch.manual_seed(3)
    B = 5
    x = torch.randn(B, C, H, H)
    eng = UNetEngine.for_model(model, H, 50, prec)
    variants = torch.tensor([0, 1, 2, 2, 0], dtype=torch.int32)
    for t in (49, 17):
        got = eng.forward(x.cuda(), t, variants.cuda()).cpu().numpy()
        tt = torch.full((1,), t, dtype=torch.long)
        for r in range(B):
            cond = None if variants[r] == 0 else torch.full((1, 1), float(variants[r] - 1))
            want = ounet.unet_forward(sd, x[r:r + 1], tt, cond).numpy()
            assert_close(got[r:r + 1], want, 0.0, FWD_TOL[prec], f"row {r} t={t} [{prec}]")
    assert umma_error_flag() == 0


@pytest.mark.parametrize("prec", ["tf32", "f16"])
@pytest.mark.parametrize("sf", [1.0, 0.5])
def test_forward_bench_sized_batch(sf, prec):
    """A batch large enough for the persistent / CTA-pair forms of every kernel (160 rows: 320 enc1 tiles, 80+ conv
    tiles at the 8x8 level; multiple tiles per CTA): sampled rows against the oracle, and the whole batch against the
    same rows pushed through in small batches (other launch shapes of the same kernels)."""
    cfg = Cfg(1, 16, 50)
    model = make_model(cfg, sf, 11, device="cuda")
    sd = cpu_sd(model)
    torch.manual_seed(5)
    R = 160
    x = torch.randn(R, 1, 16, 16)
    variants = (torch.arange(R) % 3).to(torch.int32)
    eng = UNetEngine.for_model(model, 16, 50, prec)
    got = eng.forward(x.cuda(), 23, variants.cuda()).cpu().numpy()
    tt = torch.full((1,), 23, dtype=torch.long)
    for r in (0, 1, 77, 158, 159):
        cond = None if variants[r] == 0 else torch.full((1, 1), float(variants[r] - 1))
        want = ounet.unet_forward(sd, x[r:r + 1], tt, cond).numpy()
        assert_close(got[r:r + 1], want, 0.0, FWD_TOL[prec], f"row {r} [{prec}]")
    small = np.concatenate([eng.forward(x[i:i + 8].cuda(), 23, variants[i:i + 8].cuda()).cpu().numpy() for i in range(0, R, 8)])
    # (fp16: the halo form of the 8x8-level convs sums its K blocks chunk-major, the im2col form the small batches take
    # tap-major: the fp32 accumulators differ in their last bits and an output may round to the neighbouring fp16 value)
    assert_close(got, small, 0.0, 1e-5 if prec == "tf32" else 1.5e-3, f"160-row batch vs 8-row batches [{prec}]")
    assert umma_error_flag() == 0


@pytest.mark.parametrize("C,H", [(1, 16), (3, 32)])
def test_forward_f16_unfused_first_block(C, H):
    """fp16 mode without the fused enc1 kernel (what first blocks wider than 128 channels take): k_conv_first writing
    fp16, the generic conv2 with the recomputed 1x1 residual and the pool tail (16x16) or k_pool2_h (32x32).  The supported
    models all take the fused kernel, so the plan is built through the test hook with options bit 0."""
    from test_gpu_layers import CONV_RESX, NO_ENC1, describe
    cfg = Cfg(C, H, 50)
    model = make_model(cfg, 0.3, 13, device="cuda")
    sd = cpu_sd(model)
    torch.manual_seed(4)
    x = torch.randn(4, C, H, H)
    variants = torch.tensor([0, 1, 2, 1], dtype=torch.int32)
    eng = UNetEngine.for_model(model, H, 50, "f16")
    ws = torch.empty(eng.workspace_bytes(4), dtype=torch.uint8, device="cuda")
    _, bufs, launches = describe(eng, 4, ws, NO_ENC1)
    assert launches[0]["kind"] == "FIRST" and [t["type"] for t in launches[0]["tensors"] if t["dir"] == "out"] == ["f16"]
    assert any(L["kind"] == "CONV_UMMA" and L["flags"] & CONV_RESX for L in launches)
    assert not any(L["kind"] in ("ENC1", "ENC1H") for L in launches)
    xd, vd = x.cuda(), variants.cuda()
    _lib.check(eng.lib.dtraj_test_plan_run(eng.handle, _lib.ptr(xd), 4, 31, _lib.ptr(vd), 0, _lib.ptr(ws), ws.numel(), NO_ENC1,
                                           0, len(launches), _lib.stream_ptr()))
    torch.cuda.synchronize()
    off = bufs["elow"]["off"]
    elow = ws[off:off + 4 * (H // 2) ** 2 * C * 4].view(torch.float32).view(4, H // 2, H // 2, C)
    # (eps = bilinear x2 of the half-resolution eps, k_eps_out's job in the product, here in f64)
    got = torch.nn.functional.interpolate(elow.permute(0, 3, 1, 2).double(), scale_factor=2, mode="bilinear",
                                          align_corners=True).cpu().numpy()
    tt = torch.full((1,), 31, dtype=torch.long)
    for r in range(4):
        cond = None if variants[r] == 0 else torch.full((1, 1), float(variants[r] - 1))
        want = ounet.unet_forward(sd, x[r:r + 1], tt, cond).numpy()
        assert_close(got[r:r + 1], want, 0.0, FWD_TOL["f16"], f"row {r} unfused f16")
    assert umma_error_flag() == 0


@pytest.mark.parametrize("prec", ["fp32", "tf32x3", "tf32", "f16"])
@pytest.mark.parametrize("sf,C,H,R", [(1.0, 1, 16, 37), (0.5, 1, 16, 5), (0.2, 3, 32, 3)])
def test_forward_stays_inside_its_workspace(sf, C, H, R, prec):
    """Guard bands around the caller-owned workspace and the eps output: a forward (ragged row counts: partial tiles,
    padded pair tiles) must not write a byte outside dtraj_unet_workspace_bytes / the eps tensor."""
    import ctypes as Ct
    cfg = Cfg(C, H, 8)
    model = make_model(cfg, sf, 17, device="cuda")
    eng = UNetEngine.for_model(model, H, 8, prec)
    lib = _lib.load()
    need = eng.workspace_bytes(R)
    guard = 1 << 20
    ws = torch.full((guard + need + guard,), 0xAB, dtype=torch.uint8, device="cuda")
    base = ws.data_ptr() + guard
    assert base % 256 == 0
    x = torch.randn(R, C, H, H, device="cuda")
    out = torch.full((R + 2, C, H, H), 7.0, device="cuda")           # rows 0 and R + 1 are guards
    variants = (torch.arange(R, device="cuda") % 3).to(torch.int32)
    _lib.check(lib.dtraj_unet_forward(eng.handle, _lib.ptr(x), R, 3, _lib.ptr(variants), Ct.c_void_p(out[1:].data_ptr()),
                                      Ct.c_void_p(base), need, _lib.stream_ptr()))
    torch.cuda.synchronize()
    assert bool((ws[:guard] == 0xAB).all()) and bool((ws[guard + need:] == 0xAB).all()), "wrote outside the workspace"
    assert bool((out[0] == 7.0).all()) and bool((out[R + 1] == 7.0).all()), "wrote outside the eps tensor"
    assert torch.isfinite(out[1:R + 1]).all()
    ref = eng.forward(x, 3, variants)
    assert torch.equal(out[1:R + 1], ref)
    assert umma_error_flag() == 0


def test_training_mode_and_bad_input_fail_loudly():
    from distillation_trajectories_b200 import DtrajError
    cfg = Cfg(1, 16, 4)
    m = make_model(cfg, 0.05, 1, device="cuda")
    m.train()
    with pytest.raises(DtrajError):
        m(torch.zeros(1, 1, 16, 16, device="cuda"), torch.tensor([0], device="cuda"))
    m.eval()
    # mixed timesteps in one batch are served by the per-row form and equal the rows run one at a time
    xm = torch.randn(2, 1, 16, 16, device="cuda")
    both = m(xm, torch.tensor([0, 3], device="cuda"))
    one = torch.cat([m(xm[:1], torch.tensor([0], device="cuda")), m(xm[1:], torch.tensor([3], device="cuda"))])
    assert torch.allclose(both, one, rtol=0, atol=1e-6 * float(one.abs().max()))
    with pytest.raises(DtrajError):
        m(xm, torch.tensor([0, -1], device="cuda"))                                           # negative timestep
    eng = UNetEngine.for_model(m, 16, 4, "fp32")
    with pytest.raises(DtrajError):
        eng.forward(torch.zeros(1, 1, 16, 16, device="cuda"), 9)                              # t outside the table
