"""GPU: every launch of the U-Net forward plan, run alone (dtraj_test_plan_run), against an f64 reference of THAT launch
computed from the GPU's own input maps as they were before it.  Errors do not compound from layer to layer, so the bounds
are those of one layer (test_gpu_conv.py's form), not the whole-forward FWD_TOL of test_gpu_forward.py, and a failure
names the launch, its tile form and the rows that are wrong.

Before each launch the maps it writes are filled with NaN: the product never clears its workspace, so a kernel must write
every element its readers use, channel pads included (they must be exactly 0)."""
import ctypes as C

import pytest
import torch
import torch.nn.functional as F

from oracle import unet as ounet
from distillation_trajectories_b200 import _lib, umma_error_flag
from distillation_trajectories_b200.engine import UNetEngine
from helpers import Cfg, cpu_sd, make_model

pytestmark = pytest.mark.gpu

CONV_RELU, CONV_TBIAS, CONV_RESID, CONV_POOL, CONV_NOSTORE, CONV_RESX, CONV_FINAL, CONV_RESACC = 1, 2, 4, 8, 16, 32, 64, 128
ACT_PLAIN, ACT_ROUND, ACT_SPLIT = 0, 1, 2
NO_ENC1 = 1                      # dtraj_test_plan_* options bit 0: k_conv_first + the generic enc1.conv2 (RESX tails)
T_STEPS = 50
U = 2.0 ** -11                   # unit roundoff of fp16 and of TF32 (round to nearest): one output rounding is <= U * |v|
F16_SUB = 2.0 ** -24             # fp16 subnormal step: the absolute part of one fp16 rounding
TB_RTOL = 2e-5                   # the fp32 time-bias table against the f64 oracle (test_gpu_forward.py::test_time_bias_table_matches_oracle)


def acc_bound(K, scale):
    """fp32 accumulation over K products (tensor core: round-toward-zero adds, ~2e-9 * K of max|ref|, test_gpu_conv.py)"""
    return (4e-6 + 4e-9 * K) * scale


# ----------------------------------------------------------------------------------------------------- plan description
def _kv(s):
    out = {}
    for tok in s.split():
        k, v = tok.split("=", 1)
        try:
            out[k] = int(v)
        except ValueError:
            out[k] = v
    return out


def parse_plan(text):
    plan, bufs, launches = {}, {}, []
    for ln in text.splitlines():
        rec, rest = ln.split(" ", 1)
        if rec == "launch":
            head, name = rest.split(" name=", 1)
            d = _kv(head)
            d["name"], d["tensors"] = name, []
            assert d["i"] == len(launches)
            launches.append(d)
        elif rec == "tensor":
            d = _kv(rest)
            launches[d["i"]]["tensors"].append(d)
        elif rec == "buf":
            d = _kv(rest)
            bufs[d["name"]] = d
        else:
            assert rec == "plan", ln
            plan = _kv(rest)
    assert plan["launches"] == len(launches)
    return plan, bufs, launches


def describe(eng, R, ws, options):
    buf = C.create_string_buffer(1 << 16)
    _lib.check(eng.lib.dtraj_test_plan_describe(eng.handle, R, _lib.ptr(ws), ws.numel(), options, buf, len(buf)))
    return parse_plan(buf.value.decode())


def features(launches, per_row):
    """What a plan exercises, in the vocabulary of REQUIRED below."""
    f = set()
    for L in launches:
        kind, fl = L["kind"], L["flags"]
        outs = {t["role"]: t for t in L["tensors"] if t["dir"] == "out"}
        f.add(kind)
        if kind == "FIRST":
            f.add("FIRST:" + outs["out"]["type"])
        if kind not in ("CONV_UMMA", "CONV_SIMT"):
            continue
        src0 = next(t for t in L["tensors"] if t["role"] == "src0")
        S, f16 = src0["S"], src0["type"] == "f16"
        if kind == "CONV_UMMA":
            form = L["form"]
            f.add(f"{form}@{S}")
            if L["pair"]:
                f.add(f"{form}@{S}+pair")
            if L["split"] > 1:
                f.add("split")
            if f16:
                f.add(f"f16 epi{L['epi']}")
            if fl & CONV_RESACC:
                f.add(f"RESACC {form}")
        if fl & CONV_POOL:
            f.add(f"POOL tail@{S}")
        if fl & CONV_FINAL and fl & CONV_NOSTORE:
            f.add("FINAL+NOSTORE tail")
        if fl & CONV_RESX:
            f.add("RESX tail")
        if per_row and fl & CONV_TBIAS:
            f.add("per-row time bias")
        if L["act"] == ACT_SPLIT:
            f.add("lo planes")
    return f


# Everything the case list must run.  A plan change that stops running one of them fails test_plan_coverage instead of
# silently testing less.
REQUIRED = {
    "ENC1H", "ENC1", "FIRST:f16", "FIRST:f32", "CONV_SIMT", "POOL", "POOL_H", "UP", "UP_H", "UP_H4", "FINAL",
    "generic@16", "generic@16+pair", "halo1@8", "halo1@8+pair", "halo2@16", "halo2@16+pair", "halo2@32",
    "halo2@32+pair", "posm@4", "posm@4+pair", "posm@2", "posm@2+pair", "split",
    "f16 epi0", "f16 epi1", "f16 epi2", "f16 epi3", "f16 epi4",
    "POOL tail@16", "POOL tail@8", "FINAL+NOSTORE tail", "RESX tail",
    "RESACC generic", "RESACC halo1", "RESACC halo2", "RESACC posm",
    "lo planes", "per-row time bias",
}


# ------------------------------------------------------------------------------------------------------------ the cases
# (C, H, sf, precision, R, options, per_row)
CASES = []
for _sf in (1.0, 0.5):                                        # the bench pair
    for _p in ("f16", "tf32"):
        CASES += [(1, 16, _sf, _p, 8, 0, 0),                  # generic tiles, split-N at the deep levels
                  (1, 16, _sf, _p, 160, 0, 0),                # CTA pairs, halo mode 1, several tiles per CTA
                  (1, 16, _sf, _p, 160, 0, 1)]                # ... with a timestep and a variant per row
    CASES.append((1, 16, _sf, "f16", 2350, 0, 0))             # 4x4 maps position-major: 19 image blocks padded to 20 for pairs,
                                                              # partial last block, stand-alone pool after enc3
CASES.append((1, 16, 0.5, "f16", 9500, 0, 0))                 # 2x2 maps position-major with CTA pairs: >= 2 * 148 / 4 = 74 image
                                                              # blocks per position (75 here, padded to 76), partial last block
for _p in ("fp32", "tf32x3"):                                 # exact modes: FIRST, CONV_SIMT, stand-alone pool / upsample / final
    CASES += [(1, 16, 0.5, _p, 8, 0, 0), (1, 16, 0.5, _p, 37, 0, 1)]
for _p in ("fp32", "tf32x3", "tf32", "f16"):                  # halo mode 2 at 16x16, half-filled fp16 K blocks (sf 0.3: 76 channels)
    CASES += [(3, 32, 1.0, _p, 40, 0, 0), (3, 32, 0.3, _p, 3, 0, 0)]
    if _p in ("tf32", "f16"):                                 # 16x16 maps with CTA pairs (>= 296 tiles of half an image)
        CASES.append((3, 32, 1.0, _p, 160, 0, 0))
for _p in ("f16", "tf32"):                                    # halo mode 2 at 32x32, 2-row generic tiles at 64x64
    CASES += [(3, 64, 1.0, _p, 24, 0, 0), (3, 64, 0.5, _p, 2, 0, 1)]
    if _p == "f16":                                           # 32x32 halo tiles with CTA pairs: 8 tiles per image, >= 296 tiles
        CASES.append((3, 64, 1.0, _p, 40, 0, 0))
    for _C, _H in ((1, 16), (3, 32), (3, 64)):                # k_conv_first + the RESX tails
        CASES.append((_C, _H, 0.3, _p, 4, NO_ENC1, 0))


def case_id(c):
    C_, H, sf, p, R, opt, pr = c
    return f"{C_}x{H}-sf{sf}-{p}-R{R}" + ("-noenc1" if opt else "") + ("-rows" if pr else "")


_MODELS = {}


def model_for(C_, H, sf):
    key = (C_, H, sf)
    if key not in _MODELS:
        _MODELS[key] = make_model(Cfg(C_, H, T_STEPS), sf, 31 + int(sf * 10) + H, device="cuda")
    return _MODELS[key]


# ------------------------------------------------------------------------------------------------------- f64 reference
def tf32_rna(w):
    """round-to-nearest, ties away, to TF32 (cvt.rna / tf32_rna_host), of an fp32 tensor"""
    u = w.contiguous().view(torch.int32).to(torch.int64) + 0x1000
    return (u & 0xFFFFE000).to(torch.int32).view(torch.float32)


def tf32_trunc(a):
    return (a.contiguous().view(torch.int32) & -8192).view(torch.float32)


class Layers:
    """Per-block reference weights, rounded exactly as pack_conv rounds them."""

    def __init__(self, model, prec):
        self.sd = {k: v.detach().double().cuda() for k, v in cpu_sd(model).items() if torch.is_floating_point(v)}
        self.prec = prec

    def _round(self, w32):
        if self.prec == "f16":
            return w32.half().double()
        if self.prec == "tf32":
            return tf32_rna(w32).double()
        return w32.double()                               # fp32; tf32x3 packs hi + lo = the fp32 value

    def folded(self, blk, which):
        """BN-folded conv (bn_fold): fp32 weights w * scale, fp32 bias"""
        sd, n = self.sd, f"{blk}.norm{which[-1]}"
        s = sd[n + ".weight"] / torch.sqrt(sd[n + ".running_var"] + 1e-5)
        shift = (sd[f"{blk}.{which}.bias"] - sd[n + ".running_mean"]) * s + sd[n + ".bias"]
        return (sd[f"{blk}.{which}.weight"] * s[:, None, None, None]).float(), shift.float().double()

    def conv(self, blk, which):
        """(weights as the packed operand, fp32 bias) of conv1 / conv2 / res of a generic block"""
        if which == "res":
            return self._round(self.sd[blk + ".residual_conv.weight"].float()), self.sd[blk + ".residual_conv.bias"]
        w, b = self.folded(blk, which)
        return self._round(w), b


def nchw(m, c):
    return m[..., :c].permute(0, 3, 1, 2).double()


def maxpool_nhwc(m):
    R, S, _, cp = m.shape
    return m.view(R, S // 2, 2, S // 2, 2, cp).amax(dim=(2, 4))


def up2(a):
    return F.interpolate(a, scale_factor=2, mode="bilinear", align_corners=True)


class Checker:
    def __init__(self, what):
        self.what = what

    def close(self, got, want, bound, label, real=None):
        """|got - want| <= bound elementwise; NCHW f64 tensors.  Reports the worst rows / channels."""
        d = (got - want).abs()
        bad = ~(d <= bound)
        if bool(bad.any()):
            idx = bad.nonzero()
            ex = (d - bound)[bad]
            w = int(ex.argmax())
            rows = sorted(set(int(r) for r in idx[:, 0].tolist()))
            chans = sorted(set(int(c) for c in idx[:, 1].tolist()))
            pytest.fail(f"{self.what} {label}: {int(bad.sum())}/{bad.numel()} outside the bound; worst at (row, c, y, x) = "
                        f"{tuple(int(v) for v in idx[w])}: got {float(got[tuple(idx[w])]):.6g} want {float(want[tuple(idx[w])]):.6g} "
                        f"bound {float(bound[tuple(idx[w])]):.3g}; rows {rows[:12]}{'...' if len(rows) > 12 else ''} "
                        f"channels {chans[:12]}{'...' if len(chans) > 12 else ''}")

    def equal(self, got, want, label):
        if not torch.equal(got, want):
            bad = (got != want) & ~(torch.isnan(got) & torch.isnan(want))
            idx = bad.nonzero()
            pytest.fail(f"{self.what} {label}: {int(bad.sum())} elements differ, first at {tuple(idx[0].tolist())}")


class PlanCase:
    def __init__(self, c, describe_only=False):
        C_, H, sf, prec, R, options, per_row = c
        self.case = c
        self.C, self.H, self.prec, self.R, self.options, self.per_row = C_, H, prec, R, options, per_row
        self.model = model_for(C_, H, sf)
        self.eng = UNetEngine.for_model(self.model, H, T_STEPS, prec)
        self.f16 = prec == "f16"
        self.ws = torch.empty(self.eng.workspace_bytes(R), dtype=torch.uint8, device="cuda")   # uninitialised, as the engine's
        self.plan, self.bufs, self.launches = describe(self.eng, R, self.ws, options)
        if describe_only:
            return
        g = torch.Generator().manual_seed(R * 7 + H + int(sf * 100))
        self.x = torch.randn(R, C_, H, H, generator=g).cuda()
        self.var = torch.randint(0, 3, (R,), generator=g, dtype=torch.int32)
        self.t = torch.randint(0, T_STEPS, (R,), generator=g) if per_row else torch.full((R,), 23, dtype=torch.int64)
        self.rv = ((self.t * 3 + self.var) if per_row else self.var).to(torch.int32).cuda()
        self.ref = Layers(self.model, prec)
        sd = {k: v.double() for k, v in cpu_sd(self.model).items() if torch.is_floating_point(v)}
        self.tb = {}                                       # block -> [R, cout] f64: relu(time_mlp(temb(t_i, cond_i)))
        for blk in ounet.BLOCKS:
            rows = torch.empty(R, sd[blk + ".time_mlp.bias"].numel(), dtype=torch.float64)
            for (tv, v) in set(zip(self.t.tolist(), self.var.tolist())):
                cond = None if v == 0 else torch.full((1, 1), float(v - 1), dtype=torch.float64)
                temb = ounet.time_embedding(sd, torch.tensor([float(tv)], dtype=torch.float64), cond)
                rows[(self.t == tv) & (self.var == v)] = ounet.block_time_bias(sd, blk, temb)[0]
            self.tb[blk] = rows.cuda()

    # --- workspace views
    def view(self, t, lo=False):
        if t["buf"] == "x":
            return self.x
        b = self.bufs[t["buf"]]
        esz = 2 if t["type"] == "f16" else 4
        n = self.R * t["S"] * t["S"] * t["cp"]
        off = b["off"] + (b["lo"] if lo else 0)
        assert off + n * esz <= b["off"] + b["bytes"], f"{t} outside buffer {b}"
        return self.ws[off:off + n * esz].view(torch.float16 if esz == 2 else torch.float32).view(self.R, t["S"], t["S"], t["cp"])

    def run(self, i):
        _lib.check(self.eng.lib.dtraj_test_plan_run(self.eng.handle, _lib.ptr(self.x), self.R, 23, _lib.ptr(self.rv), self.per_row,
                                                    _lib.ptr(self.ws), self.ws.numel(), self.options, i, i + 1, _lib.stream_ptr()))
        torch.cuda.synchronize()
        self.eng.check_errors()
        assert umma_error_flag() == 0

    def split_lo(self, L):
        return L["act"] == ACT_SPLIT

    # --- one launch
    def check_launch(self, L):
        i = L["i"]
        chk = Checker(f"[{case_id(self.case)}] launch {i} "
                      f"{L['kind']} '{L['name']}' form={L['form']} pair={L['pair']} split={L['split']} epi={L['epi']}")
        ins = {t["role"]: (t, self.view(t).clone()) for t in L["tensors"] if t["dir"] == "in"}
        outs = {t["role"]: t for t in L["tensors"] if t["dir"] == "out"}
        for t in outs.values():                            # NaN (fp16 0x7E00): a skipped element cannot pass
            self.view(t).fill_(float("nan"))
            if self.split_lo(L) and t["role"] != "elow" and self.bufs[t["buf"]]["lo"]:
                self.view(t, lo=True).fill_(float("nan"))
        self.run(i)
        got = {r: self.view(t) for r, t in outs.items()}
        for r, g in got.items():
            assert not bool(torch.isnan(g).any()), f"{chk.what}: NaN left in output '{r}' ({int(torch.isnan(g).sum())} elements)"
        kind = L["kind"]
        if kind in ("CONV_UMMA", "CONV_SIMT"):
            self.check_conv(L, ins, outs, got, chk)
        elif kind == "FIRST":
            self.check_first(L, outs, got, chk)
        elif kind in ("ENC1", "ENC1H"):
            self.check_enc1(L, outs, got, chk)
        elif kind in ("POOL", "POOL_H"):
            src = ins["src0"][1]
            chk.equal(got["out"], maxpool_nhwc(src), "max-pool")
        elif kind in ("UP", "UP_H", "UP_H4"):
            t_in, src = ins["src0"]
            a = src.permute(0, 3, 1, 2).double()
            want = up2(a)
            Hi = t_in["S"]
            # fp32 coordinates: s = fp32((Hi-1)/(2Hi-1)) * dst carries <= 2 * 2^-24 relative error, |s| < Hi, so a weight is off by
            # <= Hi * 2^-23; three fp32 lerps add <= 3 * 2^-24 of the larger corner; then one rounding of the stored value
            amax = a.abs().amax(dim=(1, 2, 3), keepdim=True)
            bound = (Hi * 2.0 ** -22 + 2.0 ** -21) * amax
            if self.f16 or L["act"] == ACT_ROUND:
                bound = bound + U * want.abs() + (F16_SUB if self.f16 else 0.0)
            chk.close(got["out"].permute(0, 3, 1, 2).double(), want, bound, "upsample")
        elif kind == "FINAL":
            t_in, y = ins["src0"]
            self.check_final(nchw(y, self.ref.sd["final.weight"].shape[1]), torch.zeros(1, device="cuda", dtype=torch.float64),
                             got["elow"], chk)
        else:
            pytest.fail(f"no reference for launch kind {kind}")
        if self.split_lo(L):                               # 3xTF32 low planes: exactly y - trunc_tf32(y) of the stored y
            for r, t in outs.items():
                if r in ("out", "res") and self.bufs[t["buf"]]["lo"]:
                    chk.equal(self.view(t, lo=True), got[r] - tf32_trunc(got[r]), f"'{r}' low plane")

    def pads_zero(self, g, c, chk, label):
        if g.shape[-1] > c:
            pad = g[..., c:]
            if not bool((pad == 0).all()):
                chk.equal(pad, torch.zeros_like(pad), f"'{label}' channel pads")

    def store_bound(self, L, want, pre_scale, K, dtype_f16):
        """accumulation + (when the map is rounded to fp16 / TF32) one output rounding"""
        b = acc_bound(K, pre_scale)
        if dtype_f16 or L["act"] == ACT_ROUND:
            b = b + U * want.abs() + (F16_SUB if dtype_f16 else 0.0)
        return b

    def check_conv(self, L, ins, outs, got, chk):
        blk, which = L["name"].split(" ")[0].split(".")
        fl = L["flags"]
        w, b = self.ref.conv(blk, which)
        cin = w.shape[1]
        two = "src1" in ins
        c0 = cin // 2 if two else cin
        a = nchw(ins["src0"][1], c0)
        if two:
            a = torch.cat([a, nchw(ins["src1"][1], cin - c0)], dim=1)
        pre = F.conv2d(a, w, b, padding=w.shape[-1] // 2)
        K = cin * w.shape[-1] * w.shape[-2]
        v = pre.relu() if fl & CONV_RELU else pre
        extra = torch.zeros_like(v[:, :, :1, :1])
        if fl & CONV_TBIAS:
            tb = self.tb[blk][:, :, None, None]
            v = v + tb
            extra = extra + TB_RTOL * tb.abs()
        cout = w.shape[0]
        if fl & CONV_RESID:
            v = v + nchw(ins["resid"][1], cout)
        if fl & CONV_RESX:                                 # enc1.residual_conv of the raw frame, fp32 weights, fp32 FMAs
            sd = self.ref.sd
            v = v + F.conv2d(self.x.double(), sd["enc1.residual_conv.weight"].float().double(), sd["enc1.residual_conv.bias"].float().double())
            K += self.C
        if fl & CONV_RESACC:
            rw, rb = self.ref.conv(blk, "res")
            r = nchw(ins["rsrc0"][1], rw.shape[1] // 2 if "rsrc1" in ins else rw.shape[1])
            if "rsrc1" in ins:
                r = torch.cat([r, nchw(ins["rsrc1"][1], rw.shape[1] // 2)], dim=1)
            v = v + F.conv2d(r, rw, rb)
            K += rw.shape[1]
        scale = torch.maximum(pre.abs().amax(), v.abs().amax())
        f16 = self.f16 and L["kind"] == "CONV_UMMA"
        bound = self.store_bound(L, v, scale, K, f16) + extra
        if "out" in got:
            g = got["out"]
            self.pads_zero(g, cout, chk, "out")
            chk.close(nchw(g, cout), v, bound, "output")
        if "pool" in got:
            p = got["pool"]
            self.pads_zero(p, cout, chk, "pool")
            if "out" in got:                               # the pool of the stored map, bit for bit
                chk.equal(p, maxpool_nhwc(got["out"]), "fused pool")
            else:                                          # max is 1-Lipschitz: the bound of the window's worst element
                chk.close(nchw(p, cout), F.max_pool2d(v, 2), F.max_pool2d(bound, 2), "fused pool (map not stored)")
        if "elow" in got:
            self.check_final(v, bound, got["elow"], chk)

    def check_final(self, y, y_bound, elow, chk):
        """final 1x1 at half resolution of y (whose values carry y_bound), fp32 sums over the padded width"""
        sd = self.ref.sd
        w = sd["final.weight"].float().double()
        b = sd["final.bias"].float().double()
        want = F.conv2d(y, w, b)
        mag = F.conv2d(y.abs(), w.abs(), b.abs())
        bound = F.conv2d(y_bound.expand_as(y), w.abs()) + acc_bound(y.shape[1], mag.amax())
        chk.close(elow.permute(0, 3, 1, 2).double(), want, bound, "final 1x1 (elow)")

    def enc1_conv1(self):
        sd = self.ref.sd
        w3, b3 = self.ref.folded("enc1", "conv1")
        x = self.x.double()
        h = F.conv2d(x, w3.double(), b3, padding=1).relu() + self.tb["enc1"][:, :, None, None]
        mag = F.conv2d(x.abs(), w3.double().abs(), b3.abs(), padding=1)
        r = F.conv2d(x, sd["enc1.residual_conv.weight"].float().double(), sd["enc1.residual_conv.bias"].float().double())
        return h, mag, r

    def check_first(self, L, outs, got, chk):
        h, mag, r = self.enc1_conv1()
        cout = h.shape[1]
        f16 = outs["out"]["type"] == "f16"
        bound = self.store_bound(L, h, mag.amax(), 9 * self.C, f16) + TB_RTOL * self.tb["enc1"][:, :, None, None].abs()
        self.pads_zero(got["out"], cout, chk, "out")
        chk.close(nchw(got["out"], cout), h, bound, "conv1 map h")
        if "res" in got:
            self.pads_zero(got["res"], cout, chk, "res")
            chk.close(nchw(got["res"], cout), r, acc_bound(self.C, r.abs().amax()), "residual 1x1 map")

    def check_enc1(self, L, outs, got, chk):
        """The fused enc1 block: p1 = maxpool(relu(conv2(h) + b2) + res1x1(x)), h = relu(conv1(x) + b3) + tb, h never stored.
        h carries its own error into conv2: one rounding to fp16 / TF32 (U |h|), the fp32 accumulation of conv1, the table, and in
        fp16 conv1 runs on the tensor cores with x and w3 rounded to fp16 (2U of conv1(|x|, |w3|)).  conv2 propagates
        |dh| through |w2|: conv2(e_h, |w2|)."""
        h, mag, r = self.enc1_conv1()
        w2, b2 = self.ref.conv("enc1", "conv2")
        cout = h.shape[1]
        e_h = U * h.abs() + acc_bound(9 * self.C, mag.amax()) + TB_RTOL * self.tb["enc1"][:, :, None, None].abs()
        if self.f16:
            e_h = e_h + 2 * U * mag
        pre = F.conv2d(h, w2, b2, padding=1)
        y = pre.relu() + r
        K = 9 * cout + self.C
        bound = self.store_bound(L, y, torch.maximum(pre.abs().amax(), y.abs().amax()), K, self.f16) + \
            F.conv2d(e_h, w2.abs(), padding=1)
        p = got["pool"]
        self.pads_zero(p, cout, chk, "pool")
        chk.close(nchw(p, cout), F.max_pool2d(y, 2), F.max_pool2d(bound, 2), "pooled enc1 output")

    def check_end(self):
        """the hook ran what the product runs: elow equals a plain forward's, and eps is the bilinear x2 of elow (k_eps_out)"""
        lib = self.eng.lib
        t_elow = {"buf": "elow", "S": self.H // 2, "cp": self.C, "type": "f32"}
        elow_hook = self.view(t_elow).clone()
        eps = torch.empty_like(self.x)
        if self.per_row:
            _lib.check(lib.dtraj_unet_forward_rows(self.eng.handle, _lib.ptr(self.x), self.R, _lib.ptr(self.rv), _lib.ptr(eps),
                                                   _lib.ptr(self.ws), self.ws.numel(), _lib.stream_ptr()))
        else:
            _lib.check(lib.dtraj_unet_forward(self.eng.handle, _lib.ptr(self.x), self.R, 23, _lib.ptr(self.rv), _lib.ptr(eps),
                                              _lib.ptr(self.ws), self.ws.numel(), _lib.stream_ptr()))
        torch.cuda.synchronize()
        self.eng.check_errors()
        elow = self.view(t_elow)
        if self.options == 0:
            assert torch.equal(elow_hook, elow), "launch-by-launch elow differs from dtraj_unet_forward's"
        e = elow.permute(0, 3, 1, 2).double()
        want = up2(e)
        bound = ((self.H // 2) * 2.0 ** -22 + 2.0 ** -21) * e.abs().amax(dim=(1, 2, 3), keepdim=True)
        Checker("k_eps_out").close(eps.double(), want, bound.expand_as(want), "eps")


@pytest.mark.parametrize("case", CASES, ids=case_id)
def test_plan_launch_by_launch(case):
    pc = PlanCase(case)
    assert pc.plan["R"] == pc.R and pc.plan["options"] == pc.options
    for L in pc.launches:
        pc.check_launch(L)
    pc.check_end()


def test_plan_coverage():
    covered = set()
    for c in CASES:
        pc = PlanCase(c, describe_only=True)
        covered |= features(pc.launches, pc.per_row)
    missing = REQUIRED - covered
    assert not missing, f"the case list no longer runs: {sorted(missing)}"


def test_plan_options_rebuild_and_bad_range():
    """the cached plan follows the options; a launch range outside the plan is refused"""
    pc = PlanCase((1, 16, 0.5, "f16", 4, 0, 0))
    kinds0 = [L["kind"] for L in pc.launches]
    _, _, l1 = describe(pc.eng, 4, pc.ws, NO_ENC1)
    _, _, l0 = describe(pc.eng, 4, pc.ws, 0)
    assert kinds0[0] == "ENC1H" and [L["kind"] for L in l0] == kinds0
    assert l1[0]["kind"] == "FIRST" and any(L["flags"] & CONV_RESX for L in l1)
    lib = pc.eng.lib
    for first, last in ((-1, 1), (2, 1), (0, len(l0) + 1)):
        assert lib.dtraj_test_plan_run(pc.eng.handle, _lib.ptr(pc.x), 4, 23, _lib.ptr(pc.rv), 0, _lib.ptr(pc.ws), pc.ws.numel(),
                                       0, first, last, _lib.stream_ptr()) == -1
