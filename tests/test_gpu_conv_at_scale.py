"""The tcgen05 convolutions at the geometry and batch the default plans launch them with, element by element against fp64.

Every tcgen05 `ng_conv2d` (forward with fixed-point InstanceNorm statistics, data gradient) and `ng_conv2d_wgrad` launch of
the generator and PatchGAN plans runs here at plan size: the generator at 276^2 (256 + wrap pad 10) with the training and
inference slice B = 32 and at 532^2 (512 + 10 + 10) with the smallest B that gives every CTA three work items, the
PatchGAN at 256^2 with the fake + real batch 2B = 64.  Forward and data-gradient cases assert
B * VH * VW >= 3 * 128 * SMs (VH x VW: the grid the kernel tiles; a patch holds at most 128 virtual pixels), so every
CTA of the persistent kernel drains both TMEM accumulators at least once and waits on the second phase of one of them.
The fused single-channel heads (ng_head_conv) and ng_stem_conv have their own multi-CTA tests in test_gpu_conv.py.

Operands are what the plans see: post-ReLU / LeakyReLU activations, N(0, 0.02) weights (the reference's init scale),
output gradients N(0, 1) times the power of two ng_grad_scale_pow2 picks, all rounded to the 16-bit operand type first.
Outputs are NaN-poisoned and every launch runs twice and must be bit-identical.

Reference: torch fp64 on the same rounded operands -- the forward layer itself, and the autograd of the *original* layer
for the gradients (the space-to-depth PatchGAN input layer against Conv2d(4, 64, k4, s2, p1), the generator head's tap
GEMM against Conv2d(64, 1, k7), the row-merged stem against Conv2d(3, 64, k7) on the reflect-padded tile).

Bounds, with S = |x| * |w| (the same linear map applied to absolute values, fp64) and delta = C_ACC * 2^-24 * S:
  16-bit outputs : |got - ref| <= 1/2 ulp_T(|ref| + delta) + delta      (ulp_T: spacing of the output type, subnormals
                   included -- one rounding of an fp32 accumulator that is within delta of the exact value)
  fp32 dW        : |got - ref| <= delta
C_ACC = 16.  The products of 16-bit operands are exact in fp32; what remains is the fp32 accumulation in TMEM (one rounding
per K = 16 MMA step, and for the weight gradient the fixed-order sum of the split-K partials).  A sequential fp32 sum of
K terms is bounded by K * 2^-24 * S in the worst case, but the partial sums of a zero-mean-weighted (or zero-mean-
gradient) contraction stay far below S, so the realised error is a small multiple of 2^-24 * S; 16 is that multiple with
room, and it is about 65 times tighter than the 3e-3 * max|y| of test_gpu_conv.py at a typical element of a K = 2304 conv.
Each assertion message carries the observed worst |got - ref| / bound.  Measured on a B200 (1000 W power limit): the fp32
weight gradients, where the bound is accumulation error alone, reach at most 0.46 of it (the ResnetBlock's, 152k pixels of
GEMM-K: about 7.3 * 2^-24 * S); the 16-bit outputs reach 0.99 - 0.9996, which is the half-ulp output rounding of some
element out of millions, not accumulation error -- an error of 2^-10 relative in the accumulator of one work item in three
already exceeds it.

InstanceNorm statistics (the fixed-point accumulators of every normalised forward case and the (mean, rstd) that
ng_in_apply derives from them) are checked against fp64 statistics of the *stored* 16-bit output; the bound is derived
from the epilogue's arithmetic in `_stat_bounds`.
"""
import ctypes as C
import math
import zlib

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

C_ACC = 16
U32 = 2.0 ** -24                       # unit roundoff of fp32
SLOPE = 0.2                            # LeakyReLU slope of the PatchGAN
WRAP = 10                              # the wrapper's reflect pad of the generator tiles (Data.padding_amount)


# ---------------------------------------------------------------------------------------------------------------------
# the table: forward launches of the default plans, as (Cin stored, Cout stored, K, stride, pad, input halo, form, Hin, Hout)
# form: 'gather' (ordinary tcgen05 implicit GEMM), 'merged' (ConvTranspose2d(k3, s2, p1, op1) with the four output phases
# merged into GEMM-N), 's2d' (PatchGAN input layer as a 2x2 stride-1 conv over the space-to-depth input, bias + LeakyReLU
# epilogue).  A halo > 0 is a reflect halo written into the buffer; all other padding is TMA zero fill.
def gen_forward(H1):
    H2, H3 = H1 // 2, H1 // 4
    return {
        "d1": (64, 128, 3, 2, 1, 0, "gather", H1, H2),
        "d2": (128, 256, 3, 2, 1, 0, "gather", H2, H3),
        "res": (256, 256, 3, 1, 1, 1, "gather", H3, H3),
        "u1": (256, 128, 3, 2, 1, 0, "merged", H3, 2 * H3),
        "u2": (128, 64, 3, 2, 1, 0, "merged", 2 * H3, H1),
    }


def pg_forward(H):
    H1 = H // 2
    return {
        "l0": (64, 64, 2, 1, 0, 0, "s2d", H1 + 1, H1),
        "l1": (64, 128, 4, 2, 1, 0, "gather", H1, H1 // 2),
        "l2": (128, 256, 4, 2, 1, 0, "gather", H1 // 2, H1 // 4),
        "l3": (256, 512, 4, 1, 1, 0, "gather", H1 // 4, H1 // 4 - 1),
    }


G_SMALL, G_LARGE, PG = 256 + 2 * WRAP, 512 + 2 * WRAP, 256
B_GEN, B_PG = 32, 64                   # generator slice / training batch; PatchGAN fake + real batch

FWD_CASES = ([("g%d" % G_SMALL, u) for u in gen_forward(G_SMALL)] + [("g%d" % G_LARGE, u) for u in gen_forward(G_LARGE)]
             + [("pg%d" % PG, u) for u in pg_forward(PG)])


def _row(geo, unit):
    if geo.startswith("pg"):
        return pg_forward(int(geo[2:]))[unit]
    return gen_forward(int(geo[1:]))[unit]


def _sms():
    return torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count


def _need_items(B, VH, VW, what):
    """At least three 128-pixel work items per CTA of the persistent kernel."""
    need = 3 * 128 * _sms()
    assert B * VH * VW >= need, f"{what}: B * VH * VW = {B * VH * VW} < 3 * 128 * SMs = {need}"


def _fwd_batch(geo, VH, VW):
    if geo == "g%d" % G_SMALL:
        return B_GEN
    if geo.startswith("pg"):
        return B_PG
    return -(-3 * 128 * _sms() // (VH * VW))        # config 3 / 5 tiles: the smallest B with three items per CTA


# ---------------------------------------------------------------------------------------------------------------------
# operands and launches
def _seed(*key):
    return zlib.crc32(repr(key).encode()) & 0xffffff


def _gen(seed):
    return torch.Generator(device="cuda").manual_seed(seed)


def _act(shape, seed, slope, dtype):
    """Post-activation conv input: ReLU (slope 0) / LeakyReLU of N(0, 1), rounded to the operand type."""
    import helpers as Hh
    return Hh.rnd(F.leaky_relu(torch.randn(*shape, generator=_gen(seed), device="cuda"), slope), dtype)


def _weight(shape, seed, dtype):
    import helpers as Hh
    return Hh.rnd(torch.randn(*shape, generator=_gen(seed), device="cuda") * 0.02, dtype)


def _out_grad(shape, seed, dtype):
    """N(0, 1) scaled by the power of two ng_grad_scale_pow2 picks for a target max of 8, rounded to the operand type."""
    import helpers as Hh
    g = torch.randn(*shape, generator=_gen(seed), device="cuda")
    f = 2.0 ** math.floor(math.log2(8.0 / float(g.abs().max())))
    return Hh.rnd(g * f, dtype)


def _nhwc(x, dtype, halo=0):
    import helpers as Hh
    return Hh.to_actbuf(x, halo, "reflect" if halo else "zero", dtype)


def _args(x, w, Cout, K, stride, pad, Hout, dtype, form=None, sgn=1, KW=None, pad_w=None, in_pad_w=None, **kw):
    from nirgan_b200 import _lib as L
    a = L.ConvArgs()
    a.dtype, a.impl, a.form, a.sgn = dtype, L.IMPL_TC, L.FORM_GATHER if form is None else form, sgn
    a.B, a.Hin, a.Win, a.Cin, a.in_pad = x.B, x.H, x.W, x.C, x.pad
    a.in_pad_w = x.pad if in_pad_w is None else in_pad_w
    a.Cout, a.KH, a.KW, a.stride, a.pad = Cout, K, K if KW is None else KW, stride, pad
    a.pad_w = pad if pad_w is None else pad_w
    a.Hout, a.Wout = Hout, Hout
    a.epilogue, a.act, a.slope = kw.get("epilogue", L.EPI_RAW), kw.get("act", L.ACT_NONE), kw.get("slope", 0.0)
    a.x, a.w = x.t.data_ptr(), w.data_ptr()
    a.bias = kw["bias"].data_ptr() if kw.get("bias") is not None else None
    return a


def _bits(t):
    return t.view(torch.int16) if t.element_size() == 2 else t.view(torch.int32)


def _conv_twice(a, numel, tdtype, stats=False):
    """Two launches into NaN-poisoned outputs (and zeroed statistics accumulators, as the plan's memset leaves them);
    outputs and accumulators must be bit-identical.  Returns (y, acc or None)."""
    from nirgan_b200 import _lib as L
    import helpers as Hh
    runs = []
    for _ in range(2):
        y = torch.full((numel,), float("nan"), device="cuda").to(tdtype)
        a.y = y.data_ptr()
        acc = None
        if stats:
            acc = torch.full((a.B * a.Cout * 2,), 7, dtype=torch.int64, device="cuda")
            L.call("ng_memset_zero", acc.data_ptr(), acc.numel() * 8, Hh.stream())
            a.stat_acc = acc.data_ptr()
        L.call("ng_conv2d", C.byref(a), Hh.stream())
        torch.cuda.synchronize()
        runs.append((y, acc))
    assert torch.equal(_bits(runs[0][0]), _bits(runs[1][0])), "output differs between two identical launches"
    if stats:
        assert torch.equal(runs[0][1], runs[1][1]), "statistics accumulators differ between two identical launches"
    return runs[0]


def _wgrad_twice(a, numel):
    from nirgan_b200 import _lib as L
    import helpers as Hh
    need = int(L.load().ng_conv2d_wgrad_workspace_bytes(C.byref(a)))
    assert need >= 0, L.last_error()
    ws = torch.empty(max(need, 16) // 4, dtype=torch.float32, device="cuda")
    outs = []
    for _ in range(2):
        dw = torch.full((numel,), float("nan"), device="cuda")
        L.call("ng_conv2d_wgrad", C.byref(a), dw.data_ptr(), None, ws.data_ptr(), ws.numel() * 4, Hh.stream())
        torch.cuda.synchronize()
        outs.append(dw)
    assert torch.equal(_bits(outs[0]), _bits(outs[1])), "weight gradient differs between two identical launches"
    return outs[0]


def _to_nchw(y, B, H, W, Cn):
    return y.view(B, H, W, Cn).permute(0, 3, 1, 2).double()


# ---------------------------------------------------------------------------------------------------------------------
# references and bounds
def _ulp(v, dtype):
    """Spacing of the 16-bit type at magnitude v >= 0 (fp64 tensor), subnormals included."""
    from nirgan_b200 import _lib as L
    mant, emin = (10, -14) if dtype == L.F16 else (7, -126)
    _, e = torch.frexp(v.clamp_min(2.0 ** emin))
    return torch.ldexp(torch.ones_like(v), (e - 1 - mant).clamp_min(emin - mant))


def _check16(name, got, ref, S, dtype):
    assert torch.isfinite(got).all(), f"{name}: non-finite output (unwritten elements?)"
    delta = C_ACC * U32 * S
    bound = 0.5 * _ulp(ref.abs() + delta, dtype) + delta
    ratio = float(((got - ref).abs() / bound).max())
    print(f"{name}: worst |got - ref| / bound = {ratio:.4f}")
    assert ratio <= 1.0, f"{name}: worst |got - ref| / bound = {ratio:.4f} (16-bit output, c = {C_ACC})"


def _check32(name, got, ref, S):
    assert torch.isfinite(got).all(), f"{name}: non-finite weight gradient"
    ratio = float(((got - ref).abs() / (C_ACC * U32 * S)).max())
    print(f"{name}: worst |dW - ref| / bound = {ratio:.4f}")
    assert ratio <= 1.0, f"{name}: worst |dW - ref| / bound = {ratio:.4f} (fp32 weight gradient, c = {C_ACC})"


def _vjp(fn, x, w, dy, wrt):
    """fp64 autograd of the original layer: (d/dx or d/dw) <fn(x, w), dy>, and the same map on |x|, |w|, |dy| (= S)."""
    res = []
    for xx, ww, gg in ((x, w, dy), (x.abs(), w.abs(), dy.abs())):
        xx = xx.double().detach().requires_grad_(wrt == "x")
        ww = ww.double().detach().requires_grad_(wrt == "w")
        (g,) = torch.autograd.grad(fn(xx, ww), xx if wrt == "x" else ww, gg.double())
        res.append(g)
    return res


def _stat_bounds(y, T):
    """Bounds on the per-(image, channel) mean and variance carried by the fixed-point accumulators.

    The epilogue (conv_tc.cu) sums, per tile and channel, the at most 128 *stored* 16-bit values of the tile in fp32:
    eight row groups of 16 values summed sequentially, then the seven group sums added to the first.  Each value passes
    through at most 15 + 7 = 22 fp32 additions, so the tile sum is within g22 * sum|y| and the tile sum of squares
    (fmaf: the squares are exact) within g22 * sum y^2, g22 = 22u / (1 - 22u), u = 2^-24.  Each tile's sum is then
    rounded once to a multiple of 2^-24 (__float2ll_rn of sum * 2^24, the scaling exact) and its sum of squares to a
    multiple of 2^-20: at most 2^-25 and 2^-21 per tile.  An image is covered by at most T tiles, T = ng_conv_stat_slots
    (the kernel's per-image tile count; for merged phases it counts the four phases, an over-estimate), so
        |mean_acc - mean|  <= e_m = g22 * E|y| + T 2^-25 / N
        |E2_acc - E[y^2]|  <= e_q = g22 * E[y^2] + T 2^-21 / N
    and the variance, formed as E[y^2] - mean^2, inherits both plus the cancellation term:
        |var_acc - var|    <= e_v = e_q + 2 |mean| e_m + e_m^2."""
    N = y.shape[2] * y.shape[3]
    g22 = 22 * U32 / (1 - 22 * U32)
    mean = y.mean((2, 3))
    e2 = (y * y).mean((2, 3))
    var = e2 - mean * mean
    e_m = g22 * y.abs().mean((2, 3)) + T * 2.0 ** -25 / N
    e_v = g22 * e2 + T * 2.0 ** -21 / N + 2 * mean.abs() * e_m + e_m * e_m
    return mean, var, e_m, e_v


def _check_stats(name, a, y, y_stored, acc, B, H, W, Cn, dtype):
    """Accumulators against fp64 statistics of the stored output, and the (mean, rstd) one ng_in_apply call derives."""
    from nirgan_b200 import _lib as L
    import helpers as Hh
    T = int(L.load().ng_conv_stat_slots(C.byref(a)))
    assert T > 0, L.last_error()
    mean, var, e_m, e_v = _stat_bounds(y_stored, T)
    N = H * W
    s = acc.view(B, Cn, 2).double()
    m_acc = s[..., 0] / 2.0 ** 24 / N
    v_acc = s[..., 1] / 2.0 ** 20 / N - m_acc * m_acc
    rm = float(((m_acc - mean).abs() / e_m).max())
    rv = float(((v_acc - var).abs() / e_v).max())
    print(f"{name}: statistics worst ratio mean {rm:.4f} var {rv:.4f}")
    assert rm <= 1.0, f"{name}: fixed-point mean, worst |got - ref| / bound = {rm:.4f}"
    assert rv <= 1.0, f"{name}: fixed-point variance, worst |got - ref| / bound = {rv:.4f}"
    # ng_in_apply: mean = (float) m (half an fp32 ulp), rstd = rsqrtf((float) var + 1e-5f): the two fp32 roundings of
    # the argument (2^-24 relative each) and rsqrtf's 2 ulp (2^-22 relative) on top of the variance bound
    mr = torch.full((B * Cn * 2,), float("nan"), device="cuda")
    o = torch.empty(B * H * W * Cn, dtype=Hh.TORCH_DT[dtype], device="cuda")
    L.call("ng_in_apply", y.data_ptr(), dtype, B, H, W, Cn, None, acc.data_ptr(), mr.data_ptr(), L.ACT_NONE, 0.0, None,
           0, None, L.INJECT_NONE, None, o.data_ptr(), 0, L.HALO_ZERO, Hh.stream())
    torch.cuda.synchronize()
    m = mr.view(B, Cn, 2).double()
    rstd = torch.rsqrt(var + 1e-5)
    bm = e_m + U32 * mean.abs()
    br = 0.5 * e_v / (var + 1e-5) + 2 * U32 + 2.0 ** -22
    rm2 = float(((m[..., 0] - mean).abs() / bm).max())
    rr2 = float(((m[..., 1] / rstd - 1).abs() / br).max())
    print(f"{name}: ng_in_apply mean_rstd_out worst ratio mean {rm2:.4f} rstd {rr2:.4f}")
    assert rm2 <= 1.0, f"{name}: ng_in_apply mean, worst |got - ref| / bound = {rm2:.4f}"
    assert rr2 <= 1.0, f"{name}: ng_in_apply rstd, worst relative error / bound = {rr2:.4f}"


# ---------------------------------------------------------------------------------------------------------------------
def test_table_matches_the_plans():
    """The forward rows above are the units the plans build (generator at both tile sizes, PatchGAN at 256^2)."""
    from nirgan_b200 import _lib as L
    from nirgan_b200.engine import EngineConfig
    from nirgan_b200.model import networks
    from nirgan_b200.runners import GeneratorRunner, PatchGANRunner
    dev = torch.device("cuda")
    cfg = EngineConfig("fp16", "tc")

    def row(g, u):
        if u.pack == "s2d":
            form = "s2d"
        elif g.merged_phases(u):
            form = "merged"
        else:
            assert u.form == L.FORM_GATHER and u.pack == 0 and u.KW is None, u.name
            form = "gather"
        return (u.x.C, u.cout, u.K, u.stride, u.pad, u.x.pad, form, u.x.H, u.Hout)

    netG = networks.define_G(3, 1, 64, "resnet_9blocks", "instance", False, "normal", 0.02).to(dev)
    rg = GeneratorRunner(netG, cfg)
    for H1 in (G_SMALL, G_LARGE):
        g = rg.build_graph(rg.engine(dev), 1, H1 - 2 * WRAP, H1 - 2 * WRAP, WRAP, False, 0, f"t{H1}", direct_head=False,
                           direct_stem=True, keep_rowmerged=True)
        units = {u.name: u for u in g.units}
        table = gen_forward(H1)
        for name in ("d1", "d2", "u1", "u2"):
            assert row(g, units[name]) == table[name], (H1, name)
            assert units[name].Wout == units[name].Hout and units[name].x.W == units[name].x.H
        res = [u for u in g.units if u.name.startswith("r")]
        assert len(res) == 18
        for u in res:
            assert row(g, u) == table["res"], (H1, u.name)
        # the reflect halo in front of every ResnetBlock conv is written by the unit before it
        prev = {g.units[i + 1].name: g.units[i] for i in range(len(g.units) - 1)}
        assert all(prev[u.name].halo_mode == L.HALO_REFLECT and prev[u.name].out_pad == 1 for u in res)
        assert sum(1 for u in g.units if u.kind == "norm" and u.direct is None) == len(table) - 1 + len(res)
    netD = networks.define_D(4, 64, "basic", 3, "instance", "normal", 0.02).to(dev)
    rd = PatchGANRunner(netD, cfg)
    g = rd.build_graph(rd.engine(dev), 1, ((0, 1),), (3, 1), 3, 1, PG, PG, "tpg")
    assert g.records["s2d"]
    units = {u.name: u for u in g.units}
    for name, r in pg_forward(PG).items():
        assert row(g, units[name]) == r, name
    assert units["l0"].kind == "biasact" and units["l0"].act == L.ACT_LRELU and units["l0"].slope == SLOPE
    assert all(units[n].kind == "norm" for n in ("l1", "l2", "l3"))
    assert units["out"].kind == "head" and g.tap_conv(units["out"])


@pytest.mark.parametrize("dt", ["f16", "bf16"])
@pytest.mark.parametrize("geo,unit", FWD_CASES, ids=[f"{g}-{u}" for g, u in FWD_CASES])
def test_forward(geo, unit, dt):
    from nirgan_b200 import _lib as L
    import helpers as Hh
    dtype = L.F16 if dt == "f16" else L.BF16
    Cin, Cout, K, s, p, halo, form, Hin, Hout = _row(geo, unit)
    VH = Hin if form == "merged" else Hout
    B = _fwd_batch(geo, VH, VH)
    name = f"{geo}-{unit}-{dt} B={B}"
    _need_items(B, VH, VH, name)
    seed = _seed(geo, unit, dt)
    if form == "s2d":
        H = Hout * 2
        rgb = Hh.rnd(torch.rand(B, 3, H, H, generator=_gen(seed), device="cuda") * 2 - 1, dtype)
        pred = Hh.rnd(torch.tanh(torch.randn(B, 1, H, H, generator=_gen(seed + 1), device="cuda")), dtype)
        w = _weight((64, 4, 4, 4), seed + 2, dtype)
        bias = torch.randn(64, generator=_gen(seed + 3), device="cuda") * 0.02
        x0 = torch.empty(B * Hin * Hin * 64, dtype=Hh.TORCH_DT[dtype], device="cuda")
        L.call("ng_prep_input_s2d", rgb.data_ptr(), 3, pred.data_ptr(), 1, B, H, H, dtype, x0.data_ptr(), Hh.stream())
        wp = torch.empty(4 * 64 * 64, dtype=Hh.TORCH_DT[dtype], device="cuda")
        L.call("ng_pack_weight_s2d", w.data_ptr(), 64, 4, 0, dtype, wp.data_ptr(), Hh.stream())
        from nirgan_b200.engine import ActBuf
        a = _args(ActBuf(x0, B, Hin, Hin, 64, 0), wp, Cout, K, s, p, Hout, dtype, epilogue=L.EPI_BIAS_ACT,
                  act=L.ACT_LRELU, slope=SLOPE, bias=bias)
        y, _ = _conv_twice(a, B * Hout * Hout * Cout, Hh.TORCH_DT[dtype])
        x = torch.cat([rgb, pred], 1).double()
        ref = F.leaky_relu(F.conv2d(x, w.double(), bias.double(), stride=2, padding=1), SLOPE)
        S = F.conv2d(x.abs(), w.double().abs(), bias.double().abs(), stride=2, padding=1)
        _check16(name, _to_nchw(y, B, Hout, Hout, Cout), ref, S, dtype)
        return
    slope = SLOPE if geo.startswith("pg") else 0.0
    x = _act((B, Cin, Hin, Hin), seed, slope, dtype)
    xb = _nhwc(x, dtype, halo)
    if form == "merged":
        w = _weight((Cin, Cout, 3, 3), seed + 1, dtype)                 # ConvTranspose2d (Cin, Cout, kh, kw)
        wp = torch.empty(16 * Cout * Cin, dtype=Hh.TORCH_DT[dtype], device="cuda")
        L.call("ng_pack_weight_phasemerged", w.data_ptr(), Cin, Cout, dtype, wp.data_ptr(), Hh.stream())
        a = _args(xb, wp, Cout, K, s, p, Hout, dtype, form=L.FORM_PHASED_MERGED)
        conv = lambda xx, ww: F.conv_transpose2d(xx, ww, stride=2, padding=1, output_padding=1)   # noqa: E731
    else:
        w = _weight((Cout, Cin, K, K), seed + 1, dtype)
        wp = Hh.pack_weight(w, 0, Cout, Cin, dtype)
        a = _args(xb, wp, Cout, K, s, p, Hout, dtype)
        conv = lambda xx, ww: F.conv2d(F.pad(xx, (halo,) * 4, mode="reflect") if halo else xx, ww,  # noqa: E731
                                       stride=s, padding=p - halo)
    y, acc = _conv_twice(a, B * Hout * Hout * Cout, Hh.TORCH_DT[dtype], stats=True)
    del xb, wp
    ref = conv(x.double(), w.double())
    S = conv(x.double().abs(), w.double().abs())
    del x
    got = _to_nchw(y, B, Hout, Hout, Cout)
    _check16(name, got, ref, S, dtype)
    del ref, S
    _check_stats(name, a, y, got, acc, B, Hout, Hout, Cout, dtype)


# ---------------------------------------------------------------------------------------------------------------------
# data gradients (fp16, as in the fp16 training step), restated by the rules of UnitGraph.compile_backward:
#   stride-1 conv         -> flipped-tap full correlation of dY (GATHER, sgn = -1); a reflect-haloed input gets the gradient
#                            of the whole haloed buffer (pad 0), a zero-padded one pad = the conv's pad
#   stride-2 conv         -> phased transposed conv of dY (PHASED); merged phases where the conv has 64 input channels (d1)
#   ConvTranspose2d(s2)   -> stride-2 conv of dY (GATHER)
#   generator head        -> 1x1 conv over the 64 stored taps of dz (ng_tap_scatter's layout) at the haloed 282^2 grid
#   PatchGAN input layer  -> flipped 2x2 conv over the space-to-depth grid, then ng_grad_to_nchw(s2d = 1)
# Each case: (VH, the original layer fn(x, w), its input shape, w shape, dY NCHW shape, the launch's
# (Cout stored, K, stride, pad, sgn, form, Hout), weight packing).  The packing names: ('n1', n_pad, k_pad) =
# ng_pack_weight n_axis 1; ('n0', ...) n_axis 0; 'phasemerged'; 's2d_T'; 'taps_T'.
def _conv(stride=1, padding=0):
    return lambda x, w: F.conv2d(x, w, stride=stride, padding=padding)


def _convT(x, w):
    return F.conv_transpose2d(x, w, stride=2, padding=1, output_padding=1)


def _dgrad_cases():
    H1, H2, H3, B, P = G_SMALL, G_SMALL // 2, G_SMALL // 4, B_GEN, PG
    R0, R1, R2, R3 = P // 2, P // 4, P // 8, P // 8 - 1
    return {
        "g-res": (B, _conv(), (256, H3 + 2), (256, 256, 3), (256, H3), (256, 3, 1, 0, -1, "gather", H3 + 2), ("n1", 256, 256)),
        "g-d2": (B, _conv(2, 1), (128, H2), (256, 128, 3), (256, H3), (128, 3, 2, 1, 1, "phased", H2), ("n1", 128, 256)),
        "g-d1": (B, _conv(2, 1), (64, H1), (128, 64, 3), (128, H2), (64, 3, 2, 1, 1, "merged", H1), "phasemerged"),
        "g-u1": (B, _convT, (256, H3), (256, 128, 3), (128, H2), (256, 3, 2, 1, 1, "gather", H3), ("n0", 256, 128)),
        "g-u2": (B, _convT, (128, H2), (128, 64, 3), (64, H1), (128, 3, 2, 1, 1, "gather", H2), ("n0", 128, 64)),
        "g-head": (B, _conv(), (64, H1 + 6), (1, 64, 7), (1, H1), (64, 1, 1, 0, 1, "gather", H1 + 6), "taps_T"),
        "pg-out": (B_PG, _conv(1, 1), (512, R3), (1, 512, 4), (1, R3 - 1), (512, 4, 1, 1, -1, "gather", R3), ("n1", 512, 16)),
        "pg-l3": (B_PG, _conv(1, 1), (256, R2), (512, 256, 4), (512, R3), (256, 4, 1, 1, -1, "gather", R2), ("n1", 256, 512)),
        "pg-l2": (B_PG, _conv(2, 1), (128, R1), (256, 128, 4), (256, R2), (128, 4, 2, 1, 1, "phased", R1), ("n1", 128, 256)),
        "pg-l1": (B_PG, _conv(2, 1), (64, R0), (128, 64, 4), (128, R1), (64, 4, 2, 1, 1, "phased", R0), ("n1", 64, 128)),
        "pg-l0": (B_PG, _conv(2, 1), (4, P), (64, 4, 4), (64, R0), (64, 2, 1, 0, -1, "gather", R0 + 1), "s2d_T"),
    }


DGRAD = list(_dgrad_cases())


def _pack(w, how, dtype):
    from nirgan_b200 import _lib as L
    import helpers as Hh
    d0, d1 = w.shape[:2]
    if how == "phasemerged":               # the Conv2d weight (Cout, Cin, 3, 3) read as a ConvTranspose2d (in, out, 3, 3)
        dst = torch.empty(16 * d0 * d1, dtype=Hh.TORCH_DT[dtype], device="cuda")
        L.call("ng_pack_weight_phasemerged", w.data_ptr(), d0, d1, dtype, dst.data_ptr(), Hh.stream())
        return dst
    if how == "s2d_T":
        dst = torch.empty(4 * d0 * 64, dtype=Hh.TORCH_DT[dtype], device="cuda")
        L.call("ng_pack_weight_s2d", w.data_ptr(), d0, d1, 1, dtype, dst.data_ptr(), Hh.stream())
        return dst
    if how == "taps_T":                    # (1, C, 7, 7) is a [C][49] matrix: n = channel, k = tap padded to 64
        return Hh.pack_weight(w.reshape(d1, -1, 1, 1), 0, d1, 64, dtype)
    return Hh.pack_weight(w, 1 if how[0] == "n1" else 0, how[1], how[2], dtype)


def _head_dz(g, dtype):
    """dz[n][yy][xx][kh*7 + kw] = g[n][yy - kh][xx - kw] (zero outside, taps 49..63 zero): ng_tap_scatter's layout."""
    import helpers as Hh
    taps = [F.pad(g[:, 0], (kw, 6 - kw, kh, 6 - kh)) for kh in range(7) for kw in range(7)]
    taps += [torch.zeros_like(taps[0])] * 15
    return torch.stack(taps, -1).to(Hh.TORCH_DT[dtype]).reshape(-1)


def _head_grad(B, H, seed, dtype):
    """Gradient of the head's fp32 output: zero outside the wrapper's crop window, as ng_tap_scatter leaves it."""
    g = _out_grad((B, 1, H, H), seed, dtype)
    g[..., :WRAP, :] = 0
    g[..., H - WRAP:, :] = 0
    g[..., :, :WRAP] = 0
    g[..., :, H - WRAP:] = 0
    return g


@pytest.mark.parametrize("case", DGRAD)
def test_data_gradient(case):
    from nirgan_b200 import _lib as L
    from nirgan_b200.engine import ActBuf
    import helpers as Hh
    dtype = L.F16
    B, fn, (ci, hi), wshape, (cd, hd), (Cout, K, s, p, sgn, form, Hout), how = _dgrad_cases()[case]
    VH = Hout // 2 if form == "phased" else (hd if form == "merged" else Hout)
    name = f"dgrad-{case} B={B}"
    _need_items(B, VH, VH, name)
    seed = _seed("dgrad", case)
    w = _weight(wshape + (wshape[-1],), seed, dtype)
    if case == "g-head":
        dy = _head_grad(B, hd, seed + 1, dtype)
        dyb = ActBuf(_head_dz(dy, dtype), B, hi, hi, 64, 0)
    elif case == "pg-out":
        dy = _out_grad((B, 1, hd, hd), seed + 1, dtype)
        dyb = Hh.to_actbuf(dy, 0, "zero", dtype, c_pad=16)          # ng_head_bwd_prep: channel 0 of 16 stored
    else:
        dy = _out_grad((B, cd, hd, hd), seed + 1, dtype)
        dyb = _nhwc(dy, dtype)
    frm = {"gather": L.FORM_GATHER, "phased": L.FORM_PHASED, "merged": L.FORM_PHASED_MERGED}[form]
    a = _args(dyb, _pack(w, how, dtype), Cout, K, s, p, Hout, dtype, form=frm, sgn=sgn)
    y, _ = _conv_twice(a, B * Hout * Hout * Cout, torch.float16)
    del dyb
    if case == "pg-l0":
        got = torch.full((B, 4, hi, hi), float("nan"), device="cuda")
        L.call("ng_grad_to_nchw", y.data_ptr(), dtype, B, hi, hi, 16, 0, 4, 1, 1.0, None, got.data_ptr(), Hh.stream())
        torch.cuda.synchronize()
        got = got.double()
    else:
        got = _to_nchw(y, B, Hout, Hout, Cout)
    del y
    ref, S = _vjp(fn, torch.zeros(B, ci, hi, hi, device="cuda"), w, dy, "x")
    _check16(name, got, ref, S, dtype)


# ---------------------------------------------------------------------------------------------------------------------
# weight gradients (fp16 operands, fp32 packed result) and the unpack each plan unit exports with
def _wgrad_cases():
    H1, H2, H3, P = G_SMALL, G_SMALL // 2, G_SMALL // 4, PG
    R0, R1, R2, R3 = P // 2, P // 4, P // 8, P // 8 - 1
    # (B, fn, x (C, H), halo, w shape, dY (C stored, H), launch (Cout, K, stride, pad, form), unpack (n_axis, n_pad, k_pad))
    return {
        "g-stem": (B_GEN, _conv(), None, None, (64, 3, 7), (64, H1), None, "rowmerged"),
        "g-d1": (B_GEN, _conv(2, 1), (64, H1), 0, (128, 64, 3), (128, H2), (128, 3, 2, 1, "gather"), (0, 128, 64)),
        "g-d2": (B_GEN, _conv(2, 1), (128, H2), 0, (256, 128, 3), (256, H3), (256, 3, 2, 1, "gather"), (0, 256, 128)),
        "g-res": (B_GEN, _conv(), (256, H3), 1, (256, 256, 3), (256, H3), (256, 3, 1, 1, "gather"), (0, 256, 256)),
        "g-u1": (B_GEN, _convT, (256, H3), 0, (256, 128, 3), (128, H2), (128, 3, 2, 1, "phased"), (1, 128, 256)),
        "g-u2": (B_GEN, _convT, (128, H2), 0, (128, 64, 3), (64, H1), (64, 3, 2, 1, "phased"), (1, 64, 128)),
        "g-head": (B_GEN, _conv(), (64, H1), 3, (1, 64, 7), (1, H1), None, "taps"),
        "pg-l0": (B_PG, _conv(2, 1), None, None, (64, 4, 4), (64, R0), None, "s2d"),
        "pg-l1": (B_PG, _conv(2, 1), (64, R0), 0, (128, 64, 4), (128, R1), (128, 4, 2, 1, "gather"), (0, 128, 64)),
        "pg-l2": (B_PG, _conv(2, 1), (128, R1), 0, (256, 128, 4), (256, R2), (256, 4, 2, 1, "gather"), (0, 256, 128)),
        "pg-l3": (B_PG, _conv(1, 1), (256, R2), 0, (512, 256, 4), (512, R3), (512, 4, 1, 1, "gather"), (0, 512, 256)),
        "pg-out": (B_PG, _conv(1, 1), (512, R3), 0, (1, 512, 4), (1, R3 - 1), (16, 4, 1, 1, "head"), (0, 16, 512)),
    }


WGRAD = list(_wgrad_cases())


@pytest.mark.parametrize("case", WGRAD)
def test_weight_gradient(case):
    from nirgan_b200 import _lib as L
    from nirgan_b200.engine import ActBuf
    import helpers as Hh
    dtype = L.F16
    B, fn, xs, halo, wshape, (cd, hd), launch, unpack = _wgrad_cases()[case]
    name = f"wgrad-{case} B={B}"
    seed = _seed("wgrad", case)
    wfull = wshape + (wshape[-1],)
    dst = torch.full(wfull, float("nan"), device="cuda")
    T16 = Hh.TORCH_DT[dtype]
    if case == "g-stem":
        # row-merged stem: ng_prep_stem writes [B][H1 + 6][W1][kw * 8 + c]; a 7x1 conv over 64 merged channels
        H = hd - 2 * WRAP
        src = Hh.rnd(torch.rand(B, 3, H, H, generator=_gen(seed), device="cuda") * 2 - 1, dtype)
        x0 = torch.empty(B * (hd + 6) * hd * 64, dtype=T16, device="cuda")
        L.call("ng_prep_stem", src.data_ptr(), 3, B, H, H, WRAP, 3, 7, dtype, x0.data_ptr(), Hh.stream())
        dy = _out_grad((B, cd, hd, hd), seed + 1, dtype)
        dyt = _nhwc(dy, dtype).t
        a = _args(ActBuf(x0, B, hd, hd, 64, 3), dyt, 64, 7, 1, 3, hd, dtype, KW=1, pad_w=0, in_pad_w=0)
        numel = 7 * 64 * 64
        xref = F.pad(F.pad(src, (WRAP,) * 4, mode="reflect"), (3,) * 4, mode="reflect")
    elif case == "pg-l0":
        H = 2 * hd
        rgb = Hh.rnd(torch.rand(B, 3, H, H, generator=_gen(seed), device="cuda") * 2 - 1, dtype)
        pred = Hh.rnd(torch.tanh(torch.randn(B, 1, H, H, generator=_gen(seed + 2), device="cuda")), dtype)
        x0 = torch.empty(B * (hd + 1) ** 2 * 64, dtype=T16, device="cuda")
        L.call("ng_prep_input_s2d", rgb.data_ptr(), 3, pred.data_ptr(), 1, B, H, H, dtype, x0.data_ptr(), Hh.stream())
        dy = _out_grad((B, cd, hd, hd), seed + 1, dtype)
        dyt = _nhwc(dy, dtype).t
        a = _args(ActBuf(x0, B, hd + 1, hd + 1, 64, 0), dyt, 64, 2, 1, 0, hd, dtype)
        numel = 4 * 64 * 64
        xref = torch.cat([rgb, pred], 1)
    elif case == "g-head":
        # tap form: dW[tap][c] = sum over the haloed 282^2 grid of dz[px][tap] * x[px][c], a 1x1 weight gradient
        x = _act((B, 64, xs[1], xs[1]), seed, 0.0, dtype)
        xb = _nhwc(x, dtype, 3)
        dy = _head_grad(B, hd, seed + 1, dtype)
        dyt = _head_dz(dy, dtype)
        Hz = xs[1] + 6
        a = _args(ActBuf(xb.t, B, Hz, Hz, 64, 0), dyt, 64, 1, 1, 0, Hz, dtype)
        numel = 64 * 64
        xref = F.pad(x, (3,) * 4, mode="reflect")
    else:
        Cout, K, s, p, form = launch
        x = _act((B, xs[0], xs[1], xs[1]), seed, SLOPE if case.startswith("pg") else 0.0, dtype)
        xb = _nhwc(x, dtype, halo)
        if form == "head":
            dy = _out_grad((B, 1, hd, hd), seed + 1, dtype)
            dyt = Hh.to_actbuf(dy, 0, "zero", dtype, c_pad=16).t            # ng_head_bwd_prep: channel 0 of 16 stored
        else:
            dy = _out_grad((B, cd, hd, hd), seed + 1, dtype)
            dyt = _nhwc(dy, dtype).t
        a = _args(xb, dyt, Cout, K, s, p, hd, dtype, form=L.FORM_PHASED if form == "phased" else None,
                  epilogue=L.EPI_HEAD if form == "head" else L.EPI_RAW)
        numel = K * K * Cout * xs[0]
        xref = F.pad(x, (halo,) * 4, mode="reflect") if halo else x
    a.y = dyt.data_ptr()
    dwp = _wgrad_twice(a, numel)
    if unpack == "rowmerged":
        L.call("ng_unpack_weight_grad_rowmerged", dwp.data_ptr(), *wfull, 1.0, None, 0.0, dst.data_ptr(), Hh.stream())
    elif unpack == "s2d":
        L.call("ng_unpack_weight_grad_s2d", dwp.data_ptr(), 64, 4, 1.0, None, 0.0, dst.data_ptr(), Hh.stream())
    elif unpack == "taps":              # packed [tap (64 stored)][channel] -> the reference layout [channel][tap]
        L.call("ng_unpack_weight_grad", dwp.data_ptr(), 64, 49, 1, 1, 1, 64, 64, 1.0, None, 0.0, dst.data_ptr(),
               Hh.stream())
    else:
        L.call("ng_unpack_weight_grad", dwp.data_ptr(), *wfull, *unpack, 1.0, None, 0.0, dst.data_ptr(), Hh.stream())
    torch.cuda.synchronize()
    ref, S = _vjp(fn, xref, torch.zeros(wfull, device="cuda"), dy, "w")
    _check32(name, dst.double(), ref, S)
