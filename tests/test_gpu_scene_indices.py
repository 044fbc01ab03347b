"""Index bands of whole-scene prediction on the GPU: ng_scene_blend_indices against ng_scene_blend /
ng_scene_blend_masked followed by ng_rs_index, bit for bit, and predict_scene(indices=...) end to end against
predict_scene(indices=()) and losses.rs_index of its NIR plane."""
import math

import pytest
import torch

import nirgan_b200  # noqa: F401
import nirgan_oracle as O
from nirgan_b200 import _lib as L
from nirgan_b200 import scene as S
from nirgan_b200.losses import rs_index
from test_cpu_scene_nodata import triangle_pixel_hole
from test_gpu_scene_nodata import _blend, _blend_masked, _compact, _ng, _px2px, _raw, _scene_with_nodata, _stream

pytestmark = pytest.mark.gpu

ALL = ("evi", "msavi", "ndvi", "gndvi", "ndwi", "savi")     # every index, not in RS_TERMS order


def same(a, b):
    """Bitwise equality with NaN equal to NaN (0/0 and MSAVI's square root of a negative are legitimate here)."""
    a, b = a.cpu(), b.cpu()
    if a.shape != b.shape:
        return False
    eq = (a == b) & (torch.signbit(a) == torch.signbit(b))
    return bool((eq | (torch.isnan(a) & torch.isnan(b))).all())


def _rgb(scene, dn_scale=10000.0):
    """R, G, B as the generator sees them: a uint16 scene divided by dn_scale with IEEE division on the host."""
    s = scene.cpu()
    s = s.view(torch.int16).to(torch.int32) & 0xFFFF if s.dtype == torch.uint16 else s
    return (s[:3].float() / dn_scale if scene.dtype == torch.uint16 else s[:3].clone()).cuda()


def _rs(rgb, nir, name):
    """losses.rs_index's prediction map (index mode) of the NIR plane `nir` (h, w) and `rgb` (3, h, w)."""
    return rs_index(rgb[None], nir[None, None], nir[None, None], name, loss_eps=False)[1][0, 0]


def _blend_indices(pred, slot, ys, xs, T, ov, W, y0, y1, scene_dev, row0, names, nodata=None, nodata_out=0.0,
                   dn_scale=10000.0, out=None):
    C, rows, _ = scene_dev.shape
    oy = torch.tensor(ys, dtype=torch.int32, device="cuda")
    ox = torch.tensor(xs, dtype=torch.int32, device="cuda")
    sl = None if slot is None else torch.tensor(slot, dtype=torch.int32, device="cuda")
    which = [S.INDEX_NAMES.index(n) + 1 for n in names]
    if out is None:
        out = torch.full((1 + len(which), y1 - y0, W), 7.0, device="cuda")
    L.call("ng_scene_blend_indices", pred.data_ptr(), None if sl is None else sl.data_ptr(), oy.data_ptr(), len(ys),
           ox.data_ptr(), len(xs), T, ov, W, y0, y1, _raw(scene_dev).data_ptr(), _ng(scene_dev), C, rows, row0,
           dn_scale, int(nodata is not None), 0.0 if nodata is None else float(nodata), float(nodata_out),
           (L.c_i32 * len(which))(*which), len(which), out.data_ptr(), _stream())
    return out


def _kernel_scene(kind, H, W, seed):
    """(scene, nodata mask) with nodata 0 (uint16) / NaN (float32); a float32 scene has negative reflectances too (MSAVI's
    radicand (2n - 1)^2 + 8R can then be negative) and pixels with R = G = B = 0 (0/0 where the NIR is 0)."""
    nodata = 0 if kind == "u16" else float("nan")
    scene, mask = _scene_with_nodata(kind, nodata, H, W, seed)
    if kind == "f32":
        valid = ~mask
        scene = torch.where(valid, scene * 1.2 - 0.2, scene)
        zero = valid & (torch.rand(H, W, generator=torch.Generator().manual_seed(seed)) < 0.02)
        scene[:, zero] = 0.0
    return scene, mask, nodata


@pytest.mark.parametrize("H,W,T,ov", [(150, 212, 64, 16), (77, 91, 30, 29), (131, 517, 64, 40), (192, 128, 64, 0)])
@pytest.mark.parametrize("kind", ["u16", "f32"])
@pytest.mark.parametrize("mode", ["plain", "slot", "mask", "compact"])
def test_blend_indices_equals_blend_then_rs_index(H, W, T, ov, kind, mode):
    """plain: slot NULL, no nodata (= ng_scene_blend); slot: a permuted buffer through its slot map, no nodata; mask:
    slot NULL with the nodata mask; compact: the compacted buffer with the mask (= ng_scene_blend_masked)."""
    ys, xs = S.scene_grid(H, W, T, ov)
    scene, mask, nodata = _kernel_scene(kind, H, W, seed=H + ov)
    dev = scene.cuda()
    valid = ~mask
    g = torch.Generator(device="cuda").manual_seed(H * W + ov)
    n = len(ys) * len(xs)
    pred = torch.rand(n, T, T, generator=g, device="cuda") * 2 - 1
    pred[pred.abs() < 0.05] = 0.0                            # NIR 0 over R = G = B = 0: 0/0
    full, compact, cslot = _compact(pred, valid, ys, xs, T)
    perm = torch.randperm(n, generator=torch.Generator().manual_seed(n))
    if mode == "plain":
        buf, slot, nd = pred, None, None
        nir = _blend(pred, ys, xs, T, ov, W, 0, H)
    elif mode == "slot":
        buf, slot, nd = pred[perm.cuda()].contiguous(), torch.argsort(perm).tolist(), None
        nir = _blend(pred, ys, xs, T, ov, W, 0, H)
    elif mode == "mask":
        buf, slot, nd = full, None, nodata
        nir = _blend_masked(pred, list(range(n)), ys, xs, T, ov, W, 0, H, dev, 0, nodata, -9999.0)
    else:
        buf, slot, nd = compact, cslot, nodata
        nir = _blend_masked(compact, cslot, ys, xs, T, ov, W, 0, H, dev, 0, nodata, -9999.0)
    out = _blend_indices(buf, slot, ys, xs, T, ov, W, 0, H, dev, 0, ALL, nd, -9999.0)
    assert same(out[0], nir)
    rgb = _rgb(scene)
    v = valid.cuda() if nd is not None else torch.ones(H, W, dtype=torch.bool, device="cuda")
    for i, name in enumerate(ALL):
        want = torch.where(v, _rs(rgb, nir, name), torch.full_like(nir, -9999.0))
        assert same(out[1 + i], want), name
    if nd is not None:
        assert bool((out[:, ~v] == -9999.0).all())
    if kind == "f32" and mode == "plain":                    # the corners are exercised
        assert bool(torch.isnan(out[1 + ALL.index("ndvi")]).any()) and bool(torch.isnan(out[1 + ALL.index("msavi")]).any())
    # one index, and a band from its own resident rows: the same planes
    one = _blend_indices(buf, slot, ys, xs, T, ov, W, 0, H, dev, 0, ("gndvi",), nd, -9999.0)
    assert same(one[0], out[0]) and same(one[1], out[1 + ALL.index("gndvi")])
    y0, y1 = S.band_rows(H, 1, 3)
    lo, hi = y0 - 3, y1 + 2
    part = _blend_indices(buf, slot, ys, xs, T, ov, W, y0, y1, dev[:, lo:hi].contiguous(), lo, ALL, nd, -9999.0)
    assert same(part, out[:, y0:y1])


def test_blend_indices_rejects_bad_arguments():
    H, W, T, ov = 77, 92, 30, 10
    ys, xs = S.scene_grid(H, W, T, ov)
    pred = torch.rand(len(ys) * len(xs), T, T, device="cuda")
    scene = torch.rand(3, H, W, device="cuda")
    oy = torch.tensor(ys, dtype=torch.int32, device="cuda")
    ox = torch.tensor(xs, dtype=torch.int32, device="cuda")
    buf = torch.zeros(7 * H * W + 4, device="cuda")

    def call(which, k=None, C=3, rows=H, row0=0, y0=0, y1=H, out=buf[:7 * H * W], sc=scene):
        k = len(which) if k is None else k
        return L.load().ng_scene_blend_indices(
            pred.data_ptr(), None, oy.data_ptr(), len(ys), ox.data_ptr(), len(xs), T, ov, W, y0, y1, sc.data_ptr(),
            L.F32, C, rows, row0, 1.0, 0, 0.0, 0.0, (L.c_i32 * max(len(which), 1))(*which), k, out.data_ptr(),
            _stream())

    assert call([1]) == 0
    assert call([1, 2, 3, 4, 5, 6]) == 0
    assert call([], k=0) != 0
    assert call([1, 2, 3, 4, 5, 6, 1], k=7) != 0
    assert call([0]) != 0 and call([7]) != 0 and call([1, -1]) != 0
    assert call([1], C=2, sc=scene[:2].contiguous()) != 0
    assert "channels" in L.last_error()
    assert call([1], rows=40, row0=10, y0=5, y1=30) != 0               # rows [5, 30) not inside [10, 50)
    assert call([1], rows=40, row0=10, y0=20, y1=60) != 0
    assert call([1], out=buf[1:]) != 0                                   # W % 4 == 0: 16-byte aligned planes
    assert "aligned" in L.last_error()
    torch.cuda.synchronize()
    assert torch.equal(buf[7 * H * W:], torch.zeros(4, device="cuda"))  # nothing past the planes is written


# ---- predict_scene(indices=...) end to end ---------------------------------------------------------------------------
def _scenes(H, W, seed):
    """(dn int32, host uint16, device uint16, host float32 = dn / 10000): the same R, G, B in both types."""
    dn = torch.randint(0, 10001, (3, H, W), generator=torch.Generator().manual_seed(seed), dtype=torch.int32)
    dn[:, 5:9, 20:30] = 0                                    # R = G = B = 0
    host = dn.to(torch.int16).view(torch.uint16)
    return dn, host, host.view(torch.int16).cuda().view(torch.uint16), dn.float() / 10000


@pytest.mark.parametrize("H,W", [(150, 213), (130, 256)])
@pytest.mark.parametrize("inject", [False, True], ids=["plain", "inject"])
def test_predict_scene_indices_end_to_end(inject, H, W):
    T, ov = 64, 16
    model = _px2px(inject)
    dn, host_u16, dev_u16, f32 = _scenes(H, W, 21)
    n = len(S.scene_tiles(H, W, T, ov))
    emb = torch.randn(n, 256, generator=torch.Generator().manual_seed(5)) if inject else None
    kw = dict(tile=T, overlap=ov, embeds=emb, batch_size=7)
    rgb = f32.cuda()
    plain = S.predict_scene(model, dev_u16, **kw)
    ref = None
    for scene in (dev_u16, host_u16, f32.cuda(), f32):
        out = S.predict_scene(model, scene, indices=ALL, **kw)
        assert out.shape == (1 + len(ALL), H, W) and out.dtype == torch.float32 and out.is_cuda
        assert torch.equal(out[0], plain[0])
        if ref is None:
            ref = torch.stack([plain[0]] + [_rs(rgb, plain[0], name) for name in ALL])
        assert same(out, ref)
        assert torch.equal(S.predict_scene(model, scene, **kw), plain)          # indices=() unchanged

    # the fp64 oracle on the same inputs, where no denominator (or MSAVI radicand) is near zero
    n64 = ref[0].double().cpu()[None, None]
    rgb64 = rgb.double().cpu()[None]
    R, G = rgb64[0, 0], rgb64[0, 1]
    nn = n64[0, 0]
    ndvi64 = (nn - R) / (nn + R)
    dens = {"ndvi": [nn + R], "ndwi": [nn + G], "gndvi": [nn + R, ndvi64 + G], "savi": [nn + R + 0.5],
            "msavi": [(2 * nn + 1) ** 2 - 8 * (nn - R)], "evi": [(nn + 6) * (R - 7.5)]}
    pairs = {"ndvi": O.ndvi_pair(rgb64, n64, n64, eps=0.0), "ndwi": O.ndwi_pair(rgb64, n64, n64, eps=0.0),
             "gndvi": O.gndvi_pair(rgb64, n64, n64), "savi": O.savi_pair(rgb64, n64, n64),
             "msavi": O.msavi_pair(rgb64, n64, n64), "evi": O.evi_pair(rgb64, n64, n64, loss_mode=False)}
    for i, name in enumerate(ALL):
        want = pairs[name][1][0, 0]
        good = torch.isfinite(want)
        for d in dens[name]:
            good &= d.abs() > 1e-2
        assert float(good.float().mean()) > 0.9, name
        got = ref[1 + i].double().cpu()
        err = (got - want).abs()[good]
        assert float((err / (1e-4 * want.abs()[good] + 2e-6)).max()) <= 1.0, name


def test_index_order_follows_the_caller():
    T, ov, H, W = 64, 16, 150, 213
    model = _px2px(False)
    _, host, _, _ = _scenes(H, W, 23)
    a = S.predict_scene(model, host, tile=T, overlap=ov, indices=("ndvi", "evi"))
    b = S.predict_scene(model, host, tile=T, overlap=ov, indices=["evi", "ndvi"])
    c = S.predict_scene(model, host, tile=T, overlap=ov, indices=("evi",))
    assert same(b, a[[0, 2, 1]])
    assert same(c, a[[0, 2]])


@pytest.mark.parametrize("inject", [False, True], ids=["plain", "inject"])
def test_predict_scene_indices_with_nodata(inject):
    T, ov, H, W = 64, 16, 150, 213
    model = _px2px(inject)
    nodata = torch.from_numpy(triangle_pixel_hole(H, W))
    dn = torch.randint(1, 10001, (3, H, W), generator=torch.Generator().manual_seed(11), dtype=torch.int32)
    dn[:, nodata] = 0
    host = dn.to(torch.int16).view(torch.uint16)
    dev = host.view(torch.int16).cuda().view(torch.uint16)
    f32 = dn.float() / 10000
    f32_nan = f32.clone()
    f32_nan[:, nodata] = float("nan")
    n = len(S.scene_tiles(H, W, T, ov))
    emb = torch.randn(n, 256, generator=torch.Generator().manual_seed(5)) if inject else None
    kw = dict(tile=T, overlap=ov, embeds=emb, batch_size=7, indices=ALL)
    v = ~nodata.cuda()
    unmasked = S.predict_scene(model, dev, **kw)                          # every pixel computed
    masked_nir = S.predict_scene(model, dev, tile=T, overlap=ov, embeds=emb, batch_size=7, nodata=0)
    for fill in (float("nan"), -9999.0):
        out = S.predict_scene(model, dev, nodata=0, nodata_out=fill, **kw)
        assert out.shape == (1 + len(ALL), H, W)
        assert same(out[:, v], unmasked[:, v])                           # valid pixels: the no-nodata result
        assert same(out[0], masked_nir[0].nan_to_num(fill) if not math.isnan(fill) else masked_nir[0])
        holes = out[:, ~v]
        assert bool(torch.isnan(holes).all()) if math.isnan(fill) else bool((holes == fill).all())
        for scene, nd in ((host, 0), (host.pin_memory(), 0), (f32.cuda(), 0.0), (f32, 0.0), (f32_nan, float("nan")),
                          (f32_nan.cuda(), float("nan"))):
            got = S.predict_scene(model, scene, nodata=nd, nodata_out=fill, **kw)
            if scene.dtype == torch.float32 and math.isnan(nd):
                # NaN of partly valid tiles reaches the generator as it is: compare the masking, not the values
                assert same(got[:, ~v], out[:, ~v])
            else:
                assert same(got, out)


@pytest.mark.parametrize("nodata", [None, 0], ids=["all_valid", "nodata"])
def test_index_bands_assemble_across_ranks(nodata):
    T, ov, H, W = 64, 16, 150, 213
    model = _px2px(True)
    dn, host, dev, _ = _scenes(H, W, 31)
    if nodata is not None:
        m = torch.from_numpy(triangle_pixel_hole(H, W))
        dn[:, m] = 0
        host = dn.to(torch.int16).view(torch.uint16)
        dev = host.view(torch.int16).cuda().view(torch.uint16)
    emb = torch.randn(len(S.scene_tiles(H, W, T, ov)), 256, generator=torch.Generator().manual_seed(7))
    kw = dict(tile=T, overlap=ov, embeds=emb, batch_size=7, nodata=nodata, indices=("ndwi", "msavi", "evi"))
    whole = S.predict_scene(model, dev, **kw)
    assert whole.shape == (4, H, W)
    for world in (2, 3):
        for scene in (dev, host):
            parts = [S.predict_scene(model, scene, rank=r, world=world, **kw) for r in range(world)]
            for r, (y0, y1, band) in enumerate(parts):
                assert (y0, y1) == S.band_rows(H, r, world) and band.shape == (4, y1 - y0, W)
            assert same(S.assemble_bands(parts), whole), world
            assert same(S.gather_bands(parts[0])[:, :parts[0][1]], whole[:, :parts[0][1]])
