"""Nodata in whole-scene prediction on the GPU: ng_scene_tile_valid against a torch count, ng_scene_blend_masked against
ng_scene_blend over the full grid, and predict_scene(nodata=...) end to end against predict_scene(nodata=None)."""
import math

import numpy as np
import pytest
import torch

import nirgan_b200  # noqa: F401
from nirgan_b200 import _lib as L
from nirgan_b200 import scene as S
from test_cpu_scene_nodata import computed_tiles, masked_blend_reference, triangle_pixel_hole

pytestmark = pytest.mark.gpu


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _raw(scene_dev):
    return scene_dev.view(torch.int16) if scene_dev.dtype == torch.uint16 else scene_dev


def _ng(scene_dev):
    return L.U16 if scene_dev.dtype == torch.uint16 else L.F32


def _valid_counts(scene_dev, row0, origins, T, nodata):
    C, rows, W = scene_dev.shape
    org = torch.tensor(origins, dtype=torch.int32, device="cuda")
    cnt = torch.full((len(origins),), -7, dtype=torch.int32, device="cuda")
    L.call("ng_scene_tile_valid", _raw(scene_dev).data_ptr(), _ng(scene_dev), C, rows, W, row0, org.data_ptr(),
           len(origins), T, float(nodata), cnt.data_ptr(), _stream())
    return cnt.cpu()


def _torch_valid(scene, nodata):
    """(H, W) bool: not every channel equals nodata (NaN matches NaN)."""
    s = scene.float() if scene.dtype == torch.uint16 else scene
    eq = torch.isnan(s) if math.isnan(nodata) else s == nodata
    return ~eq.all(0)


def _scene_with_nodata(kind, nodata, H, W, seed):
    """(C, H, W) scene with whole-nodata pixels (a triangle, a hole, scattered pixels) and partly-nodata pixels."""
    g = torch.Generator().manual_seed(seed)
    C = 3
    mask = torch.from_numpy(triangle_pixel_hole(H, W)) | (torch.rand(H, W, generator=g) < 0.05)
    part = torch.rand(C, H, W, generator=g) < 0.3                      # some channels equal nodata: still valid
    if kind == "u16":
        dn = torch.randint(1, 10001, (C, H, W), generator=g, dtype=torch.int32)
        dn[part] = nodata
        dn[:, mask] = nodata
        return dn.to(torch.int16).view(torch.uint16), mask | part.all(0)
    s = torch.rand(C, H, W, generator=g)
    s[part] = nodata
    s[:, mask] = nodata
    if nodata == 0.0:
        s[:, mask & (torch.rand(H, W, generator=g) < 0.5)] = -0.0      # -0.0 matches 0.0
    return s, mask | part.all(0)


@pytest.mark.parametrize("kind,nodata", [("f32", float("nan")), ("f32", 0.0), ("f32", -9999.0), ("u16", 0)])
@pytest.mark.parametrize("T", [32, 30])
def test_tile_valid_counts_match_torch(kind, nodata, T):
    C, H, W, row0, rows = 3, 77, 91, 5, 61                   # odd scene; rows [5, 66) resident
    scene, mask = _scene_with_nodata(kind, nodata, H, W, seed=T)
    valid = _torch_valid(scene, nodata)
    assert torch.equal(valid, ~mask)
    band = scene[:, row0:row0 + rows].contiguous()
    dev = band.view(torch.int16).cuda().view(torch.uint16) if kind == "u16" else band.cuda()
    g = torch.Generator().manual_seed(T + 1)
    origins = [(row0, 0), (row0 + rows - T, W - T), (row0 + 7, 13), (row0 + 1, W - T - 1), (row0 + 20, 0)]
    origins += [(int(row0 + torch.randint(0, rows - T + 1, (1,), generator=g)),
                 int(torch.randint(0, W - T + 1, (1,), generator=g))) for _ in range(40)]
    got = _valid_counts(dev, row0, origins, T, nodata)
    want = torch.tensor([int(valid[y:y + T, x:x + T].sum()) for y, x in origins], dtype=torch.int32)
    assert torch.equal(got, want)
    assert int(want[0]) == 1 and int(want[4]) == 0                 # the lone valid pixel; a window inside the triangle
    assert len(set(want.tolist())) > 10
    assert torch.equal(_valid_counts(dev, row0, origins, T, nodata), got)          # repeated launch: same counts
    # windows outside the resident rows: -1, nothing read
    bad = _valid_counts(dev, row0, [(row0 - 1, 0), (row0 + rows - T + 1, 0), (row0, W - T + 1)], T, nodata)
    assert bad.tolist() == [-1, -1, -1]


def _blend(pred, ys, xs, T, ov, W, y0, y1):
    oy = torch.tensor(ys, dtype=torch.int32, device="cuda")
    ox = torch.tensor(xs, dtype=torch.int32, device="cuda")
    out = torch.full((y1 - y0, W), 7.0, device="cuda")
    L.call("ng_scene_blend", pred.data_ptr(), oy.data_ptr(), len(ys), ox.data_ptr(), len(xs), T, ov, W, y0, y1,
           out.data_ptr(), _stream())
    return out


def _blend_masked(pred, slot, ys, xs, T, ov, W, y0, y1, scene_dev, row0, nodata, nodata_out):
    C, rows, _ = scene_dev.shape
    oy = torch.tensor(ys, dtype=torch.int32, device="cuda")
    ox = torch.tensor(xs, dtype=torch.int32, device="cuda")
    sl = torch.tensor(slot, dtype=torch.int32, device="cuda")
    out = torch.full((y1 - y0, W), 7.0, device="cuda")
    L.call("ng_scene_blend_masked", pred.data_ptr(), sl.data_ptr(), oy.data_ptr(), len(ys), ox.data_ptr(), len(xs), T,
           ov, W, y0, y1, _raw(scene_dev).data_ptr(), _ng(scene_dev), C, rows, row0, float(nodata),
           float(nodata_out), out.data_ptr(), _stream())
    return out


def _compact(pred, valid, ys, xs, T):
    """(pred with skipped tiles poisoned to NaN, compacted pred, slot map) of the grid (ys, xs)."""
    keep = [bool(valid[y:y + T, x:x + T].any()) for y in ys for x in xs]
    full = pred.clone()
    full[torch.tensor([not k for k in keep], device=pred.device)] = float("nan")
    slot, rows = [], []
    for t, k in enumerate(keep):
        slot.append(len(rows) if k else -1)
        if k:
            rows.append(t)
    compact = pred[torch.tensor(rows, dtype=torch.long, device=pred.device)].contiguous() if rows else \
        torch.empty(1, T, T, device=pred.device)
    return full, compact, slot


@pytest.mark.parametrize("H,W,T,ov", [(150, 213, 64, 16), (77, 91, 30, 29), (131, 517, 64, 40), (192, 128, 64, 0)])
@pytest.mark.parametrize("kind,nodata,nodata_out", [("u16", 0, float("nan")), ("f32", float("nan"), -9999.0)])
def test_blend_masked_equals_the_full_blend_at_valid_pixels(H, W, T, ov, kind, nodata, nodata_out):
    ys, xs = S.scene_grid(H, W, T, ov)
    scene, mask = _scene_with_nodata(kind, nodata, H, W, seed=H + ov)
    dev = scene.cuda()
    valid = ~mask
    g = torch.Generator(device="cuda").manual_seed(H * W + ov)
    pred = torch.rand(len(ys) * len(xs), T, T, generator=g, device="cuda") * 2 - 1
    full, compact, slot = _compact(pred, valid, ys, xs, T)
    assert -1 in slot
    ref = _blend(full, ys, xs, T, ov, W, 0, H)
    out = _blend_masked(compact, slot, ys, xs, T, ov, W, 0, H, dev, 0, nodata, nodata_out)
    v = valid.cuda()
    assert torch.equal(out[v], ref[v])
    assert not bool(torch.isnan(out[v]).any())
    fill = out[~v]
    assert bool(torch.isnan(fill).all()) if math.isnan(nodata_out) else bool((fill == nodata_out).all())
    assert torch.equal(_blend_masked(compact, slot, ys, xs, T, ov, W, 0, H, dev, 0, nodata, nodata_out).nan_to_num(3.0),
                       out.nan_to_num(3.0))
    # sub-bands from their own resident rows and their own compacted tiles: bit-identical to the full masked blend
    for world in (2, 3):
        for r in range(world):
            y0, y1 = S.band_rows(H, r, world)
            k0, k1 = S.band_tile_rows(ys, T, y0, y1)
            lo, hi = ys[k0], ys[k1 - 1] + T                 # the rows a host scene keeps resident for this band
            _, c_band, s_band = _compact(pred[k0 * len(xs):k1 * len(xs)], valid, ys[k0:k1], xs, T)
            part = _blend_masked(c_band, s_band, ys[k0:k1], xs, T, ov, W, y0, y1, dev[:, lo:hi].contiguous(), lo,
                                 nodata, nodata_out)
            assert torch.equal(part.nan_to_num(3.0), out[y0:y1].nan_to_num(3.0)), (world, r)


# ---- predict_scene(nodata=...) end to end ----------------------------------------------------------------------------
def _px2px(inject):
    from nirgan_b200.config import px2px_config
    from nirgan_b200.model.pix2pix import Px2Px
    torch.manual_seed(3)
    m = Px2Px(px2px_config(inject=inject, scale_init=1.0) if inject else px2px_config()).cuda().eval()
    m.netG.configure_b200(precision="fp16", impl="tc")
    return m


class _Spy:
    """Wraps model.forward_async: records each call's input tiles (and embeddings)."""

    def __init__(self, model):
        self.model, self.orig, self.x, self.e = model, model.forward_async, [], []
        model.forward_async = self

    def __call__(self, x, e, ready):
        ready.synchronize()
        self.x.append(x.clone())
        self.e.append(None if e is None else e.clone())
        return self.orig(x, e, ready)

    def close(self):
        del self.model.forward_async


@pytest.mark.parametrize("inject", [False, True], ids=["plain", "inject"])
def test_predict_scene_nodata_end_to_end(inject):
    T, ov, H, W = 64, 16, 150, 213
    model = _px2px(inject)
    g = torch.Generator().manual_seed(11)
    nodata = torch.from_numpy(triangle_pixel_hole(H, W))
    dn = torch.randint(1, 10001, (3, H, W), generator=g, dtype=torch.int32)
    dn[:, nodata] = 0
    dn[0, 140, 200] = 0                                      # one channel 0: still valid
    host_u16 = dn.to(torch.int16).view(torch.uint16)
    dev_u16 = host_u16.view(torch.int16).cuda().view(torch.uint16)
    f32 = dn.float() / 10000                                # nodata pixels 0.0
    f32_nan = f32.clone()
    f32_nan[:, nodata] = float("nan")
    ys, xs = S.scene_grid(H, W, T, ov)
    tiles = S.scene_tiles(H, W, T, ov)
    n = len(tiles)
    comp = computed_tiles(~nodata.numpy(), H, W, T, ov)
    assert 0 < len(comp) < n
    emb = torch.randn(n, 256, generator=torch.Generator().manual_seed(5)) if inject else None
    kw = dict(tile=T, overlap=ov, embeds=emb)
    v = ~nodata.cuda()

    plain = S.predict_scene(model, dev_u16, batch_size=64, **kw)
    spy = _Spy(model)
    try:
        out = S.predict_scene(model, dev_u16, batch_size=7, nodata=0, **kw)
    finally:
        spy.close()
    # valid pixels bit-identical to nodata=None, nodata pixels nodata_out (NaN by default)
    assert torch.equal(out[0][v], plain[0][v])
    assert bool(torch.isnan(out[0][~v]).all()) and not bool(torch.isnan(out[0][v]).any())
    # the generator saw exactly the tiles with a valid pixel, in order, in ceil(n_valid / batch_size) calls
    assert len(spy.x) == math.ceil(len(comp) / 7)
    seen = torch.cat(spy.x)[:len(comp)].cpu()
    want = torch.stack([dn[:, y:y + T, x:x + T].float() / 10000 for y, x in (tiles[t] for t in comp)])
    assert torch.equal(seen, want)
    assert bool((torch.cat(spy.x)[len(comp):].cpu() == want[-1]).all())            # tail padding: last computed tile
    if inject:
        assert torch.equal(torch.cat(spy.e)[:len(comp)].cpu(), emb[comp])

    # the fp64 masked blend of the per-tile predictions
    pred, *_ , done, _ = S._scene_predictions(model, dev_u16, batch_size=64, **kw)
    torch.cuda.current_stream().wait_event(done)
    ref = masked_blend_reference(pred[:n].cpu().numpy(), ys, xs, T, ov, W, 0, H, nodata.numpy(), np.nan)
    vv = ~nodata.numpy()
    assert np.abs(out[0].cpu().numpy()[vv] - ref[vv]).max() <= 2e-6

    def same(a, b):
        return torch.equal(a.nan_to_num(3.0), b.nan_to_num(3.0))

    for bs in (1, 64):
        assert same(S.predict_scene(model, dev_u16, batch_size=bs, nodata=0, **kw), out), bs
    for world in (2, 3):
        parts = [S.predict_scene(model, dev_u16, batch_size=7, rank=r, world=world, nodata=0, **kw)
                 for r in range(world)]
        assert same(S.assemble_bands(parts), out.cpu()), world
        parts = [S.predict_scene(model, host_u16, batch_size=7, rank=r, world=world, nodata=0, **kw)
                 for r in range(world)]
        assert same(S.assemble_bands(parts), out.cpu()), world
    # host pageable, host pinned, float32 (device and host): the same result
    assert same(S.predict_scene(model, host_u16, batch_size=7, nodata=0, **kw), out)
    assert same(S.predict_scene(model, host_u16.pin_memory(), batch_size=64, nodata=0, **kw), out)
    assert same(S.predict_scene(model, f32.cuda(), batch_size=7, nodata=0.0, **kw), out)
    assert same(S.predict_scene(model, f32, batch_size=7, nodata=0.0, **kw), out)
    # NaN nodata: the same tiles are skipped and the same pixels masked; the NaN of a partly valid tile enters the
    # generator as it is, so valid pixels match nodata=None on that scene (NaN included), not the zero-filled one
    spy = _Spy(model)
    try:
        nan_out = S.predict_scene(model, f32_nan.cuda(), batch_size=7, nodata=float("nan"), **kw)
    finally:
        spy.close()
    assert len(spy.x) == math.ceil(len(comp) / 7)
    nan_plain = S.predict_scene(model, f32_nan.cuda(), batch_size=7, **kw)
    assert same(nan_out[0][v], nan_plain[0][v]) and bool(torch.isnan(nan_out[0][~v]).all())
    assert same(S.predict_scene(model, f32_nan, batch_size=64, nodata=float("nan"), **kw), nan_out)
    if inject:                                               # skipped tiles' embeddings are never read
        poisoned = emb.clone()
        poisoned[[t for t in range(n) if t not in comp]] = float("nan")
        kwp = dict(kw, embeds=poisoned)
        assert same(S.predict_scene(model, dev_u16, batch_size=7, nodata=0, **kwp), out)
        assert same(S.predict_scene(model, host_u16, batch_size=7, nodata=0, **kwp), out)
    filled = S.predict_scene(model, host_u16, batch_size=7, nodata=0, nodata_out=-9999.0, **kw)
    assert torch.equal(filled[0][v], plain[0][v]) and bool((filled[0][~v] == -9999.0).all())


@pytest.mark.parametrize("where", ["device", "host"])
def test_all_nodata_scene_makes_no_generator_call(where):
    T, ov, H, W = 64, 16, 150, 213
    model = _px2px(True)
    scene = torch.zeros(3, H, W, dtype=torch.int16).view(torch.uint16)
    if where == "device":
        scene = scene.view(torch.int16).cuda().view(torch.uint16)
    emb = torch.full((len(S.scene_tiles(H, W, T, ov)), 256), float("nan"))
    spy = _Spy(model)
    try:
        out = S.predict_scene(model, scene, tile=T, overlap=ov, embeds=emb, nodata=0, nodata_out=-9999.0)
        parts = [S.predict_scene(model, scene, tile=T, overlap=ov, embeds=emb, nodata=0, nodata_out=-9999.0, rank=r,
                                 world=2) for r in range(2)]
    finally:
        spy.close()
    assert spy.x == []
    assert out.shape == (1, H, W) and bool((out == -9999.0).all())
    assert bool((S.assemble_bands(parts) == -9999.0).all())


@pytest.mark.parametrize("inject", [False, True], ids=["plain", "inject"])
def test_nodata_on_a_scene_without_nodata_pixels_changes_nothing(inject):
    T, ov, H, W = 64, 16, 150, 213
    model = _px2px(inject)
    dn = torch.randint(1, 10001, (3, H, W), generator=torch.Generator().manual_seed(13), dtype=torch.int32)
    host = dn.to(torch.int16).view(torch.uint16)
    emb = torch.randn(len(S.scene_tiles(H, W, T, ov)), 256) if inject else None
    kw = dict(tile=T, overlap=ov, embeds=emb, batch_size=7)
    plain = S.predict_scene(model, host, **kw)
    assert torch.equal(S.predict_scene(model, host, nodata=0, **kw), plain)
    assert torch.equal(S.predict_scene(model, host.view(torch.int16).cuda().view(torch.uint16), nodata=0, **kw), plain)
    assert torch.equal(S.predict_scene(model, dn.float() / 10000, nodata=0.0, **kw), plain)
