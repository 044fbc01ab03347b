"""Whole-scene prediction on the GPU (csrc/scene.cu, nirgan_b200/scene.py): the cut against torch slicing, the blend
against an fp64 reference, and predict_scene end to end against per-tile model calls."""
import numpy as np
import pytest
import torch

import nirgan_b200  # noqa: F401
from nirgan_b200 import _lib as L
from nirgan_b200 import scene as S
from scene_ref import blend_reference

pytestmark = pytest.mark.gpu


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _cut(scene_dev, dtype, row0, origins, T):
    C, rows, W = scene_dev.shape
    org = torch.tensor(origins, dtype=torch.int32, device="cuda")
    dst = torch.full((len(origins), C, T, T), float("nan"), device="cuda")
    raw = scene_dev.view(torch.int16) if dtype == L.U16 else scene_dev
    L.call("ng_scene_tiles", raw.data_ptr(), dtype, C, rows, W, row0, org.data_ptr(), len(origins), T, 10000.0,
           dst.data_ptr(), _stream())
    return dst


@pytest.mark.parametrize("kind", ["f32", "u16"])
@pytest.mark.parametrize("T", [32, 30])
def test_scene_tiles_matches_torch_slicing(kind, T):
    g = torch.Generator().manual_seed(T)
    C, H, W, row0, rows = 3, 77, 91, 5, 61                   # odd scene; rows [5, 66) resident
    if kind == "u16":
        dn = torch.randint(0, 65536, (C, H, W), generator=g, dtype=torch.int32)
        scene = dn.to(torch.int16).view(torch.uint16)
        ref = dn.float() / 10000                             # IEEE fp32 division on the host
        dtype = L.U16
    else:
        scene = torch.rand(C, H, W, generator=g) * 2 - 0.5
        ref = scene
        dtype = L.F32
    band = scene[:, row0:row0 + rows].contiguous()
    dev = (band.view(torch.int16).cuda().view(torch.uint16) if kind == "u16" else band.cuda())
    origins = [(row0, 0), (row0 + rows - T, W - T), (row0 + 7, 13), (row0 + 1, W - T - 1)]
    origins += [(int(row0 + torch.randint(0, rows - T + 1, (1,), generator=g)),
                 int(torch.randint(0, W - T + 1, (1,), generator=g))) for _ in range(12)]
    out = _cut(dev, dtype, row0, origins, T)
    for t, (y, x) in enumerate(origins):
        assert torch.equal(out[t].cpu(), ref[:, y:y + T, x:x + T]), (t, y, x)
    assert torch.equal(_cut(dev, dtype, row0, origins, T), out)           # repeated launch: same bits
    # a window outside the resident rows is written as NaN, not read out of bounds
    bad = _cut(dev, dtype, row0, [(row0 - 1, 0), (row0 + rows - T + 1, 0), (row0, W - T + 1)], T)
    assert bool(torch.isnan(bad).all())


def _blend(pred, ys, xs, T, ov, W, y0, y1):
    oy = torch.tensor(ys, dtype=torch.int32, device="cuda")
    ox = torch.tensor(xs, dtype=torch.int32, device="cuda")
    out = torch.full((y1 - y0, W), float("nan"), device="cuda")
    L.call("ng_scene_blend", pred.data_ptr(), oy.data_ptr(), len(ys), ox.data_ptr(), len(xs), T, ov, W, y0, y1,
           out.data_ptr(), _stream())
    return out


@pytest.mark.parametrize("H,W,T,ov", [(150, 213, 64, 16), (192, 128, 64, 0), (600, 301, 256, 32), (77, 91, 30, 29),
                                      (300, 256, 256, 255), (131, 517, 64, 40)])
def test_scene_blend_matches_fp64(H, W, T, ov):
    ys, xs = S.scene_grid(H, W, T, ov)
    g = torch.Generator(device="cuda").manual_seed(H * W + ov)
    pred = torch.rand(len(ys) * len(xs), T, T, generator=g, device="cuda") * 2 - 1
    out = _blend(pred, ys, xs, T, ov, W, 0, H)
    ref = blend_reference(pred.cpu().numpy(), ys, xs, T, ov, W, 0, H)
    assert not bool(torch.isnan(out).any())
    assert np.abs(out.cpu().numpy() - ref).max() <= 2e-6
    assert torch.equal(_blend(pred, ys, xs, T, ov, W, 0, H), out)
    if ov == 0 and H % T == 0 and W % T == 0:              # pure stitching
        st = pred.view(len(ys), len(xs), T, T).permute(0, 2, 1, 3).reshape(H, W)
        assert torch.equal(out, st)
    # a pixel covered by one tile is that tile's value exactly: the scene's top-left corner
    assert torch.equal(out[0, 0], pred[0, 0, 0])
    # sub-bands: only the tile rows meeting the band, bit-identical to the full blend
    for world in (2, 3):
        for r in range(world):
            y0, y1 = S.band_rows(H, r, world)
            k0, k1 = S.band_tile_rows(ys, T, y0, y1)
            part = _blend(pred[k0 * len(xs):k1 * len(xs)].contiguous(), ys[k0:k1], xs, T, ov, W, y0, y1)
            assert torch.equal(part, out[y0:y1]), (world, r)


def _px2px(inject):
    from nirgan_b200.config import px2px_config
    from nirgan_b200.model.pix2pix import Px2Px
    torch.manual_seed(3)
    m = Px2Px(px2px_config(inject=inject, scale_init=1.0) if inject else px2px_config()).cuda().eval()
    m.netG.configure_b200(precision="fp16", impl="tc")
    return m


def _embeds(n, seed=5):
    return torch.randn(n, 256, generator=torch.Generator().manual_seed(seed))


@pytest.mark.parametrize("inject", [False, True], ids=["plain", "inject"])
def test_predict_scene_end_to_end(inject):
    T, ov, H, W = 64, 16, 150, 213                           # pad 10: 84-row generator tiles; non-square, unaligned
    model = _px2px(inject)
    g = torch.Generator().manual_seed(11)
    dn = torch.randint(0, 10001, (3, H, W), generator=g, dtype=torch.int32)
    host_u16 = dn.to(torch.int16).view(torch.uint16)
    scene = (dn.float() / 10000).cuda()
    ys, xs = S.scene_grid(H, W, T, ov)
    n = len(ys) * len(xs)
    emb = _embeds(n) if inject else None
    kw = dict(tile=T, overlap=ov, embeds=emb)

    # every tile of the scene loop is bit-identical to model(tile[None])
    pred, _, _, (k0, k1), _, done, _ = S._scene_predictions(model, scene, batch_size=7, **kw)
    torch.cuda.current_stream().wait_event(done)
    assert (k0, k1) == (0, len(ys))
    with torch.no_grad():
        for t, (y, x) in enumerate(S.scene_tiles(H, W, T, ov)):
            one = model(scene[:, y:y + T, x:x + T][None], emb[t:t + 1].cuda() if inject else None)
            assert torch.equal(pred[t], one[0, 0]), t

    out = S.predict_scene(model, scene, batch_size=64, **kw)
    assert out.shape == (1, H, W) and out.dtype == torch.float32 and out.is_cuda
    ref = blend_reference(pred[:n].cpu().numpy(), ys, xs, T, ov, W, 0, H)
    assert np.abs(out[0].cpu().numpy() - ref).max() <= 2e-6
    for bs in (1, 7):
        assert torch.equal(S.predict_scene(model, scene, batch_size=bs, **kw), out), bs
    for world in (2, 3):
        parts = [S.predict_scene(model, scene, batch_size=7, rank=r, world=world, **kw) for r in range(world)]
        assert torch.equal(S.assemble_bands(parts), out.cpu()), world
    # uint16 digital numbers from the host (pageable: pinned staging; pinned: direct copies) = the fp32 scene
    assert torch.equal(S.predict_scene(model, host_u16, batch_size=7, **kw), out)
    assert torch.equal(S.predict_scene(model, host_u16.pin_memory(), batch_size=64, **kw), out)
    assert torch.equal(S.predict_scene(model, scene.cpu(), batch_size=7, **kw), out)


def test_predict_scene_realistic_size():
    T, ov, H = 256, 32, 2048
    model = _px2px(True)
    g = torch.Generator().manual_seed(21)
    host = torch.randint(0, 10001, (3, H, H), generator=g, dtype=torch.int32).to(torch.int16).view(torch.uint16)
    emb = _embeds(len(S.scene_tiles(H, H, T, ov)))
    out = S.predict_scene(model, host.pin_memory(), tile=T, overlap=ov, embeds=emb)
    assert out.shape == (1, H, H)
    assert bool(torch.isfinite(out).all()) and float(out.abs().max()) <= 1.0
    parts = [S.predict_scene(model, host, tile=T, overlap=ov, embeds=emb, rank=r, world=2) for r in range(2)]
    assert torch.equal(S.assemble_bands(parts), out.cpu())
