"""Index bands of whole-scene prediction (nirgan_b200/scene.py, `indices=`): argument checks, the name-to-term mapping
and plane order, and the numpy index-mode reference the GPU tests compare against, pinned to the oracle's restatement
of the reference's RemoteSensingIndices."""
import numpy as np
import pytest
import torch

import nirgan_b200  # noqa: F401
import nirgan_oracle as O
from nirgan_b200 import losses
from nirgan_b200 import scene as S


# ---- reference ---------------------------------------------------------------------------------------------------
def index_reference(name, n, R, G, B):
    """Index-mode RemoteSensingIndices (epsilon 0) of NIR n and bands R, G, B, elementwise in the arrays' dtype.  The
    epsilon is added as 0.0, as the reference does in index mode (it turns a -0 denominator into +0)."""
    with np.errstate(divide="ignore", invalid="ignore"):
        if name == "ndvi":
            return (n - R) / (n + R + 0.0)
        if name == "ndwi":
            return (n - G) / (n + G + 0.0)
        if name == "gndvi":
            return (n - G) / ((n - R) / (n + R) + G)
        if name == "savi":
            return 1.5 * (n - R) / (n + R + 0.5)
        if name == "msavi":
            return (2 * n + 1 - np.sqrt((2 * n + 1) ** 2 - 8 * (n - R))) / 2
        if name == "evi":
            return 2.5 * ((n - R) / ((n + 6) * (R - 7.5) * (B + 1) + 0.0))
    raise ValueError(name)


_ORACLE = {"ndvi": lambda rgb, n: O.ndvi_pair(rgb, n, n, eps=0.0), "ndwi": lambda rgb, n: O.ndwi_pair(rgb, n, n, eps=0.0),
           "gndvi": lambda rgb, n: O.gndvi_pair(rgb, n, n), "savi": lambda rgb, n: O.savi_pair(rgb, n, n),
           "msavi": lambda rgb, n: O.msavi_pair(rgb, n, n), "evi": lambda rgb, n: O.evi_pair(rgb, n, n, loss_mode=False)}


def _pixels(seed):
    """(rgb (1, 3, H, W), nir (1, 1, H, W)) float64 with reflectance-like values plus the corners of the formulas: 0/0,
    a negative MSAVI radicand (it needs R < 0), n = -R, n = -6."""
    g = np.random.default_rng(seed)
    rgb = g.uniform(0, 1, (1, 3, 8, 16))
    nir = g.uniform(-0.2, 1.2, (1, 1, 8, 16))
    rgb[0, :, 0, 0], nir[0, 0, 0, 0] = 0.0, 0.0              # 0/0 in NDVI, NDWI, SAVI's numerator only
    rgb[0, 0, 0, 1], nir[0, 0, 0, 1] = -0.1, 0.5             # (2n + 1)^2 - 8 (n - R) = (2n - 1)^2 + 8R < 0: NaN
    rgb[0, 0, 0, 2], nir[0, 0, 0, 2] = 0.3, -0.3             # n + R = 0: NDVI +-inf
    nir[0, 0, 0, 3] = -6.0                                   # EVI's denominator 0
    return rgb, nir


@pytest.mark.parametrize("name", S.INDEX_NAMES)
def test_index_reference_is_the_oracles_index_mode(name):
    rgb, nir = _pixels(1)
    ref = index_reference(name, nir[0, 0], rgb[0, 0], rgb[0, 1], rgb[0, 2])
    it, ip = _ORACLE[name](torch.from_numpy(rgb), torch.from_numpy(nir))
    np.testing.assert_array_equal(ip[0, 0].numpy(), ref)
    np.testing.assert_array_equal(it[0, 0].numpy(), ref)


def test_index_reference_keeps_the_formulas_non_finite_values():
    rgb, nir = _pixels(2)
    n, R, G, B = nir[0, 0], rgb[0, 0], rgb[0, 1], rgb[0, 2]
    assert np.isnan(index_reference("ndvi", n, R, G, B)[0, 0]) and np.isnan(index_reference("ndwi", n, R, G, B)[0, 0])
    assert np.isnan(index_reference("msavi", n, R, G, B)[0, 1])
    assert np.isinf(index_reference("ndvi", n, R, G, B)[0, 2])
    assert np.isinf(index_reference("evi", n, R, G, B)[0, 3])
    assert np.isfinite(index_reference("savi", n, R, G, B)).all()


def test_index_names_are_the_reference_terms():
    assert S.INDEX_NAMES == ("ndvi", "ndwi", "gndvi", "savi", "msavi", "evi") == losses.RS_TERMS[1:]


def test_names_map_to_term_ids_in_the_callers_order():
    assert S._index_ids(()) == []
    assert S._index_ids(["ndvi"]) == [1]
    assert S._index_ids(("evi", "ndvi")) == [6, 1]
    assert S._index_ids(("msavi", "savi", "gndvi", "ndwi", "ndvi", "evi")) == [5, 4, 3, 2, 1, 6]
    assert S._index_ids(n for n in ("ndwi", "gndvi")) == [2, 3]
    assert all(losses.RS_TERMS[i] == n for n, i in zip(S.INDEX_NAMES, S._index_ids(S.INDEX_NAMES)))


# ---- argument checks ---------------------------------------------------------------------------------------------
def _model(input_nc=3, **kw):
    from nirgan_b200.config import px2px_config
    from nirgan_b200.model.pix2pix import Px2Px
    cfg = px2px_config(**kw)
    cfg.base_configs.input_nc = input_nc
    return Px2Px(cfg).eval()


U16 = torch.zeros(3, 70, 70, dtype=torch.int16).view(torch.uint16)
F32 = torch.zeros(3, 70, 70)


@pytest.mark.parametrize("indices", [("ndvi", "foo"), ("NDVI",), ("l1",), ("ndvi", "ndvi"), ("evi", "ndwi", "evi"),
                                     ("ndvi", 1), (None,), (b"ndvi",), "ndvi", b"ndvi", None, 3])
@pytest.mark.parametrize("scene", [U16, F32], ids=["u16", "f32"])
def test_bad_indices_are_rejected_before_device_work(indices, scene):
    with pytest.raises(ValueError, match="indices|index"):
        S.predict_scene(_model(), scene, tile=64, overlap=0, indices=indices)


def test_index_bands_need_an_rgb_generator():
    m = _model(input_nc=4)
    with pytest.raises(ValueError, match="input_nc"):
        S.predict_scene(m, torch.zeros(4, 70, 70), tile=64, overlap=0, indices=("ndvi",))
    # without indices the four-channel model gets past the argument checks to the device check
    with pytest.raises(RuntimeError, match="CUDA device"):
        S.predict_scene(m, torch.zeros(4, 70, 70), tile=64, overlap=0)


@pytest.mark.parametrize("indices", [(), ["ndvi"], ("evi", "ndvi"), S.INDEX_NAMES])
@pytest.mark.parametrize("nodata", [None, 0])
def test_accepted_indices_reach_the_device_check(indices, nodata):
    with pytest.raises(RuntimeError, match="CUDA device"):
        S.predict_scene(_model(), U16, tile=64, overlap=0, nodata=nodata, indices=indices)


def test_existing_checks_hold_with_indices():
    m = _model()
    kw = dict(tile=64, overlap=0, indices=("ndvi", "evi"))
    with pytest.raises(ValueError, match="divisible by 4"):
        S.predict_scene(m, U16, tile=66, overlap=0, indices=("ndvi",))
    with pytest.raises(ValueError, match="overlap"):
        S.predict_scene(m, U16, tile=64, overlap=64, indices=("ndvi",))
    with pytest.raises(ValueError, match="channels"):
        S.predict_scene(m, torch.zeros(4, 70, 70), **kw)
    with pytest.raises(ValueError, match="nodata"):
        S.predict_scene(m, U16, nodata=0.5, **kw)
    with pytest.raises(ValueError, match="nodata_out"):
        S.predict_scene(m, U16, nodata=0, nodata_out="nan", **kw)
    with pytest.raises(ValueError, match="needs embeds"):
        S.predict_scene(_model(inject=True), U16, **kw)


def test_assemble_bands_stacks_multi_plane_bands():
    H, W, k = 10, 6, 3
    full = torch.arange((1 + k) * H * W, dtype=torch.float32).view(1 + k, H, W)
    parts = [(y0, y1, full[:, y0:y1]) for y0, y1 in (S.band_rows(H, r, 3) for r in range(3))]
    assert torch.equal(S.assemble_bands(parts[::-1]), full)
    assert torch.equal(S.gather_bands((0, H, full)), full)
