"""Whole-scene NIR prediction: overlapping tiles cut and blended on the device, sharded by row bands.

The reference (and ``synth.run_shard``) only runs pre-cut tiles (create_synthetic_dataset.py:93,100-118).  Here a
``(C, H, W)`` RGB scene -- float32 reflectance, or uint16 digital numbers read as ``dn / dn_scale`` -- becomes one
``(1, H, W)`` NIR band:

* Tile grid.  Tile ``T``, ``overlap`` in ``[0, T)``, stride ``s = T - overlap``; row origins
  ``oy_k = min(k*s, H - T)`` for ``k = 0 .. ceil((H - T) / s)``, columns the same, tile index row-major over
  ``(k_y, k_x)`` (``scene_tiles``).  Every pixel is covered; the last tile of a row / column is clamped to the border.
* Per tile, exactly ``model(tile[None])`` (``Px2Px`` in eval mode, its reflect pad / crop wrapper included).  A tile's
  bits do not depend on its batch slot or rank, so every tile of the scene loop is bit-identical to that single call.
* Blend.  ``out(y, x) = sum_t w_t p_t / sum_t w_t`` over the covering tiles, ``w(i, j) = w1(i) w1(j)``,
  ``w1(i) = min(1, (i + 1) / (overlap + 1), (T - i) / (overlap + 1))``; fp32 sums in ascending ``(k_y, k_x)`` order
  (deterministic); a pixel covered by one tile gets that tile's value exactly.
* Several GPUs: output rows are split into ``world`` contiguous bands balanced to within one row (``band_rows``).  A
  rank computes every tile whose rows meet its band and blends only its band; tiles at band edges are computed by both
  neighbours, with the same bits, so the assembled bands (``assemble_bands`` / ``gather_bands``) equal the ``world = 1``
  result bit for bit.  No collective on the data path.

* Nodata (``nodata=``, off by default).  A pixel is nodata when every channel equals ``nodata`` (GDAL's per-dataset
  mask; NaN matches NaN; uint16 scenes compare the raw digital number).  A tile without a valid pixel is skipped: never
  cut, never run, its ``embeds`` row never read.  Nodata pixels come out as ``nodata_out``; every valid pixel is
  bit-identical to ``nodata=None``, because each tile covering it contains it and so is computed: the blend sees the
  same tiles in the same order with the same weights.
* Index bands (``indices=``, none by default): names from ``INDEX_NAMES`` (``losses.RS_TERMS[1:]``), each at most once.
  The result gains one plane per name, after the NIR plane and in the caller's order.  Each is the reference's
  index-mode formula (``RemoteSensingIndices(mode="index")``, ``losses.rs_index(..., loss_eps=False)``: epsilon 0), with
  ``n`` the blended NIR of plane 0 and ``R, G, B`` channels 0, 1, 2 of the scene exactly as the generator saw them
  (``dn / dn_scale`` for uint16, the raw value for float32): NDVI ``(n - R)/(n + R)``, NDWI ``(n - G)/(n + G)``, GNDVI
  ``(n - G)/(ndvi + G)``, SAVI ``1.5 (n - R)/(n + R + 0.5)``, MSAVI ``(2n + 1 - sqrt((2n + 1)^2 - 8 (n - R)))/2``, EVI
  ``2.5 (n - R)/((n + 6)(R - 7.5)(B + 1))``.  A value the formula makes non-finite (0/0, the square root of a negative)
  stays so.  Every plane is bit-identical to ``rs_index`` of plane 0; plane 0 is bit-identical to ``indices=()``;
  nodata pixels are ``nodata_out`` in every plane.  Needs ``input_nc = 3``.

Cutting (``ng_scene_tiles``: conversion + cut in one pass) and blending (``ng_scene_blend``: gather form, every pixel
written once) are CUDA kernels of ``csrc/scene.cu``; the generator runs through ``Px2Px.forward_async``.  A host scene
is copied to the device one tile row at a time on a copy stream (through pinned staging when it is not pinned itself),
so the copy overlaps the generator.  With ``nodata`` the valid pixels of each tile are counted on the device
(``ng_scene_tile_valid``: once over a device scene, per tile row right after its copy for a host scene), the computed
tiles are batched in tile-index order, and ``ng_scene_blend_masked`` blends the compacted predictions.  With
``indices`` the blend is ``ng_scene_blend_indices``: the same blend kernel writes the index planes from the NIR value it
has just computed and the R, G, B of the resident scene rows, which it reads once per pixel for the nodata test too.  The
band grows to ``(1 + k) (y1 - y0) W`` floats; nothing else grows.
"""
from __future__ import annotations

import numbers
from typing import Dict, List, NamedTuple, Optional, Sequence, Tuple

import torch

from . import _lib as L
from .losses import RS_TERMS


def _check_grid(H: int, W: int, T: int, overlap: int) -> None:
    if T <= 0:
        raise ValueError(f"tile size must be positive, got {T}")
    if not 0 <= overlap < T:
        raise ValueError(f"overlap must lie in [0, {T}) for tile {T}, got {overlap}")
    if H < T or W < T:
        raise ValueError(f"scene {H}x{W} is smaller than the tile {T}x{T}")


def _axis_origins(n: int, T: int, overlap: int) -> List[int]:
    s = T - overlap
    return [min(k * s, n - T) for k in range(-(-(n - T) // s) + 1)]


def scene_grid(H: int, W: int, T: int, overlap: int) -> Tuple[List[int], List[int]]:
    """Row origins and column origins of the tile grid (see the module docstring)."""
    _check_grid(H, W, T, overlap)
    return _axis_origins(H, T, overlap), _axis_origins(W, T, overlap)


def scene_tiles(H: int, W: int, T: int, overlap: int) -> List[Tuple[int, int]]:
    """``(y0, x0)`` of every tile in tile-index order (row-major over ``(k_y, k_x)``); e.g. to compute per-tile lon/lat
    for the SatCLIP encoder of an injected generator."""
    ys, xs = scene_grid(H, W, T, overlap)
    return [(y, x) for y in ys for x in xs]


def band_rows(H: int, rank: int, world: int) -> Tuple[int, int]:
    """Output rows ``[y0, y1)`` of ``rank``'s band: ``world`` contiguous bands balanced to within one row."""
    if not 1 <= world <= H:
        raise ValueError(f"world must lie in [1, {H}] for a scene of {H} rows, got {world}")
    if not 0 <= rank < world:
        raise ValueError(f"rank {rank} out of range for world {world}")
    base, extra = divmod(H, world)
    y0 = rank * base + min(rank, extra)
    return y0, y0 + base + (1 if rank < extra else 0)


def band_tile_rows(row_origins: Sequence[int], T: int, y0: int, y1: int) -> Tuple[int, int]:
    """``[k0, k1)``: the tile rows whose rows meet ``[y0, y1)`` (the origins are ascending)."""
    ks = [k for k, o in enumerate(row_origins) if o < y1 and o + T > y0]
    return ks[0], ks[-1] + 1


INDEX_NAMES = RS_TERMS[1:]          # ("ndvi", "ndwi", "gndvi", "savi", "msavi", "evi")


def _index_ids(indices) -> List[int]:
    """``RS_TERMS`` numbers (1 = NDVI .. 6 = EVI) of the index names, in the caller's order."""
    if isinstance(indices, (str, bytes)):
        raise ValueError(f"indices must be a sequence of index names, not the string {indices!r}")
    try:
        names = list(indices)
    except TypeError:
        raise ValueError(f"indices must be a sequence of index names, got {indices!r}") from None
    for v in names:
        if not isinstance(v, str) or v not in INDEX_NAMES:
            raise ValueError(f"unknown index {v!r}: indices are names from {INDEX_NAMES}")
    if len(set(names)) != len(names):
        raise ValueError(f"indices must not repeat a name, got {tuple(names)}")
    return [RS_TERMS.index(v) for v in names]


def _padding(model) -> int:
    d = model.config.Data
    return d.padding_amount if d.padding else 0


def _stream(s) -> int:
    return s.cuda_stream


class _HostRows:
    """Copies scene rows ``[r_lo, r_hi)`` of a host scene to a device buffer, a chunk per tile row, on a copy stream;
    ``ensure(k)`` issues every chunk up to tile row ``k`` and returns the event after which its rows are resident."""

    def __init__(self, scene: torch.Tensor, ys: Sequence[int], k0: int, k1: int, T: int, device):
        self.scene, self.ys, self.T, self.k1 = scene, ys, T, k1
        C, _, W = scene.shape
        self.r_lo = ys[k0]
        self.dev = torch.empty(C, ys[k1 - 1] + T - self.r_lo, W, dtype=scene.dtype, device=device)
        self.stream = torch.cuda.Stream(device)
        self.stream.wait_stream(torch.cuda.current_stream(device))    # the buffer comes from the caller's stream
        self.events: Dict[int, torch.cuda.Event] = {}
        self.next_k, self.have = k0, self.r_lo
        self.staging = []
        if not scene.is_pinned():
            # two pinned chunks of at most T rows: the host fills one while the other is being copied
            self.staging = [[torch.empty(C, T, W, dtype=scene.dtype).pin_memory(), None] for _ in range(2)]
        self.n_chunks = 0

    def ensure(self, k: int) -> torch.cuda.Event:
        while self.next_k <= min(k, self.k1 - 1):
            a, b = self.have, self.ys[self.next_k] + self.T
            if b > a:
                self._copy(a, b)
            ev = torch.cuda.Event()
            ev.record(self.stream)
            self.events[self.next_k] = ev
            self.have = max(self.have, b)
            self.next_k += 1
        return self.events[min(k, self.k1 - 1)]

    def _copy(self, a: int, b: int) -> None:
        dst = self.dev[:, a - self.r_lo:b - self.r_lo]
        if self.staging:
            slot = self.staging[self.n_chunks % 2]
            if slot[1] is not None:
                slot[1].synchronize()                 # its previous chunk has left for the device
            src = slot[0][:, :b - a]
            src.copy_(self.scene[:, a:b])
        else:
            src = self.scene[:, a:b]
        with torch.cuda.stream(self.stream):
            for c in range(dst.shape[0]):             # one contiguous run of rows per channel: plain async copies
                dst[c].copy_(src[c], non_blocking=True)
            if self.staging:
                done = torch.cuda.Event()
                done.record(self.stream)
                slot[1] = done
        self.n_chunks += 1


def _as_scene(scene) -> torch.Tensor:
    if not isinstance(scene, torch.Tensor):
        import numpy as np
        scene = torch.from_numpy(np.ascontiguousarray(scene))
    if scene.dim() != 3:
        raise ValueError(f"scene must be (C, H, W), got shape {tuple(scene.shape)}")
    if scene.dtype not in (torch.float32, torch.uint16):
        raise ValueError(f"scene must be float32 reflectance or uint16 digital numbers, got {scene.dtype}")
    return scene.contiguous()


def _nodata_value(nodata, dtype: torch.dtype) -> float:
    """``nodata`` as the float the kernels compare with: an integer in [0, 65535] for uint16 scenes (the raw digital
    number), any float for float32 scenes (compared in fp32)."""
    if isinstance(nodata, bool) or not isinstance(nodata, numbers.Real):
        raise ValueError(f"nodata must be a number, got {nodata!r}")
    v = float(nodata)
    if dtype == torch.uint16 and not (v.is_integer() and 0 <= v <= 65535):
        raise ValueError(f"nodata of a uint16 scene must be an integer in [0, 65535], got {nodata!r}")
    return v


class _TileCounts:
    """Valid-pixel counts (``ng_scene_tile_valid``) of the tiles of tile rows ``[k0, k1)``, local tile index
    ``(k - k0) * nx + kx``.  A device scene is counted in one launch and read back at once; a host scene one tile row at
    a time on the copy stream right after that row's copy, read back into pinned memory behind an event, so that
    ``row(k)`` waits for row ``k`` only while the next row's copy is already in flight."""

    def __init__(self, src, dtype, row0, origins, nx, k0, k1, T, nodata, host: Optional[_HostRows], stream):
        self.src, self.dtype, self.row0, self.origins = src, dtype, row0, origins
        self.nx, self.k0, self.k1, self.T, self.nodata, self.host = nx, k0, k1, T, nodata, host
        n = (k1 - k0) * nx
        self.dev = torch.empty(n, dtype=torch.int32, device=src.device)
        if host is None:
            self._launch(0, n, stream)
            with torch.cuda.stream(stream):
                self.counts = self.dev.cpu()
            return
        self.dev.record_stream(host.stream)
        self.counts = torch.empty(n, dtype=torch.int32, pin_memory=True)
        self.events: Dict[int, torch.cuda.Event] = {}
        self.next_k = k0

    def _launch(self, lo: int, hi: int, stream) -> None:
        C, rows, W = self.src.shape
        L.call("ng_scene_tile_valid", self.src.data_ptr(), self.dtype, C, rows, W, self.row0,
               self.origins[lo].data_ptr(), hi - lo, self.T, self.nodata, self.dev[lo:].data_ptr(), _stream(stream))

    def _issue(self, k: int) -> None:
        while self.next_k <= min(k, self.k1 - 1):
            self.host.ensure(self.next_k)             # the row's copy, then its count, on the copy stream
            lo = (self.next_k - self.k0) * self.nx
            hi = lo + self.nx
            self._launch(lo, hi, self.host.stream)
            with torch.cuda.stream(self.host.stream):
                self.counts[lo:hi].copy_(self.dev[lo:hi], non_blocking=True)
                ev = torch.cuda.Event()
                ev.record(self.host.stream)
            self.events[self.next_k] = ev
            self.next_k += 1

    def row(self, k: int) -> List[int]:
        if self.host is not None:
            self._issue(k + 1)                        # keep the next tile row's copy in flight
            self.events[k].synchronize()
        lo = (k - self.k0) * self.nx
        return self.counts[lo:lo + self.nx].tolist()


class _Run(NamedTuple):
    pred: torch.Tensor            # [rows][T][T] fp32, tile at its slot (every tile's own index without nodata)
    ys: List[int]
    xs: List[int]
    k: Tuple[int, int]            # tile rows [k0, k1) of the band
    band: Tuple[int, int]         # output rows [y0, y1)
    done: torch.cuda.Event
    stream: torch.cuda.Stream
    slot: Optional[List[int]]     # nodata only: local tile index -> row of pred, -1 for a skipped tile
    mask: Optional[tuple]         # nodata only: (resident scene rows, NG dtype, row0, nodata)
    rows: Optional[tuple]         # nodata or scene_rows: (resident scene rows, NG dtype, row0), complete on stream


@torch.no_grad()
def _scene_run(model, scene, tile: int, overlap: int, batch_size: int, embeds: Optional[torch.Tensor], dn_scale: float,
               rank: int, world: int, nodata, scene_rows: bool = False) -> _Run:
    """Per-tile predictions of ``rank``'s computed tiles (every tile without ``nodata``), complete on ``stream`` and
    after the event ``done``; with ``nodata`` or ``scene_rows`` the resident scene rows are complete there too."""
    if getattr(model, "concat", False):
        raise NotImplementedError("predict_scene: concat-style SatCLIP generators are not supported")
    if model.training:
        raise RuntimeError("predict_scene: the model is in training mode, call model.eval() first")
    inject = bool(getattr(model, "inject", False))
    T = int(tile)
    scene = _as_scene(scene)
    nd = None if nodata is None else _nodata_value(nodata, scene.dtype)
    C, H, W = scene.shape
    ys, xs = scene_grid(H, W, T, overlap)
    cin = model.opt.input_nc
    if C != cin:
        raise ValueError(f"scene has {C} channels, the model takes input_nc = {cin}")
    pad = _padding(model)
    if (T + 2 * pad) % 4:
        raise ValueError(f"tile {T} with the wrapper's reflect pad {pad} gives {T + 2 * pad} rows, which the generator "
                         f"refuses (must be divisible by 4)")
    if batch_size < 1:
        raise ValueError("batch_size must be >= 1")
    if scene.dtype == torch.uint16 and not dn_scale > 0:
        raise ValueError("dn_scale must be positive")
    n_all = len(ys) * len(xs)
    if inject:
        if embeds is None:
            raise ValueError("predict_scene: a SatCLIP-injected generator needs embeds of shape (n_tiles, 256) in "
                             "tile-index order (scene_tiles gives the origins)")
        if tuple(embeds.shape) != (n_all, 256):
            raise ValueError(f"embeds must have shape ({n_all}, 256), got {tuple(embeds.shape)}")
    elif embeds is not None:
        raise ValueError("predict_scene: embeds given for a generator without SatCLIP injection")
    device = next(model.parameters()).device
    if device.type != "cuda":
        raise RuntimeError("predict_scene: the model must be on a CUDA device (there is no CPU fallback)")
    if scene.is_cuda and scene.device != device:
        raise ValueError(f"scene is on {scene.device}, the model on {device}")

    y0, y1 = band_rows(H, rank, world)
    k0, k1 = band_tile_rows(ys, T, y0, y1)
    nx = len(xs)
    n = (k1 - k0) * nx
    local = [(ys[k], x) for k in range(k0, k1) for x in xs]
    emb = embeds.detach().to(device=device, dtype=torch.float32) if inject else None

    main = torch.cuda.current_stream(device)
    cut, gather = torch.cuda.Stream(device), torch.cuda.Stream(device)
    raw = scene.view(torch.int16) if scene.dtype == torch.uint16 else scene      # copies move the raw 16-bit words
    host = None
    if scene.is_cuda:
        src, row0 = raw, 0
    else:
        host = _HostRows(raw, ys, k0, k1, T, device)
        src, row0 = host.dev, host.r_lo
    dtype = L.U16 if scene.dtype == torch.uint16 else L.F32
    rows = src.shape[1]
    cut.wait_stream(main)                 # embeddings / a device scene were produced on the caller's stream
    gather.wait_stream(main)
    counts = None
    if nd is not None:
        all_origins = torch.tensor(local, dtype=torch.int32).to(device)
        counts = _TileCounts(src, dtype, row0, all_origins, nx, k0, k1, T, nd, host, cut)
        all_origins.record_stream(cut if host is None else host.stream)
    # a host scene learns its computed tiles one tile row at a time while the generator runs: its prediction buffer is
    # sized for every tile of the band, a device scene's for the computed tiles only
    n_pred = n if counts is None or host is not None else sum(c > 0 for c in counts.counts.tolist())
    cap = -(-n_pred // batch_size) * batch_size
    pred = torch.empty(max(cap, 1), T, T, dtype=torch.float32, device=device)
    # batch b's origins (and embedding rows) at [b * batch_size, (b + 1) * batch_size): pinned, then one async copy
    org_h = torch.empty(max(cap, 1), 2, dtype=torch.int32, pin_memory=True)
    org = torch.empty_like(org_h, device=device)
    idx_h = torch.empty(max(cap, 1), dtype=torch.int64, pin_memory=True) if inject else None
    idx = torch.empty_like(idx_h, device=device) if inject else None
    slot = [-1] * n if nd is not None else None
    nb = 0

    def run(tiles: List[int]) -> None:
        nonlocal nb
        lo = nb * batch_size
        # tail padding: the last computed window is repeated so that every batch has batch_size tiles (one plan shape)
        tiles = tiles + [tiles[-1]] * (batch_size - len(tiles))
        org_h[lo:lo + batch_size] = torch.tensor([local[t] for t in tiles], dtype=torch.int32)
        if inject:
            idx_h[lo:lo + batch_size] = torch.tensor(tiles, dtype=torch.int64) + k0 * nx
        with torch.cuda.stream(cut):
            if host is not None:
                last = tiles[-1] // nx + k0
                cut.wait_event(host.ensure(last))
                host.ensure(last + 1)                 # keep the next tile row's copy in flight
            org[lo:lo + batch_size].copy_(org_h[lo:lo + batch_size], non_blocking=True)
            x = torch.empty(batch_size, C, T, T, dtype=torch.float32, device=device)
            L.call("ng_scene_tiles", src.data_ptr(), dtype, C, rows, W, row0, org[lo].data_ptr(), batch_size, T,
                   float(dn_scale), x.data_ptr(), _stream(cut))
            e = None
            if inject:
                idx[lo:lo + batch_size].copy_(idx_h[lo:lo + batch_size], non_blocking=True)
                e = emb.index_select(0, idx[lo:lo + batch_size])
            ready = torch.cuda.Event()
            ready.record(cut)
        out, done = model.forward_async(x, e, ready)
        with torch.cuda.stream(gather):
            for ev in done:
                gather.wait_event(ev)
            out.record_stream(gather)
            pred[lo:lo + batch_size].copy_(out.view(batch_size, T, T))
        nb += 1

    # batches: consecutive runs of computed tiles in tile-index order
    pending: List[int] = []
    for k in range(k0, k1):
        base = (k - k0) * nx
        if counts is None:
            pending += range(base, base + nx)
        else:
            for kx, c in enumerate(counts.row(k)):
                if c > 0:
                    slot[base + kx] = nb * batch_size + len(pending)
                    pending.append(base + kx)
        while len(pending) >= batch_size:
            run(pending[:batch_size])
            pending = pending[batch_size:]
    if pending:
        run(pending)
    org.record_stream(cut)
    if inject:
        idx.record_stream(cut)
        emb.record_stream(cut)
    if host is not None:
        src.record_stream(cut)
    mask = rows = None
    if nd is not None or scene_rows:
        if host is not None:
            gather.wait_event(host.ensure(k1 - 1))    # the blend reads the mask / R, G, B from every resident row
            src.record_stream(gather)
        rows = (src, dtype, row0)
    if nd is not None:
        mask = (src, dtype, row0, nd)
    fin = torch.cuda.Event()
    fin.record(gather)
    return _Run(pred, ys, xs, (k0, k1), (y0, y1), fin, gather, slot, mask, rows)


@torch.no_grad()
def _scene_predictions(model, scene, tile: int = 256, overlap: int = 32, batch_size: int = 64,
                       embeds: Optional[torch.Tensor] = None, dn_scale: float = 10000.0, rank: int = 0, world: int = 1):
    """Per-tile predictions of ``rank``'s tiles.  Returns ``(pred, ys, xs, (k0, k1), (y0, y1), done, stream)``:
    ``pred`` ``[(k1 - k0) * len(xs) (+ tail padding)][T][T]`` fp32 holds tile ``(k_y, k_x)`` at
    ``(k_y - k0) * len(xs) + k_x`` and is complete on ``stream`` and after the event ``done``."""
    r = _scene_run(model, scene, tile, overlap, batch_size, embeds, dn_scale, rank, world, None)
    return r.pred, r.ys, r.xs, r.k, r.band, r.done, r.stream


@torch.no_grad()
def predict_scene(model, scene, tile: int = 256, overlap: int = 32, batch_size: int = 64,
                  embeds: Optional[torch.Tensor] = None, dn_scale: float = 10000.0, rank: int = 0, world: int = 1,
                  nodata=None, nodata_out: float = float("nan"), indices: Sequence[str] = ()):
    """NIR band of a whole scene, and optionally index bands computed from it (module docstring: grid, blend, bands,
    nodata, index bands).

    ``model``: a ``Px2Px`` in eval mode on a CUDA device (plain or SatCLIP-injected; for the latter ``embeds`` is
    ``(n_tiles, 256)`` in tile-index order).  ``scene``: ``(C, H, W)`` float32 reflectance or uint16 digital numbers
    (read as ``dn / dn_scale``), host or device, ``C = input_nc``.  ``batch_size`` tiles per generator call.
    ``nodata``: ``None`` (every pixel holds data), or the value that marks a nodata pixel in every channel -- an integer
    in [0, 65535] compared with the raw digital numbers of a uint16 scene, any float (NaN included) for a float32 scene.
    Tiles without a valid pixel are skipped (their ``embeds`` rows are never read) and nodata pixels are ``nodata_out``.
    ``indices``: ``k`` distinct names from ``INDEX_NAMES`` = ("ndvi", "ndwi", "gndvi", "savi", "msavi", "evi"); plane
    ``1 + i`` of the result is index ``indices[i]`` in the reference's index mode (epsilon 0; NDWI ``(n - G)/(n + G)``,
    GNDVI over ``ndvi + G``, EVI over ``(n + 6)(R - 7.5)(B + 1)``, verbatim), of the pixel's blended NIR ``n`` (plane 0)
    and its ``R, G, B`` = channels 0-2 as the generator saw them (``dn / dn_scale`` for uint16); a non-finite value of
    the formula (0/0, MSAVI's square root of a negative) stays as it is, and a nodata pixel is ``nodata_out`` in every
    plane.  Plane 0 is bit-identical to ``indices=()``, plane ``1 + i`` to ``losses.rs_index(rgb, nir, nir, name,
    loss_eps=False)[1]`` of it.  Needs ``input_nc = 3``; the default ``()`` runs exactly the NIR-only blend.
    Returns the ``(1 + k, H, W)`` float32 device tensor for ``world = 1``, else ``(y0, y1, band)`` with ``band`` the
    ``(1 + k, y1 - y0, W)`` rows of this rank (``gather_bands`` / ``assemble_bands`` put the bands together).  The
    result is valid on the caller's current stream.  Bad arguments raise ``ValueError`` before any device work."""
    if nodata is not None and (isinstance(nodata_out, bool) or not isinstance(nodata_out, numbers.Real)):
        raise ValueError(f"nodata_out must be a number, got {nodata_out!r}")
    ids = _index_ids(indices)
    if ids and model.opt.input_nc != 3:
        raise ValueError(f"index bands need an RGB generator (input_nc = 3: channels 0, 1, 2 are R, G, B), this one "
                         f"takes input_nc = {model.opt.input_nc}")
    r = _scene_run(model, scene, tile, overlap, batch_size, embeds, dn_scale, rank, world, nodata, bool(ids))
    (k0, k1), (y0, y1), gather = r.k, r.band, r.stream
    device = r.pred.device
    W = r.xs[-1] + tile
    main = torch.cuda.current_stream(device)
    band = torch.empty(1 + len(ids), y1 - y0, W, dtype=torch.float32, device=device)
    with torch.cuda.stream(gather):
        oy = torch.tensor(r.ys[k0:k1], dtype=torch.int32).to(device)
        ox = torch.tensor(r.xs, dtype=torch.int32).to(device)
        band.record_stream(gather)
        if ids:
            src, dtype, row0 = r.rows
            slot = None if r.slot is None else torch.tensor(r.slot, dtype=torch.int32).to(device)
            nd = 0.0 if r.mask is None else r.mask[3]
            L.call("ng_scene_blend_indices", r.pred.data_ptr(), None if slot is None else slot.data_ptr(),
                   oy.data_ptr(), k1 - k0, ox.data_ptr(), len(r.xs), tile, overlap, W, y0, y1, src.data_ptr(), dtype,
                   src.shape[0], src.shape[1], row0, float(dn_scale), int(r.mask is not None), nd, float(nodata_out),
                   (L.c_i32 * len(ids))(*ids), len(ids), band.data_ptr(), _stream(gather))
        elif r.mask is None:
            L.call("ng_scene_blend", r.pred.data_ptr(), oy.data_ptr(), k1 - k0, ox.data_ptr(), len(r.xs), tile, overlap,
                   W, y0, y1, band.data_ptr(), _stream(gather))
        else:
            src, dtype, row0, nd = r.mask
            slot = torch.tensor(r.slot, dtype=torch.int32).to(device)
            L.call("ng_scene_blend_masked", r.pred.data_ptr(), slot.data_ptr(), oy.data_ptr(), k1 - k0, ox.data_ptr(),
                   len(r.xs), tile, overlap, W, y0, y1, src.data_ptr(), dtype, src.shape[0], src.shape[1], row0, nd,
                   float(nodata_out), band.data_ptr(), _stream(gather))
    main.wait_stream(gather)
    if world == 1:
        return band
    return y0, y1, band


def assemble_bands(parts: Sequence[Tuple[int, int, torch.Tensor]]) -> torch.Tensor:
    """``(1, H, W)`` CPU tensor from the ``(y0, y1, band)`` of every rank; the bands must tile ``[0, H)`` exactly."""
    parts = sorted(parts, key=lambda p: p[0])
    at = 0
    for y0, y1, band in parts:
        if y0 != at or y1 <= y0 or band.shape[-2] != y1 - y0:
            raise ValueError(f"bands do not tile the scene's rows: expected one starting at row {at}, got [{y0}, {y1})")
        at = y1
    return torch.cat([band.detach().cpu() for _, _, band in parts], dim=-2)


def gather_bands(local: Tuple[int, int, torch.Tensor], group=None) -> torch.Tensor:
    """Host-side assembly of the per-rank bands (the only cross-rank step; not on the GPU data path), like
    ``synth.gather_shards``: with ``torch.distributed`` initialised every rank receives the whole ``(1, H, W)`` scene."""
    import torch.distributed as dist
    y0, y1, band = local
    mine = (y0, y1, band.detach().cpu())
    if not dist.is_available() or not dist.is_initialized() or dist.get_world_size(group) == 1:
        return assemble_bands([mine])
    parts = [None] * dist.get_world_size(group)
    dist.all_gather_object(parts, mine, group=group)
    return assemble_bands(parts)
