#!/usr/bin/env python
"""Whole-scene prediction rate (nirgan_b200.scene.predict_scene) next to bench.py's tile rate, in one run.

Workload: a seeded synthetic 8192 x 8192 uint16 scene (3 bands of digital numbers) in pinned host memory, tile 256,
overlap 32 (37 x 37 = 1369 tiles), batch 64, the SatCLIP-injected generator of BASELINE.json configs[1] behind the Px2Px
pad-10 wrapper (random init, per-tile random embeddings).  After --warmup scenes, --scenes scenes are timed as one
window ending in a device synchronise.  Reported besides: the generator alone on resident 256 x 256 tiles with the same
wrapper (where the scene loop's time goes), ng_scene_tiles / ng_scene_blend kernel times from CUDA events with their
algorithmic bytes against a device-to-device copy measured in the same run, the card's name, power limit and clocks,
and the `value` of `bench.py --steps K` run right after.

--nodata-frac F adds a swath edge: a corner triangle of area fraction F (legs sqrt(2 F) N, F <= 0.5) set to DN 0 in
every band of a copy of the scene, predicted with nodata=0.  Recorded besides: the tiles computed and skipped, that
scene's time and its rate over the computed tiles, the ng_scene_tile_valid time (one tile row of windows, as a host
scene runs it after each row's copy, and the whole scene in one launch), and nodata=0 against nodata=None on the fully
valid scene, alternated scene by scene, which shows the cost of the validity pass.

--indices ndvi,ndwi,evi (any subset of ndvi, ndwi, gndvi, savi, msavi, evi) adds index bands: the scene with those
indices against indices=(), alternated scene by scene (medians), and ng_scene_blend_indices against ng_scene_blend on the
same predictions of the resident scene, with their algorithmic bytes (predictions, plus 2 B per channel and pixel of the
uint16 scene and (1 + k) 4 B per pixel written for the index blend) against the device-to-device copy.

    python tools/bench_scene.py --out profiles/scene_bench.json
    python tools/bench_scene.py --nodata-frac 0.4 --out profiles/scene_bench_nodata.json
    python tools/bench_scene.py --indices ndvi,ndwi,evi --out profiles/scene_bench_indices.json
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")
import torch  # noqa: E402


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", f"--query-gpu={q}", "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        f = [x.strip() for x in out.splitlines()[0].split(",")]
        return {"name": f[0], "power_limit_w": float(f[1]), "sm_mhz": float(f[2]), "sm_max_mhz": float(f[3])}
    except Exception as e:                          # the numbers below are still valid, only unlabeled
        return {"error": repr(e)}


def event_ms(fn, reps):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    fn()
    torch.cuda.synchronize()
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


def nodata_section(frac, scene, one_scene, model, emb, sdev, tiles, N, T, ov, B, args, copy_gbs):
    import math
    from nirgan_b200 import _lib as L
    from nirgan_b200 import scene as S

    dev = sdev.device
    n = len(tiles)
    i = torch.arange(N, dtype=torch.int32)
    edge = math.sqrt(2 * frac) * N
    mask = (i[:, None] + i[None, :]) < edge                  # pixels (y, x) with y + x < sqrt(2 F) N: the swath edge
    swath = scene.clone().pin_memory()
    swath.view(torch.int16).masked_fill_(mask, 0)
    ys, xs = S.scene_grid(N, N, T, ov)
    nx = len(xs)

    def swath_scene():
        return S.predict_scene(model, swath, tile=T, overlap=ov, batch_size=B, embeds=emb, nodata=0)

    for _ in range(args.warmup):
        swath_scene()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(args.scenes):
        out = swath_scene()
    torch.cuda.synchronize()
    s = (time.perf_counter() - t0) / args.scenes
    nan = torch.isnan(out[0])
    mask_ok = bool(torch.equal(nan, mask.to(dev)))

    # nodata=0 against nodata=None on the fully valid scene, alternated scene by scene
    def valid_scene():
        return S.predict_scene(model, scene, tile=T, overlap=ov, batch_size=B, embeds=emb, nodata=0)

    valid_scene()
    times = {"none": [], "nodata0": []}
    for _ in range(args.scenes):
        for key, fn in (("none", one_scene), ("nodata0", valid_scene)):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            o = fn()
            torch.cuda.synchronize()
            times[key].append(time.perf_counter() - t0)
    masked_pixels = int(torch.isnan(o).sum())

    # ng_scene_tile_valid alone on the swath scene: one tile row of windows (a host scene's launch), and the whole
    # scene in one launch (its counts give the skipped tiles)
    st = torch.cuda.current_stream().cuda_stream
    swd = swath.view(torch.int16).to(dev)
    org = torch.tensor(tiles, dtype=torch.int32, device=dev)
    cnt = torch.empty(n, dtype=torch.int32, device=dev)
    row_ms = event_ms(lambda: L.call("ng_scene_tile_valid", swd.data_ptr(), L.U16, 3, N, N, 0, org.data_ptr(), nx, T,
                                     0.0, cnt.data_ptr(), st), 200)
    all_ms = event_ms(lambda: L.call("ng_scene_tile_valid", swd.data_ptr(), L.U16, 3, N, N, 0, org.data_ptr(), n, T,
                                     0.0, cnt.data_ptr(), st), 20)
    skipped = int((cnt == 0).sum())
    skipped_grid = sum(1 for y, x in tiles if (y + T - 1) + (x + T - 1) < edge)
    del swd
    row_bytes = nx * (3 * T * T * 2 + 4)
    all_bytes = n * (3 * T * T * 2 + 4)
    med = {k: sorted(v)[len(v) // 2] for k, v in times.items()}
    return {
        "nodata_frac": frac, "triangle_legs_px": edge, "nodata_pixel_frac": float(mask.float().mean()),
        "tiles": n, "tiles_skipped": skipped, "tiles_computed": n - skipped, "tiles_skipped_by_grid_arithmetic": skipped_grid,
        "scene_s": s, "computed_tiles_per_s": (n - skipped) / s, "output_mask_equals_triangle": mask_ok,
        "valid_output_finite": bool(torch.isfinite(out[0][~nan]).all()),
        "ab_fully_valid_scene": {"scene_s_nodata_none": times["none"], "scene_s_nodata_0": times["nodata0"],
                                 "median_none": med["none"], "median_nodata_0": med["nodata0"],
                                 "median_ratio": med["nodata0"] / med["none"], "pixels_masked": masked_pixels},
        "ng_scene_tile_valid": {
            "tile_row": {"windows": nx, "ms": row_ms, "bytes": row_bytes, "gbs": row_bytes / row_ms / 1e6,
                         "frac_of_copy_peak": row_bytes / row_ms / 1e6 / copy_gbs, "ms_per_scene": row_ms * n / nx,
                         "note": "one tile row's 12.6 MB of scene rows stays in the L2, as right after its copy"},
            "whole_scene": {"windows": n, "ms": all_ms, "bytes": all_bytes, "gbs": all_bytes / all_ms / 1e6,
                            "frac_of_copy_peak": all_bytes / all_ms / 1e6 / copy_gbs}},
    }


def indices_section(names, scene, one_scene, model, emb, sdev, pred, oy, ox, ys, xs, N, T, ov, B, args, copy_gbs,
                    blend_ms):
    from nirgan_b200 import _lib as L
    from nirgan_b200 import scene as S

    def idx_scene():
        return S.predict_scene(model, scene, tile=T, overlap=ov, batch_size=B, embeds=emb, indices=names)

    idx_scene()
    times = {"none": [], "indices": []}
    for _ in range(args.scenes):
        for key, fn in (("none", one_scene), ("indices", idx_scene)):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            o = fn()
            torch.cuda.synchronize()
            times[key].append(time.perf_counter() - t0)
            if key == "none":
                nir = o
    plane0_same = bool(torch.equal(o[0], nir[0]))
    del o, nir

    # the blend kernels alone on the same predictions of the resident scene
    st = torch.cuda.current_stream().cuda_stream
    k = len(names)
    which = (L.c_i32 * k)(*[S.INDEX_NAMES.index(n) + 1 for n in names])
    out = torch.empty(1 + k, N, N, device=sdev.device)
    idx_ms = event_ms(lambda: L.call("ng_scene_blend_indices", pred.data_ptr(), None, oy.data_ptr(), len(ys),
                                     ox.data_ptr(), len(xs), T, ov, N, 0, N, sdev.data_ptr(), L.U16, 3, N, 0, 10000.0,
                                     0, 0.0, 0.0, which, k, out.data_ptr(), st), 10)
    del out
    idx_bytes = len(ys) * len(xs) * T * T * 4 + N * N * (3 * 2 + (1 + k) * 4)
    med = {key: sorted(v)[len(v) // 2] for key, v in times.items()}
    return {
        "indices": list(names), "scene_s_indices_none": times["none"], "scene_s_indices": times["indices"],
        "median_none": med["none"], "median_indices": med["indices"], "median_ratio": med["indices"] / med["none"],
        "plane0_equals_indices_none": plane0_same,
        "ng_scene_blend_indices": {"ms_per_scene": idx_ms, "bytes": idx_bytes, "gbs": idx_bytes / idx_ms / 1e6,
                                   "frac_of_copy_peak": idx_bytes / idx_ms / 1e6 / copy_gbs,
                                   "over_ng_scene_blend": idx_ms / blend_ms},
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--size", type=int, default=8192)
    ap.add_argument("--tile", type=int, default=256)
    ap.add_argument("--overlap", type=int, default=32)
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--scenes", type=int, default=4)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--bench-steps", type=int, default=20)
    ap.add_argument("--nodata-frac", type=float, default=None)
    ap.add_argument("--indices", default=None)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    names = None
    if args.indices is not None:
        names = tuple(v.strip() for v in args.indices.split(",") if v.strip())
        valid = ("ndvi", "ndwi", "gndvi", "savi", "msavi", "evi")
        if not names or any(v not in valid for v in names) or len(set(names)) != len(names):
            raise SystemExit(f"bench_scene.py: --indices takes distinct names from {','.join(valid)}")
    if args.nodata_frac is not None and not 0 < args.nodata_frac <= 0.5:
        raise SystemExit("bench_scene.py: --nodata-frac must lie in (0, 0.5] (a corner triangle)")
    if not torch.cuda.is_available():
        raise SystemExit("bench_scene.py: no CUDA device")
    import nirgan_b200  # noqa: F401
    from nirgan_b200 import _lib as L
    from nirgan_b200 import scene as S
    from nirgan_b200.config import satclip_inject_config
    from nirgan_b200.model.pix2pix import Px2Px

    dev = torch.device("cuda", 0)
    torch.manual_seed(0)
    model = Px2Px(satclip_inject_config()).to(dev).eval()
    model.netG.configure_b200(precision="fp16", impl="tc")
    N, T, ov, B = args.size, args.tile, args.overlap, args.batch
    g = torch.Generator().manual_seed(1)
    scene = torch.randint(0, 10001, (3, N, N), generator=g, dtype=torch.int32).to(torch.int16)
    scene = scene.view(torch.uint16).pin_memory()
    tiles = S.scene_tiles(N, N, T, ov)
    n = len(tiles)
    emb = torch.randn(n, 256, generator=g)
    padded = -(-n // B) * B

    def one_scene():
        return S.predict_scene(model, scene, tile=T, overlap=ov, batch_size=B, embeds=emb)

    for _ in range(args.warmup):
        one_scene()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(args.scenes):
        out = one_scene()
    torch.cuda.synchronize()
    s = (time.perf_counter() - t0) / args.scenes
    finite = bool(torch.isfinite(out).all())

    # the generator alone: resident batches of B tiles through the same wrapper (pad 10), streamed like the scene loop
    x = torch.rand(B, 3, T, T, generator=g).to(dev)
    e = torch.randn(B, 256, generator=g).to(dev)
    steps = padded // B
    last = {}

    def gen_step():
        last["y"], last["done"] = model.forward_async(x, e)

    for _ in range(3):
        gen_step()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(steps * args.scenes):
        gen_step()
    torch.cuda.synchronize()
    gen_tps = B * steps * args.scenes / (time.perf_counter() - t0)

    # kernels on their own: one batch cut from the resident u16 scene; the blend of the whole scene
    st = torch.cuda.current_stream().cuda_stream
    sdev = scene.view(torch.int16).to(dev)
    org = torch.tensor(tiles[:B], dtype=torch.int32, device=dev)
    xb = torch.empty(B, 3, T, T, device=dev)
    cut_ms = event_ms(lambda: L.call("ng_scene_tiles", sdev.data_ptr(), L.U16, 3, N, N, 0, org.data_ptr(), B, T,
                                     10000.0, xb.data_ptr(), st), 50)
    cut_bytes = B * 3 * T * T * (2 + 4)
    ys, xs = S.scene_grid(N, N, T, ov)
    pred = torch.rand(n, T, T, generator=torch.Generator(device=dev).manual_seed(2), device=dev) * 2 - 1
    oy = torch.tensor(ys, dtype=torch.int32, device=dev)
    ox = torch.tensor(xs, dtype=torch.int32, device=dev)
    band = torch.empty(N, N, device=dev)
    blend_ms = event_ms(lambda: L.call("ng_scene_blend", pred.data_ptr(), oy.data_ptr(), len(ys), ox.data_ptr(),
                                       len(xs), T, ov, N, 0, N, band.data_ptr(), st), 10)
    blend_bytes = n * T * T * 4 + N * N * 4
    big = torch.empty(1 << 28, device=dev)                   # 1 GiB: well beyond the L2
    big2 = torch.empty_like(big)
    copy_ms = event_ms(lambda: big2.copy_(big), 10)
    copy_gbs = 2 * big.numel() * 4 / copy_ms / 1e6
    h2d_bytes = scene.numel() * 2
    nodata_rec = None
    if args.nodata_frac is not None:
        nodata_rec = nodata_section(args.nodata_frac, scene, one_scene, model, emb, sdev, tiles, N, T, ov, B, args,
                                    copy_gbs)
    indices_rec = None
    if names is not None:
        indices_rec = indices_section(names, scene, one_scene, model, emb, sdev, pred, oy, ox, ys, xs, N, T, ov, B,
                                      args, copy_gbs, blend_ms)
    info = gpu_info()
    del pred, band, big, big2, sdev
    torch.cuda.empty_cache()

    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(args.bench_steps),
           "--warmup", "5", "--no-train", "--no-cpu-baseline"]
    r = subprocess.run(cmd, capture_output=True, text=True, cwd=ROOT)
    bench_value = None
    for line in r.stdout.splitlines():
        if line.startswith("{"):
            bench_value = json.loads(line).get("value")
    tps = n / s
    rec = {
        "workload": f"predict_scene: {N}x{N} uint16 scene in pinned host memory, tile {T}, overlap {ov} ({n} tiles, "
                    f"{padded} with tail padding), batch {B}, SatCLIP-injected generator behind the pad-10 wrapper, "
                    f"fp16 / tcgen05",
        "gpu": info,
        "scene_s": s, "scenes_timed": args.scenes, "output_finite": finite,
        "tiles_per_s": tps, "output_mpix_per_s": N * N / s / 1e6,
        "generator_alone_pad10_tiles_per_s": gen_tps,
        "tail_padding_share": (padded - n) / padded,
        "h2d_bytes_per_scene": h2d_bytes,
        "kernels": {
            "copy_peak_gbs_d2d": copy_gbs,
            "ng_scene_tiles": {"ms_per_batch": cut_ms, "bytes": cut_bytes, "gbs": cut_bytes / cut_ms / 1e6,
                               "frac_of_copy_peak": cut_bytes / cut_ms / 1e6 / copy_gbs,
                               "ms_per_scene": cut_ms * padded / B},
            "ng_scene_blend": {"ms_per_scene": blend_ms, "bytes": blend_bytes, "gbs": blend_bytes / blend_ms / 1e6,
                               "frac_of_copy_peak": blend_bytes / blend_ms / 1e6 / copy_gbs}},
        "bench_py": {"cmd": " ".join(cmd[1:]), "value": bench_value, "returncode": r.returncode},
        "scene_over_bench_value": tps / bench_value if bench_value else None,
        "scene_over_generator_alone": tps / gen_tps,
    }
    if nodata_rec is not None:
        rec["nodata"] = nodata_rec
    if indices_rec is not None:
        rec["index_bands"] = indices_rec
    if r.returncode != 0:
        rec["bench_py"]["stderr_tail"] = r.stderr[-2000:]
    txt = json.dumps(rec, indent=1)
    print(txt)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(txt + "\n")


if __name__ == "__main__":
    main()
