#!/usr/bin/env python
"""bench.py -- NIR-GAN hot path on B200: 256x256 RGB->NIR tiles/sec (+ the training step as a sub-record).

Headline workload (N=1): BASELINE.json configs[1] -- SatCLIP-injected ResnetGenerator inference, 64 synthetic
3x256x256 tiles + 64 random (256,) embeddings per step, random-init weights, through the reference-
compatible API (`define_G_inject(config)(x, embeds)`).  N>1: the same per-GPU workload on every rank
(tile-sharded, no collective; scaling = weak).

One JSON line on stdout (rank 0).  `value` = tiles/s with inputs resident in HBM; `e2e` = the same through
host (pinned) buffers incl. H2D of tiles+embeddings and D2H of the NIR band every step.  Each is timed over one
window of exactly --steps steps after the warm-up (barrier + synchronize on both sides of the window, CUDA events,
max over ranks).  A clock sampler (nvidia-smi) runs beside every timed loop alike.
`--dump-outputs DIR` writes the NIR prediction of the last timed `value` step (rank 0) to DIR/nir_pred.npy (float32,
at most 64 MB: the leading tiles of a larger batch); inputs and weights are seeded, so two builds can be compared
output for output.
`train` sub-record: BASELINE.json configs[3] (full Pix2Pix training step, batch 32, 256x256) and configs[4]
(data-parallel training, batch 32 per GPU, seeded mixed 128..512 px resolutions, NCCL gradient all-reduce over
N ranks) through `nirgan_b200.trainer.Trainer`.
`--impl reference` times the CPU oracle port of the reference on the host cores (the reference is pure
Python/torch and cannot travel to the GPU box; SURVEY.md 8c).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

# more hardware queues than streams (compute slices + copy streams): no false dependencies between streams
os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")
import torch  # noqa: E402

TILE = 256
BATCH = 64
METRIC = "rgb2nir_256px_tiles_per_sec"
UNIT = "tiles/s"
WORKLOAD = ("configs[1]: SatCLIP-injected ResnetGenerator (9 blocks, ngf 64) inference, 64x3x256x256 tiles + 64x256 "
            "random embeddings per GPU per step, random-init weights")
TRAIN_RES = (128, 192, 256, 384, 512)
GFLOP_PER_SAMPLE_256 = 391.6          # SURVEY.md 8d: minimal training-step op count (one G forward), 256x256 tile
DUMP_LIMIT_BYTES = 64 << 20           # --dump-outputs: leading tiles of the last step's prediction up to this size


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        d = json.load(open(path))
        return {"hbm_gbs": d["hbm_gbs"], "tf_burst": d["bf16_tflops"], "tf_sustained": d["bf16_tflops_sustained"],
                "src": "MEASURED_PEAKS.json"}
    return {"hbm_gbs": 6650.0, "tf_burst": 1590.0, "tf_sustained": 1400.0, "src": "fallback (B200_PROFILING.md)"}


class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.p = None
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(gpu_index), f"--query-gpu={self.Q}",
                                       "--format=csv,noheader,nounits", "-lms", "100"],
                                      stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.p = None

    def stop(self):
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"], "samples": 0}
        self.p.terminate()
        try:
            out, _ = self.p.communicate(timeout=5)
        except Exception:
            self.p.kill()
            out = ""
        sm, mx, reasons = [], 0.0, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in out.strip().splitlines():
            f = [x.strip() for x in line.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx = max(mx, float(f[1]))
            except ValueError:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx or None, "reasons": sorted(reasons),
                "samples": len(sm)}


def merge_clocks(parts: dict):
    """One `clocks` object for the line: median of the per-loop medians, union of the reasons, plus the per-loop records."""
    meds = sorted(c["sm_mhz"] for c in parts.values() if c and c.get("sm_mhz"))
    out = {"sm_mhz": meds[len(meds) // 2] if meds else None,
           "sm_max_mhz": max([c["sm_max_mhz"] for c in parts.values() if c and c.get("sm_max_mhz")] or [None]),
           "reasons": sorted({r for c in parts.values() if c for r in c.get("reasons", [])}),
           "samples": sum(c.get("samples", 0) for c in parts.values() if c),
           "per_loop": parts}
    return out


def build_model(dev):
    import nirgan_b200  # noqa: F401
    from nirgan_b200.config import satclip_inject_config
    from nirgan_b200.model.generator_inject import define_G_inject
    import contextlib
    torch.manual_seed(0)
    with contextlib.redirect_stdout(sys.stderr):   # the reference prints its scale-param init; stdout is JSON only
        net = define_G_inject(satclip_inject_config())     # random-init, N(0, 0.02) like the reference
    return net.to(dev).eval()


def cpu_oracle_tiles_per_sec(budget_s=12.0, batch=4):
    """The reference's CPU path on the host cores: a bounded sample of the same workload.  Runs the reference's OWN modules
    (oracle/_ref: unmodified model/networks.py + model/generator_inject.py placed there by oracle/make_ref.py, kind
    "reference") when that tree travelled with the snapshot, else the oracle port (kind "port").
    Returns (tiles/s, cores, sample description, kind)."""
    import contextlib
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    g = torch.Generator().manual_seed(1)
    x = torch.rand(batch, 3, TILE, TILE, generator=g)
    e = torch.randn(batch, 256, generator=g)
    fwd, kind = None, "port"
    try:
        import make_ref
        mods = make_ref.load()
        if mods is not None:
            from nirgan_b200.config import satclip_inject_config      # attribute-style mirror of config_px2px_SatCLIP.yaml
            torch.manual_seed(0)
            with contextlib.redirect_stdout(sys.stderr):
                net = mods[1].define_G_inject(satclip_inject_config()).eval()
            fwd, kind = (lambda xb, eb: net(xb, eb)), "reference"
    except Exception as ex:                    # the reference tree is optional: say why the port is used instead
        print(f"bench.py: oracle/_ref not usable ({type(ex).__name__}: {ex}); timing the oracle port", file=sys.stderr)
    if fwd is None:
        import nirgan_oracle as O
        sd = O.random_state_dict(O.generator_param_shapes(inject=True), seed=0)
        fwd = lambda xb, eb: O.resnet_generator_forward(sd, xb, embeds=eb)
    with torch.no_grad():
        fwd(x[:1], e[:1])                                             # warm-up
        n, t0 = 0, time.perf_counter()
        while True:
            fwd(x, e)
            n += batch
            el = time.perf_counter() - t0
            if el >= budget_s or n >= 64:
                break
    what = "the reference's own nn.Modules (oracle/_ref)" if kind == "reference" else "oracle port"
    return n / el, cores, (f"{n} tiles ({n // batch} batches of {batch}) of the 64-tile step, {what}, fp32, "
                           f"torch {torch.__version__} CPU, {el:.1f} s"), kind


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    vals = []
    sample = ""
    kind = "port"
    for i in range(args.warmup + args.steps):
        v, cores, sample, kind = cpu_oracle_tiles_per_sec(budget_s=6.0, batch=4)
        if i >= args.warmup:
            vals.append(v)
    v = sum(vals) / len(vals)
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": BATCH / v * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD,
                       "note": "the reference's CPU implementation of the path (its own modules from oracle/_ref when "
                               "present, else the oracle port); each step is a bounded sample of the 64-tile step on all "
                               "host cores"},
            "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample},
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit(line)


_REAL_STDOUT = [None]


def _quiet_stdout():
    """stdout must carry exactly one JSON line.  Libraries print there too (NCCL's version banner, the reference's
    constructor messages), so file descriptor 1 is pointed at stderr for the whole run and the JSON line is written
    to a saved duplicate of the real stdout."""
    if _REAL_STDOUT[0] is None:
        sys.stdout.flush()
        _REAL_STDOUT[0] = os.dup(1)
        os.dup2(2, 1)


def emit(line: dict):
    data = (json.dumps(line) + "\n").encode()
    sys.stdout.flush()
    if _REAL_STDOUT[0] is None:
        os.write(1, data)
    else:
        os.write(_REAL_STDOUT[0], data)


def pct(sorted_vals, q):
    if not sorted_vals:
        return None
    i = min(len(sorted_vals) - 1, max(0, int(round(q * (len(sorted_vals) - 1)))))
    return sorted_vals[i]


class Timing:
    """Window timing shared by every loop of the bench: W warm-up steps (then more, until >= `settle_s` of work has run, so
    the SM clocks have ramped), then windows of exactly K steps -- barrier + synchronize, event, K steps, join, event,
    barrier + synchronize; max over ranks -- until >= min_windows windows and >= min_total_s of timed work."""

    def __init__(self, dev, dist, main_stream, extra_streams=()):
        self.dev, self.dist, self.main, self.extra = dev, dist, main_stream, tuple(extra_streams)

    def barrier(self):
        torch.cuda.synchronize(self.dev)
        if self.dist is not None:
            self.dist.barrier()
        torch.cuda.synchronize(self.dev)

    def max_over_ranks(self, ms):
        if self.dist is None:
            return ms
        t = torch.tensor([ms], device=self.dev, dtype=torch.float64)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def windows(self, fn, steps, warm, join=None, min_windows=5, min_total_s=2.0, max_windows=60, settle_s=1.0):
        t0 = time.perf_counter()
        n = 0
        while n < warm or self.max_over_ranks(time.perf_counter() - t0) < settle_s:
            fn()
            n += 1
            if n % 4 == 0:
                torch.cuda.synchronize(self.dev)
        ms_all = []
        while True:
            self.barrier()
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            ev0.record(self.main)
            for _ in range(steps):
                fn()
            if join is not None:
                join()
            for st in self.extra:
                self.main.wait_stream(st)
            ev1.record(self.main)
            self.barrier()
            ms_all.append(self.max_over_ranks(ev0.elapsed_time(ev1)))      # identical on every rank after the reduce
            if len(ms_all) >= max_windows or (len(ms_all) >= min_windows and sum(ms_all) >= min_total_s * 1e3):
                break
        s = sorted(ms_all)
        return {"ms_p50": pct(s, 0.5), "ms_p10": pct(s, 0.1), "ms_p90": pct(s, 0.9), "n": len(s),
                "total_s": sum(s) / 1e3, "warm_steps": n, "first_ms": ms_all[0]}


# =====================================================================================================================
# training sub-record (BASELINE.json configs[3] and configs[4])
# =====================================================================================================================
def train_record(args, dev, rank, world, dist, tm: Timing, samplers: dict):
    import contextlib
    import nirgan_b200  # noqa: F401
    from nirgan_b200.config import px2px_config
    from nirgan_b200.model.pix2pix import Px2Px
    from nirgan_b200.trainer import Trainer
    torch.manual_seed(0)                       # same initial weights on every rank (DDP)
    with contextlib.redirect_stdout(sys.stderr):
        model = Px2Px(px2px_config()).to(dev).train()
    model.netG.configure_b200(precision=args.precision, impl=args.conv)
    model.netD.configure_b200(precision=args.precision, impl=args.conv)
    trainer = Trainer(model, time_exchange=True)
    B = args.train_batch
    gen = torch.Generator().manual_seed(200 + rank)
    # host (pinned) copies of every resolution's batch: the e2e loop feeds the step from them
    host = {s: {"rgb": torch.rand(B, 3, s, s, generator=gen).pin_memory(),
                "nir": torch.rand(B, 1, s, s, generator=gen).pin_memory()} for s in TRAIN_RES}
    data = {s: {k: v.to(dev) for k, v in host[s].items()} for s in TRAIN_RES}
    losses = torch.zeros(2, device=dev)
    losses_host = torch.zeros(2).pin_memory()
    state = {"last": None}

    def step_at(s):
        ld, lg = trainer.step(data[s])
        state["last"] = (ld, lg)

    # every resolution once, largest first (plan compilation, pool sizing, graph capture are one-off costs)
    for s in sorted(TRAIN_RES, reverse=True):
        for _ in range(2):
            step_at(s)
    torch.cuda.synchronize(dev)
    rec = {}

    # ---- configs[3]: fixed 256x256, batch 32 per GPU ----
    def flop(s):
        return GFLOP_PER_SAMPLE_256 * (s / 256.0) ** 2 if model.reuse_g_forward else 505.8 * (s / 256.0) ** 2

    samplers["train"] = ClockSampler(int(os.environ.get("LOCAL_RANK", "0"))) if rank == 0 else None
    k4 = max(2, args.train_steps)
    w = tm.windows(lambda: step_at(256), k4, 3, min_windows=5, min_total_s=1.5, settle_s=0.5)
    ms4 = w["ms_p50"] / k4
    torch.cuda.synchronize(dev)
    ld, lg = state["last"]
    exposed4 = trainer.exposed_exchange_ms()
    rec["config4"] = {
        "workload": f"configs[3]: full Pix2Pix training step (D pass + G pass, LSGAN + 100*L1 + NDVI/NDWI/EVI, Adam), "
                    f"batch {B} per GPU, 256x256, plain generator behind the pad-10 wrapper",
        "ms_per_step": ms4, "samples_per_s": B * world / ms4 * 1e3, "steps_per_window": k4, "windows": w,
        "tflops": B * world * flop(256) / ms4, "gflop_per_sample": flop(256),
        "frac_of_sustained_peak": B * flop(256) / ms4 / peaks()["tf_sustained"],
        "allreduce_exposed_ms_per_step": exposed4, "loss_D": float(ld), "loss_G": float(lg)}
    # the same step fed from pinned host memory (H2D of the batch, D2H of the two losses every step)
    hstream = torch.cuda.Stream(dev)
    dbuf = [{k: torch.empty_like(v) for k, v in data[256].items()} for _ in range(2)]
    hev = [torch.cuda.Event() for _ in range(2)]
    fev = [None, None]
    ctr = {"i": 0}

    def step_e2e():
        i = ctr["i"] & 1
        ctr["i"] += 1
        with torch.cuda.stream(hstream):
            if fev[i] is not None:
                hstream.wait_event(fev[i])
            for k in dbuf[i]:
                dbuf[i][k].copy_(host[256][k], non_blocking=True)
            hev[i].record(hstream)
        tm.main.wait_event(hev[i])
        ld_, lg_ = trainer.step(dbuf[i])
        fev[i] = torch.cuda.Event()
        fev[i].record(tm.main)
        losses[0].copy_(ld_)
        losses[1].copy_(lg_)
        losses_host.copy_(losses, non_blocking=True)

    w = tm.windows(step_e2e, k4, 2, min_windows=3, min_total_s=1.0, settle_s=0.2)
    ms4e = w["ms_p50"] / k4
    rec["config4"]["e2e"] = {"samples_per_s": B * world / ms4e * 1e3, "ms_per_step": ms4e,
                             "h2d_bytes_per_step": sum(v.numel() * 4 for v in host[256].values()),
                             "d2h_bytes_per_step": 8}

    # ---- configs[4]: mixed resolutions, data parallel over `world` ranks ----
    seq_gen = torch.Generator().manual_seed(1234)
    k5 = 10
    seq = [TRAIN_RES[int(torch.randint(0, len(TRAIN_RES), (1,), generator=seq_gen))] for _ in range(k5)]
    it = {"i": 0}

    def step_mixed():
        step_at(seq[it["i"] % k5])
        it["i"] += 1

    def run_cfg5():
        it["i"] = 0
        return tm.windows(step_mixed, k5, k5, min_windows=3, min_total_s=1.5, settle_s=0.2)

    w = run_cfg5()
    ms5 = w["ms_p50"] / k5
    torch.cuda.synchronize(dev)
    ld, lg = state["last"]
    gf5 = sum(flop(s) for s in seq) / k5
    rec["config5"] = {
        "workload": f"configs[4]: data-parallel Pix2Pix training, batch {B} per GPU x {world} GPU(s), per-step resolution "
                    f"from the seeded sequence {seq} (same on every rank), bucketed NCCL all-reduce of the D and G "
                    "gradients overlapped with the backward pass",
        "ms_per_step": ms5, "samples_per_s": B * world / ms5 * 1e3, "steps_per_window": k5, "windows": w,
        "tflops": B * world * gf5 / ms5, "gflop_per_sample_mean": gf5,
        "frac_of_sustained_peak": B * gf5 / ms5 / peaks()["tf_sustained"],
        "loss_D": float(ld), "loss_G": float(lg)}
    if world > 1:
        # cost of the gradient exchange: the same windows without the collectives (ranks diverge afterwards, measurement
        # only) and the device-timed wait of the training stream for the last bucket
        rec["config5"]["allreduce_exposed_ms_per_step_last"] = trainer.exposed_exchange_ms()
        trainer.exchange = False
        w0 = run_cfg5()
        trainer.exchange = True
        rec["config5"]["ms_per_step_without_allreduce"] = w0["ms_p50"] / k5
        rec["config5"]["allreduce_exposed_ms_per_step"] = max(0.0, ms5 - w0["ms_p50"] / k5)
        rec["config5"]["nccl_buckets_per_step"] = {k: r.last_buckets for k, r in trainer.reducers.items()}
    rec["clocks"] = samplers["train"].stop() if samplers.get("train") else None
    rec["mem_gb"] = {"max_allocated": torch.cuda.max_memory_allocated(dev) / 1e9,
                     "generator_pool": model.netG._runner.pool_bytes() / 1e9,
                     "discriminator_pool": model.netD._runner.pool_bytes() / 1e9}
    rec["skipped_steps"] = [trainer.opt_d.skipped_steps, trainer.opt_g.skipped_steps]
    rec["cuda_graphs"] = bool(__import__("nirgan_b200").engine.TRAIN_GRAPHS[0])
    rec["launches_per_step_256"] = sum(c["fwd"].launches + c["bwd"].launches for r in (model.netG._runner, model.netD._runner)
                                       for k, c in r._train.items() if c["geom"][2] in (256,))
    return rec


def main():
    _quiet_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--precision", default=os.environ.get("NIRGAN_B200_PRECISION", "fp16"))
    ap.add_argument("--conv", default=os.environ.get("NIRGAN_B200_IMPL", "tc"), choices=["tc", "simt"])
    ap.add_argument("--chunk", type=int, default=int(os.environ.get("NIRGAN_B200_CHUNK", "0")))
    ap.add_argument("--batch", type=int, default=BATCH)
    ap.add_argument("--streams", type=int, default=int(os.environ.get("NIRGAN_B200_STREAMS", "0")),
                    help="batch slices run concurrently on separate CUDA streams (0 = engine default: 2 for >= 32 tiles)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-train", action="store_true", help="skip the training sub-record (configs[3] / configs[4])")
    ap.add_argument("--train-batch", type=int, default=32)
    ap.add_argument("--train-steps", type=int, default=10, help="steps per timed window of the configs[3] loop")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the NIR prediction of the last timed step to DIR/nir_pred.npy (float32, <= 64 MB)")
    ap.add_argument("--settle", type=float, default=1.0,
                    help="seconds of untimed work before the first window of a loop (clock ramp); 0 under a profiler")
    ap.add_argument("--sync-calls", action="store_true",
                    help="issue steps with net(x, e) (joins the caller's stream every step) instead of forward_async")
    ap.add_argument("--no-graph", action="store_true")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3)
    if args.impl == "reference":
        return run_reference(args)

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the hot path has no CPU fallback)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist = None
    if world > 1:
        import torch.distributed as dist_
        dist = dist_
        # stdout carries exactly one JSON line: keep NCCL's banner ("NCCL version ...") off it
        if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
            os.environ["NCCL_DEBUG"] = "WARN"
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        dist.init_process_group("nccl", device_id=dev)
    if args.no_graph:
        import nirgan_b200
        nirgan_b200.engine.GRAPHS[0] = False

    B = args.batch
    net = build_model(dev).configure_b200(precision=args.precision, impl=args.conv, chunk=args.chunk,
                                           streams=args.streams)
    g = torch.Generator().manual_seed(1 + rank)
    x_host = torch.rand(B, 3, TILE, TILE, generator=g).pin_memory()
    e_host = torch.randn(B, 256, generator=g).pin_memory()
    y_host = torch.empty(B, 1, TILE, TILE).pin_memory()
    x = x_host.to(dev)
    e = e_host.to(dev)

    # Both loops use the streaming call of the public API (``forward_async``): a step's slices queue behind the same
    # slices of the previous step on the generator's own streams, so consecutive steps overlap instead of meeting at a
    # barrier on the caller's stream; a timed window ends when its last step's results are complete.
    # (--sync-calls: the plain ``net(x, e)`` call, which joins the caller's stream after every step.)
    last_done = {"ev": [], "y": None}

    def step_resident():
        with torch.no_grad():
            if args.sync_calls:
                y = net(x, e)
            else:
                y, done = net.forward_async(x, e)
                last_done["ev"] = done
            last_done["y"] = y

    # end-to-end: every step copies its tiles + embeddings from pinned host memory and reads the NIR band back.  The
    # copies run on their own streams (double-buffered device inputs) so that step i+1's H2D and step i-1's D2H
    # overlap step i's kernels -- the way a user of the API would feed a GPU from a host-side loader.
    main_stream = torch.cuda.current_stream(dev)
    h2d_stream, d2h_stream = torch.cuda.Stream(dev), torch.cuda.Stream(dev)
    xd = [torch.empty_like(x) for _ in range(2)]
    ed = [torch.empty_like(e) for _ in range(2)]
    ev_in = [torch.cuda.Event() for _ in range(2)]
    ev_free = [[], []]
    e2e_state = {"i": 0}

    def step_e2e():
        i = e2e_state["i"]
        e2e_state["i"] = i + 1
        slot = i & 1
        with torch.no_grad():
            with torch.cuda.stream(h2d_stream):
                for ev in ev_free[slot]:
                    h2d_stream.wait_event(ev)                  # the step that last read this slot has finished
                xd[slot].copy_(x_host, non_blocking=True)
                ed[slot].copy_(e_host, non_blocking=True)
                ev_in[slot].record(h2d_stream)
            if args.sync_calls:
                main_stream.wait_event(ev_in[slot])
                y = net(xd[slot], ed[slot])
                done = [torch.cuda.Event()]
                done[0].record(main_stream)
            else:
                y, done = net.forward_async(xd[slot], ed[slot], ready=ev_in[slot])
            ev_free[slot] = done
            last_done["ev"] = done
            y.record_stream(d2h_stream)
            with torch.cuda.stream(d2h_stream):
                for ev in done:
                    d2h_stream.wait_event(ev)
                y_host.copy_(y, non_blocking=True)

    def join_last():
        for ev in last_done["ev"]:
            main_stream.wait_event(ev)                         # the last step's slices

    tm = Timing(dev, dist, main_stream, (h2d_stream, d2h_stream))
    samplers = {}
    clock_parts = {}
    # identical conditions for both loops: a clock sampler beside each, the same warm-up rule, the same window rule
    samplers["value"] = ClockSampler(local) if rank == 0 else None
    w_val = tm.windows(step_resident, args.steps, args.warmup, join=join_last, min_windows=1, min_total_s=0.0,
                       settle_s=args.settle)
    clock_parts["value"] = samplers["value"].stop() if samplers["value"] else None
    # the window ends with a device synchronize: the last step's prediction is complete
    y_last = last_done["y"].cpu() if args.dump_outputs and rank == 0 else None
    samplers["e2e"] = ClockSampler(local) if rank == 0 else None
    w_e2e = tm.windows(step_e2e, args.steps, args.warmup, join=join_last, min_windows=1, min_total_s=0.0,
                       settle_s=args.settle)
    clock_parts["e2e"] = samplers["e2e"].stop() if samplers["e2e"] else None
    ms, ms_e2e = w_val["ms_p50"], w_e2e["ms_p50"]
    # diagnostic: the host link alone (one H2D of a step's tiles from pinned memory), to read e2e against
    tm.barrier()
    c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    c0.record()
    for _ in range(3):
        xd[0].copy_(x_host, non_blocking=True)
    c1.record()
    torch.cuda.synchronize(dev)
    h2d_gbs = 3 * x_host.numel() * 4 / (c0.elapsed_time(c1) * 1e-3) / 1e9

    # ---- per-kernel device times over the same steps (CUDA events on the launching stream) ----
    runner = net._runner
    plan = runner.last_plan
    stream = torch.cuda.current_stream(dev).cuda_stream
    per_op = {}
    nprof = max(3, min(args.steps, 10))
    for it in range(nprof):
        evs = [torch.cuda.Event(enable_timing=True) for _ in range(len(plan.ops) + 1)]
        evs[0].record()
        for i, (fn, a, name) in enumerate(plan.ops):
            fn(*a, stream)
            evs[i + 1].record()
        torch.cuda.synchronize(dev)
        for i, (fn, a, name) in enumerate(plan.ops):
            per_op.setdefault(i, []).append(evs[i].elapsed_time(evs[i + 1]))
    op_ms = {i: sum(v) / len(v) for i, v in per_op.items()}
    by_name = {}
    for i, (fn, a, name) in enumerate(plan.ops):
        by_name.setdefault(name, []).append(op_ms[i])
    # dominant kernel: the 18 ResnetBlock 3x3 convs (256->256 at H/4): 4.832 GFLOP per tile per launch
    import re
    conv_idx = [i for i, (fn, a, name) in enumerate(plan.ops) if name in ("ng_conv2d", "ng_stem_conv", "ng_head_conv")]
    res_idx = [i for i in conv_idx if re.search(r"\.r\d+[ab]$", plan.labels[i])]
    assert len(res_idx) == 18, [plan.labels[i] for i in conv_idx]
    Bc = plan.records["src"].numel() // (3 * TILE * TILE)      # tiles per plan run (batch slice)

    # average launch duration of one kernel family: its launches of a step back to back between ONE pair of events
    # (a pair of events around every single launch adds the event + launch gap, ~10 % of a 30 us kernel)
    def grouped_ms(indices):
        # replayed as a CUDA graph, the way the product launches them (Plan.run_graphed): launch gaps of ~1 us
        gr = torch.cuda.CUDAGraph()
        with torch.cuda.graph(gr, capture_error_mode="thread_local"):
            cs = torch.cuda.current_stream(dev).cuda_stream
            for i in indices:
                fn, a, _ = plan.ops[i]
                fn(*a, cs)
        reps = []
        for _ in range(nprof + 1):
            g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            g0.record()
            gr.replay()
            g1.record()
            torch.cuda.synchronize(dev)
            reps.append(g0.elapsed_time(g1))
        reps = sorted(reps[1:])
        return reps[len(reps) // 2]

    res_ms = grouped_ms(res_idx) / len(res_idx)
    res_flop = 2.0 * Bc * (TILE // 4) ** 2 * 256 * 256 * 9
    pk = peaks()
    achieved = res_flop / (res_ms * 1e-3) / 1e12
    share = sum(op_ms[i] for i in res_idx) / sum(op_ms.values())
    small_idx = [i for i in conv_idx if i not in res_idx]
    small_ms = grouped_ms(small_idx)

    # HBM-bound companion: the fused InstanceNorm-apply launches; algorithmic bytes from their own arguments
    # (read y [+ residual], write the haloed output; 16-bit elements) -- DESIGN.md section 3.3
    esz = 4 if args.precision == "fp32" else 2
    ap_bytes = 0.0
    for i, (fn, a, name) in enumerate(plan.ops):
        if name != "ng_in_apply":
            continue
        _, _, b_, h_, w_, c_ = a[:6]
        res_, opad = a[11], a[17]
        ap_bytes += b_ * c_ * esz * (h_ * w_ * (2 if res_ else 1) + (h_ + 2 * opad) * (w_ + 2 * opad))
    ap_idx = [i for i, (fn, a, name) in enumerate(plan.ops) if name == "ng_in_apply"]
    ap_ms = grouped_ms(ap_idx)
    hbm_achieved = ap_bytes / (ap_ms * 1e-3) / 1e9 if ap_ms > 0 else 0.0
    plan_launches = plan.launches

    # ---- training sub-record ----
    train = None
    if not args.no_train:
        try:
            train = train_record(args, dev, rank, world, dist, tm, samplers)
            clock_parts["train"] = train.pop("clocks", None)
        except Exception as ex:           # the headline must still be printed; the failure is part of the record
            import traceback
            traceback.print_exc()
            train = {"error": f"{type(ex).__name__}: {ex}"}
            if samplers.get("train"):
                samplers["train"].stop()

    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return

    tiles_per_window = B * world * args.steps
    value = tiles_per_window / (ms * 1e-3)
    e2e = tiles_per_window / (ms_e2e * 1e-3)
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import nirgan_oracle as O
    gflop_tile = O.g_forward_gflop(TILE, TILE) + 2 * 256 * 16384 / 1e9
    # dram__bytes_read.sum + dram__bytes_write.sum of the dominant kernel from the committed `ncu --set full` capture
    traffic, traffic_src = None, None
    tpath = os.path.join(ROOT, "profiles", "roofline_traffic.json")
    if os.path.exists(tpath):
        tj = json.load(open(tpath))
        traffic = tj["dram_bytes_per_launch"] * Bc / tj["tiles_per_launch"]
        traffic_src = tj["source"]
    checks = {"value_ge_0p97_e2e": bool(value >= 0.97 * e2e),
              "value_over_e2e": value / e2e,
              "value_spread_p90_over_p10": w_val["ms_p90"] / w_val["ms_p10"],
              "e2e_spread_p90_over_p10": w_e2e["ms_p90"] / w_e2e["ms_p10"]}
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": args.precision if args.precision != "fp32" else "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD if B == BATCH else WORKLOAD.replace("64x", f"{B}x"),
                   "global_batch": B * world, "tile": TILE, "parallelism": f"tile-sharded x{world}, no collective",
                   "conv_impl": args.conv, "operands": args.precision + " operands, fp32 accumulate (TMEM)",
                   "chunk": Bc, "streams": B // Bc if args.chunk <= 0 else args.streams,
                   "timing": "one window of exactly `steps` steps after the warm-up (barrier + synchronize around the "
                             "window, CUDA events on the launching stream, max over ranks)",
                   "l2": "every layer's tensors (hundreds of MB per 32-tile slice) exceed the 126 MB L2; no explicit flush",
                   "inference_buffers_gb": runner.inference_bytes() / 1e9},
        "windows": {"value": w_val, "e2e": w_e2e},
        "checks": checks,
        "e2e": {"value": e2e, "unit": UNIT, "h2d_bytes_per_step": x_host.numel() * 4 + e_host.numel() * 4,
                "d2h_bytes_per_step": y_host.numel() * 4, "ms_per_step": ms_e2e / args.steps,
                "h2d_link_gbs_measured": h2d_gbs,
                "pipelining": "double-buffered H2D / D2H on copy streams overlap the kernels of neighbouring steps; steps issued with forward_async (slices of consecutive steps overlap)"},
        "gpu_launches": plan_launches * (B // Bc) * args.steps,
        "clocks": merge_clocks(clock_parts),
        "roofline": {"bound": "tensor", "kernel": "conv_tc_kernel<256,64> (ResnetBlock 3x3, 256->256)",
                     "achieved": achieved, "peak": pk["tf_sustained"], "unit": "TFLOP/s",
                     "frac": achieved / pk["tf_sustained"], "frac_of_burst_peak": achieved / pk["tf_burst"],
                     "traffic": traffic, "traffic_source": traffic_src,
                     "ms_per_launch": res_ms, "flop_per_launch": res_flop, "share_of_step": share,
                     "timing": "the kernel's launches of a step slice replayed as one CUDA graph between one CUDA-event pair, median of repeats",
                     "peak_source": pk["src"] + " (sustained bf16; fp16/bf16 share one tcgen05 rate)"},
        "roofline_hbm": {"bound": "hbm", "kernel": "in_apply_kernel (InstanceNorm + inject + act + residual + halo; all launches of a step)",
                         "achieved": hbm_achieved, "peak": pk["hbm_gbs"], "unit": "GB/s", "frac": hbm_achieved / pk["hbm_gbs"],
                         "bytes_per_step_slice": ap_bytes, "ms_per_step_slice": ap_ms, "peak_source": pk["src"]},
        "small_convs": {"kernels": "stem, down x2, up x2, fused head (the non-ResnetBlock convolutions)",
                        "ms_per_step_slice": small_ms,
                        "tflops": (gflop_tile - 18 * 4.832) * Bc / small_ms if small_ms > 0 else None},
        "model_tflops": value * gflop_tile / 1e3,
        "model_frac_of_sustained_peak": value * gflop_tile / 1e3 / (pk["tf_sustained"] * world),
        "op_ms": {k: round(sum(v), 4) for k, v in by_name.items()},
        "train": train,
    }
    if os.path.isdir(os.path.join(ROOT, "gpurun_out")):
        with open(os.path.join(ROOT, "gpurun_out", "op_times.json"), "w") as f:
            json.dump([{"op": name, "label": plan.labels[i], "ms": round(op_ms[i], 5)}
                       for i, (fn, a, name) in enumerate(plan.ops)], f, indent=0)
    if not args.no_cpu_baseline:
        v, cores, sample, kind = cpu_oracle_tiles_per_sec()
        line["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample}
    if y_last is not None:
        import numpy as np
        tile_bytes = y_last[0].numel() * 4
        n = min(y_last.shape[0], DUMP_LIMIT_BYTES // tile_bytes)
        os.makedirs(args.dump_outputs, exist_ok=True)
        np.save(os.path.join(args.dump_outputs, "nir_pred.npy"), y_last[:n].float().numpy())
    emit(line)
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
