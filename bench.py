#!/usr/bin/env python
"""bench.py -- rendered views/sec, rasterizer forward+backward @256x256, 3 Gaussians/pixel.

Workload = BASELINE.json configs[1]: 2 context views -> 1 target view, 256x256, P = 393 216
Gaussians, SH degree 4, synthetic re10k-like scenes (pixelsplat_b200/synthetic.py).  A "step" is
one forward + backward of the rasterizer hot path over one batch of `--views` target views of one
scene (default 1, exactly configs[1]).

  value     : whole-job views/s, inputs resident in HBM, K steps back to back between two CUDA
              events (a pool of scenes larger than L2 is cycled, so no step re-reads a hot L2).
  e2e       : same metric through the reference-facing `render_cuda` call with HOST (pinned)
              buffers: per step H2D of every input, forward, backward, D2H of the image and of a
              gradient checksum -- all inside the timed region.
  roofline  : the dominant kernel (found live with the library's per-stage CUDA events).
  cpu_baseline : the pure-PyTorch CPU oracle (oracle/raster_torch.py, kind "port") on one view.
  --impl reference : the reference arm.  The reference's own rasterizer is an un-vendored CUDA
              dependency that cannot be installed offline, so this arm times the CPU restatement
              (the "pure-PyTorch CPU composite" BASELINE.json names), kind "port".

Multi-GPU: replicas only (the rasterizer has no trainable parameters, so there is no gradient
all-reduce on this path); ranks render disjoint scenes, time is the max over ranks.

--dump-outputs DIR writes what the last timed step returned (rank 0) as DIR/<name>.npy, float32, so
that two builds run with the same arguments (hence the same seeded inputs) can be compared output for
output: `image` [1, V, 3, H, W] whole, and `grad_<input>` for each Gaussian input, at a fixed seeded
sample of Gaussians (dump_rows) that keeps the files under 64 MB.
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

METRIC = "rendered views/sec fwd+bwd @256x256, 3 gauss/px"
WORKLOAD = ("configs[1]: re10k-like 2-view -> 1 target, 256x256, 3 gauss/px, batch 1, rasterizer fwd+bwd "
            "(SH degree 4)")          # the SAME string in both arms (driver's same_config check)
ISSUE_PEAK = 148 * 4 * 1.965e9        # warp instructions / s: SMs x schedulers x max SM clock
UNIT = "views/s"
IMAGE = (256, 256)
STAGES = ["preprocess", "count_scan_scatter", "tile_sort", "composite_fwd", "grad_zero_fill",
          "composite_bwd", "preprocess_bwd"]


def peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        return json.loads(p.read_text()), "measured"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0}, "fallback"


def csrc_sha() -> str:
    """Hash of the CUDA sources the library is built from (same function as tools/summarize_launches.py)."""
    import hashlib
    root = ROOT / "pixelsplat_b200" / "csrc"
    h = hashlib.sha1()
    for f in sorted(list(root.glob("*.cu")) + list(root.glob("*.cuh")) + [root / "Makefile"]):
        h.update(f.name.encode() + b"\0" + f.read_bytes())
    return h.hexdigest()[:16]


def kernel_profile():
    """(per-kernel ncu metrics of this build | None, provenance note)."""
    p = ROOT / "profiles" / "kernel_metrics_V1.json"
    if not p.exists():
        return None, "profiles/kernel_metrics_V1.json absent: traffic / issue_frac not reported"
    data = json.loads(p.read_text())
    if data.get("csrc_sha") != csrc_sha():
        return None, (f"profiles/kernel_metrics_V1.json was captured from other CUDA sources "
                      f"({data.get('csrc_sha')} != {csrc_sha()}): ignored")
    return data, f"profiles/kernel_metrics_V1.json (ncu launch list {data.get('source')}, same CUDA sources {data['csrc_sha']})"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region."""

    def __init__(self, index: int):
        self.rows, self.proc, self.index = [], None, index

    def __enter__(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "50",
                 "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.monotonic(), [c.strip() for c in line.split(",")]))

    def count_between(self, t0: float, t1: float) -> int:
        return sum(1 for t, _ in self.rows if t0 <= t <= t1)

    def __exit__(self, *exc):
        if self.proc is not None:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except subprocess.TimeoutExpired:
                self.proc.kill()

    def summary(self, t0: float = float("-inf"), t1: float = float("inf"), window: str = "timed region"):
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for t, r in self.rows:
            if not (t0 <= t <= t1):
                continue
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
            except (ValueError, IndexError):
                continue
            for n, v in zip(names, r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0, "window": window}
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(mx), "reasons": sorted(reasons),
                "samples": len(sm), "window": window}


CONTEXT_VIEWS = 2


def make_scene(seed: int, views: int):
    from pixelsplat_b200 import synthetic
    return synthetic.scene_re10k_like(seed=seed, image_hw=IMAGE, context_views=CONTEXT_VIEWS,
                                      gaussians_per_pixel=3, sh_degree=4, target_views=views)


def scene_host_tensors(sc, pin: bool):
    t = dict(extrinsics=sc.extrinsics, intrinsics=sc.intrinsics, near=sc.near, far=sc.far,
             means=sc.means[None], covariances=sc.covariances[None], harmonics=sc.harmonics[None],
             opacities=sc.opacities[None])
    t = {k: v.contiguous().float() for k, v in t.items()}
    return {k: (v.pin_memory() if pin else v) for k, v in t.items()}


GAUSS_KEYS = ("means", "covariances", "harmonics", "opacities")


def render_step(d, d_img, views, state_out=None):
    """One forward + backward of the hot path through the public API; returns (image, grads)."""
    from pixelsplat_b200.decoder import render_views
    leaves = [d[k] for k in GAUSS_KEYS]
    bg = torch.zeros((1, views, 3), device=d["means"].device)
    img = render_views(d["extrinsics"][None], d["intrinsics"][None], d["near"][None], d["far"][None],
                       IMAGE, bg, *leaves, state_out=state_out)
    grads = torch.autograd.grad(img, leaves, d_img)
    return img, grads


DUMP_GAUSSIANS = 65536          # gradient rows written by --dump-outputs (1/6 of configs[1]'s Gaussians)
DUMP_LIMIT = 64 * 10**6         # bytes


def dump_rows(P: int) -> torch.Tensor:
    """The Gaussians whose gradients --dump-outputs writes: a fixed seeded sample, in ascending order."""
    g = torch.Generator().manual_seed(0)
    return torch.randperm(P, generator=g)[:DUMP_GAUSSIANS].sort().values


def step_outputs(img, grads, rows) -> dict:
    """Host float32 copies of what one step returns to its caller: the image whole, and the gradient of each
    Gaussian input at `rows` (axis 1 is the Gaussian axis of every input)."""
    out = {"image": img.detach()}
    for k, gr in zip(GAUSS_KEYS, grads):
        out["grad_" + k] = gr.index_select(1, rows.to(gr.device))
    return {k: v.float().cpu().numpy() for k, v in out.items()}


def capture_step(d, d_img, views):
    """The same step captured once into a CUDA graph (inputs are the scene's resident tensors)."""
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(2):
            render_step(d, d_img, views)
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    graph, states = torch.cuda.CUDAGraph(), []
    with torch.cuda.graph(graph):
        out = render_step(d, d_img, views, state_out=states)
    return graph, out, states


def algorithmic_bytes(P, M, N, vis, HW, cov_floats=9):
    """Per-view algorithmic HBM bytes of each timed stage (DESIGN.md section 5)."""
    return {
        "preprocess": P * (12 + 4 * cov_floats + 4 + 4) + vis * 41,        # k_preprocess (k_sh_color overlaps binning)
        "count_scan_scatter": P * 4 + vis * (8 + 4) + N * 8,
        "tile_sort": N * 16 + vis * (12 * M + 12 + 17),                     # sort + the concurrent k_sh_color
        "composite_fwd": N * (8 + 8 + 16 + 16) + HW * 20,
        "grad_zero_fill": P * 40,
        "composite_bwd": N * (8 + 8 + 16 + 16) + N * 36 + HW * 20,
        "preprocess_bwd": vis * (52 + 40 + 12 * M) + vis * (52 + 12 * M),
    }


def build_roofline(stage_ms: dict, V: int, P: int, N: float, vis: float, HW: int, standard_workload: bool) -> dict:
    """The `roofline` object of the bench line for the stage the live per-stage CUDA events found dominant.
    Pure function of its arguments + profiles/kernel_metrics_V1.json + MEASURED_PEAKS.json (unit-tested on the CPU:
    tests/test_abi_cpu.py)."""
    ab = algorithmic_bytes(P, 25, N, vis, HW)
    dom = max(stage_ms, key=stage_ms.get)
    pk, pk_kind = peaks()
    achieved = V * ab[dom] / (stage_ms[dom] * 1e-3) / 1e9
    # Measured-by-ncu properties of the stage's kernel -- DRAM bytes and warp instructions per launch -- come
    # from profiles/kernel_metrics_V1.json, written by tools/summarize_launches.py from an ncu launch list of
    # THIS build (the file carries a hash of the CUDA sources; a stale file is ignored, never a literal here).
    kern = {"composite_bwd": "k_composite_bwd2", "composite_fwd": "k_composite_fwd2",
            "preprocess_bwd": "k_preprocess_bwd", "tile_sort": "k_tile_sort", "preprocess": "k_preprocess",
            "count_scan_scatter": "k_scatter"}.get(dom)
    if os.environ.get("PIXELSPLAT_B200_COMPOSITE", "") == "1" and kern:
        kern = kern.replace("2", "")
    prof, prof_note = kernel_profile()
    kp = prof.get(kern) if (prof and standard_workload and kern) else None
    if not (isinstance(kp, dict) and "warp_inst" in kp and "dram_bytes" in kp):
        kp = None
    traffic = kp["dram_bytes"] if kp else None
    issue_frac = (kp["warp_inst"] / (stage_ms[dom] * 1e-3) / ISSUE_PEAK) if kp else None
    hbm_frac = achieved / pk["hbm_gbs"]
    bound = "issue" if (issue_frac is not None and issue_frac > hbm_frac) else "hbm"
    return {"kernel": dom, "bound": bound, "achieved": achieved, "peak": pk["hbm_gbs"],
            "unit": "GB/s", "frac": hbm_frac, "traffic": traffic,
            "issue_frac": issue_frac,
            "issue": None if kp is None else {
                "warp_inst_per_launch": kp["warp_inst"], "peak_warp_inst_per_s": ISSUE_PEAK,
                "achieved_warp_inst_per_s": kp["warp_inst"] / (stage_ms[dom] * 1e-3),
                "warps_active_pct": kp.get("warps_active_pct")},
            "profile": prof_note,
            "note": "the composite is SIMT fp32 work on L2-resident gathers: its DRAM traffic is at or below the "
                    "algorithmic bytes (no re-reads) and what bounds it is instruction issue, so `frac` (HBM) is "
                    "small by construction and `issue_frac` (warp instructions / s over SMs x 4 x clock) is the "
                    "roofline that moves; see profiles/README.md",
            "peak_source": f"{pk_kind} (MEASURED_PEAKS.json hbm_gbs, burst copy)",
            "algorithmic_bytes_per_launch": V * ab[dom], "avg_launch_ms": stage_ms[dom],
            "pair_evals_per_s": (V * N * 256 / (stage_ms[dom] * 1e-3) if dom.startswith("composite") else None),
            "all_stages_gbs": {s: V * ab[s] / (stage_ms[s] * 1e-3) / 1e9 for s in STAGES if stage_ms[s] > 0}}


def cpu_threads() -> int:
    """Threads used for the CPU arm: the oracle's per-tile tensors are small (256 x ~1.5k), and
    on a 128-core host torch's intra-op pool over-subscribes badly (measured: 325 s per view with
    128 threads vs 9 s with 8), so the pool is capped at 8."""
    return min(os.cpu_count() or 1, 8)


def cpu_baseline_sample(threads: int, seed: int = 0):
    """The pure-PyTorch CPU oracle, forward + backward of ONE configs[1] view."""
    from oracle import raster_torch as rt
    torch.set_num_threads(threads)
    sc = make_scene(seed, 1)
    a = rt.prepare_view(sc.means, sc.covariances, sc.harmonics, sc.opacities, sc.extrinsics[0],
                        sc.intrinsics[0], sc.near[0], sc.far[0])
    leaves = {k: a[k].clone().requires_grad_(True) for k in ("means", "cov6", "opac", "sh")}
    g = torch.Generator().manual_seed(1)
    d_img = torch.randn(3, *IMAGE, generator=g)
    t0 = time.perf_counter()
    color, _ = rt.rasterize(leaves["means"], leaves["cov6"], leaves["opac"], leaves["sh"], None,
                            a["vm"], a["pm"], a["campos"], a["tanfovx"], a["tanfovy"], torch.zeros(3),
                            IMAGE[1], IMAGE[0], a["sh_degree"])
    (color * d_img).sum().backward()
    return time.perf_counter() - t0


def run_reference(args, rank, world):
    if rank != 0:
        return
    threads = cpu_threads()
    times = []
    for i in range(args.warmup + args.steps):
        dt = cpu_baseline_sample(threads, seed=i)
        if i >= args.warmup:
            times.append(dt)
    total = sum(times)
    value = len(times) / total
    sample = (f"{len(times)} timed steps, each 1 view of configs[1] (256x256, P=393216), fwd+bwd, "
              f"pure-PyTorch CPU oracle (oracle/raster_torch.py)")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": len(times), "warmup": args.warmup, "ms_per_step": 1e3 * total / len(times),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic",
        "config": {"workload": WORKLOAD, "views_per_step": 1},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port",
                         "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "note": "the reference's CUDA rasterizer (diff-gaussian-rasterization-modified) is an "
                "un-vendored dependency that cannot be installed offline; this arm is the CPU "
                "restatement (kind=port), not the reference's CUDA path",
    }
    emit(line)


_RESULT_OUT = None


def isolate_stdout():
    """stdout must carry exactly one JSON line.  Libraries write to file descriptor 1 behind Python's back
    (NCCL prints its version banner there at NCCL_DEBUG=VERSION / WARN), so keep a private duplicate of the
    real stdout for the result line and point fd 1 at stderr for everything else."""
    global _RESULT_OUT
    if _RESULT_OUT is None:
        sys.stdout.flush()
        _RESULT_OUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)


def emit(line: dict):
    out = _RESULT_OUT if _RESULT_OUT is not None else sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def main():
    isolate_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None, help="timed steps (default 400; 2 with --impl reference)")
    ap.add_argument("--warmup", type=int, default=None, help="warm-up steps (default 10; 1 with --impl reference)")
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--views", type=int, default=1, help="target views per step (one scene)")
    ap.add_argument("--pool", type=int, default=4, help="distinct scenes cycled (> L2 in total)")
    ap.add_argument("--streams", type=int, default=4, help="extra leg: steps issued over N streams")
    ap.add_argument("--image", type=int, default=256, help="square image size (512 with --context-views 3 = configs[4])")
    ap.add_argument("--context-views", type=int, default=2)
    ap.add_argument("--batched-views", type=int, default=4, help="extra leg: V target views per call")
    ap.add_argument("--no-graph", action="store_true", help="issue every step from Python instead of replaying a CUDA graph")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the last timed step's outputs to DIR/<name>.npy (see the module docstring)")
    args = ap.parse_args()
    reference = args.impl == "reference"
    if args.steps is None:
        args.steps = 2 if reference else 400
    if args.warmup is None:
        args.warmup = 1 if reference else 10
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and reference:
        ap.error("--dump-outputs writes the native path's outputs; it does not apply to --impl reference")
    global IMAGE, CONTEXT_VIEWS
    IMAGE, CONTEXT_VIEWS = (args.image, args.image), args.context_views
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if reference:
        run_reference(args, rank, world)
        return
    if args.warmup < 3:
        args.warmup = 3
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: pixelsplat_b200 has no CPU path "
                         "(use --impl reference for the CPU arm)")
    import torch.distributed as dist
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        # (NCCL's version banner goes to fd 1: see isolate_stdout)
        dist.init_process_group("nccl", device_id=dev)

    from pixelsplat_b200 import _lib, rasterizer
    from pixelsplat_b200.decoder import render_views  # noqa: F401  (loads the CUDA library)

    K, W_, V = args.steps, args.warmup, args.views
    pool_host = [scene_host_tensors(make_scene(1000 * rank + i, V), pin=True) for i in range(args.pool)]
    P = pool_host[0]["means"].shape[1]
    pool_dev = []
    for h in pool_host:
        d = {k: v.to(dev) for k, v in h.items()}
        for k in GAUSS_KEYS:
            d[k].requires_grad_(True)
        pool_dev.append(d)
    g = torch.Generator(device="cpu").manual_seed(7)
    d_img = torch.randn((1, V, 3, *IMAGE), generator=g).to(dev)
    rows = None
    if args.dump_outputs:               # checked on every rank: all ranks have the same shapes, so all stop together
        rows = dump_rows(P)
        dump_bytes = 4 * (d_img.numel() + len(rows) * sum(pool_dev[0][k][0, 0].numel() for k in GAUSS_KEYS))
        if dump_bytes > DUMP_LIMIT:
            raise SystemExit(f"--dump-outputs: {dump_bytes / 1e6:.0f} MB of outputs at this size, over "
                             f"{DUMP_LIMIT / 1e6:.0f} MB (the image is written whole)")

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---------------- value: device-resident inputs, K steps back to back
    rasterizer.set_capacity_check("sync")
    for i in range(W_):
        render_step(pool_dev[i % args.pool], d_img, V)
    rasterizer.set_capacity_check("deferred")   # capacity known from warm-up; verified at backward
    for i in range(W_):
        render_step(pool_dev[i % args.pool], d_img, V)
    barrier()
    # the step is launch-bound from Python (~0.4 ms of host work for ~0.4 ms of kernels), so each
    # scene's forward+backward is captured once into a CUDA graph and replayed
    graphs = None
    if not args.no_graph:
        l0 = _lib.lib.ps_launch_count()
        graphs = [capture_step(d, d_img, V) for d in pool_dev]
        launches_per_step = (_lib.lib.ps_launch_count() - l0) // (3 * len(pool_dev))
        for i in range(W_):
            graphs[i % args.pool][0].replay()
    barrier()
    launches0 = _lib.lib.ps_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    def run_steps(n):
        """Runs n steps; returns the (image, gradients) of the last."""
        if graphs is not None:
            for i in range(n):
                graphs[i % args.pool][0].replay()
            return graphs[(n - 1) % args.pool][1]
        for i in range(n):
            out = render_step(pool_dev[i % args.pool], d_img, V)
        return out

    with ClockSampler(local_rank) as clk:
        barrier()
        t_begin = time.monotonic()
        e0.record()
        last = run_steps(K)
        e1.record()
        barrier()
        t_end = time.monotonic()
        launches_timed = _lib.lib.ps_launch_count() - launches0
        # read now: the steps below replay the same graphs and overwrite their outputs
        outputs = step_outputs(*last, rows) if (rows is not None and rank == 0) else None
        clock_window = "timed region"
        if clk.proc is not None and clk.count_between(t_begin, t_end) < 3:
            # the timed region is shorter than a few nvidia-smi sampling periods: keep the SAME load running,
            # untimed, until the sampler has seen it (at most ~1 s), and say so
            t_c = time.monotonic()
            while time.monotonic() - t_c < 1.0 and clk.count_between(t_begin, time.monotonic()) < 6:
                run_steps(min(K, 100))
                torch.cuda.synchronize()
            t_end = time.monotonic()
            clock_window = "timed region + identical untimed continuation (timed region shorter than the sampling period)"
        clocks = clk.summary(t_begin, t_end, clock_window)
    ms_total = e0.elapsed_time(e1)
    launches = (launches_per_step * K) if graphs is not None else launches_timed
    if graphs is not None:
        for _, _, states in graphs:      # capacity check of the replayed forwards (count is in pinned memory)
            for st_ in states:
                st_.verify()
    if world > 1:
        t = torch.tensor([ms_total], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_total = float(t.item())
    value = world * K * V / (ms_total * 1e-3)

    # ---------------- extra: the same steps issued round-robin on several CUDA streams.  A single
    # 256x256 view is only 2048 warps (0.3 waves of the composite grid), so independent scenes
    # overlap well; reported separately because configs[1] is batch 1, strictly sequential.
    concurrent = None
    if args.streams > 1:
        streams = [torch.cuda.Stream(dev) for _ in range(args.streams)]
        def run(n):
            for i in range(n):
                with torch.cuda.stream(streams[i % args.streams]):
                    if graphs is not None:
                        graphs[i % args.pool][0].replay()
                    else:
                        render_step(pool_dev[i % args.pool], d_img, V)
        for st_ in streams:
            st_.wait_stream(torch.cuda.current_stream())
        run(W_)
        barrier()
        t0 = time.perf_counter()
        run(K)
        barrier()
        dtc = time.perf_counter() - t0
        concurrent = {"streams": args.streams, "value": world * K * V / dtc, "unit": UNIT,
                      "how": "wall clock, steps round-robin over CUDA streams, same pool of scenes"}

    # ---------------- extra: the training shape -- 4 target views of one scene share its Gaussians
    # in ONE call (V cameras per Gaussian set; the reference repeats every Gaussian tensor per
    # view, decoder_splatting_cuda.py:53-56).  Reported separately; configs[1] is 1 view per step.
    batched = None
    if args.batched_views > 1 and not args.no_graph:
        Vb = args.batched_views
        hb = scene_host_tensors(make_scene(1000 * rank + 500, Vb), pin=False)
        db = {k: v.to(dev) for k, v in hb.items()}
        for k in GAUSS_KEYS:
            db[k].requires_grad_(True)
        d_img_b = torch.randn((1, Vb, 3, *IMAGE), generator=g).to(dev)
        rasterizer.set_capacity_check("sync")
        render_step(db, d_img_b, Vb)
        rasterizer.set_capacity_check("deferred")
        gb, _, states_b = capture_step(db, d_img_b, Vb)
        for _ in range(W_):
            gb.replay()
        barrier()
        b0, b1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        nb = max(K // Vb, 10)
        b0.record()
        for _ in range(nb):
            gb.replay()
        b1.record()
        barrier()
        for st_ in states_b:
            st_.verify()
        batched = {"views_per_call": Vb, "value": world * nb * Vb / (b0.elapsed_time(b1) * 1e-3), "unit": UNIT,
                   "how": "one scene, V target cameras sharing its Gaussians in a single forward+backward"}

    # ---------------- e2e: host buffers, H2D + fwd + bwd + D2H per step, prefetch on a side stream
    e2e = None
    if not args.no_e2e:
        copy_stream = torch.cuda.Stream(dev)
        img_host = torch.empty((1, V, 3, *IMAGE), dtype=torch.float32).pin_memory()
        chk_host = torch.empty((1,), dtype=torch.float32).pin_memory()
        h2d_bytes = sum(v.numel() * 4 for v in pool_host[0].values())
        d2h_bytes = img_host.numel() * 4 + 4

        # two device-resident input sets, allocated ONCE and refilled by H2D copies on a side stream while the
        # other set is being rendered (no per-step device allocations); a set is reused only after the step
        # that read it has finished (event), so the copy never races the kernels
        bufs = []
        for _ in range(2):
            d = {k: torch.empty_like(v, device=dev) for k, v in pool_host[0].items()}
            for k in GAUSS_KEYS:
                d[k].requires_grad_(True)
            bufs.append({"d": d, "ready": torch.cuda.Event(), "free": torch.cuda.Event()})
            bufs[-1]["free"].record(torch.cuda.current_stream())

        def upload(h, slot):
            b = bufs[slot]
            with torch.cuda.stream(copy_stream), torch.no_grad():
                copy_stream.wait_event(b["free"])
                for k, v in h.items():
                    b["d"][k].copy_(v, non_blocking=True)
                b["ready"].record(copy_stream)

        def e2e_loop(n):
            upload(pool_host[0], 0)
            for i in range(n):
                b = bufs[i & 1]
                if i + 1 < n:
                    upload(pool_host[(i + 1) % args.pool], (i + 1) & 1)
                cur = torch.cuda.current_stream()
                cur.wait_event(b["ready"])
                img, grads = render_step(b["d"], d_img, V)
                img_host.copy_(img.detach(), non_blocking=True)
                chk_host.copy_(sum(gr.sum() for gr in grads).reshape(1), non_blocking=True)
                b["free"].record(cur)
            torch.cuda.current_stream().synchronize()

        e2e_loop(W_)
        barrier()
        # the timed loop runs at least one second (a 20-step loop is ~50 ms: start-up effects and the host
        # allocator dominate it), K steps at a time
        Ke, dt = 0, 0.0
        t0 = time.perf_counter()
        while True:
            e2e_loop(K)
            Ke += K
            dt = time.perf_counter() - t0
            if dt >= 1.0 or Ke >= 100 * K:
                break
        barrier()
        dt = time.perf_counter() - t0
        if world > 1:
            t = torch.tensor([dt], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dt = float(t.item())
        e2e = {"value": world * Ke * V / dt, "unit": UNIT, "h2d_bytes_per_step": h2d_bytes,
               "d2h_bytes_per_step": d2h_bytes, "steps": Ke, "seconds": dt,
               "how": "render_views(...) public API on pinned host inputs; H2D into two reused device buffer sets, "
                      "prefetched on a side stream; image + gradient checksum read back every step; wall clock over "
                      ">= 1 s of steps, max over ranks"}

    # ---------------- roofline: per-stage CUDA events inside the library
    roofline, stage_ms, stats = None, None, None
    if rank == 0:
        rasterizer.set_capacity_check("sync")
        _lib.lib.ps_timing_enable(1)
        acc = [0.0] * 7
        buf = (ctypes.c_float * 7)()
        n_prof = min(K, 20)
        states = []
        for i in range(n_prof):
            render_step(pool_dev[i % args.pool], d_img, V)
            _lib.check(_lib.lib.ps_timing_read(buf), "ps_timing_read")
            for j in range(7):
                acc[j] += buf[j]
        _lib.lib.ps_timing_enable(0)
        stage_ms = {s: acc[j] / n_prof for j, s in enumerate(STAGES)}
        # workload statistics (N, visible) from one more forward
        from pixelsplat_b200.decoder import render_views as rv
        d = pool_dev[0]
        rv(d["extrinsics"][None], d["intrinsics"][None], d["near"][None], d["far"][None], IMAGE,
           torch.zeros((1, V, 3), device=dev), *[d[k] for k in GAUSS_KEYS], state_out=states)
        im = states[0].intermediates()
        N = im["num_instances"] / V
        vis = float((im["radii"] > 0).sum().item()) / V
        stats = {"instances_per_view": N, "visible_per_view": vis, "gaussians": P}
        roofline = build_roofline(stage_ms, V, P, N, vis, IMAGE[0] * IMAGE[1],
                                  standard_workload=(args.image, args.context_views, V) == (256, 2, 1))
    torch.cuda.synchronize()

    # ---------------- CPU baseline (rank 0, N=1 only)
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        threads = cpu_threads()
        dt = cpu_baseline_sample(threads)
        cpu = {"value": 1.0 / dt, "unit": UNIT, "cores": threads, "kind": "port",
               "sample": "1 view of configs[1] (256x256, P=393216) forward+backward, pure-PyTorch CPU "
                         f"oracle (oracle/raster_torch.py), torch.set_num_threads({threads}), {dt:.1f} s"}

    if outputs is not None:
        out_dir = Path(args.dump_outputs)
        out_dir.mkdir(parents=True, exist_ok=True)
        for name, a in outputs.items():
            np.save(out_dir / f"{name}.npy", a)

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W_,
            "ms_per_step": ms_total / K, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD if (args.image, args.context_views) == (256, 2)
                       else f"re10k-like {args.context_views}-view -> 1 target, {args.image}x{args.image}, 3 gauss/px, "
                            "batch 1, rasterizer fwd+bwd (SH degree 4)",
                       "views_per_step": V, "gaussians": P, "parallelism": f"replicas x{world}",
                       "l2": f"pool of {args.pool} scenes ({args.pool * P * 352 // 10**6} MB of inputs) cycled: "
                             "inputs larger than L2, no flush",
                       "capacity_check": "deferred (verified at backward)",
                       "launch": "eager python" if args.no_graph else "one CUDA graph per scene (fwd+bwd), replayed"},
            "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches),
            "roofline": roofline, "cpu_baseline": cpu, "stage_ms": stage_ms, "workload_stats": stats, "throughput_concurrent_streams": concurrent, "throughput_batched_views": batched,
        }
        emit(line)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
