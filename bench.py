#!/usr/bin/env python
"""bench.py — `python bench.py --gpus N --steps K --warmup W [--impl reference] [--workload NAME] [--dump-outputs DIR]`.

Prints ONE JSON line (rank 0).  A "step" = one pass of the hot path over one batch of synthetic images per GPU; the
resident and e2e loops of every workload, sub-benchmarks included, time K steps.  `--dump-outputs DIR` writes what the last timed step of the selected workload returned (rank 0)
as DIR/<name>.npy: the same seeded inputs on every run, so two builds can be compared output for output.

Workloads (BASELINE.json configs):
  depth_beit512     dpt_beit_large_512 @512x512, batch 32/GPU, depth only            (configs[1], the default once built)
  dav2_stereo       depth_anything_v2 vitl @518 + SBS stereo (polylines) + normal map (configs[2])
  zoedepth_nk768    zoedepth_nk @768 (pad + flip TTA, 64 core forwards) + red-cyan anaglyph, batch 32/GPU (configs[3])
  stereo2048        normalise -> stereo SBS (div 2.5, polylines_sharp) -> normal map on 2048x2048, batch 16/GPU
                    (north_star's "2048x2048 stereo warp" HBM-roofline target)
The default run (depth_beit512) carries the other three as `sub_benchmarks`, so one driver run covers BASELINE's
"depth+stereo 512^2 & 2048^2"; `e2e_funnel` is the same workload through core_generation_funnel with PIL images in and out.

`value` = images/s with inputs resident in HBM; `e2e` = same through the public batched API from pinned HOST buffers,
H2D and D2H inside the timed region; `roofline` = dominant kernel vs MEASURED_PEAKS.json; `cpu_baseline` = the oracle
(C restatement of the reference's CPU path) timed on this box's host cores on a bounded sample.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np  # noqa: E402


def _peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm_gbs": d["hbm_gbs"], "bf16_tflops": d["bf16_tflops"], "bf16_tflops_sustained": d.get("bf16_tflops_sustained", d["bf16_tflops"]), "source": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, gpu_index):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "100",
                                       "-i", str(gpu_index)], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if self.p is None:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        rows = [r.strip().split(",") for r in open(self.f.name).read().strip().splitlines() if r.strip()]
        os.unlink(self.f.name)
        sm, reasons, mx = [], set(), None
        for r in rows:
            try:
                sm.append(float(r[1])); mx = float(r[2])
            except Exception:
                continue
            for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], r[5:9]):
                if "Active" in v and "Not" not in v:
                    reasons.add(name)
        if sm:
            out["sm_mhz"] = float(np.median(sm))
            out["sm_max_mhz"] = mx
        out["reasons"] = sorted(reasons)
        out["samples"] = len(sm)
        return out


# ---------------------------------------------------------------------------------------------------------------------
# synthetic data
# ---------------------------------------------------------------------------------------------------------------------
def make_images(B, H, W, rank):
    from synth import synth_depth_u16, synth_rgb
    nuniq = min(B, 4)
    rgbs = [synth_rgb(H, W, 100 * rank + i) for i in range(nuniq)]
    preds = [(synth_depth_u16(H, W, 100 * rank + i).astype(np.float32) / 1000.0 - 7.0) for i in range(nuniq)]
    rgb = np.stack([rgbs[i % nuniq] for i in range(B)])
    pred = np.stack([preds[i % nuniq] for i in range(B)])
    return rgb, pred


# ---------------------------------------------------------------------------------------------------------------------
# workload: stereo2048  (normalise -> stereo SBS -> normal map), all HBM-side kernels
# ---------------------------------------------------------------------------------------------------------------------
class Stereo2048:
    name = "stereo2048"
    H = W = 2048
    B = 16
    dtype = "f64"  # the stereo / normal-map arithmetic type (fp64, truncating to u8); normalise is f32
    fill = "polylines_sharp"
    launches_per_step = 3 + 3 + 1  # normalise (init, minmax, quantise) + stereo (init, minmax, row) + normal map
    outputs = ("depth", "stereo_sbs", "normal")

    def __init__(self, dev, rank):
        import torch
        self.dev = dev
        rgb, pred = make_images(self.B, self.H, self.W, rank)
        self.rgb_h = torch.from_numpy(rgb).pin_memory()
        self.pred_h = torch.from_numpy(pred).pin_memory()
        self.rgb = self.rgb_h.to(dev)
        self.pred = self.pred_h.to(dev)
        self.kernel_ms = []

    def config(self):
        return {"workload": "synthetic 2048x2048 RGB + float32 prediction -> u16 depth -> SBS stereo (divergence 2.5, "
                            "polylines_sharp) -> normal map (Sobel 3)", "batch_per_gpu": self.B, "height": self.H,
                "width": self.W, "l2_policy": "inputs+outputs per step (1.0 GB) exceed the 126 MB L2"}

    def step(self, rgb, pred, time_kernel=False):
        import torch
        from depthmap_b200.core import normalize_prediction_batch
        from depthmap_b200.normalmap_generation import create_normalmap_batch
        from depthmap_b200.stereoimage_generation import create_stereoimages_batch
        depth = normalize_prediction_batch(pred, False)
        if time_kernel:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
        sbs = create_stereoimages_batch(rgb, depth, 2.5, 0.0, ['left-right'], 0.0, 1.0, self.fill)[0]
        if time_kernel:
            e1.record()
            self._ev = (e0, e1)
        normal = create_normalmap_batch(depth)
        return depth, sbs, normal

    def step_resident(self, time_kernel=False):
        return self.step(self.rgb, self.pred, time_kernel)

    def step_e2e(self):
        rgb = self.rgb_h.to(self.dev, non_blocking=True)
        pred = self.pred_h.to(self.dev, non_blocking=True)
        outs = self.step(rgb, pred)
        return [o.to("cpu", non_blocking=True) for o in outs]

    def e2e_bytes(self):
        h2d = self.rgb_h.numel() + self.pred_h.numel() * 4
        d2h = self.B * self.H * self.W * (2 + 6 + 3)
        return h2d, d2h

    def roofline(self, peaks, kernel_ms):
        alg = 11.0 * self.H * self.W * self.B  # SURVEY §8d: 3 (RGB) + 2 (depth) in, 6 (two eyes) out per pixel
        achieved = alg / (kernel_ms * 1e-3) / 1e9
        return {"bound": "hbm", "kernel": "stereo_row_kernel (+ u16 min/max pre-pass)", "achieved": achieved,
                "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": achieved / peaks["hbm_gbs"],
                # dram read + write of the row kernel for this batch (profiles/r01_ncu_stereo2048.txt): no re-reads
                "traffic": 692.5e6 if (self.B == 16 and self.fill == "polylines_sharp") else None, "traffic_unit": "bytes/launch (ncu --set full)",
                "peak_source": peaks["source"], "algorithmic_bytes_per_launch": alg, "kernel_ms": kernel_ms,
                "note": "exact-fp64 polylines is FP64/latency bound, not HBM bound; see DESIGN.md"}

    def cpu_sample(self, nthreads):
        """oracle on one 2048^2 image (normalise + stereo + normal map)."""
        from oracle import normalmap as onm
        from oracle import stereo as ost
        rgb = self.rgb_h[0].numpy()
        pred = self.pred_h[0].numpy()
        t0 = time.perf_counter()
        d = onm.normalize_to_u16(pred, False)
        ost.create_stereoimages(rgb, d, 2.5, 0.0, ['left-right'], 0.0, 1.0, self.fill, return_arrays=True, nthreads=nthreads)
        onm.create_normalmap(d, return_array=True)
        return 1, time.perf_counter() - t0


def host_threads():
    """Threads the CPU arm may really use: scheduler affinity and the cgroup CPU quota, not the machine's core count."""
    n = os.cpu_count() or 1
    try:
        n = min(n, len(os.sched_getaffinity(0)))
    except (AttributeError, OSError):
        pass
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if quota != "max":
            n = min(n, max(1, int(int(quota) / int(period))))
    except (OSError, ValueError):
        pass
    return max(1, n)


def pick_torch_threads(limit):
    """torch's intra-op pool is fastest well below the hardware thread count on big hosts (SMT siblings, NUMA): time one
    fp32 GEMM at a few pool sizes and keep the best, so the CPU arm is not handicapped by oversubscription."""
    import torch
    a = torch.randn(1536, 1536)
    best, best_t = limit, None
    for n in sorted({limit, min(limit, 64), min(limit, 32), min(limit, 16), min(limit, 8)}, reverse=True):
        torch.set_num_threads(n)
        a @ a
        t0 = time.perf_counter()
        for _ in range(3):
            a @ a
        dt = time.perf_counter() - t0
        if best_t is None or dt < best_t * 0.9:
            best, best_t = n, dt
    torch.set_num_threads(best)
    return best


class GraphedStep:
    """Captures one full step (every kernel launch of the hot path, allocations included) into a CUDA graph and replays
    it: same kernels, same work per step, without ~700 host-side launches per step.  Falls back to eager if capture fails."""

    def __init__(self, fn):
        import torch
        self.fn = fn
        self.graph = None
        self.outs = None
        try:
            s = torch.cuda.Stream()
            s.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(s):
                for _ in range(2):
                    fn()
            torch.cuda.current_stream().wait_stream(s)
            torch.cuda.synchronize()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                self.outs = fn()
            self.graph = g
        except Exception as e:  # noqa: BLE001
            sys.stderr.write(f"[bench] CUDA graph capture failed ({e}); running eagerly\n")
            torch.cuda.synchronize()
            self.graph = None

    def __call__(self):
        if self.graph is None:
            return self.fn()
        self.graph.replay()
        return self.outs


DUMP_BYTES = 64 << 20


def dump_outputs(dirname, names, outs):
    """Writes one step's outputs (CUDA tensors) as <dirname>/<name>.npy in float32 (float64 stays float64), 64 MB at most
    in all: an output larger than its even share of that is written as its values at a fixed, seeded sample of its
    flattened positions (the same positions on every run)."""
    os.makedirs(dirname, exist_ok=True)
    share = DUMP_BYTES // len(outs) - 4096                    # room for each file's .npy header
    for name, o in zip(names, outs):
        a = o.detach().cpu().numpy()
        dt = np.float64 if a.dtype == np.float64 else np.float32
        k = share // np.dtype(dt).itemsize
        if a.size > k:
            a = a.reshape(-1)[np.sort(np.random.default_rng(0).choice(a.size, k, replace=False))]
        np.save(os.path.join(dirname, f"{name}.npy"), a.astype(dt))


WORKLOADS = {"stereo2048": Stereo2048}
try:
    from bench_models import MODEL_WORKLOADS  # depth-network workloads, added once the tensor-core path is built
    WORKLOADS.update(MODEL_WORKLOADS)
except ImportError:
    pass
DEFAULT_WORKLOAD = "depth_beit512" if "depth_beit512" in WORKLOADS else ("dav2_stereo" if "dav2_stereo" in WORKLOADS else "stereo2048")


def run_reference(args, rank, world):
    """--impl reference: the reference's CPU implementation of the path (oracle port) on this box's host cores."""
    if rank != 0:
        return
    import oracle
    oracle.build()
    wl_cls = WORKLOADS[args.workload]
    wl = wl_cls.__new__(wl_cls)
    import torch
    cores = pick_torch_threads(host_threads())
    rgb, pred = make_images(1, wl_cls.H, wl_cls.W, 0)
    wl.rgb_h, wl.pred_h = torch.from_numpy(rgb), torch.from_numpy(pred)
    wl.rgb = rgb[0]                       # the single-image workloads (BOOST) keep a numpy image
    # every step is one image through the CPU path; the whole run is held to ~4 minutes: if the first (untimed) image
    # shows that warmup + steps would not fit, the step count is cut and the cut is reported in "steps"
    budget_s = float(os.environ.get("DEPTHMAP_B200_REF_BUDGET_S", "240"))
    t_start = time.perf_counter()
    warm = max(args.warmup, 1)
    per_image = None
    sample_note = None
    for _ in range(warm):
        t0 = time.perf_counter()
        res = wl.cpu_sample(cores)
        per_image = time.perf_counter() - t0            # wall time of one sample (a workload may extrapolate its figure from a part)
        if time.perf_counter() - t_start + per_image * 2 > budget_s * 0.5:
            break
    left = budget_s - (time.perf_counter() - t_start)
    steps = max(1, min(args.steps, int(left / max(per_image, 1e-6))))
    t = []
    for _ in range(steps):
        res = wl.cpu_sample(cores)
        n, dt = res[0], res[1]
        sample_note = res[2] if len(res) > 2 else None
        t.append(dt / n)
    ms = float(np.mean(t)) * 1e3
    val = 1000.0 / ms
    cfg = dict(wl_cls.config(wl))
    cfg.pop("batch_per_gpu", None)
    cfg["sample"] = "1 image per step (the reference's own loop is one image at a time, src/core.py:133)"
    sample = sample_note or ("1 image per step: fp32 torch CPU forward of the same network (oracle/ restatement of the reference module) + "
                             "oracle/ C restatement of the reference's numba / cv2 post-processing, all host threads")
    line = {"metric": "images/sec", "value": val, "unit": "images/s", "n_gpus": args.gpus, "steps": steps,
            "steps_requested": args.steps, "warmup": warm, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "fp32" if wl_cls.dtype == "fp16" else wl_cls.dtype, "data": "synthetic",
            "impl": "reference", "config": cfg,
            "cpu_baseline": {"value": val, "unit": "images/s", "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": val, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


class Gatherer:
    """The path's one exchange (north_star): ONE NCCL all-gather per batch of the finished tensors, packed into a single
    buffer, issued on a SIDE stream so that it overlaps the next batch's compute (SURVEY.md §5 / §8e).  The compute stream
    only waits for the cheap device-to-device pack of the previous batch before it overwrites the outputs."""

    def __init__(self, world, dev):
        import torch
        self.world, self.dev = world, dev
        self.side = torch.cuda.Stream(device=dev)
        self.pack = [None, None]
        self.gathered = [None, None]
        self.pack_done = [None, None]
        self.k = 0
        self.bytes_per_rank = 0

    def submit(self, outs):
        import torch
        import torch.distributed as dist
        flat = [o.reshape(-1).view(torch.uint8) if o.dtype != torch.uint8 else o.reshape(-1) for o in outs]
        total = sum(f.numel() for f in flat)
        k = self.k & 1
        if self.pack[k] is None or self.pack[k].numel() != total:
            self.pack[k] = torch.empty(total, dtype=torch.uint8, device=self.dev)
            self.gathered[k] = torch.empty(self.world * total, dtype=torch.uint8, device=self.dev)
        self.bytes_per_rank = total
        main = torch.cuda.current_stream()
        ready = torch.cuda.Event()
        ready.record(main)
        with torch.cuda.stream(self.side):
            self.side.wait_event(ready)
            off = 0
            for f in flat:
                self.pack[k][off:off + f.numel()].copy_(f, non_blocking=True)
                off += f.numel()
            done = torch.cuda.Event()
            done.record(self.side)
            dist.all_gather_into_tensor(self.gathered[k], self.pack[k])
        main.wait_event(done)            # the next batch may overwrite `outs` once they are packed; the gather itself overlaps it
        self.pack_done[k] = done
        self.k += 1
        return self.gathered[k]

    def drain(self):
        import torch
        torch.cuda.current_stream().wait_stream(self.side)


def measure(wl, args, world, dev, rank, local_rank, peaks, steps, with_cpu_baseline, with_funnel, dump_dir=None):
    """One workload: resident-input throughput, dominant-kernel roofline, host-buffer e2e (+ funnel e2e, CPU baseline).
    With `dump_dir`, rank 0 writes the outputs of the last timed step there (dump_outputs)."""
    import torch
    import torch.distributed as dist
    dump = (lambda outs: dump_outputs(dump_dir, wl.outputs, outs)) if (dump_dir and rank == 0) else None
    if hasattr(wl, "measure"):       # a workload with its own step structure (BOOST: one image, patch-parallel, strong scaling)
        return wl.measure(args, world, dev, rank, local_rank, peaks, steps, with_cpu_baseline, ClockSampler, dump)
    graphed = None
    if not args.no_graph:
        graphed = GraphedStep(lambda: wl.step_resident(False))
    gatherer = Gatherer(world, dev) if world > 1 else None

    def full_step(time_kernel=False):
        outs = wl.step_resident(True) if (time_kernel or graphed is None) else graphed()
        if gatherer is not None:
            gatherer.submit(outs)
        return outs

    for _ in range(args.warmup):
        full_step()
    if gatherer is not None:
        gatherer.drain()
    torch.cuda.synchronize()

    # ---- timed region: device-resident inputs ------------------------------------------------------------------
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    sampler = ClockSampler(local_rank) if rank == 0 else None
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        outs = full_step(time_kernel=False)
    if gatherer is not None:
        gatherer.drain()
    e1.record()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    clocks = sampler.stop() if sampler else None
    if dump is not None:
        dump(outs)
    ms_total = e0.elapsed_time(e1)
    t = torch.tensor([ms_total], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_step = float(t.item()) / steps

    # ---- dominant-kernel probe: same kernels, eager, CUDA events around the launches (events cannot be captured) ----
    roofline = None
    if rank == 0:
        if hasattr(wl, "probe"):
            roofline = wl.roofline_from_probe(peaks, wl.probe(20), ms_step)
        else:
            evs = []
            wl.step_resident(True)                      # warm the eager path (allocator) before the measured launches
            torch.cuda.synchronize()
            for _ in range(3):
                wl.step_resident(True)
                evs.append(wl._ev)
            torch.cuda.synchronize()
            roofline = wl.roofline(peaks, float(np.mean([a.elapsed_time(b) for a, b in evs])))

    # ---- e2e: host buffers, H2D + D2H inside the timed region ----------------------------------------------------
    for _ in range(2):
        wl.step_e2e()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0.record()
    for _ in range(steps):
        wl.step_e2e()
    e1.record()
    torch.cuda.synchronize()
    t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_e2e = float(t.item()) / steps
    h2d, d2h = wl.e2e_bytes()
    if rank != 0:
        return None
    value = wl.B * world / (ms_step * 1e-3)
    line = {"metric": "images/sec", "value": value, "unit": "images/s", "n_gpus": world, "steps": steps,
            "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": wl.dtype, "data": "synthetic", "config": wl.config(),
            "clocks": clocks, "gpu_launches": (wl.launches_per_step or 0) * steps,
            "launch_mode": "cuda_graph" if (graphed is not None and graphed.graph is not None) else "eager",
            "e2e": {"value": wl.B * world / (ms_e2e * 1e-3), "unit": "images/s", "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": d2h, "ms_per_step": ms_e2e,
                    "api": "public batched API (ModelHolder / create_*_batch) from pinned host buffers, H2D + D2H in the timed region"}}
    if roofline is not None:
        line["roofline"] = roofline
    if gatherer is not None:
        line["collective"] = {"backend": "nccl", "nccl_version": ".".join(str(v) for v in torch.cuda.nccl.version()),
                              "op": "all_gather_into_tensor, one per batch, packed buffer, side stream overlapped with the next batch",
                              "bytes_per_rank_per_step": gatherer.bytes_per_rank}
    if hasattr(wl, "extra"):
        line.update(wl.extra(ms_step, peaks))
    if with_funnel and world == 1 and hasattr(wl, "funnel_e2e"):
        try:
            line["e2e_funnel"] = wl.funnel_e2e(2)
        except Exception as e:  # noqa: BLE001
            line["e2e_funnel"] = {"error": str(e)[:200]}
    if world == 1 and with_cpu_baseline:
        import oracle
        oracle.build()
        cores = pick_torch_threads(host_threads())
        wl.cpu_sample(cores)
        n, dt = wl.cpu_sample(cores)
        line["cpu_baseline"] = {"value": n / dt, "unit": "images/s", "cores": cores, "kind": "port",
                                "sample": f"{n} image(s) of the same workload through oracle/ (restatement of the reference CPU path: fp32 torch network, C + OpenMP stereo / normal map / normalise), {dt:.2f} s"}
    return line


# sub-benchmarks carried in the default run so that the driver's record covers BASELINE's "depth+stereo 512^2 & 2048^2"
SUB_WORKLOADS = {"depth_beit512": ["stereo2048", "dav2_stereo", "zoedepth_nk768", "boost_res101_2048"]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default=DEFAULT_WORKLOAD, choices=sorted(WORKLOADS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-sub", action="store_true", help="skip the sub-benchmarks (stereo2048, dav2_stereo) of the default run")
    ap.add_argument("--no-funnel", action="store_true", help="skip the core_generation_funnel (PIL in / PIL out) end-to-end measurement")
    ap.add_argument("--no-graph", action="store_true", help="launch every kernel eagerly instead of replaying a CUDA graph")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step of --workload to DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the b200 path")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        # a collective that cannot complete (a sick link, a rank that died) raises after 5 minutes instead of hanging the job
        import datetime
        dist.init_process_group("nccl", device_id=dev, timeout=datetime.timedelta(minutes=5))

    import __graft_entry__ as ge
    if rank == 0:
        ge.build()
    if world > 1:
        dist.barrier()
    peaks = _peaks()
    wl = WORKLOADS[args.workload](dev, rank)
    line = measure(wl, args, world, dev, rank, local_rank, peaks, args.steps, not args.no_cpu_baseline, not args.no_funnel,
                   args.dump_outputs)
    if rank == 0 and world == 1 and not args.no_sub:
        subs = []
        for name in SUB_WORKLOADS.get(args.workload, []):
            del wl
            import gc
            gc.collect()
            torch.cuda.empty_cache()
            try:
                wl = WORKLOADS[name](dev, rank)
                sub = measure(wl, args, world, dev, rank, local_rank, peaks, args.steps, not args.no_cpu_baseline, False)
                sub["workload"] = name
                subs.append(sub)
            except Exception as e:  # noqa: BLE001
                subs.append({"workload": name, "error": str(e)[:300]})
                wl = None
        line["sub_benchmarks"] = subs
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
