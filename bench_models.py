"""Depth-network workloads for bench.py (kept separate so bench.py stays importable before the tensor-core path exists).

Timed region: the model-level C-ABI handle (NativeDepthModel -> dm_depth_forward) + the HBM-side kernels.  A second, op-level
instance of the same network (the Python engine that issues the same kernels one C call at a time) exists only for the PROBE
pass after the timed region: CUDA events around every attention launch and around the block-0 fc1 GEMM, which gives the
dominant kernel's share of the step and its roofline live, in this run."""
from __future__ import annotations

import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))


class _NetWorkload:
    """Shared parts of the network workloads: native model for the timed region, op-level engine for the kernel probe."""
    heads = 16
    C = 1024

    def probe(self, n=20):
        """Dominant-kernel timing, live in this run: the op-level engine runs one forward (so its buffers hold this workload's
        real activations), then the fused attention kernel of the LAST block and the fc1 GEMM are launched n times back to back
        on those buffers with CUDA events around the loop (GPU-bound: no host gaps inside the interval); the forward itself is
        timed on the native model (the thing the timed region runs)."""
        import torch
        from depthmap_b200 import _lib
        eng = self.engine
        for _ in range(2):
            self._engine_forward()
        torch.cuda.synchronize()
        b = eng._bufs
        cfg = eng.cfg
        C, heads = cfg['embed_dim'], cfg['heads']
        _, nh, nw = eng._buf_key
        gh, gw = nh // eng.PATCH, nw // eng.PATCH
        N = gh * gw + 1
        last = cfg['depth'] - 1
        blk = eng.w['blocks'][last]
        PB = getattr(self, 'probe_batch', self.B)
        rows = PB * N

        def timed(fn):
            fn()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(n):
                fn()
            e1.record()
            torch.cuda.synchronize()
            return e0.elapsed_time(e1) / n
        attn_ms = timed(lambda: eng.attention(last, b, PB, N, heads, C, gh, gw))
        fc1_ms = timed(lambda: eng.ops.gemm(b['h'], C, blk['fc1_w'], C, rows, 4 * C, C, act=_lib.ACT_GELU, bias=blk['fc1_b'], C=b['mlp'], ldc=4 * C))
        fwd_ms = timed(self._model_forward)
        return {"attn_ms_per_launch": float(attn_ms), "attn_launches": cfg['depth'], "fc1_ms": float(fc1_ms), "forward_ms": float(fwd_ms)}

    def roofline_from_probe(self, peaks, pr, ms_step):
        """Dominant kernel = the fused attention kernel (largest share of the step, measured here); fc1 reported beside it."""
        N = self.N
        attn_flops = 4.0 * getattr(self, 'probe_batch', self.B) * self.heads * N * N * 64          # QK^T + PV, 2 flops per MAC (SURVEY 8d: 2.15 + 2.15 GFLOP / image / block)
        a = attn_flops / (pr["attn_ms_per_launch"] * 1e-3) / 1e12
        f = self.fc1_flops / (pr["fc1_ms"] * 1e-3) / 1e12
        share = pr["attn_ms_per_launch"] * pr["attn_launches"] / pr["forward_ms"]
        return {"bound": "tensor", "kernel": self.ATTN_KERNEL, "achieved": a, "peak": peaks["bf16_tflops"], "unit": "TFLOP/s",
                "frac": a / peaks["bf16_tflops"], "traffic": None, "traffic_note": "see profiles/r02_ncu_attention_fwd4.txt (one ncu --set full capture per kernel)",
                "peak_source": peaks["source"] + " (cuBLAS bf16 burst)", "algorithmic_flops_per_launch": attn_flops,
                "kernel_ms": pr["attn_ms_per_launch"], "launches_per_step": pr["attn_launches"],
                "share_of_step": share, "share_note": "attention launches per forward x kernel time / forward time of the model handle, all CUDA events, this run",
                "secondary": {"kernel": self.FC1_KERNEL, "achieved": f, "frac": f / peaks["bf16_tflops"], "kernel_ms": pr["fc1_ms"],
                              "algorithmic_flops_per_launch": self.fc1_flops}}

    def _model_forward(self):
        return self.model.forward_batch(self.rgb, self.W, self.H)

    def extra(self, ms_step, peaks):
        fwd = self.FLOP_PER_IMAGE * self.B / (ms_step * 1e-3) / 1e12
        return {"whole_step_tflops": fwd, "whole_step_frac_of_sustained_peak": fwd / peaks["bf16_tflops_sustained"]}

    def funnel_e2e(self, steps=2):
        """The reference-facing entry point itself: PIL images in, PIL images out through core_generation_funnel (src/core.py:83)."""
        import torch
        from PIL import Image
        from depthmap_b200 import core
        holder = core.get_model_holder()
        holder.unload_models()
        holder.weights_provider = lambda t: self._state_dict()
        imgs = [Image.fromarray(self.rgb_h[i].numpy()) for i in range(self.B)]
        inp = self.funnel_options()
        n_out = 0
        times = []
        for it in range(steps + 1):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            n_out = sum(1 for _ in core.core_generation_funnel(None, list(imgs), None, None, inp, ops={}))
            torch.cuda.synchronize()
            times.append(time.perf_counter() - t0)
        holder.unload_models()
        holder.weights_provider = None
        dt = float(np.mean(times[1:]))             # first pass loads / packs the model, as the reference's first call does
        return {"value": self.B / dt, "unit": "images/s", "ms_per_step": dt * 1e3, "results_per_step": n_out,
                "note": "core_generation_funnel(PIL in -> PIL out), wall clock incl. PIL<->tensor conversion, H2D/D2H and the funnel's bounded batches"}


class Dav2Stereo(_NetWorkload):
    """BASELINE.json configs[2]: depth_anything_v2 vitl @518x518 + SBS stereo (divergence 2.5, polylines fill) + normal map,
    batch 64 per GPU."""
    name = "dav2_stereo"
    encoder = "vitl"
    H = W = 518
    B = 64
    dtype = "fp16"  # tensor-core operands fp16, fp32 accumulate / residual stream (the reference's GPU path is .half())
    fill = "polylines_sharp"
    outputs = ("depth", "stereo_sbs", "normal")
    FLOP_PER_IMAGE = 1304.2e9  # SURVEY §8d, cross-checked there against FlopCounterMode on the reference module
    MODEL_TYPE = 14
    ATTN_KERNEL = "attention_fwd4_kernel<0> (fused softmax(QK^T)V, tcgen05 + TMEM, N = 1370, 16 heads x 64)"
    FC1_KERNEL = "gemm_tcgen05_2sm_kernel (cta_group::2, 256x256 tile pair; block-0 MLP fc1: M=B*1370, N=4096, K=1024, GELU epilogue)"

    def _state_dict(self):
        from oracle import synth_weights  # synthetic checkpoint-layout weights (data generation, not compute)
        return synth_weights.make_dav2_state_dict(self.encoder, seed=0)

    def funnel_options(self):
        return dict(compute_device='GPU', model_type=self.MODEL_TYPE, net_width=self.W, net_height=self.H, do_output_depth=True,
                    gen_stereo=True, stereo_modes=['left-right'], stereo_divergence=2.5, stereo_fill_algo=self.fill, gen_normalmap=True)

    def __init__(self, dev, rank):
        import torch
        from bench import make_images
        from depthmap_b200.depthmap_generation import DepthAnythingV2Engine, NativeDepthModel
        self.dev = dev
        sd = self._state_dict()
        self.model = NativeDepthModel(sd, self.MODEL_TYPE, dev)
        self.engine = DepthAnythingV2Engine(sd, self.encoder, dev)      # probe pass only
        del sd
        rgb, _ = make_images(self.B, self.H, self.W, rank)
        self.rgb_h = torch.from_numpy(rgb).pin_memory()
        self.rgb = self.rgb_h.to(dev)
        cfg = self.engine.cfg
        C = cfg['embed_dim']
        self.N = (self.H // 14) * (self.W // 14) + 1
        self.fc1_flops = 2.0 * self.B * self.N * C * 4 * C
        self.launches_per_step = None

    def config(self):
        return {"workload": "depth_anything_v2 vitl 518x518 -> u16 depth -> SBS stereo (divergence 2.5, polylines_sharp) -> "
                            "normal map (Sobel 3)", "batch_per_gpu": self.B, "height": self.H, "width": self.W,
                "weights": "seeded synthetic, upstream checkpoint layout",
                "l2_policy": "activations per step (>10 GB) far exceed the 126 MB L2"}

    def step(self, rgb, time_kernel=False):
        import torch
        from depthmap_b200.core import normalize_prediction_batch
        from depthmap_b200.normalmap_generation import create_normalmap_batch
        from depthmap_b200.stereoimage_generation import create_stereoimages_batch
        n0 = self.model.launches
        pred = self.model.forward_batch(rgb, self.W, self.H)
        depth = normalize_prediction_batch(pred, False)
        sbs = create_stereoimages_batch(rgb, depth, 2.5, 0.0, ['left-right'], 0.0, 1.0, self.fill)[0]
        normal = create_normalmap_batch(depth)
        n1 = self.model.launches
        if n1 > n0:
            self.launches_per_step = (n1 - n0) + 3 + 3 + 1
        return depth, sbs, normal

    def _engine_forward(self):
        return self.engine.forward_batch(self.rgb, self.W)

    def step_resident(self, time_kernel=False):
        return self.step(self.rgb, time_kernel)

    def step_e2e(self):
        rgb = self.rgb_h.to(self.dev, non_blocking=True)
        outs = self.step(rgb)
        return [o.to("cpu", non_blocking=True) for o in outs]

    def e2e_bytes(self):
        return self.rgb_h.numel(), self.B * self.H * self.W * (2 + 6 + 3)

    def cpu_sample(self, nthreads):
        """reference CPU path on one image: fp32 torch forward (oracle restatement) + C oracle stereo / normal map."""
        import torch
        from oracle import dav2 as odav2
        from oracle import normalmap as onm
        from oracle import stereo as ost
        from oracle import synth_weights
        if not hasattr(self, "_sd_cpu"):
            self._sd_cpu = synth_weights.make_dav2_state_dict(self.encoder, seed=0)
        rgb = self.rgb_h[0].numpy()
        torch.set_num_threads(nthreads)
        t0 = time.perf_counter()
        pred, inv = odav2.get_raw_prediction(rgb, self._sd_cpu, self.encoder, self.W)
        d = onm.normalize_to_u16(pred, inv)
        ost.create_stereoimages(rgb, d, 2.5, 0.0, ['left-right'], 0.0, 1.0, self.fill, return_arrays=True, nthreads=nthreads)
        onm.create_normalmap(d, return_array=True)
        return 1, time.perf_counter() - t0


class DepthBeit512(_NetWorkload):
    """BASELINE.json configs[1]: dpt_beit_large_512 @512x512, batch 32 per GPU, depth only (prediction -> 16-bit depth)."""
    name = "depth_beit512"
    model_name = "beitl16_512"
    H = W = 512
    B = 32
    dtype = "fp16"
    outputs = ("depth",)
    FLOP_PER_IMAGE = 962.7e9  # SURVEY §8d
    MODEL_TYPE = 1
    ATTN_KERNEL = "attention_fwd4_kernel<3> (fused softmax(QK^T + rel-pos bias)V, tcgen05 + TMEM, N = 1025, 16 heads x 64; + class-row kernel)"
    FC1_KERNEL = "gemm_tcgen05_2sm_kernel (cta_group::2, 256x256 tile pair; block-0 MLP fc1: M=B*1025, N=4096, K=1024, GELU epilogue)"

    def _state_dict(self):
        from oracle import synth_weights  # synthetic checkpoint-layout weights (data generation, not compute)
        return synth_weights.make_beit_dpt_state_dict(self.model_name, seed=0)

    def funnel_options(self):
        return dict(compute_device='GPU', model_type=self.MODEL_TYPE, net_width=self.W, net_height=self.H, do_output_depth=True)

    def __init__(self, dev, rank):
        import torch
        from bench import make_images
        from depthmap_b200.depthmap_generation import DptBeitEngine, NativeDepthModel
        self.dev = dev
        sd = self._state_dict()
        self.model = NativeDepthModel(sd, self.MODEL_TYPE, dev)
        self.engine = DptBeitEngine(sd, self.model_name, dev)           # probe pass only
        del sd
        rgb, _ = make_images(self.B, self.H, self.W, rank)
        self.rgb_h = torch.from_numpy(rgb).pin_memory()
        self.rgb = self.rgb_h.to(dev)
        C = self.engine.cfg['embed_dim']
        self.N = (self.H // 16) * (self.W // 16) + 1
        self.fc1_flops = 2.0 * self.B * self.N * C * 4 * C
        self.launches_per_step = None

    def config(self):
        return {"workload": "dpt_beit_large_512 (MiDaS 3.1) 512x512 -> float32 prediction -> u16 depth", "batch_per_gpu": self.B,
                "height": self.H, "width": self.W, "weights": "seeded synthetic, MiDaS checkpoint layout",
                "l2_policy": "activations per step (>5 GB) far exceed the 126 MB L2"}

    def step(self, rgb, time_kernel=False):
        import torch
        from depthmap_b200.core import normalize_prediction_batch
        n0 = self.model.launches
        pred = self.model.forward_batch(rgb, self.W, self.H)
        depth = normalize_prediction_batch(pred, False)
        n1 = self.model.launches
        if n1 > n0:
            self.launches_per_step = (n1 - n0) + 3
        return (depth,)

    def _engine_forward(self):
        return self.engine.forward_batch(self.rgb, self.W, self.H)

    def step_resident(self, time_kernel=False):
        return self.step(self.rgb, time_kernel)

    def step_e2e(self):
        rgb = self.rgb_h.to(self.dev, non_blocking=True)
        outs = self.step(rgb)
        return [o.to("cpu", non_blocking=True) for o in outs]

    def e2e_bytes(self):
        return self.rgb_h.numel(), self.B * self.H * self.W * 2

    def cpu_sample(self, nthreads):
        """reference CPU path on one image: fp32 torch forward (oracle restatement of DPT-BEiT) + C oracle normalise."""
        import torch
        from oracle import beit_dpt
        from oracle import normalmap as onm
        from oracle import synth_weights
        if not hasattr(self, "_sd_cpu"):
            self._sd_cpu = synth_weights.make_beit_dpt_state_dict(self.model_name, seed=0)
        rgb = self.rgb_h[0].numpy()
        torch.set_num_threads(nthreads)
        t0 = time.perf_counter()
        pred, inv = beit_dpt.get_raw_prediction(rgb, self._sd_cpu, self.model_name, self.W, self.H)
        onm.normalize_to_u16(pred, inv)
        return 1, time.perf_counter() - t0


class ZoeAnaglyph(_NetWorkload):
    """BASELINE.json configs[3]: zoedepth_nk at 768x768 + anaglyph stereo, 32 images per GPU (256 over 8 GPUs, sharded, one
    NCCL gather).  Every image runs twice through the DPT-BEiT-L-384 core (flip TTA): 64 forwards at the 512x512 net size
    that PrepForMidas picks for the reflect-padded 884x884 input with the UI default net (w 384, h 512)."""
    name = "zoedepth_nk768"
    H = W = 768
    B = 32
    dtype = "fp16"
    NET_W, NET_H = 384, 512
    outputs = ("depth", "anaglyph")
    FLOP_PER_IMAGE = 2 * 962.7e9 + 2 * 10e9      # SURVEY 8d: two core forwards at 512x512 + the metric head (~1%)
    ATTN_KERNEL = "attention_fwd4_kernel<3> (fused softmax(QK^T + rel-pos bias)V of the BEiT-L-384 core at a 32x32 window, 64 forwards)"
    FC1_KERNEL = "gemm_tcgen05_2sm_kernel (block MLP fc1: M=64*1025, N=4096, K=1024, GELU epilogue)"

    def _state_dict(self):
        from oracle import beit_dpt, synth_weights
        csd = synth_weights.make_beit_dpt_state_dict('beitl16_384', seed=0)
        hsd = synth_weights.make_zoedepth_head_state_dict(feat_ch=beit_dpt.CONFIGS['beitl16_384']['features'], seed=100, gain=1.5)
        sd = {"core.core." + k: v for k, v in csd.items()}
        sd.update(hsd)
        return sd

    def funnel_options(self):
        return dict(compute_device='GPU', model_type=9, net_width=self.NET_W, net_height=self.NET_H, do_output_depth=True, gen_stereo=True,
                    stereo_modes=['red-cyan-anaglyph'], stereo_divergence=2.5, stereo_fill_algo='polylines_sharp')

    def __init__(self, dev, rank):
        import torch
        from bench import make_images
        from depthmap_b200.depthmap_generation import ZoeDepthNKEngine
        self.dev = dev
        self.engine = ZoeDepthNKEngine(self._state_dict(), dev)
        self.model = self.engine
        rgb, _ = make_images(self.B, self.H, self.W, rank)
        self.rgb_h = torch.from_numpy(rgb).pin_memory()
        self.rgb = self.rgb_h.to(dev)
        self.probe_batch = 2 * self.B
        self.N = 32 * 32 + 1
        self.fc1_flops = 2.0 * self.probe_batch * self.N * 1024 * 4096
        self.launches_per_step = None

    def config(self):
        return {"workload": "zoedepth_nk (DPT-BEiT-L-384 core + metric head, pad + flip TTA) 768x768 -> u16 depth -> red-cyan anaglyph "
                            "(divergence 2.5, polylines_sharp)", "batch_per_gpu": self.B, "height": self.H, "width": self.W,
                "net": "384x512 (UI default) -> 512x512 for the padded 884x884 input", "weights": "seeded synthetic, ZoeD_M12_NK checkpoint layout",
                "l2_policy": "activations per step (>20 GB) far exceed the 126 MB L2"}

    def step(self, rgb, time_kernel=False):
        from depthmap_b200.core import normalize_prediction_batch
        from depthmap_b200.stereoimage_generation import create_stereoimages_batch
        n0 = self.engine.ops.launches
        pred = self.engine.forward_batch(rgb, self.NET_W, self.NET_H)
        depth = normalize_prediction_batch(pred, True)
        ana = create_stereoimages_batch(rgb, depth, 2.5, 0.0, ['red-cyan-anaglyph'], 0.0, 1.0, 'polylines_sharp')[0]
        self.launches_per_step = (self.engine.ops.launches - n0) + 3 + 3
        return depth, ana

    def step_resident(self, time_kernel=False):
        return self.step(self.rgb, time_kernel)

    def step_e2e(self):
        rgb = self.rgb_h.to(self.dev, non_blocking=True)
        outs = self.step(rgb)
        return [o.to("cpu", non_blocking=True) for o in outs]

    def e2e_bytes(self):
        return self.rgb_h.numel(), self.B * self.H * self.W * (2 + 3)

    def _engine_forward(self):
        return self.engine.forward_batch(self.rgb, self.NET_W, self.NET_H)

    def _model_forward(self):
        return self.engine.forward_batch(self.rgb, self.NET_W, self.NET_H)

    def cpu_sample(self, nthreads):
        """reference CPU path on one image: fp32 torch ZoeDepth-NK (oracle restatement, 2 core forwards) + C oracle normalise / stereo."""
        import torch
        from oracle import normalmap as onm
        from oracle import stereo as ost
        from oracle import zoedepth as ozd
        if not hasattr(self, "_sd_cpu"):
            self._sd_cpu = self._state_dict()
        rgb = self.rgb_h[0].numpy()
        torch.set_num_threads(nthreads)
        t0 = time.perf_counter()
        pred, inv = ozd.get_raw_prediction(rgb, self._sd_cpu, self.NET_W, self.NET_H, core_name='beitl16_384')
        d = onm.normalize_to_u16(pred, inv)
        ost.create_stereoimages(rgb, d, 2.5, 0.0, ['red-cyan-anaglyph'], 0.0, 1.0, 'polylines_sharp', return_arrays=True, nthreads=nthreads)
        return 1, time.perf_counter() - t0


class Dav2StereoSmall(Dav2Stereo):
    """ViT-S variant for quick functional runs."""
    name = "dav2s_stereo"
    encoder = "vits"
    B = 8
    FLOP_PER_IMAGE = 0.0
    MODEL_TYPE = 12
    heads, C = 6, 384


class BoostRes101:
    """BASELINE.json configs[4]: BoostingMonocularDepth multi-resolution merge (LeReS res101 base + pix2pix merge net) on a 2048x2048
    synthetic image.  One image per step; with N GPUs the image's patches are dealt to the ranks (patch-parallel, one all-gather of the
    fitted patches, every rank replays the blend): STRONG scaling.  `value` = images/s with the image resident and the host control plane
    (R_x search + patch selection, a function of the RGB image only) computed once outside the timed region; `e2e` = the public call
    ModelHolder.get_raw_prediction(PIL image) including that control plane, the H2D of the image and the D2H of the depth map."""
    name = "boost_res101_2048"
    H = W = 2048
    B = 1
    dtype = "fp16 (LeReS operands) / split fp16 = fp32-class (merge net), fp32 accumulate"
    RMAX = 1600                                   # the reference's default boost_rmax (src/backbone.py:36-49)
    outputs = ("depth",)

    def __init__(self, dev, rank):
        from bench import make_images
        from depthmap_b200.depthmap_generation import ModelHolder
        from oracle import synth_weights
        self.dev = dev
        lsd = synth_weights.make_leres_state_dict(seed=2)
        psd = synth_weights.make_pix2pix_state_dict(seed=1)
        self.holder = ModelHolder()
        self.holder.weights_provider = lambda t: psd if t == "pix2pix" else lsd
        self.holder.update_settings(boost_rmax=self.RMAX)
        self.holder.ensure_models(0, dev, True)
        self.pipe = self.holder.pix2pix_model
        rgb, _ = make_images(1, self.H, self.W, 0)            # every rank works on the SAME image
        self.rgb = rgb[0]

    def config(self):
        return {"workload": "BOOST: LeReS res101 double estimation + pix2pix merge net, 2048x2048 -> 2048x2048 fp32 depth", "images_per_step": 1,
                "height": self.H, "width": self.W, "boost_rmax": self.RMAX, "weights": "seeded synthetic, res101.pth / latest_net_G.pth layouts",
                "l2_policy": "per-image activations (several GB) far exceed the 126 MB L2"}

    def measure(self, args, world, dev, rank, local_rank, peaks, steps, with_cpu_baseline, ClockSampler, dump=None):
        import torch
        import torch.distributed as dist
        from PIL import Image
        from depthmap_b200 import boost
        import cv2
        group = dist.group.WORLD if world > 1 else None
        info = {}
        self.pipe.run(self.rgb, self.RMAX, group=group, info=info)           # warm-up 1 (allocations), also yields the plan
        plan = {k: info[k] for k in ("rf", "whole", "patch_scale", "factor", "target", "work", "rects", "scaled_rects")}
        for _ in range(max(args.warmup - 1, 1)):
            self.pipe.run(self.rgb, self.RMAX, group=group, precomputed=plan, to_host=False)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        n0 = self.pipe.launches + self.pipe.depth.ops.launches + self.pipe.merge.ops.launches
        sampler = ClockSampler(local_rank) if rank == 0 else None
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            depth = self.pipe.run(self.rgb, self.RMAX, group=group, precomputed=plan, to_host=False)
        e1.record()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        clocks = sampler.stop() if sampler else None
        if dump is not None:
            dump((depth,))
        launches = self.pipe.launches + self.pipe.depth.ops.launches + self.pipe.merge.ops.launches - n0
        t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_step = float(t.item()) / steps
        # e2e through the public API (rank 0's wall clock around the call; the call ends with a D2H copy, i.e. it is synchronous)
        pil = Image.fromarray(self.rgb)
        if world == 1:
            self.holder.get_raw_prediction(pil, 448, 448)
            t0 = time.perf_counter()
            for _ in range(steps):
                pred, _ = self.holder.get_raw_prediction(pil, 448, 448)
            ms_e2e = (time.perf_counter() - t0) / steps * 1e3
        else:
            t0 = time.perf_counter()
            for _ in range(steps):
                self.pipe.run(self.rgb, self.RMAX, group=group)
            ms_e2e = (time.perf_counter() - t0) / steps * 1e3
        if rank != 0:
            return None
        n_patches = len(plan["rects"])
        # algorithmic FLOPs (SURVEY 8d, FlopCounterMode on the reference modules): LeReS 290.0 GFLOP at 448^2 scaling with the pixel count,
        # merge net 191.1 GFLOP per 1024^2 call; whole image: 2 LeReS + 1 merge; per patch: 2 LeReS (448, 896) + 2 merges
        leres = lambda s: 290.0e9 * (s / 448.0) ** 2
        flops = leres(448) + leres(plan["whole"]) + 191.1e9 + n_patches * (leres(448) + leres(896) + 2 * 191.1e9)
        line = {"metric": "images/sec", "value": 1000.0 / ms_step, "unit": "images/s", "n_gpus": world, "steps": steps, "warmup": args.warmup,
                "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": self.dtype, "data": "synthetic",
                "config": dict(self.config(), patches=n_patches, whole_size=plan["whole"], target=list(plan["target"]),
                               parallelism=("patch-parallel over %d ranks, one all-gather" % world) if world > 1 else "single GPU, patches one by one"),
                "clocks": clocks, "gpu_launches": launches, "launch_mode": "cuda_graph per network (LeReS per net size, merge net); glue kernels eager",
                "e2e": {"value": 1000.0 / ms_e2e, "unit": "images/s", "h2d_bytes_per_step": self.H * self.W * 3, "d2h_bytes_per_step": self.H * self.W * 4,
                        "ms_per_step": ms_e2e, "api": "ModelHolder.get_raw_prediction(PIL image) with boost: host control plane (cv2 Sobel / integral image on the "
                                                      "3136-px work image) + H2D + every network pass + D2H, wall clock"},
                "roofline": {"bound": "tensor", "kernel": "whole step (no single dominant kernel: ~%d launches per image, B = 1)" % (launches // max(steps, 1)),
                             "achieved": flops / (ms_step * 1e-3) / 1e12, "peak": peaks["bf16_tflops_sustained"], "unit": "TFLOP/s",
                             "frac": flops / (ms_step * 1e-3) / 1e12 / peaks["bf16_tflops_sustained"], "traffic": None, "peak_source": peaks["source"],
                             "algorithmic_flops_per_launch": flops,
                             "note": "algorithmic FLOPs of the fp32 reference networks; the merge net spends 3x that on the tensor core (split operands)"}}
        if world == 1 and with_cpu_baseline:
            import oracle
            from bench import host_threads, pick_torch_threads
            oracle.build()
            cores = pick_torch_threads(host_threads())
            n, dt, what = self.cpu_sample(cores)
            line["cpu_baseline"] = {"value": n / dt, "unit": "images/s", "cores": cores, "kind": "port", "sample": what}
        return line

    def cpu_sample(self, nthreads):
        """Bounded sample of the reference CPU path: ONE patch's network work (LeReS at 448 and 896 + two merge-net calls, fp32 torch through
        oracle/), scaled to the image by the patch count + the whole-image prefix at the same per-FLOP rate."""
        import torch
        from oracle import leres, pix2pix as op2p, synth_weights
        torch.set_num_threads(nthreads)
        lsd = synth_weights.make_leres_state_dict(seed=2)
        psd = synth_weights.make_pix2pix_state_dict(seed=1)
        crop = (self.rgb[:900, :900].astype(np.float64) / 255.0)[:, :, ::-1]
        t0 = time.perf_counter()
        with torch.no_grad():
            a = leres.estimateleres(crop, lsd, 448, 448)
            b = leres.estimateleres(crop, lsd, 896, 896)
            import cv2
            a = cv2.resize(a, (1024, 1024), interpolation=cv2.INTER_CUBIC)
            b = cv2.resize(b, (1024, 1024), interpolation=cv2.INTER_CUBIC)
            m = op2p.unet(psd, op2p.merge_input(a, b))[0, 0].numpy()
            op2p.unet(psd, op2p.merge_input(a, m))
        dt = time.perf_counter() - t0
        per_patch_flops = 290.0e9 * (1 + 4) + 2 * 191.1e9
        info = {}
        from depthmap_b200 import boost
        import cv2
        p = boost.plan(cv2.cvtColor(self.rgb, cv2.COLOR_BGR2RGB) / 255.0, 0, self.RMAX)
        total = 290.0e9 * (1 + (p["whole"] / 448.0) ** 2) + 191.1e9 + len(p["rects"]) * per_patch_flops
        est = dt * total / per_patch_flops
        return 1, est, (f"one patch's double estimation + merge measured ({dt:.1f} s, fp32 torch CPU through oracle/), extrapolated by FLOPs to the image's "
                        f"{len(p['rects'])} patches + whole-image prefix = {est:.0f} s per image")


MODEL_WORKLOADS = {"boost_res101_2048": BoostRes101, "depth_beit512": DepthBeit512, "dav2_stereo": Dav2Stereo, "dav2s_stereo": Dav2StereoSmall, "zoedepth_nk768": ZoeAnaglyph}
