"""Tool: images/s of the three ZoeDepth model types at batch 32 per call, metric depth only (pad + flip TTA, so 64 core forwards
per call), DPT-BEiT-L-384 core with seeded synthetic weights:
    ZoeDepth-N  (type 7)  768 x 768 images,          UI default net 384 x 512
    ZoeDepth-K  (type 8)  1536 x 512 (W x H) images, UI default net 384 x 768
    ZoeDepth-NK (type 9)  the zoedepth_nk768 workload's 768 x 768 images, net 384 x 512
Device-event timing of the 32 images through engine.forward_batch after warm-up, one engine at a time, the median call
reported.  ZoeDepth-K takes them in 4 calls of 8: PrepForMidas scales the reflect-padded 1702 x 608 input to a 768 x 2144 net
(6433 tokens per forward), where 64 forwards in one call do not fit in the card's memory.  The card's name and power limit are
read in the same run.
usage: python tools/bench_zoedepth.py [--rounds N] [--warmup W] [--out FILE]"""
import argparse
import gc
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

B = 32
CASES = [  # (label, model type, image H, image W, net_w, net_h, images per forward_batch call)
    ("zoedepth_n", 7, 768, 768, 384, 512, 32),
    ("zoedepth_k", 8, 512, 1536, 384, 768, 8),
    ("zoedepth_nk", 9, 768, 768, 384, 512, 32),
]


def card():
    import torch
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=60)
        name, power, clock = [x.strip() for x in q.stdout.strip().split(",")]
        info.update(smi_name=name, power_limit=power, max_sm_clock=clock)
    except Exception as e:      # the measurement stays valid; say that the limit is unknown
        info.update(power_limit=f"unknown ({type(e).__name__})")
    return info


def engine(model_type, dev):
    from bench_models import ZoeAnaglyph
    from depthmap_b200.depthmap_generation import ZoeDepthEngine, ZoeDepthNKEngine
    from oracle import synth_weights, zoedepth_single
    if model_type == 9:
        return ZoeDepthNKEngine(ZoeAnaglyph._state_dict(None), dev)
    sd = {"core.core." + k: v for k, v in synth_weights.make_beit_dpt_state_dict('beitl16_384', seed=0).items()}
    sd.update(zoedepth_single.make_zoedepth_single_state_dict(model_type, feat_ch=256, seed=100))
    return ZoeDepthEngine(sd, model_type, dev)


def main():
    import numpy as np
    import torch
    from bench import make_images
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=7, help="timed calls per model")
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_zoedepth: no CUDA device (nothing is measured without one)")
    dev = torch.device("cuda")
    runs = []
    for label, t, H, W, nw, nh, chunk in CASES:
        rgb, _ = make_images(B, H, W, 0)
        r = dict(label=label, type=t, net=(nw, nh), hw=(H, W), chunk=chunk, ms=[])
        chunks = [torch.from_numpy(np.ascontiguousarray(rgb[i:i + chunk])).to(dev) for i in range(0, B, chunk)]
        eng = engine(t, dev)

        def run():
            for c in chunks:
                eng.forward_batch(c, nw, nh)
        for _ in range(a.warmup):
            run()
        torch.cuda.synchronize()
        for _ in range(a.rounds):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            run()
            e1.record()
            torch.cuda.synchronize()
            r["ms"].append(e0.elapsed_time(e1))
        del eng, chunks, run
        gc.collect()
        torch.cuda.empty_cache()
        runs.append(r)
    res = {"tool": "tools/bench_zoedepth.py", "card": card(), "batch": B, "rounds": a.rounds, "warmup": a.warmup,
           "timing": "CUDA events around the forward_batch calls of the 32 images (uint8 resident on the device -> float32 metric depth), median",
           "weights": "seeded synthetic (oracle/synth_weights.py, oracle/zoedepth_single.py), checkpoint layouts of ZoeD_M12_N / _K / _NK", "results": []}
    for r in runs:
        ms = float(np.median(r["ms"]))
        res["results"].append(dict(model=r["label"], model_type=r["type"], image_hw=list(r["hw"]), net_wh=list(r["net"]),
                                   images_per_call=r["chunk"], ms_per_batch=round(ms, 2),
                                   ms_min=round(min(r["ms"]), 2), ms_max=round(max(r["ms"]), 2), images_per_s=round(B * 1000.0 / ms, 2)))
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
