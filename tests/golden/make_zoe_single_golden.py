"""Mints tests/golden/zoe_single_pin_golden.npz: what the original extension's own ZoeDepth module (the single metric head of
ZoeDepth-N and ZoeDepth-K, model types 7 and 8) computes on the seeded inputs of tests/test_zoe_single_pin.py, which compares
oracle/zoedepth.py against it.  Minting needs a checkout of the original extension (oracle/ref_loader.py finds it through
DEPTHMAP_REFERENCE_ROOT):

    python tests/golden/make_zoe_single_golden.py

The module is built as the original builds it: ZoeDepth(core, **get_config("zoedepth", "infer"[, config_version="kitti"])),
around a stub core that hands the head fixed activations and a non-zero relative depth (the head consumes it).  Its weights
are oracle/zoedepth_single.make_zoedepth_single_state_dict, loaded strictly (so the key names and shapes are the module's own);
inputs and weights are rebuilt from the seeds on both sides and not stored.  Storage follows tests/golden/make_pin_golden.py
(sampled values, shape, max |value|; one intra-op thread), plus the layout of the module's state_dict and the resolved
configuration of each variant.  The archive is written with fixed member timestamps so that minting again gives the same bytes.
"""
import io
import json
import os
import sys
import warnings
import zipfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from golden import make_pin_golden as mk  # noqa: E402

PATH = os.path.join(HERE, "zoe_single_pin_golden.npz")
VARIANTS = {7: None, 8: "kitti"}                 # model type -> config_version of get_config("zoedepth", "infer")
HEADS = [(0, (3, 4)), (1, (4, 3))]               # (seed, base size of the stub core's bottleneck)
TTA = [(True, True), (True, False), (False, True)]
TTA_SEED, TTA_BASE = 2, (2, 3)


def inputs(model_type, seed, base_hw):
    """(features, rel_depth, head state_dict) of one case: the activations MidasCore hands the head
    (dzoedepth/models/base_models/midas.py:258-276) and the relative depth, a post-ReLU map at out_conv's size"""
    import torch
    from oracle import zoedepth_single
    g = torch.Generator().manual_seed(1000 * model_type + seed)
    feats = mk.zoe_features(g, base_hw)
    rel = torch.rand(feats[0].shape[0], feats[0].shape[2], feats[0].shape[3], generator=g) * 2.0 + 0.1
    sd = zoedepth_single.make_zoedepth_single_state_dict(model_type, feat_ch=256, seed=50 + 10 * model_type + seed)
    return feats, rel, sd


def _model(model_type, feats, rel, sd):
    import torch
    import torch.nn as nn
    from dzoedepth.models.zoedepth.zoedepth_v1 import ZoeDepth
    from dzoedepth.utils.config import get_config

    class StubCore(nn.Module):                 # MidasCore.forward(x, denorm, return_rel_depth=True) -> (rel_depth, out)
        output_channels = (256, 256, 256, 256, 256)

        def forward(self, x, denorm=False, return_rel_depth=False):
            return rel.clone(), [f.clone() for f in feats]

    version = VARIANTS[model_type]
    conf = get_config("zoedepth", "infer", config_version=version) if version else get_config("zoedepth", "infer")
    model = ZoeDepth(StubCore(), **conf).eval()
    full = model.state_dict()
    buffers = {k for k, _ in model.named_buffers()}
    assert set(full) - set(sd) - buffers == set(), "the synthetic state_dict misses parameters"
    full.update(sd)                            # strict: an unexpected key or a wrong shape raises
    model.load_state_dict(full, strict=True)
    return model


def put_config(out, model_type, model):
    out[f"config_{model_type}"] = np.array(json.dumps(dict(
        variant={7: "zoedepth_n", 8: "zoedepth_k"}[model_type], bin_centers_type=model.bin_centers_type,
        min_depth=float(model.min_depth), max_depth=float(model.max_depth),
        n_attractors=[int(a.n_attractors) for a in model.attractors], attractor_layer=type(model.attractors[0]).__name__,
        attractor_alpha_applied=300.0, seed_layer=type(model.seed_bin_regressor).__name__,
        memory_efficient=[bool(a.memory_efficient) for a in model.attractors], kind=model.attractors[0].kind)))


def save(path, arrays):
    """np.savez_compressed with fixed member timestamps"""
    with zipfile.ZipFile(path, "w", zipfile.ZIP_DEFLATED) as zf:
        for k in sorted(arrays):
            buf = io.BytesIO()
            np.lib.format.write_array(buf, np.asanyarray(arrays[k]), allow_pickle=False)
            info = zipfile.ZipInfo(k + ".npy", date_time=(1980, 1, 1, 0, 0, 0))
            info.compress_type = zipfile.ZIP_DEFLATED
            info.external_attr = 0o644 << 16
            zf.writestr(info, buf.getvalue())


def main():
    import torch
    from oracle import ref_loader
    warnings.filterwarnings("ignore")
    torch.set_num_threads(mk.THREADS)
    ref_loader.bootstrap()
    out = {}
    for model_type in VARIANTS:
        for seed, base_hw in HEADS:
            feats, rel, sd = inputs(model_type, seed, base_hw)
            model = _model(model_type, feats, rel, sd)
            if f"config_{model_type}" not in out:
                put_config(out, model_type, model)
                sd_all = {k: v for k, v in model.state_dict().items() if not k.startswith("core.")}
                mk.put_layout(out, f"zoe_single_{model_type}", sd_all, {k for k, _ in model.named_parameters()})
            with torch.no_grad():
                want = model(torch.zeros(2, 3, feats[0].shape[2], feats[0].shape[3]))["metric_depth"]
            mk.put(out, f"head_{model_type}_{seed}", want.numpy())
        feats, rel, sd = inputs(model_type, TTA_SEED, TTA_BASE)
        model = _model(model_type, feats, rel, sd)
        for pad, flip in TTA:
            with torch.no_grad():
                want = model.infer(mk.zoe_tta_input(), pad_input=pad, with_flip_aug=flip)
            mk.put(out, f"tta_{model_type}_{int(pad)}{int(flip)}", want.numpy())
        print("model type", model_type, "done", flush=True)
    save(PATH, out)
    print("wrote", len(out), "arrays,", os.path.getsize(PATH), "bytes")


if __name__ == "__main__":
    main()
