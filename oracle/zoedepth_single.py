"""ORACLE (test infrastructure only — the product never imports this): plain-torch fp32 functional restatement of the
single metric head of ZoeDepth-N and ZoeDepth-K (model types 7 / 8, dzoedepth/models/zoedepth/zoedepth_v1.py:38-186),
composed with the DPT-BEiT core of oracle/beit_dpt.py and the pad + flip TTA / PrepForMidas of oracle/zoedepth.py, plus
seeded single-head weights in the checkpoint layout.

Follows the reference:
  dzoedepth/models/zoedepth/zoedepth_v1.py:120-186        ZoeDepth.forward after the core (seed bins, attractors, log-binomial)
  dzoedepth/models/layers/localbins_layers.py:29-94       SeedBinRegressor (normed), SeedBinRegressorUnnormed, Projector
  dzoedepth/models/layers/attractor.py:60-208             AttractorLayer (normed), AttractorLayerUnnormed
  dzoedepth/models/layers/dist_layers.py                  ConditionalLogBinomial (shared with the NK oracle)
Pinned against the reference module itself, built around a stub core, by tests/test_zoe_single_pin.py."""
from __future__ import annotations

import torch
import torch.nn.functional as F

from .zoedepth import _conditional_log_binomial, _conv1x1, _inv_attractor, _mlp2, infer, prep_for_midas

# ---------------------------------------------------------------------------------------------------------------------
# the single metric head of dzoedepth/models/zoedepth/zoedepth_v1.py:38-186, built by
# the reference from get_config("zoedepth", "infer"[, config_version="kitti"]) (src/depthmap_generation.py:196-205).
# Resolved configs: 64 bins, 128-d bin embedding, temperatures 0.0212 .. 50, attractor kind "mean", type "inv";
# min / max depth are the constructor defaults 1e-3 / 10 for BOTH variants (infer mode merges no dataset config, so K does
# not get KITTI's 80).  The counts [16, 8, 4, 1] are passed by keyword, so the levels really have 16, 8, 4 and 1
# attractors.  `memory_efficient` is not forwarded to the layers, which therefore take the torch.mean branch.
# ---------------------------------------------------------------------------------------------------------------------
SINGLE_CONFIG = {
    7: dict(variant="n", bin_centers_type="softplus", n_attractors=[16, 8, 4, 1], min_depth=1e-3, max_depth=10),
    8: dict(variant="k", bin_centers_type="normed", n_attractors=[16, 8, 4, 1], min_depth=1e-3, max_depth=10),
}


def _seed_bins_normed(x, sd, prefix, min_depth, max_depth):
    """SeedBinRegressor.forward (localbins_layers.py:29-68): bin centres bounded to (min_depth, max_depth)."""
    B = F.relu(_mlp2(x, sd, prefix, F.relu)) + 1e-3
    widths = (max_depth - min_depth) * (B / B.sum(dim=1, keepdim=True))
    widths = F.pad(widths, (0, 0, 0, 0, 1, 0), mode="constant", value=min_depth)
    edges = torch.cumsum(widths, dim=1)
    return 0.5 * (edges[:, :-1, ...] + edges[:, 1:, ...])


def _attractor_single(x, b_prev, prev_emb, sd, prefix, n_attractors, normed, min_depth, max_depth):
    """AttractorLayer (normed) / AttractorLayerUnnormed with interpolate=True, memory_efficient=False, kind='mean', type 'inv'
    (attractor.py:60-136 / 139-208); returns (b_new for the next level, bin centres of this level)."""
    x = x + F.interpolate(prev_emb, x.shape[-2:], mode="bilinear", align_corners=True)
    if normed:
        A = F.relu(_mlp2(x, sd, prefix, F.relu)) + 1e-3
        n, c, h, w = A.shape
        A = A.view(n, n_attractors, 2, h, w)[:, :, 0, ...]      # the normalisation line of the reference is overwritten
    else:
        A = F.softplus(_mlp2(x, sd, prefix, F.relu))
        h, w = A.shape[-2:]
    b_centers = F.interpolate(b_prev, (h, w), mode="bilinear", align_corners=True)
    delta = torch.mean(_inv_attractor(A.unsqueeze(2) - b_centers.unsqueeze(1)), dim=1)
    b_new = b_centers + delta
    if not normed:
        return b_new, b_new
    B = (max_depth - min_depth) * b_new + min_depth
    B, _ = torch.sort(B, dim=1)
    return b_new, torch.clip(B, min_depth, max_depth)


def metric_head_single(features, rel_depth, sd, model_type):
    """ZoeDepth.forward after the core (zoedepth_v1.py:139-186).  features = [out_conv, btlnck, x_block4..1] (fp32 NCHW),
    rel_depth [N, h, w] the core's relative depth; sd: head weights (checkpoint keys minus "core.").  -> metric depth [N,1,H,W]"""
    cfg = SINGLE_CONFIG[model_type]
    normed, mn, mx = cfg["bin_centers_type"] == "normed", cfg["min_depth"], cfg["max_depth"]
    outconv, btlnck, x_blocks = features[0], features[1], features[2:]
    x = _conv1x1(btlnck, sd, "conv2")
    if normed:
        b_prev = (_seed_bins_normed(x, sd, "seed_bin_regressor", mn, mx) - mn) / (mx - mn)
    else:
        b_prev = F.softplus(_mlp2(x, sd, "seed_bin_regressor", F.relu))           # SeedBinRegressorUnnormed
    prev_emb = _mlp2(x, sd, "seed_projector", F.relu)
    b_centers = b_emb = None
    for i, xb in enumerate(x_blocks):
        b_emb = _mlp2(xb, sd, f"projectors.{i}", F.relu)
        b_prev, b_centers = _attractor_single(b_emb, b_prev, prev_emb, sd, f"attractors.{i}", cfg["n_attractors"][i], normed, mn, mx)
        prev_emb = b_emb
    rel_cond = F.interpolate(rel_depth.unsqueeze(1), size=outconv.shape[2:], mode="bilinear", align_corners=True)
    last = torch.cat([outconv, rel_cond], dim=1)
    b_emb = F.interpolate(b_emb, last.shape[-2:], mode="bilinear", align_corners=True)
    probs = _conditional_log_binomial(last, b_emb, sd, "conditional_log_binomial", 64)
    b_centers = F.interpolate(b_centers, probs.shape[-2:], mode="bilinear", align_corners=True)
    return torch.sum(probs * b_centers, dim=1, keepdim=True)


@torch.no_grad()
def get_raw_prediction_single(rgb_uint8, sd, model_type, net_w=512, net_h=384, core_name="beitl16_384"):
    """ModelHolder.get_raw_prediction for model types 7 (zoedepth_n) / 8 (zoedepth_k): (float32 metric depth [H,W], invert=True).
    sd: checkpoint layout — MiDaS weights under "core.core.", head weights at the top level."""
    import numpy as np
    from oracle import beit_dpt
    core_sd = {k[len("core.core."):]: v for k, v in sd.items() if k.startswith("core.core.")}
    head_sd = {k: v for k, v in sd.items() if not k.startswith("core.")}

    def model_fn(x):
        xin = prep_for_midas(x, net_w, net_h)
        rel, feats = beit_dpt.forward(core_sd, xin, core_name, return_features=True)
        return metric_head_single(feats, rel, head_sd, model_type)

    img = np.asarray(rgb_uint8)
    x = torch.from_numpy(np.ascontiguousarray(img)).permute(2, 0, 1).float().div(255.0).unsqueeze(0)      # transforms.ToTensor
    out = infer(model_fn, x, pad_input=True, with_flip_aug=True)
    return out.squeeze().cpu().numpy(), True


def make_zoedepth_single_state_dict(model_type, feat_ch=256, out_conv_ch=32, seed=0, dtype=torch.float32, gain=1.5):
    """Seeded ZoeDepth-N (model_type 7) / ZoeDepth-K (8) metric-head weights in the checkpoint layout of
    dzoedepth/models/zoedepth/zoedepth_v1.py (keys as `ZoeDepth.state_dict()` minus "core."): seed regressor hidden 256,
    projector hidden 128, attractor layers of 16, 8, 4, 1 attractors (2 channels each for K's normed layers), log-binomial
    MLP 161 -> 80 -> 4.  Fan-in scaled weights times `gain`; K's attractor outputs are scaled so that the normed attractor
    points stay inside [0, 1] and the bin centres spread over (min, max) instead of piling up at a clip bound."""
    normed = model_type == 8
    if model_type not in (7, 8):
        raise ValueError(f"model_type {model_type}: 7 (ZoeDepth-N) or 8 (ZoeDepth-K)")
    g = torch.Generator().manual_seed(seed)
    sd = {}

    def conv(key, cout, cin, gain_=gain, bias_std=0.3, bias_mean=0.0):
        sd[key + ".weight"] = (torch.randn(cout, cin, 1, 1, generator=g) * (gain_ * cin ** -0.5)).to(dtype)
        sd[key + ".bias"] = (torch.randn(cout, generator=g) * bias_std + bias_mean).to(dtype)

    emb, nb, bott = 128, 64, (out_conv_ch + 1 + 128) // 2
    conv("conv2", feat_ch, feat_ch)
    conv("seed_bin_regressor._net.0", 256, feat_ch)
    conv("seed_bin_regressor._net.2", nb, 256)
    if not normed:   # N's softplus centres increase over the bins, as in a trained model: the expectation then moves with p
        sd["seed_bin_regressor._net.2.bias"] = (torch.linspace(-2.0, 3.0, nb) + torch.randn(nb, generator=g) * 0.1).to(dtype)
    conv("seed_projector._net.0", 128, feat_ch)
    conv("seed_projector._net.2", emb, 128)
    for i, n in enumerate((16, 8, 4, 1)):
        conv(f"projectors.{i}._net.0", 128, feat_ch)
        conv(f"projectors.{i}._net.2", emb, 128)
        conv(f"attractors.{i}._net.0", 128, emb)
        if normed:     # relu(.) + 1e-3 of these should land in [0, 1]: small weights around a mid-range bias
            conv(f"attractors.{i}._net.2", 2 * n, 128, gain_=0.1, bias_std=0.1, bias_mean=0.45)
        else:
            conv(f"attractors.{i}._net.2", n, 128)
    conv("conditional_log_binomial.mlp.0", bott, out_conv_ch + 1 + emb)
    # small output gain: temperatures mostly well above min_temp, so the softmax over the bins is not a near-argmax that turns
    # rounding in the core into bin switches
    conv("conditional_log_binomial.mlp.2", 4, bott, gain_=0.5, bias_std=0.1)
    return sd
