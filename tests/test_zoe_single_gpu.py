"""GPU: ZoeDepth-N / -K (model types 7 / 8): the single-head kernels against torch fp32, the engine against the fp32 oracle
(oracle/zoedepth_single.py:get_raw_prediction_single, its head and TTA pinned to the reference module by test_zoe_single_pin.py),
batch independence, the real DPT-BEiT-L-384 configuration through ModelHolder and one funnel run.
Bar: max |d - oracle| / range <= 3.5e-3 and mean <= 8.3e-4, the worst ZoeDepth-NK figures of DESIGN.md (c).  The error of
the reference's own fp16 policy is printed beside ours where it is finite (the reference runs N / K halved, and N in fp16
is known to break down)."""
import math

import numpy as np
import pytest

import precision

pytestmark = pytest.mark.gpu

BAR_MAX, BAR_MEAN = 3.5e-3, 8.3e-4


def make_sd(core, model_type, seed):
    from oracle import beit_dpt, synth_weights, zoedepth_single
    csd = synth_weights.make_beit_dpt_state_dict(core, seed=seed)
    hsd = zoedepth_single.make_zoedepth_single_state_dict(model_type, feat_ch=beit_dpt.CONFIGS[core]['features'], seed=seed + 100)
    sd = {"core.core." + k: v for k, v in csd.items()}
    sd.update(hsd)
    return sd


def fp16_policy_error(img, sd, model_type, net_w, net_h, core_name, want, dev):
    """the oracle network in fp16 on the GPU (core, head, TTA): the reference's `.half()` precision policy"""
    import torch
    from oracle import beit_dpt
    from oracle import zoedepth as ozd
    from oracle import zoedepth_single as ozs
    core_sd = precision.HalfView({k[len("core.core."):]: v for k, v in sd.items() if k.startswith("core.core.")}, dev)
    head_sd = {k: v.to(dev, torch.float16) for k, v in sd.items() if not k.startswith("core.")}

    def model_fn(x):
        rel, feats = beit_dpt.forward(core_sd, ozd.prep_for_midas(x, net_w, net_h), core_name, return_features=True)
        return ozs.metric_head_single(feats, rel, head_sd, model_type)

    x = torch.from_numpy(np.ascontiguousarray(np.asarray(img))).permute(2, 0, 1).float().div(255.0).unsqueeze(0).to(dev, torch.float16)
    with torch.no_grad():
        out = ozd.infer(model_fn, x, pad_input=True, with_flip_aug=True)
    return precision.norm_err(out.squeeze().float().cpu().numpy(), want)


def check(label, got, want, ref16=None):
    mx, mean = precision.norm_err(got, want)
    line = f"[precision] {label}: ours max {mx:.3e} mean {mean:.3e}"
    if ref16 is not None and all(math.isfinite(v) for v in ref16):
        line += f" | reference fp16 policy max {ref16[0]:.3e} mean {ref16[1]:.3e}"
    print(line)
    assert np.isfinite(got).all() and mx <= BAR_MAX and mean <= BAR_MEAN, (label, mx, mean)


# ---- kernel units ------------------------------------------------------------------------------------------------------
def _attractor_torch(A, n, normed, b_prev, H, W, mn, mx):
    import torch
    import torch.nn.functional as F
    Fw = b_prev.shape[0]
    if normed:
        a = torch.relu(A[:, 0:2 * n:2]) + 1e-3
    else:
        a = F.softplus(A[:, :n])
    a = a.reshape(Fw, H, W, n).permute(0, 3, 1, 2)                               # [F, n, H, W]
    b = F.interpolate(b_prev.permute(0, 3, 1, 2), (H, W), mode="bilinear", align_corners=True)
    dx = a.unsqueeze(2) - b.unsqueeze(1)
    b_new = b + torch.mean(dx / (1 + 300.0 * dx * dx), dim=1)
    B = torch.clip(torch.sort((mx - mn) * b_new + mn, dim=1)[0], mn, mx)
    return b_new.permute(0, 2, 3, 1), B.permute(0, 2, 3, 1)


@pytest.mark.parametrize("normed", [False, True])
@pytest.mark.parametrize("n", [16, 8, 4, 1])
def test_attractor_single_kernel(cuda_device, n, normed):
    import torch
    from depthmap_b200 import _lib
    L = _lib.load()
    g = torch.Generator(device=cuda_device).manual_seed(10 * n + normed)
    Fw, Hp, Wp, H, W, mn, mx = 3, 5, 7, 9, 13, 1e-3, 10.0
    A = (torch.randn(Fw * H * W, 32, generator=g, device=cuda_device) * 0.6 + 0.3).contiguous()
    b_prev = torch.rand(Fw, Hp, Wp, 64, generator=g, device=cuda_device) * 1.4 - 0.2     # partly outside [0, 1]: clipped bins
    b_prev[0, 1, 2, :] = 0.5                                                           # equal centres: sort ties
    b_prev[1, :, :, 10:20] = 0.25
    b_out = torch.empty(Fw, H, W, 64, device=cuda_device)
    B_out = torch.full((Fw, H, W, 64), float("nan"), device=cuda_device)
    _lib.check(L.dm_zoe_attractor_single(A.data_ptr(), 32, n, int(normed), b_prev.data_ptr(), Fw, Hp, Wp, H, W, mn, mx, b_out.data_ptr(),
                                         B_out.data_ptr() if normed else None, _lib.stream_ptr()), "dm_zoe_attractor_single")
    torch.cuda.synchronize()
    want_b, want_B = _attractor_torch(A, n, normed, b_prev, H, W, mn, mx)
    assert torch.allclose(b_out, want_b, rtol=1e-5, atol=2e-6), float((b_out - want_b).abs().max())
    if normed:
        assert torch.allclose(B_out, want_B, rtol=1e-5, atol=2e-5), float((B_out - want_B).abs().max())
        assert (B_out == mn).any() and (B_out == mx).any() and (B_out[:, :, :, 1:] >= B_out[:, :, :, :-1]).all()


def test_seed_normed_kernel(cuda_device):
    import torch
    from depthmap_b200 import _lib
    L = _lib.load()
    g = torch.Generator(device=cuda_device).manual_seed(3)
    rows, ld, mn, mx = 1000, 68, 1e-3, 10.0
    seed = torch.randn(rows, ld, generator=g, device=cuda_device)
    out = torch.empty(rows, 64, device=cuda_device)
    _lib.check(L.dm_zoe_seed_normed(seed.data_ptr(), ld, rows, mn, mx, out.data_ptr(), _lib.stream_ptr()), "dm_zoe_seed_normed")
    torch.cuda.synchronize()
    w = torch.relu(seed[:, :64]) + 1e-3
    w = (mx - mn) * (w / w.sum(dim=1, keepdim=True))
    edges = torch.cumsum(torch.cat([torch.full((rows, 1), mn, device=cuda_device), w], dim=1), dim=1)
    want = (0.5 * (edges[:, :-1] + edges[:, 1:]) - mn) / (mx - mn)
    assert torch.allclose(out, want, rtol=1e-5, atol=2e-6), float((out - want).abs().max())
    assert (out[:, 1:] > out[:, :-1]).all() and float(out.min()) > 0 and float(out.max()) < 1


# ---- engine against the oracle -------------------------------------------------------------------------------------------
@pytest.mark.parametrize("model_type", [7, 8])
@pytest.mark.parametrize("seed,hw,net", [(1, (96, 128), (64, 64)), (3, (70, 50), (64, 96)), (1, (64, 64), (96, 96))])
def test_zoe_single_tiny_core_vs_oracle(cuda_device, model_type, seed, hw, net):
    import torch
    from depthmap_b200.depthmap_generation import ZoeDepthEngine
    from oracle import zoedepth_single as ozs
    from synth import synth_rgb
    sd = make_sd('beit_tiny', model_type, seed)
    eng = ZoeDepthEngine(sd, model_type, cuda_device, core_name='beit_tiny')
    imgs = [synth_rgb(hw[0], hw[1], 5 + s) for s in range(2)]
    got = eng.forward_batch(torch.from_numpy(np.stack(imgs)).to(cuda_device), net[0], net[1]).cpu().numpy()
    assert got.shape == (2, hw[0], hw[1]) and got.dtype == np.float32
    for i, img in enumerate(imgs):
        want, invert = ozs.get_raw_prediction_single(img, sd, model_type, net[0], net[1], core_name='beit_tiny')
        assert invert is True and want.max() - want.min() > 0.05
        ref16 = fp16_policy_error(img, sd, model_type, net[0], net[1], 'beit_tiny', want, cuda_device)
        check(f"zoedepth type {model_type} tiny seed{seed} {hw} net {net} img{i}", got[i], want, ref16)


@pytest.mark.parametrize("model_type", [7, 8])
def test_zoe_single_batch_equals_single_images(cuda_device, model_type):
    import torch
    from depthmap_b200.depthmap_generation import ZoeDepthEngine
    from synth import synth_rgb
    eng = ZoeDepthEngine(make_sd('beit_tiny', model_type, 2), model_type, cuda_device, core_name='beit_tiny')
    rgb = torch.from_numpy(np.stack([synth_rgb(80, 112, 30 + i) for i in range(3)])).to(cuda_device)
    batch = eng.forward_batch(rgb, 64, 96).cpu()
    for i in range(3):
        one = eng.forward_batch(rgb[i:i + 1].contiguous(), 64, 96).cpu()
        assert torch.equal(batch[i], one[0]), (i, float((batch[i] - one[0]).abs().max()))


def test_zoe_single_rejects_bad_checkpoints(cuda_device):
    from depthmap_b200.depthmap_generation import ZoeDepthEngine
    sd = make_sd('beit_tiny', 8, 1)
    missing = {k: v for k, v in sd.items() if k != 'attractors.2._net.2.weight'}
    with pytest.raises(ValueError, match=r"attractors\.2\._net\.2\.weight"):
        ZoeDepthEngine(missing, 8, cuda_device, core_name='beit_tiny')
    # N's attractor layers have n outputs, K's 2n: a K checkpoint is not an N checkpoint
    with pytest.raises(ValueError, match=r"attractors\.0\._net\.2\.weight"):
        ZoeDepthEngine(sd, 7, cuda_device, core_name='beit_tiny')
    with pytest.raises(ValueError, match="model types 7"):
        ZoeDepthEngine(sd, 9, cuda_device, core_name='beit_tiny')


# ---- the real configuration ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("model_type,hw", [(7, (384, 320)), (8, (200, 600))])
def test_zoe_single_beit384_core(cuda_device, model_type, hw):
    """DPT-BEiT-L-384 core through ModelHolder at the UI default net size of the type (7: 384 x 512, 8: 384 x 768), PIL in."""
    from PIL import Image
    from depthmap_b200.depthmap_generation import ModelHolder
    from oracle import zoedepth_single as ozs
    from synth import synth_rgb
    sd = make_sd('beitl16_384', model_type, 3)
    mh = ModelHolder()
    mh.weights_provider = lambda t: sd
    mh.ensure_models(model_type, cuda_device, False)
    net = ModelHolder.get_default_net_size(model_type)
    assert net == {7: [384, 512], 8: [384, 768]}[model_type]
    img = synth_rgb(hw[0], hw[1], 21)
    pred, invert = mh.get_raw_prediction(Image.fromarray(img), net[0], net[1])
    assert invert is True and pred.shape == hw and pred.dtype == np.float32
    want, _ = ozs.get_raw_prediction_single(img, sd, model_type, net[0], net[1], core_name='beitl16_384')
    ref16 = fp16_policy_error(img, sd, model_type, net[0], net[1], 'beitl16_384', want, cuda_device)
    check(f"zoedepth type {model_type} beitl16_384 ({hw[0]}x{hw[1]} image, net {net})", pred, want, ref16)
    mh.unload_models()


def test_zoe_single_boost_still_raises(cuda_device):
    from depthmap_b200.depthmap_generation import ModelHolder
    mh = ModelHolder()
    mh.weights_provider = lambda t: {}
    for t in (7, 8):
        with pytest.raises(NotImplementedError):
            mh.ensure_models(t, cuda_device, True)


def test_zoe_n_funnel_yields_depth(cuda_device):
    from PIL import Image
    from depthmap_b200 import core
    from synth import synth_rgb
    sd = make_sd('beitl16_384', 7, 1)
    holder = core.get_model_holder()
    holder.unload_models()
    holder.weights_provider = lambda t: sd
    try:
        inp = dict(compute_device='GPU', model_type=7, net_width=64, net_height=96, net_size_match=False, boost=False,
                   do_output_depth=True, gen_stereo=False, gen_normalmap=False)
        out = list(core.core_generation_funnel(None, [Image.fromarray(synth_rgb(70, 90, 4))], None, None, inp, ops={}))
    finally:
        holder.unload_models()
        holder.weights_provider = None
    kinds = [k for _, k, _ in out]
    assert 'depth' in kinds
    d = np.asarray([v for _, k, v in out if k == 'depth'][0])
    assert d.shape[:2] == (70, 90) and d.max() > d.min()
