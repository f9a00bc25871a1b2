"""Mints tests/golden/oracle_pin_golden.npz: what the original extension's own functions and modules compute on the seeded
inputs of tests/test_oracle_pin.py, which compares the oracle against it.  Minting needs a checkout of the original
extension (oracle/ref_loader.py finds it through DEPTHMAP_REFERENCE_ROOT):

    python tests/golden/make_pin_golden.py

Inputs and weights are not stored: both sides rebuild them from the seeds and builders below.  Where weights are drawn in
a module's parameter order, the fixture stores that order ("layout_*": name, shape, parameter or buffer) and the values of
buffers the module computes itself.  An output the test compares exactly is stored as the SHA-256 of its dtype, shape and
bytes.  An output compared within a tolerance is stored as values; one of more than SAMPLE values at SAMPLE fixed, seeded
positions, with its shape and its max |value| (the scale of the tolerances).
"""
import hashlib
import json
import os
import sys
import warnings

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from synth import noise_depth_u16, noise_rgb, synth_depth_u16, synth_rgb  # noqa: E402

PATH = os.path.join(HERE, "oracle_pin_golden.npz")
SAMPLE = 2048
THREADS = 1      # torch intra-op threads on both sides: a reduction split over another thread count rounds differently
STEREO_FILLS = ['none', 'naive', 'naive_interpolating', 'polylines_soft', 'polylines_sharp']
STEREO_MODES = ['left-right', 'red-cyan-anaglyph']
NORMAL_CASES = [(None, 3, None, False), (None, 5, None, True), (None, None, None, False), (3, 3, 3, False),
                (None, 11, None, False), (9, 3, None, True), (None, 3, 11, False), (None, 31, None, False), (31, 3, 31, False)]
ZOE_HEADS = [(0, (3, 4)), (1, (4, 3)), (2, (2, 2))]
ZOE_TTA = [(True, True), (True, False), (False, True)]
VIDEO_SMOOTHENING = ["none", "experimental", "something-else"]
DAV2_CASES = [("vits", (70, 98), 70), ("vits", (84, 56), 56), ("vitb", (70, 70), 70)]
BOOST_SELECTION = [((300, 420), 1600), ((520, 360), 1200)]


def sample_index(n):
    return np.sort(np.random.default_rng(n).choice(n, SAMPLE, replace=False))


def sample(a):
    """`a` flattened, at the positions an output of its size is stored at (all of it when it is small)"""
    a = np.asarray(a).reshape(-1)
    return a if a.size <= SAMPLE else a[sample_index(a.size)]


def digest(a):
    a = np.ascontiguousarray(a)
    return f"{a.dtype.str} {list(a.shape)} {hashlib.sha256(a.tobytes()).hexdigest()}"


def put_exact(out, key, a):
    out[key] = np.array(digest(a))


def put(out, key, a):
    a = np.asarray(a)
    out[key] = sample(a)
    out[key + "_shape"] = np.array(a.shape, np.int64)
    out[key + "_absmax"] = np.abs(a).max().astype(np.float64)


def put_layout(out, key, sd, param_names):
    out["layout_" + key] = np.array(json.dumps([[k, list(v.shape), k in param_names] for k, v in sd.items()]))


def layout(gold, key):
    return json.loads(str(gold["layout_" + key]))


# ---------------------------------------------------------------------------------------------------------------------
# seeded inputs and weights, shared with tests/test_oracle_pin.py
# ---------------------------------------------------------------------------------------------------------------------
def stereo_cases():
    """(image, depth, divergence, separation, balance, exponent) of every stereo case, the same for each fill technique"""
    rng = np.random.default_rng(11)
    for (h, w, seed, kind) in [(21, 67, 10, 'smooth'), (16, 50, 11, 'noise')]:
        img = synth_rgb(h, w, seed) if kind == 'smooth' else noise_rgb(h, w, seed)
        dep = synth_depth_u16(h, w, seed) if kind == 'smooth' else noise_depth_u16(h, w, seed)
        for _ in range(3):
            div, sep = float(rng.uniform(0.05, 15)), float(rng.uniform(-5, 5))
            bal, ex = float(rng.uniform(-1, 1)), float(rng.choice([1.0, 2.0]))
            yield img, dep, div, sep, bal, ex


def stereo_float_depth_case():
    return noise_rgb(12, 40, 5), np.random.default_rng(5).random((12, 40)).astype(np.float32)


def normal_depth(seed):
    return synth_depth_u16(30, 41, seed) if seed else noise_depth_u16(30, 41, seed)


def zoe_features(g, base_hw):
    import torch
    h, w = base_hw
    shapes = [(32, 16 * h, 16 * w), (256, h, w), (256, 2 * h, 2 * w), (256, 4 * h, 4 * w), (256, 8 * h, 8 * w), (256, 16 * h, 16 * w)]
    feats = [torch.randn(2, c, hh, ww, generator=g) * 0.7 for c, hh, ww in shapes]
    feats[0] = feats[0].abs()                      # out_conv is a post-ReLU activation in the core
    return feats


def zoe_head_weights(g, lay, buffers):
    """the metric head's state_dict: parameters drawn from `g` in the module's parameter order, with enough spread to
    exercise every branch; buffers as the module computes them"""
    import torch
    sd = {}
    for name, shape, is_param in lay:
        if is_param:
            p = torch.randn(shape, generator=g) * (0.05 if len(shape) > 1 else 0.02)
            sd[name] = p + 1.0 if name.endswith("norm1.weight") or name.endswith("norm2.weight") else p
        else:
            sd[name] = torch.from_numpy(buffers[name].copy())
    return sd


def zoe_head_inputs(seed, base_hw, lay, buffers):
    import torch
    g = torch.Generator().manual_seed(seed)
    feats = zoe_features(g, base_hw)
    return feats, zoe_head_weights(g, lay, buffers)


def zoe_tta_input():
    import torch
    return torch.rand(2, 3, 40, 56, generator=torch.Generator().manual_seed(5))


def video_frames():
    rng = np.random.default_rng(11)
    return [(rng.standard_normal((24, 32)) * (1 + 0.3 * i) + 0.1 * i).astype(np.float32) for i in range(7)]


def leres_weights(lay):
    """seeded LeReS weights and running statistics that keep activations O(1) through 100+ layers"""
    import torch
    g = torch.Generator().manual_seed(21)
    sd = {}
    for name, shape, is_param in lay:
        if not is_param:
            continue
        if len(shape) == 4:
            fan_in = shape[1] * shape[2] * shape[3]
            sd[name] = torch.randn(shape, generator=g) * (1.0 / fan_in ** 0.5)
        elif name.endswith(".weight"):
            sd[name] = (0.3 if "bn3" in name else 1.0) + 0.05 * torch.randn(shape, generator=g)
        else:
            sd[name] = 0.05 * torch.randn(shape, generator=g)
    for name, shape, is_param in lay:
        if is_param:
            continue
        if name.endswith("running_mean"):
            sd[name] = 0.1 * torch.randn(shape, generator=g)
        elif name.endswith("running_var"):
            sd[name] = 0.5 + torch.rand(shape, generator=g)
        else:
            sd[name] = torch.zeros(shape, dtype=torch.long)     # num_batches_tracked
    return {name: sd[name] for name, _, _ in lay}


def leres_synth_input():
    import torch
    return torch.randn(1, 3, 64, 96, generator=torch.Generator().manual_seed(4))


def leres_network_input():
    import torch
    return torch.randn(1, 3, 96, 128, generator=torch.Generator().manual_seed(4))


def pix2pix_weights(lay):
    import torch
    g = torch.Generator().manual_seed(31)
    return {name: torch.randn(shape, generator=g) * (1.6 / (shape[1] * 16) ** 0.5) if len(shape) == 4
            else 0.05 * torch.randn(shape, generator=g) for name, shape, _ in lay}


def pix2pix_input():
    from oracle import pix2pix as op2p
    rng = np.random.default_rng(5)
    outer = rng.standard_normal((1024, 1024)).astype(np.float32)
    inner = (outer * 0.5 + rng.standard_normal((1024, 1024)).astype(np.float32)).astype(np.float32)
    return op2p.merge_input(outer, inner)


class FakeLeres:
    """stands for RelDepthModel in BOOST: estimateleres calls model.depth_model(normalised [1,3,h,w])"""

    @staticmethod
    def depth_model(x):
        import torch
        import torch.nn.functional as F
        g = x.mean(dim=1, keepdim=True)
        return F.avg_pool2d(g, 9, 1, 4) + 0.25 * torch.sin(3.0 * x[:, :1]) + 0.1 * x[:, 2:3]


class FakePix2Pix:
    """stands for Pix2Pix4DepthModel: set_input / test / get_current_visuals (pix2pix/models/pix2pix4depth_model.py:96-116)"""

    def set_input(self, outer, inner):
        from oracle import pix2pix as op2p
        self.real_A = op2p.merge_input(outer, inner)

    def test(self):
        import torch
        o, i = self.real_A[:, :1], self.real_A[:, 1:]
        self.fake_B = torch.tanh(0.7 * o + 0.5 * i + 0.1 * o * i)

    def get_current_visuals(self):
        return {"fake_B": self.fake_B}


def fake_estimate(img, msize):
    """FakeLeres through the oracle's estimateleres pre- and post-processing"""
    import cv2
    import torch
    from oracle import leres
    with torch.no_grad():
        pred = FakeLeres.depth_model(leres.preprocess(img, msize, msize)).squeeze().numpy()
    return cv2.resize(pred, (img.shape[1], img.shape[0]), interpolation=cv2.INTER_CUBIC)


def fake_merge(outer, inner):
    p = FakePix2Pix()
    p.set_input(outer, inner)
    p.test()
    return p.fake_B.squeeze().numpy()


def boost_image(hw, seed):
    import cv2
    return cv2.cvtColor(synth_rgb(hw[0], hw[1], seed), cv2.COLOR_BGR2RGB) / 255.0


def boost_big_image(img, whole_size, rmax):
    """the image resized for patch selection at the resolution calculateprocessingres chose"""
    import cv2
    from oracle import boost
    factor = max(min(1, 4 * whole_size[1] * whole_size[0] / rmax), 0.2)
    a, b = boost.target_size(img.shape, whole_size[0], factor)
    return cv2.resize(img, (b, a), interpolation=cv2.INTER_CUBIC), factor


# ---------------------------------------------------------------------------------------------------------------------
# the original's side
# ---------------------------------------------------------------------------------------------------------------------
def _stereo(out, ref_loader):
    rs, rn = ref_loader.stereo_module(), ref_loader.normalmap_module()
    for fill in STEREO_FILLS:
        for ci, (img, dep, div, sep, bal, ex) in enumerate(stereo_cases()):
            res = rs.create_stereoimages(img, dep, div, sep, STEREO_MODES, bal, ex, fill)
            for m, r in zip(STEREO_MODES, res):
                put_exact(out, f"stereo_{fill}_{ci}_{m}", np.asarray(r))
    img, dep = stereo_float_depth_case()
    for fill in ['naive', 'polylines_sharp']:
        put_exact(out, f"stereo_float_{fill}", np.asarray(rs.create_stereoimages(img, dep, 3.0, fill_technique=fill)[0]))
    for seed in range(3):
        for ci, (pb, sb, qb, inv) in enumerate(NORMAL_CASES):
            put_exact(out, f"normal_{seed}_{ci}", np.asarray(rn.create_normalmap(normal_depth(seed), pb, sb, qb, inv)))


def _zoedepth(out, ref_loader):
    import torch
    import torch.nn as nn
    ref_loader.bootstrap()
    from dzoedepth.models.zoedepth_nk.zoedepth_nk_v1 import ZoeDepthNK
    from oracle import zoedepth as ozd

    def head(seed, base_hw):
        g = torch.Generator().manual_seed(seed)
        feats = zoe_features(g, base_hw)

        class StubCore(nn.Module):                 # hands the head fixed activations (MidasCore.forward, midas.py:258-276)
            output_channels = (256, 256, 256, 256, 256)

            def forward(self, x, denorm=False, return_rel_depth=False):
                return torch.zeros(x.shape[0], x.shape[2], x.shape[3]), [f.clone() for f in feats]

        cfg = {k: ozd.CONFIG[k] for k in ("bin_embedding_dim", "n_attractors", "attractor_alpha", "attractor_gamma", "min_temp", "max_temp")}

        class AttrDict(dict):                      # the original reads its config entries as attributes (EasyDict)
            __getattr__ = dict.__getitem__

        model = ZoeDepthNK(StubCore(), bin_conf=[AttrDict(c) for c in ozd.CONFIG["bin_conf"]], bin_centers_type="softplus",
                           attractor_kind="mean", attractor_type="inv", memory_efficient=True, **cfg).eval()
        with torch.no_grad():
            for name, p in model.named_parameters():
                p.copy_(torch.randn(p.shape, generator=g) * (0.05 if p.ndim > 1 else 0.02))
                if name.endswith("norm1.weight") or name.endswith("norm2.weight"):
                    p.add_(1.0)
        sd = {k: v.detach().clone() for k, v in model.state_dict().items() if not k.startswith("core.")}
        params = {k for k, _ in model.named_parameters()}
        if "layout_zoe_head" not in out:
            put_layout(out, "zoe_head", sd, params)
            for k, v in sd.items():
                if k not in params:
                    out["zoe_buffer_" + k] = v.numpy()
        # the test rebuilds the weights from the layout: check that it gets these
        lay = layout(out, "zoe_head")
        buffers = {k[len("zoe_buffer_"):]: v for k, v in out.items() if k.startswith("zoe_buffer_")}
        feats2, sd2 = zoe_head_inputs(seed, base_hw, lay, buffers)
        assert list(sd2) == list(sd) and all(torch.equal(sd[k], sd2[k]) for k in sd)
        assert all(torch.equal(a, b) for a, b in zip(feats, feats2))
        return model, feats

    for seed, base_hw in ZOE_HEADS:
        model, feats = head(seed, base_hw)
        with torch.no_grad():
            want = model(torch.zeros(2, 3, feats[0].shape[2], feats[0].shape[3]))
        put(out, f"zoe_head_{seed}_logits", want["domain_logits"].numpy())
        put(out, f"zoe_head_{seed}_depth", want["metric_depth"].numpy())
    model, _ = head(3, (2, 3))
    for pad, flip in ZOE_TTA:
        with torch.no_grad():
            want = model.infer(zoe_tta_input(), pad_input=pad, with_flip_aug=flip)
        put(out, f"zoe_tta_{int(pad)}{int(flip)}", want.numpy())


def _video(out, ref_loader):
    ref_loader.bootstrap()
    from src import video_mode
    for sm in VIDEO_SMOOTHENING:
        frames = video_mode.process_predicitons(video_frames(), sm)
        out[f"video_{sm}_count"] = np.array(len(frames))
        for i, f in enumerate(frames):
            put_exact(out, f"video_{sm}_{i}", f)


def _leres(out, ref_loader):
    import cv2
    import torch
    ref_loader.bootstrap()
    from lib.multi_depth_model_woauxi import RelDepthModel
    from src import depthmap_generation as dg
    from oracle import leres
    dg.depthmap_device = torch.device("cpu")
    model = RelDepthModel(backbone="resnext101").eval()
    sd = model.state_dict()
    params = {k for k, _ in model.named_parameters()}
    put_layout(out, "leres", sd, params)
    # module with the synthetic weights of oracle/synth_weights.py
    from oracle import synth_weights
    model.load_state_dict(synth_weights.make_leres_state_dict(seed=2), strict=False)
    with torch.no_grad():
        put(out, "leres_synth", model.depth_model(leres_synth_input()).numpy())
    # module with the seeded weights the test rebuilds from the layout
    g = torch.Generator().manual_seed(21)
    with torch.no_grad():
        for name, p in model.named_parameters():
            if p.ndim == 4:
                fan_in = p.shape[1] * p.shape[2] * p.shape[3]
                p.copy_(torch.randn(p.shape, generator=g) * (1.0 / fan_in ** 0.5))
            elif name.endswith(".weight"):
                p.copy_((0.3 if "bn3" in name else 1.0) + 0.05 * torch.randn(p.shape, generator=g))
            else:
                p.copy_(0.05 * torch.randn(p.shape, generator=g))
        for name, b in model.named_buffers():
            if name.endswith("running_mean"):
                b.copy_(0.1 * torch.randn(b.shape, generator=g))
            elif name.endswith("running_var"):
                b.copy_(0.5 + torch.rand(b.shape, generator=g))
            else:
                b.zero_()
    sd = model.state_dict()
    sd2 = leres_weights(layout(out, "leres"))
    assert list(sd2) == list(sd) and all(torch.equal(sd[k], sd2[k]) for k in sd)
    del sd2
    with torch.no_grad():
        put(out, "leres_network", model.depth_model(leres_network_input()).numpy())
    rgb = synth_rgb(70, 90, 3)
    img = cv2.cvtColor(rgb, cv2.COLOR_BGR2RGB) / 255.0       # what ModelHolder.get_raw_prediction hands over (:381)
    put(out, "leres_estimate_img", dg.estimateleres(img, model, 64, 96))
    put(out, "leres_estimate_u8", dg.estimateleres(rgb, model, 96, 64))


def _pix2pix(out, ref_loader):
    import torch
    ref_loader.bootstrap()
    from pix2pix.models import networks
    net = networks.define_G(2, 1, 64, 'unet_1024', 'none', False, 'normal', 0.02, []).eval()
    params = {k for k, _ in net.named_parameters()}
    put_layout(out, "pix2pix", net.state_dict(), params)
    net.load_state_dict(pix2pix_weights(layout(out, "pix2pix")), strict=True)
    with torch.no_grad():
        put(out, "pix2pix_unet", net(pix2pix_input()).numpy())


def _dav2(out, ref_loader):
    import cv2
    import torch
    import torch.nn.functional as F
    from oracle import dav2 as odav2
    from oracle import synth_weights
    cls = ref_loader.dav2_class()
    for encoder, hw, net in DAV2_CASES:
        cfg = odav2.CONFIGS[encoder]
        model = cls(encoder=encoder, features=cfg['features'], out_channels=cfg['out_channels']).eval()
        if "layout_dav2_" + encoder not in out:
            put_layout(out, "dav2_" + encoder, model.state_dict(), {k for k, _ in model.named_parameters()})
        model.load_state_dict(synth_weights.make_dav2_state_dict(encoder, seed=1), strict=True)
        rgb = synth_rgb(hw[0], hw[1], 3)
        # the original's call chain, verbatim: get_raw_prediction (:381) -> estimatedepthanything_v2 (:548-559)
        img = cv2.cvtColor(np.asarray(rgb), cv2.COLOR_BGR2RGB) / 255.0
        with torch.no_grad():
            image = cv2.cvtColor((img * 255.1).astype('uint8'), cv2.COLOR_BGR2RGB)
            image, (h, w) = model.image2tensor(image, net)
            depth = model.forward(image.to('cpu'))
            depth = F.interpolate(depth[:, None], (h, w), mode="bilinear", align_corners=True)[0, 0]
        put(out, f"dav2_{encoder}_{hw[0]}x{hw[1]}_{net}", depth.numpy())


def _boost(out, ref_loader):
    import torch
    ref_loader.bootstrap()
    from src import depthmap_generation as dg
    dg.depthmap_device = torch.device("cpu")
    import skimage.measure as sm
    from oracle import boost
    sm.block_reduce = lambda img, block, func: boost.block_reduce_max(img, block[0])   # skimage stand-in: zero-padded max pool
    dg.skimage = __import__("skimage")
    for hw, rmax in BOOST_SELECTION:
        img = boost_image(hw, 11)
        whole = dg.calculateprocessingres(img, 448, 0.2, 3, rmax)
        out[f"boost_res_{hw[0]}x{hw[1]}"] = np.array(whole[:2], np.float64)
        big, factor = boost_big_image(img, whole, rmax)
        out[f"boost_rects_{hw[0]}x{hw[1]}"] = np.array([kv[1]["rect"] for kv in dg.generatepatchs(big, 896, factor)], np.int64)
    put_exact(out, "boost_mask", dg.generatemask((300, 300)))
    put(out, "boost_estimate", dg.estimateboost(boost_image((300, 420), 12), FakeLeres(), 0, FakePix2Pix(), 1600))


def main():
    import torch
    from oracle import ref_loader
    warnings.filterwarnings("ignore")
    torch.set_num_threads(THREADS)
    out = {}
    for part in (_stereo, _zoedepth, _video, _leres, _pix2pix, _dav2, _boost):
        part(out, ref_loader)
        print(part.__name__[1:], "done", flush=True)
    np.savez_compressed(PATH, **out)
    print("wrote", len(out), "arrays,", os.path.getsize(PATH), "bytes")


if __name__ == "__main__":
    main()
