"""CPU: pins the oracle to the original extension's own code.  Every case recomputes through oracle/ what the original's
functions and modules computed on the same seeded inputs, as recorded in tests/golden/oracle_pin_golden.npz by
tests/golden/make_pin_golden.py (which runs the original).  Exact outputs are compared through their SHA-256; outputs
compared within a tolerance of more than golden.make_pin_golden.SAMPLE values at a fixed, seeded sample of positions."""
import os
import warnings

import numpy as np
import pytest

from golden import make_pin_golden as mk
from oracle import normalmap as onm
from oracle import stereo as ost
from synth import synth_rgb


@pytest.fixture(scope="module")
def gold():
    warnings.filterwarnings("ignore")
    return np.load(os.path.join(os.path.dirname(__file__), "golden", "oracle_pin_golden.npz"))


@pytest.fixture(autouse=True)
def _recorded_thread_count():
    """the outputs were recorded with mk.THREADS torch threads, which keeps fp32 reductions in the same order here"""
    import torch
    n = torch.get_num_threads()
    torch.set_num_threads(mk.THREADS)
    yield
    torch.set_num_threads(n)


def _exact(gold, key, got):
    assert mk.digest(got) == str(gold[key]), key


def _close(gold, key, got, rel=None, abs_=None):
    """`got` has the recorded output's shape and is within rel * max|output| (or abs_) of it at every stored position;
    returns max|output|"""
    got = np.asarray(got)
    assert got.shape == tuple(gold[key + "_shape"]), key
    scale = float(gold[key + "_absmax"])
    err = float(np.abs(mk.sample(got).astype(np.float64) - gold[key].astype(np.float64)).max())
    assert err <= (abs_ if abs_ is not None else rel * scale), (key, err, scale)
    return scale


@pytest.mark.parametrize("fill", mk.STEREO_FILLS)
def test_stereo_oracle_equals_reference(gold, fill):
    for ci, (img, dep, div, sep, bal, ex) in enumerate(mk.stereo_cases()):
        b = ost.create_stereoimages(img, dep, div, sep, mk.STEREO_MODES, bal, ex, fill)
        assert len(b) == len(mk.STEREO_MODES)
        for m, y in zip(mk.STEREO_MODES, b):
            _exact(gold, f"stereo_{fill}_{ci}_{m}", np.asarray(y))


def test_stereo_oracle_float_depth_equals_reference(gold):
    img, dep = mk.stereo_float_depth_case()
    for fill in ['naive', 'polylines_sharp']:
        _exact(gold, f"stereo_float_{fill}", np.asarray(ost.create_stereoimages(img, dep, 3.0, fill_technique=fill)[0]))


def test_normalmap_oracle_equals_reference(gold):
    for seed in range(3):
        for ci, (pb, sb, qb, inv) in enumerate(mk.NORMAL_CASES):
            _exact(gold, f"normal_{seed}_{ci}", onm.create_normalmap(mk.normal_depth(seed), pb, sb, qb, inv, return_array=True))


# ---------------------------------------------------------------------------------------------------------------------
# D7 (round-2 row): the ZoeDepth-NK metric head oracle against the original module built around a stub core
# ---------------------------------------------------------------------------------------------------------------------
def _zoedepth_head(gold, seed, base_hw):
    lay = mk.layout(gold, "zoe_head")
    buffers = {k[len("zoe_buffer_"):]: gold[k] for k in gold.files if k.startswith("zoe_buffer_")}
    return mk.zoe_head_inputs(seed, base_hw, lay, buffers)


@pytest.mark.parametrize("seed,base_hw", mk.ZOE_HEADS)
def test_zoedepth_head_oracle_equals_reference(gold, seed, base_hw):
    import torch
    from oracle import zoedepth as ozd
    feats, sd = _zoedepth_head(gold, seed, base_hw)
    with torch.no_grad():
        got_depth, got_logits, name = ozd.metric_head(feats, sd)
    _close(gold, f"zoe_head_{seed}_logits", got_logits.numpy(), abs_=1e-5)
    _close(gold, f"zoe_head_{seed}_depth", got_depth.numpy(), rel=1e-5)


@pytest.mark.parametrize("pad,flip", mk.ZOE_TTA)
def test_zoedepth_tta_wrapper_equals_reference(gold, pad, flip):
    """DepthModel.infer (pad + flip augmentation) around the same head: the stub core ignores its input, so this pins the
    padding arithmetic, the bicubic resize back to the padded size, the crop and the flip average."""
    import torch
    from oracle import zoedepth as ozd
    feats, sd = _zoedepth_head(gold, 3, (2, 3))
    with torch.no_grad():
        got = ozd.infer(lambda t: ozd.metric_head(feats, sd)[0], mk.zoe_tta_input(), pad_input=pad, with_flip_aug=flip)
    assert got.shape == (2, 1, 40, 56)
    _close(gold, f"zoe_tta_{int(pad)}{int(flip)}", got.numpy(), rel=1e-5)


@pytest.mark.parametrize("smoothening", mk.VIDEO_SMOOTHENING)
def test_video_normalisation_equals_reference(gold, smoothening):
    """§8(f) rank 1 groundwork: cross-frame normalisation of video mode (src/video_mode.py:103-128)."""
    from oracle import video as ovid
    got = ovid.process_predictions(mk.video_frames(), smoothening)
    assert len(got) == int(gold[f"video_{smoothening}_count"])
    for i, g in enumerate(got):
        _exact(gold, f"video_{smoothening}_{i}", g)


# ---------------------------------------------------------------------------------------------------------------------
# D8 (round-2 row): LeReS ResNeXt-101 32x8d + decoder oracle against the original module with the same state_dict
# ---------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def leres_weights(gold):
    return mk.leres_weights(mk.layout(gold, "leres"))


def test_leres_synthetic_state_dict_matches_reference_module(gold):
    """oracle.synth_weights.make_leres_state_dict has exactly the original module's keys and shapes (strict load, only the
    BatchNorm step counters are left out) and the oracle reproduces the original module with it."""
    import torch
    from oracle import leres, synth_weights
    sd = synth_weights.make_leres_state_dict(seed=2)
    want = {name: shape for name, shape, _ in mk.layout(gold, "leres")}
    assert set(sd) <= set(want) and all(k.endswith("num_batches_tracked") for k in set(want) - set(sd))
    assert all(list(v.shape) == want[k] for k, v in sd.items())
    with torch.no_grad():
        got = leres.forward(sd, mk.leres_synth_input())
    assert _close(gold, "leres_synth", got.numpy(), rel=1e-5) > 1e-3


def test_leres_network_oracle_equals_reference(gold, leres_weights):
    import torch
    from oracle import leres
    with torch.no_grad():
        got = leres.forward(leres_weights, mk.leres_network_input())
    assert got.shape == (1, 1, 96, 128)
    assert _close(gold, "leres_network", got.numpy(), rel=1e-5) > 0


def test_leres_estimate_equals_reference(gold, leres_weights):
    """estimateleres (BGR flip, cv2 resize, scale_torch, cubic resize back) around the same network."""
    from oracle import leres
    rgb = synth_rgb(70, 90, 3)
    got, invert = leres.get_raw_prediction(rgb, leres_weights, 64, 96)
    assert invert is True and got.shape == (70, 90)
    _close(gold, "leres_estimate_img", got, rel=1e-5)
    _close(gold, "leres_estimate_u8", leres.estimateleres(rgb, leres_weights, 96, 64), rel=1e-5)


def test_pix2pix_unet_oracle_equals_reference(gold):
    """D9 groundwork: the BOOST merge network (10-level U-Net, norm 'none') and its input preparation."""
    import torch
    from oracle import pix2pix as op2p
    sd = mk.pix2pix_weights(mk.layout(gold, "pix2pix"))
    x = mk.pix2pix_input()
    assert x.shape == (1, 2, 1024, 1024) and float(x.min()) == -1.0 and float(x.max()) == 1.0
    with torch.no_grad():
        got = op2p.unet(sd, x.clone())
    assert got.shape == (1, 1, 1024, 1024)
    assert _close(gold, "pix2pix_unet", got.numpy(), abs_=1e-5) > 1e-3     # the seeded weights keep a signal through the 20 layers


# ---------------------------------------------------------------------------------------------------------------------
# Depth-Anything-V2 (D5 / D6): the oracle restatement against the original's own DepthAnythingV2 module
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("encoder,hw,net", mk.DAV2_CASES)
def test_dav2_oracle_equals_reference(gold, encoder, hw, net):
    """ddepth_anything_v2/depth_anything_v2/dpt.py:176-221 + src/depthmap_generation.py:375-403,548-559: the synthetic
    weights have exactly the original module's keys and shapes (it loads them strictly), and its own pre-processing /
    forward / final resize on them matches oracle.dav2.get_raw_prediction on the same uint8 image."""
    from oracle import dav2 as odav2
    from oracle import synth_weights
    sd = synth_weights.make_dav2_state_dict(encoder, seed=1)
    assert {k: list(v.shape) for k, v in sd.items()} == {name: shape for name, shape, _ in mk.layout(gold, "dav2_" + encoder)}
    got, invert = odav2.get_raw_prediction(synth_rgb(hw[0], hw[1], 3), sd, encoder, net)
    assert invert is False
    key = f"dav2_{encoder}_{hw[0]}x{hw[1]}_{net}"
    assert got.shape == tuple(hw)
    assert float(gold[key].max() - gold[key].min()) > 0.1      # a non-degenerate map (default init would be identically zero)
    _close(gold, key, got, rel=1e-6)


# ---------------------------------------------------------------------------------------------------------------------
# D9: the BOOST driver (resolution search, patch selection, double estimation, merge + blend) against the original's own
# functions.  The two networks are stand-ins (cheap, deterministic, the same on both sides): the real ones are pinned above.
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("hw,rmax", mk.BOOST_SELECTION)
def test_boost_selection_equals_reference(gold, hw, rmax):
    """calculateprocessingres + generatepatchs + generatemask: integer / index results, compared exactly."""
    from oracle import boost
    img = mk.boost_image(hw, 11)
    got = boost.calculateprocessingres(img, 448, 0.2, 3, rmax)
    want = gold[f"boost_res_{hw[0]}x{hw[1]}"]
    assert got[0] == want[0] and got[1] == want[1]
    big, factor = mk.boost_big_image(img, got, rmax)
    gotp = boost.generatepatchs(big, 896, factor)
    wantp = gold[f"boost_rects_{hw[0]}x{hw[1]}"]
    assert len(gotp) == len(wantp) and len(gotp) > 0
    assert [list(kv[1]["rect"]) for kv in gotp] == wantp.tolist()
    _exact(gold, "boost_mask", boost.generatemask((300, 300)))


def test_boost_estimate_equals_reference(gold):
    """estimateboost end to end (model type 0: receptive field 448, patches at 896) with the stand-in networks."""
    from oracle import boost
    info = {}
    got = boost.estimateboost(mk.boost_image((300, 420), 12), 0, mk.fake_estimate, mk.fake_merge, 1600, info=info)
    assert got.shape == (300, 420) and len(info["patches"]) >= 2
    _close(gold, "boost_estimate", got, rel=1e-6)


def test_pix2pix_synthetic_state_dict_matches_reference_module(gold):
    """oracle.synth_weights.make_pix2pix_state_dict loads strictly into the original generator"""
    from oracle import synth_weights
    sd = synth_weights.make_pix2pix_state_dict(seed=1)
    assert {k: list(v.shape) for k, v in sd.items()} == {name: shape for name, shape, _ in mk.layout(gold, "pix2pix")}
