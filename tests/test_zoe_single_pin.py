"""CPU: the oracle of ZoeDepth-N / -K (model types 7 / 8; oracle/zoedepth_single.py:metric_head_single) equals what the original
extension's own ZoeDepth module computes on the same seeded inputs, as recorded in tests/golden/zoe_single_pin_golden.npz by
tests/golden/make_zoe_single_golden.py: the head for two seeds per variant and the pad / flip test-time augmentation, within
1e-5 of the output's max |value|.  Also pins the resolved configuration (K keeps max_depth 10, the counts are 16, 8, 4, 1) and
the checkpoint layout the synthetic weights and the engine follow."""
import json
import os

import numpy as np
import pytest

from golden import make_pin_golden as mk
from golden import make_zoe_single_golden as mz


@pytest.fixture(scope="module")
def gold():
    return np.load(os.path.join(os.path.dirname(__file__), "golden", "zoe_single_pin_golden.npz"))


@pytest.fixture(autouse=True)
def _recorded_thread_count():
    import torch
    n = torch.get_num_threads()
    torch.set_num_threads(mk.THREADS)
    yield
    torch.set_num_threads(n)


def _close(gold, key, got, rel):
    got = np.asarray(got)
    assert got.shape == tuple(gold[key + "_shape"]), key
    scale = float(gold[key + "_absmax"])
    err = float(np.abs(mk.sample(got).astype(np.float64) - gold[key].astype(np.float64)).max())
    assert err <= rel * scale, (key, err, scale)
    return scale


@pytest.mark.parametrize("model_type", [7, 8])
@pytest.mark.parametrize("seed,base_hw", mz.HEADS)
def test_zoe_single_head_oracle_equals_reference(gold, model_type, seed, base_hw):
    import torch
    from oracle import zoedepth_single as ozs
    feats, rel, sd = mz.inputs(model_type, seed, base_hw)
    with torch.no_grad():
        got = ozs.metric_head_single(feats, rel, sd, model_type)
    key = f"head_{model_type}_{seed}"
    _close(gold, key, got.numpy(), rel=1e-5)
    assert float(gold[key].max() - gold[key].min()) > 0.05 * float(gold[key + "_absmax"])     # a depth map that varies


@pytest.mark.parametrize("model_type", [7, 8])
@pytest.mark.parametrize("pad,flip", mz.TTA)
def test_zoe_single_tta_equals_reference(gold, model_type, pad, flip):
    import torch
    from oracle import zoedepth as ozd
    from oracle import zoedepth_single as ozs
    feats, rel, sd = mz.inputs(model_type, mz.TTA_SEED, mz.TTA_BASE)
    with torch.no_grad():
        got = ozd.infer(lambda t: ozs.metric_head_single(feats, rel, sd, model_type), mk.zoe_tta_input(), pad_input=pad, with_flip_aug=flip)
    _close(gold, f"tta_{model_type}_{int(pad)}{int(flip)}", got.numpy(), rel=1e-5)


@pytest.mark.parametrize("model_type", [7, 8])
def test_zoe_single_recorded_config(gold, model_type):
    from oracle import zoedepth_single as ozs
    cfg = json.loads(str(gold[f"config_{model_type}"]))
    want = ozs.SINGLE_CONFIG[model_type]
    assert cfg["bin_centers_type"] == want["bin_centers_type"]
    assert cfg["n_attractors"] == want["n_attractors"] == [16, 8, 4, 1]
    assert cfg["min_depth"] == want["min_depth"] and cfg["max_depth"] == want["max_depth"]
    assert cfg["kind"] == "mean" and not any(cfg["memory_efficient"])


def test_zoe_k_recorded_max_depth_is_10(gold):
    """ZoeDepth-K in infer mode keeps the constructor's max_depth (no dataset config is merged), not KITTI's 80"""
    assert json.loads(str(gold["config_8"]))["max_depth"] == 10


@pytest.mark.parametrize("model_type", [7, 8])
def test_synthetic_single_head_state_dict_matches_reference_module(gold, model_type):
    from oracle import zoedepth_single
    sd = zoedepth_single.make_zoedepth_single_state_dict(model_type, feat_ch=256, seed=0)
    want = {name: shape for name, shape, is_param in mk.layout(gold, f"zoe_single_{model_type}") if is_param}
    assert {k: list(v.shape) for k, v in sd.items()} == want
