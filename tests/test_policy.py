"""The policy modules stay PyTorch (SURVEY section 2); this only checks that they are
state_dict-compatible with, and numerically identical to, the reference modules when the
reference is installed (tools/install_reference.sh)."""
import sys

import pytest
import torch

import reference_live as RL

REF = RL.REF_DIR


def test_build_model_shapes_and_param_count():
    import minesweeper_ppo_b200 as m
    net = m.build_model("cnn_residual", obs_shape=(10, 16, 16),
                        model_cfg=dict(stem_channels=96, blocks=5, dropout=0.05, value_hidden=256))
    assert sum(p.numel() for p in net.parameters()) == 950_947          # SURVEY section 2 [measured]
    logits, value, mine = net.eval()(torch.zeros(2, 10, 16, 16), return_mine=True)
    assert logits.shape == (2, 256) and value.shape == (2,) and mine.shape == (2, 1, 16, 16)
    with pytest.raises(ValueError):
        m.build_model("nope", obs_shape=(10, 8, 8))


@pytest.mark.skipif(not RL.available(), reason=RL.SKIP_REASON)
@pytest.mark.parametrize("name,cfg,shape", [
    ("cnn_residual", dict(stem_channels=96, blocks=5, dropout=0.05, value_hidden=256), (10, 16, 16)),
    ("cnn", dict(hidden=64), (10, 8, 8)),
])
def test_matches_reference_module(name, cfg, shape):
    import minesweeper_ppo_b200 as m
    sys.path.insert(0, REF)
    try:
        from minesweeper.models import build_model as ref_build
    finally:
        sys.path.remove(REF)
    torch.manual_seed(0)
    ref = ref_build(name, obs_shape=shape, model_cfg=dict(cfg)).eval()
    net = m.build_model(name, obs_shape=shape, model_cfg=dict(cfg)).eval()
    net.load_state_dict(ref.state_dict())
    x = torch.rand(4, *shape)
    for a, b in zip(net(x, return_mine=True), ref(x, return_mine=True)):
        assert torch.equal(a, b)
