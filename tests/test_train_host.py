"""Host-side pieces of the PPO driver (CPU): YAML parsing, the PPO loss against the reference's
ppo_update when the reference tree is present, and the flat-gradient all-reduce over gloo."""
import os
import socket
import sys
from types import SimpleNamespace

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from minesweeper_ppo_b200 import train as T
from minesweeper_ppo_b200.policy import build_model
import reference_live as RL

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = RL.REF_DIR


def test_load_config_medium_yaml():
    cfg, env_d, model_d, extras = T.load_config(os.path.join(ROOT, "configs", "medium_16x16x40.yaml"))
    assert (cfg.H, cfg.W, cfg.mine_count, cfg.num_envs, cfg.steps_per_env) == (16, 16, 40, 128, 64)
    assert cfg.mini_batches == 8 and cfg.ppo_epochs == 3 and cfg.gamma == 0.995 and cfg.gae_lambda == 0.95
    assert cfg.aux_mine_weight == 0.05 and cfg.aux_mine_calib_weight == 0.01 and cfg.ent_decay_updates == 400
    assert model_d == {"name": "cnn_residual", "stem_channels": 96, "blocks": 5, "dropout": 0.05, "value_hidden": 256}
    assert env_d["step_penalty"] == 1e-4 and extras["training"]["rollout"]["num_envs"] == 128


def _batch(n=64, seed=0):
    g = torch.Generator().manual_seed(seed)
    mask = torch.rand((n, 64), generator=g) < 0.6
    mask[:, 0] = True
    acts = torch.stack([torch.nonzero(mask[i])[0, 0] for i in range(n)])
    return SimpleNamespace(
        obs=(torch.rand((n, 10, 8, 8), generator=g) < 0.3).float(), action_mask=mask, actions=acts,
        old_logp=-torch.rand(n, generator=g), advantages=torch.randn(n, generator=g),
        returns=torch.randn(n, generator=g), values=torch.randn(n, generator=g),
        mine_labels=(torch.rand((n, 8, 8), generator=g) < 0.15).float(),
        mine_valid=torch.rand((n, 8, 8), generator=g) < 0.7)


@pytest.mark.skipif(not RL.available(), reason=RL.SKIP_REASON)
def test_ppo_update_matches_reference_cpu():
    sys.path.insert(0, REF)
    try:
        from minesweeper.ppo import PPOConfig as RefCfg, ppo_update as ref_update
    finally:
        sys.path.remove(REF)
    kw = dict(aux_mine_weight=0.05, aux_mine_calib_weight=0.01, ent_coef=0.003)
    torch.manual_seed(0)
    a = build_model("cnn_residual", obs_shape=(10, 8, 8), model_cfg=dict(stem_channels=32, blocks=2, dropout=0.0, value_hidden=32))
    b = build_model("cnn_residual", obs_shape=(10, 8, 8), model_cfg=dict(stem_channels=32, blocks=2, dropout=0.0, value_hidden=32))
    b.load_state_dict(a.state_dict())
    oa, ob = torch.optim.AdamW(a.parameters(), lr=3e-4), torch.optim.AdamW(b.parameters(), lr=3e-4)
    for step in range(3):
        batch = _batch(seed=step)
        sa = T.ppo_update(a, oa, batch, T.PPOConfig(**kw), grads=T.FlatGradAllReduce(a) if step == 0 else None)
        sb = ref_update(b, ob, batch, RefCfg(**kw))
        for k in sb:
            assert abs(sa[k] - sb[k]) <= 1e-6 * max(1.0, abs(sb[k])), (k, sa[k], sb[k])
    for pa, pb in zip(a.parameters(), b.parameters()):
        assert torch.allclose(pa, pb, rtol=0, atol=1e-6)


def _free_port():
    s = socket.socket(); s.bind(("127.0.0.1", 0)); p = s.getsockname()[1]; s.close(); return p


def _worker(rank, world, port, out):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        torch.manual_seed(0)
        m = build_model("cnn", obs_shape=(10, 8, 8))
        opt = torch.optim.SGD(m.parameters(), lr=0.1)
        grads = T.FlatGradAllReduce(m)
        T.ppo_update(m, opt, _batch(seed=100 + rank), T.PPOConfig(), grads=grads)     # different data per rank
        flat = torch.cat([p.detach().reshape(-1) for p in m.parameters()])
        gathered = [torch.zeros_like(flat) for _ in range(world)]
        dist.all_gather(gathered, flat)
        if rank == 0:
            torch.save(gathered, out)
    finally:
        dist.destroy_process_group()


def test_flat_grad_allreduce_keeps_replicas_identical_gloo(tmp_path):
    out = str(tmp_path / "p.pt")
    mp.spawn(_worker, args=(2, _free_port(), out), nprocs=2, join=True)
    p0, p1 = torch.load(out)
    assert torch.equal(p0, p1)
    # and equals a single-process step on the averaged gradient
    torch.manual_seed(0)
    m = build_model("cnn", obs_shape=(10, 8, 8))
    gs = []
    for r in range(2):
        m.zero_grad()
        loss, _ = T.ppo_loss(m, _batch(seed=100 + r), T.PPOConfig())
        loss.backward()
        gs.append(torch.cat([(p.grad if p.grad is not None else torch.zeros_like(p)).reshape(-1)
                             for p in m.parameters()]).clone())
    g = (gs[0] + gs[1]) / 2
    g = g * min(1.0, 0.5 / (float(g.norm()) + 1e-6))                  # clip_grad_norm_(0.5)
    expect = torch.cat([p.detach().reshape(-1) for p in m.parameters()]) - 0.1 * g
    assert torch.allclose(p0, expect, atol=1e-6)


def test_lazy_infos_list_behaves_like_the_reference_list():
    """VecMinesweeper.step's per-env infos lists (env.py:485-505) are lazy sequences: same indexing, slicing, len,
    iteration and equality as the lists the reference builds; they pickle as plain lists."""
    import copy
    import pickle
    from minesweeper_ppo_b200.env import _LazyList
    made = []

    def item(i):
        made.append(i)
        return {"step": i, "last_new_reveals": 2 * i, "revealed_frac": i / 8}

    lz = _LazyList(5, item)
    want = [{"step": i, "last_new_reveals": 2 * i, "revealed_frac": i / 8} for i in range(5)]
    assert made == [] and len(lz) == 5                      # nothing is built until somebody looks
    assert lz[3] == want[3] and lz[-1] == want[4] and made == [3, 4]
    assert lz[1:4] == want[1:4] and list(lz) == want and lz == want and want == lz and not (lz != want)
    assert lz != want[:4] and lz != [0] * 5 and (lz == "abcde") is False
    assert int(lz[2].get("last_new_reveals", 0)) == 4       # the access pattern of eval.py:407-409
    with pytest.raises(IndexError):
        lz[5]
    assert pickle.loads(pickle.dumps(lz)) == want and type(pickle.loads(pickle.dumps(lz))) is list
    assert copy.deepcopy(lz) == want and repr(lz) == repr(want)
