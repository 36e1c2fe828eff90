"""Host-side logic of the trainer callers (CPU): policy layout, rollout buffer, PPO update, CLI surface."""
import importlib.util
import json
import os

import numpy as np
import pytest
import torch
import yaml

from tests.helpers import GOLDEN, ROOT
from solorl_b200.agents.policy import Policy
from solorl_b200.agents.ppo import PPO
from solorl_b200.agents.storage import OPBuffer
from solorl_b200.agents.train import EpisodeTracker, default_args
from solorl_b200.agents import utils
from solorl_b200.envs import Box


def _load(path):
    spec = importlib.util.spec_from_file_location(os.path.basename(path)[:-3], path)
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


def test_policy_parameter_counts_match_reference_golden():
    gold = json.load(open(os.path.join(GOLDEN, "policy_shapes.json")))
    assert gold["76x12"]["n_params"] == 19033                    # SURVEY §8e
    for key, case in gold.items():
        obs_dim, act_dim = (int(x) for x in key.split("x"))
        ac = Policy((obs_dim,), Box(-np.ones(act_dim), np.ones(act_dim)), None, {"hidden_size": 64})
        assert sum(p.numel() for p in ac.parameters()) == case["n_params"]
        assert {k: list(v.shape) for k, v in ac.state_dict().items()} == case["state_dict"]


def test_policy_forward_and_ppo_update_match_reference_golden():
    """tests/golden/ppo_update.npz was produced by the reference's own Policy / OPBuffer / PPO
    (agents/ppo/policy.py, storage.py, ppo.py) with full-batch mini-batches (order-independent)."""
    g = np.load(os.path.join(GOLDEN, "ppo_update.npz"))
    T, N, D, A = (int(x) for x in g["meta"])
    ac = Policy((D,), Box(-np.ones(A), np.ones(A)), None, {"hidden_size": 64})
    ac.load_state_dict({k[5:]: torch.from_numpy(g[k]) for k in g.files if k.startswith("init/")})
    obs, act = torch.from_numpy(g["obs"]), torch.from_numpy(g["actions"])
    with torch.no_grad():
        v, lp, ent = ac.evaluate_actions(obs[:-1].reshape(-1, D), act.reshape(-1, A))
    assert np.abs(v.numpy() - g["fwd_value"]).max() < 1e-5
    assert np.abs(lp.numpy() - g["fwd_logp"]).max() < 2e-5
    assert abs(float(ent) - float(g["fwd_entropy"])) < 1e-6
    buf = OPBuffer(T, N, (D,), A, "cpu")
    buf.obs.copy_(obs); buf.actions.copy_(act)
    buf.value_preds.copy_(torch.from_numpy(g["value_preds"]))
    buf.action_log_probs.copy_(torch.from_numpy(g["action_log_probs"]))
    buf.returns.copy_(torch.from_numpy(g["returns"]))
    agent = PPO(ac, 0.1, 3, T * N, 0.5, 0.01, lr=1e-3, l2_coef=0.0, max_grad_norm=0.5)
    losses = agent.update(buf)
    assert np.abs(np.array(losses) - g["losses"]).max() < 1e-5
    for k in g.files:
        if k.startswith("final/"):
            assert np.abs(ac.state_dict()[k[6:]].numpy() - g[k]).max() < 1e-5, k


def test_policy_log_prob_and_entropy_match_torch_normal():
    torch.manual_seed(0)
    ac = Policy((10,), Box(-np.ones(3), np.ones(3)), None, {"hidden_size": 8})
    ac.pi_dist.logstd.data.normal_()
    x = torch.randn(5, 10)
    v, a, lp = ac.act(x)
    _, feat = ac.base(x)
    mean, logstd = ac.pi_dist(feat)
    dist = torch.distributions.Normal(mean, logstd.exp())
    assert torch.allclose(lp, dist.log_prob(a).sum(-1, keepdim=True), atol=1e-5)     # policy.py:36-38
    v2, lp2, ent = ac.evaluate_actions(x, a)
    assert torch.allclose(lp2, lp, atol=1e-6) and torch.allclose(v2, v)
    assert abs(float(ent) - float(dist.entropy().mean())) < 1e-6                       # policy.py:55
    _, a_det, _ = ac.act(x, deterministic=True)
    assert torch.allclose(a_det, mean)


def test_opbuffer_shapes_append_reset_and_sampler():
    T, N, D, A = 5, 6, 7, 3
    buf = OPBuffer(T, N, (D,), A, "cpu")
    assert buf.obs.shape == (T + 1, N, D) and buf.rewards.shape == (T, N, 1)              # storage.py:9-19
    assert buf.value_preds.shape == (T + 1, N, 1) and buf.actions.shape == (T, N, A)
    for t in range(T):
        buf.append(torch.full((N, D), float(t + 1)), torch.zeros(N, A), torch.zeros(N, 1), torch.zeros(N, 1),
                   torch.full((N, 1), float(t)), torch.ones(N, 1) * (t % 2))
    assert buf.step == 0 and float(buf.obs[T][0, 0]) == T and float(buf.masks[T][0, 0]) == (T - 1) % 2
    buf.reset()
    assert torch.equal(buf.obs[0], buf.obs[-1]) and torch.equal(buf.masks[0], buf.masks[-1])   # storage.py:31-33
    adv = torch.arange(T * N, dtype=torch.float32).reshape(T, N, 1)
    seen = []
    for ob, ac, v, r, m, lp, ad in buf.batch_generator(adv, 8):
        assert ob.shape == (8, D) and ac.shape == (8, A) and ad.shape == (8, 1)
        seen += ad.reshape(-1).tolist()
    assert len(seen) == (T * N // 8) * 8 and len(set(seen)) == len(seen)                   # no replacement, drop_last
    with pytest.raises(RuntimeError):
        buf.compute_returns(torch.zeros(N, 1))                                           # CUDA kernel only


def test_ppo_update_improves_surrogate_on_cpu():
    torch.manual_seed(1)
    T, N, D, A = 8, 16, 6, 2
    ac = Policy((D,), Box(-np.ones(A), np.ones(A)), None, {"hidden_size": 16})
    agent = PPO(ac, 0.2, 4, 32, 0.5, 0.0, lr=3e-3, max_grad_norm=0.5)
    buf = OPBuffer(T, N, (D,), A, "cpu")
    buf.obs.normal_()
    with torch.no_grad():
        for t in range(T):
            v, a, lp = ac.act(buf.obs[t])
            buf.actions[t], buf.action_log_probs[t], buf.value_preds[t] = a, lp, v
    # reward the first action dimension: returns = advantage signal
    buf.returns[:-1] = buf.value_preds[:-1] + buf.actions[..., :1]
    before = float(ac.evaluate_actions(buf.obs[:-1].reshape(-1, D), buf.actions.reshape(-1, A))[1].mean())
    v, a, e = agent.update(buf)
    assert np.isfinite([v, a, e]).all()
    w = buf.actions[..., :1].reshape(-1) > 0.5
    lp_after = ac.evaluate_actions(buf.obs[:-1].reshape(-1, D), buf.actions.reshape(-1, A))[1].reshape(-1)
    lp_before = buf.action_log_probs.reshape(-1)
    assert float((lp_after - lp_before)[w].mean()) > 0.0        # actions with positive advantage became likelier
    assert before == before


def test_linear_schedule_and_init_layer():
    lin = utils.init_layer(torch.nn.Linear(4, 4))
    assert torch.allclose(lin.weight @ lin.weight.T, 2.0 * torch.eye(4), atol=1e-5)      # orthogonal, gain sqrt 2
    assert float(lin.bias.abs().sum()) == 0.0
    opt = torch.optim.Adam(lin.parameters(), lr=1.0)
    utils.update_linear_schedule(opt, 3, 10, 2.0)
    assert abs(opt.param_groups[0]["lr"] - 2.0 * 0.7) < 1e-12                             # agents/utils.py:14-18


class _FakeSim:
    def __init__(self, f, i):
        self.f, self.i = f, i

    def episode_stats_device(self):
        return self.f, self.i


def test_episode_tracker_accumulates_done_envs_only():
    n = 5
    f = torch.zeros(n, 12); i = torch.zeros(n, 12, dtype=torch.int32)
    f[:, 0] = torch.tensor([1., 2., 3., 4., 5.]); f[:, 1] = torch.tensor([10., 20., 30., 40., 50.])
    i[:, 2] = torch.tensor([5, 6, 7, 8, 9]); i[:, 3] = torch.tensor([1, 0, 1, 0, 1])
    f[:, 6] = 0.5
    tr = EpisodeTracker("cpu")
    tr.update(_FakeSim(f, i), torch.tensor([1., 0., 1., 0., 0.]))
    tr.update(_FakeSim(f, i), torch.tensor([0., 0., 0., 0., 1.]))
    st = tr.fetch()
    assert st["episodes"] == 3 and abs(st["episode_return"] - 30.0) < 1e-9 and abs(st["episode_reward"] - 3.0) < 1e-9
    assert abs(st["episode_length"] - 7.0) < 1e-9 and st["success"] == 1.0
    assert st["return_min"] == 10.0 and st["return_max"] == 50.0 and st["length_max"] == 9.0
    assert abs(st["dr/stand_rew"] - 0.5) < 1e-9
    assert tr.fetch()["episodes"] == 0                                               # cleared in place


def test_cli_defaults_are_the_reference_defaults():
    m = _load(os.path.join(ROOT, "training", "train_ppo.py"))
    a = m.get_ppo_args([])
    ref = dict(num_agents=32, output_size=64, hidden_size=64, env_name="base", gamma=0.99, tau=0.95, clip_param=0.1,
               ppo_epoch=10, mini_batch_size=32, lr=1e-3, l2_coef=0.0, value_loss_coef=0.5, entropy_coef=0.01,
               max_grad_norm=0.5, num_env_steps=1e6, seed=2301, curriculum_schedule=0, log_interval=10,
               save_interval=20, logdir=None, base_checkpoint=None, timestamp=None, task=None)   # train_ppo.py:9-45
    for k, v in ref.items():
        assert getattr(a, k) == v, k
    d = default_args()
    for k, v in ref.items():
        assert getattr(d, k) == v, k


@pytest.mark.parametrize("name,robot,task,control,H", [("basic", "solo8", "walk", "torque", 1),
                                                       ("basic12", "solo12", "pointgoal", "torque", 1),
                                                       ("basic_pd", "solo8", "stand", "pd", 0)])
def test_shipped_configs_keep_the_reference_keys(name, robot, task, control, H):
    from solorl_b200.abi import dims, params_from_config, _TASK_NAMES, _CONTROL_NAMES
    from solorl_b200.model import SoloModel
    cfg = yaml.safe_load(open(os.path.join(ROOT, "configs", name + ".yaml")))
    ref = json.load(open(os.path.join(GOLDEN, "reference_configs.json")))[name]    # the reference's configs/<name>.yaml
    assert set(cfg) == set(ref)
    for k in ref:
        if k != "model_urdf":
            assert cfg[k] == ref[k], k
    m = SoloModel.resolve(cfg["model_urdf"])
    p = params_from_config(cfg, m)
    assert m.name == robot and p.task == _TASK_NAMES[task] and p.control == _CONTROL_NAMES[control]
    assert p.num_history_stack == H and p.episode_length == 400


def test_td3_replay_ring_batched_append_and_wrap():
    from solorl_b200.agents.td3 import ReplayBuffer
    rb = ReplayBuffer(10, 3, 2, "cpu")
    for k in range(3):                                   # 3 x 4 transitions into a ring of 10: wraps once
        o = torch.full((4, 3), float(k)) + torch.arange(4).reshape(4, 1) * 0.1
        rb.append_batch(o, torch.zeros(4, 2), torch.full((4,), float(k)), o + 1, torch.ones(4))
    assert len(rb) == 10 and rb._top == 2
    assert torch.allclose(rb._observations[0], torch.full((3,), 2.2)) and torch.allclose(rb._observations[1], torch.full((3,), 2.3))
    assert torch.allclose(rb._observations[2], torch.full((3,), 0.2))            # oldest surviving transition
    assert torch.allclose(rb._next_observations[9], torch.full((3,), 3.1))
    o, a, r, o2, nt = rb.sample(64)
    assert o.shape == (64, 3) and a.shape == (64, 2) and r.shape == (64, 1) and nt.shape == (64, 1)
    assert torch.allclose(o2, o + 1)                                             # rows stay aligned
    rb2 = ReplayBuffer(5, 3, 2, "cpu")                                           # reference per-transition API
    rb2.append([(torch.ones(3), torch.zeros(2), torch.tensor(1.0), torch.ones(3) * 2, torch.tensor(0.0))])
    assert len(rb2) == 1 and float(rb2._not_terminal[0]) == 0.0


def test_td3_models_keep_reference_layout_and_update_runs():
    from solorl_b200.agents.td3 import TD3, ReplayBuffer
    torch.manual_seed(0)
    pol = TD3(10, 4, device="cpu")
    assert sorted(pol.actor.state_dict()) == ["l1.bias", "l1.weight", "l2.bias", "l2.weight", "l3.bias", "l3.weight"]
    assert pol.critic.l4.weight.shape == (256, 14) and pol.critic.l6.weight.shape == (1, 256)   # models.py:20-33
    rb = ReplayBuffer(512, 10, 4, "cpu")
    rb.append_batch(torch.randn(300, 10), torch.randn(300, 4).tanh(), torch.randn(300), torch.randn(300, 10),
                    (torch.rand(300) > 0.1).float())
    w0 = pol.actor.l3.weight.clone(); t0 = pol.actor_target.l3.weight.clone()
    q, a = pol.train(rb, 1, 64)                      # odd step: critic only (policy_freq 2)
    assert a is None and torch.equal(pol.actor.l3.weight, w0)
    q, a = pol.train(rb, 2, 64)
    assert a is not None and not torch.equal(pol.actor.l3.weight, w0)
    # soft target update: target moved by tau towards the actor
    assert torch.allclose(pol.actor_target.l3.weight, 0.995 * t0 + 0.005 * pol.actor.l3.weight, atol=1e-6)
    assert (pol.select_action(torch.randn(5, 10)).abs() <= 1).all()


def test_td3_cli_defaults_are_the_reference_defaults():
    m = _load(os.path.join(ROOT, "training", "train_td3.py"))
    a = m.get_td3_args([])
    ref = dict(env_name="base", seed=0, start_timesteps=25e3, eval_freq=5e3, num_env_steps=1e6, expl_noise=0.1,
               batch_size=256, gamma=0.99, tau=0.005, policy_noise=0.2, noise_clip=0.5, policy_freq=2, load_model="",
               max_replay_size=1000000, num_agents=32, logdir=None, timestamp=None, log_interval=1000,
               save_interval=2000, task=None)                                     # train_td3.py:10-39
    for k, v in ref.items():
        assert getattr(a, k) == v, k


def test_flat_parameter_buffers_alias_and_change_nothing():
    """PPO keeps parameters and gradients as views of two flat buffers (one all-reduce, no pack / unpack): the
    update is bit-identical to the unflattened one, the views survive it, state_dict keys are unchanged."""
    from solorl_b200.agents.policy import Policy
    from solorl_b200.agents.ppo import PPO
    from solorl_b200.agents.storage import OPBuffer
    from solorl_b200.envs import Box
    T, N, D, A = 6, 8, 10, 4
    ws = []
    for flat in (True, False):
        torch.manual_seed(3)
        ac = Policy((D,), Box(-np.ones(A), np.ones(A)), None, {"hidden_size": 16})
        keys = list(ac.state_dict().keys())
        agent = PPO(ac, 0.1, 2, 16, 0.5, 0.01, lr=1e-3, max_grad_norm=0.5, flat_parameters=flat)
        assert list(ac.state_dict().keys()) == keys
        buf = OPBuffer(T, N, (D,), A, "cpu")
        g = torch.Generator().manual_seed(5)
        for t in (buf.obs, buf.actions, buf.rewards, buf.value_preds, buf.returns):
            t.copy_(torch.randn(t.shape, generator=g))
        buf.action_log_probs.copy_(torch.randn(buf.action_log_probs.shape, generator=g) * 0.1 - 5.0)
        torch.manual_seed(11)                      # the mini-batch permutation
        agent.update(buf)
        if flat:
            assert agent.flat.intact() and agent.flat.numel == sum(p.numel() for p in ac.parameters())
            assert torch.equal(agent.flat.data, torch.cat([p.detach().reshape(-1) for p in ac.parameters()]))
            sd = {k: v.clone() for k, v in ac.state_dict().items()}
            ac.load_state_dict(sd)                 # an in-place copy: the views must survive it
            assert agent.flat.intact()
        ws.append(torch.cat([p.detach().reshape(-1) for p in ac.parameters()]).clone())
    assert torch.equal(ws[0], ws[1])
