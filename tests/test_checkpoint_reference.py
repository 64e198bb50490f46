"""SURVEY.md §8f-1 (CPU): a checkpoint WRITTEN by a jorldy_b200 agent on a B200 (tests/golden/ckpt/<agent>/ckpt, produced
by scripts/make_ckpt_fixtures.py) loads the way the reference's `load` does it (dqn.py:193-199 / reinforce.py:138-142:
torch.load, a strict load_state_dict into modules keyed like the reference's, the torch optimizer's load_state_dict),
and the reference network's eval-mode forward on the recorded input equals what the B200 agent computed (fp32 tolerance
2e-5), i.e. the reference's --eval can run B200-trained weights.  The reference modules are stood in for by their
key/shape tables (tests/golden/gen_inputs.py) and their forward by the oracle (oracle/nets.py, oracle/actor_critic.py),
both pinned to the unmodified reference classes by the golden tests, so this runs from the repository alone."""
import os

import numpy as np
import pytest
import torch

import gen_inputs as G
from oracle import actor_critic as oac
from oracle import collect as ocol
from oracle import nets

HERE = os.path.dirname(os.path.abspath(__file__))
CKPT = os.path.join(HERE, "golden", "ckpt")
CASES = {
    "ppo": ("ppo", dict(state_size=4, action_size=2, hidden_size=64, batch_size=32, n_step=8)),
    "ppo_continuous": ("ppo", dict(state_size=11, action_size=3, hidden_size=64, batch_size=32, n_step=8,
                                   network="continuous_policy_value")),
    "dqn": ("dqn", dict(state_size=4, action_size=3, hidden_size=64, buffer_size=64, batch_size=8)),
    "rainbow": ("rainbow", dict(state_size=4, action_size=3, hidden_size=64, buffer_size=64, batch_size=8, n_step=3,
                                v_min=-1, v_max=10, num_support=51)),
    "ape_x": ("ape_x", dict(state_size=4, action_size=3, hidden_size=64, buffer_size=64, batch_size=8, n_step=3,
                            network="dueling", num_workers=2,
                            optim_config={"name": "rmsprop", "lr": 1e-3, "eps": 1.5e-7, "centered": True})),
}


def _shapes(name, kw):
    """The reference module's state_dict keys, in order, with their shapes."""
    case = {"H": kw["hidden_size"], "D": kw["state_size"], "A": kw["action_size"], "K": kw.get("num_support", 51),
            "agent": name, "continuous": kw.get("network") == "continuous_policy_value"}
    if name == "ppo":
        return G.ppo_shapes(case)
    case["net"] = {"dqn": "discrete_q_network", "rainbow": "rainbow", "ape_x": "dueling"}[name]
    return G.q_shapes(case)


def _load_module(sd, shapes):
    """nn.Module.load_state_dict(strict=True) restated: same keys, same shapes; returns the parameters in module order."""
    assert list(sd.keys()) == list(shapes.keys())
    for k, s in shapes.items():
        assert tuple(sd[k].shape) == tuple(s), k
    return {k: torch.nn.Parameter(sd[k].detach().clone().float()) for k in shapes}


def _load_optimizer(sd, params, optim_config=None):
    """The reference's optimizer (a torch.optim class over the module's parameters) and its load_state_dict."""
    cfg = dict(optim_config or {"name": "adam", "lr": 1e-3})
    cls = {"adam": torch.optim.Adam, "rmsprop": torch.optim.RMSprop}[cfg.pop("name")]
    opt = cls(list(params.values()), **cfg)
    opt.load_state_dict(sd)
    return opt


@pytest.mark.parametrize("tag", list(CASES))
def test_reference_loads_b200_checkpoint(tag):
    d = os.path.join(CKPT, tag)
    name, kw = CASES[tag]
    ck = torch.load(os.path.join(d, "ckpt"), map_location="cpu", weights_only=False)
    assert set(ck.keys()) == {"network", "optimizer"}
    p = _load_module(ck["network"], _shapes(name, kw))
    optimizer = _load_optimizer(ck["optimizer"], p, kw.get("optim_config"))
    exp = dict(np.load(os.path.join(d, "outputs.npz")))
    x = torch.from_numpy(exp["state"])
    with torch.no_grad():
        if name == "ppo" and "network" not in kw:
            pi, v = nets.discrete_policy_value(p, x)
            ho = torch.from_numpy(exp["head_out"])
            np.testing.assert_allclose(pi.numpy(), torch.softmax(ho[:, :-1], -1).numpy(), rtol=2e-5, atol=2e-6)
            np.testing.assert_allclose(v.numpy(), ho[:, -1:].numpy(), rtol=2e-5, atol=2e-6)
            act = ocol.act_ppo(p, exp["state"], False, training=False)
        elif name == "ppo":
            mu, std, v = nets.continuous_policy_value(p, x)
            ho, A = torch.from_numpy(exp["head_out"]), kw["action_size"]
            np.testing.assert_allclose(mu.numpy(), ho[:, :A].clamp(-5, 5).numpy(), rtol=2e-5, atol=2e-6)
            np.testing.assert_allclose(std.numpy(), torch.exp(torch.tanh(ho[:, A:2 * A])).numpy(), rtol=2e-5, atol=2e-6)
            np.testing.assert_allclose(v.numpy(), ho[:, -1:].numpy(), rtol=2e-5, atol=2e-6)
            act = ocol.act_ppo(p, exp["state"], True, training=False)
        elif name == "rainbow":
            A, K = kw["action_size"], kw["num_support"]
            logits = nets.rainbow_network(p, x, None, A, K)
            np.testing.assert_allclose(logits.numpy(), exp["logits"], rtol=2e-5, atol=2e-5)
            act = ocol.act_rainbow(p, exp["state"], A, K, kw["v_min"], kw["v_max"], None)
        else:
            q = nets.dueling(p, x) if kw.get("network") == "dueling" else nets.discrete_q_network(p, x)
            np.testing.assert_allclose(q.numpy(), exp["q"], rtol=2e-5, atol=2e-6)
            act = torch.argmax(q, -1, keepdim=True).numpy()
    # the reference's greedy act() on the loaded weights picks the actions the B200 agent picked
    if act.dtype.kind == "f":
        np.testing.assert_allclose(act, exp["action_eval"], rtol=0, atol=2e-6)
    else:
        np.testing.assert_array_equal(act.reshape(-1), exp["action_eval"].reshape(-1))
    # optimizer state came along (one step taken before saving)
    st = optimizer.state_dict()["state"]
    assert len(st) == len(p)


AC_CASES = {
    "ddpg": dict(state_size=3, action_size=2, hidden_size=64, buffer_size=64, batch_size=8),
    "td3": dict(state_size=3, action_size=2, hidden_size=64, buffer_size=64, batch_size=8),
    "sac": dict(state_size=3, action_size=2, hidden_size=64, buffer_size=64, batch_size=8, use_dynamic_alpha=True),
}


@pytest.mark.parametrize("tag", list(AC_CASES))
def test_reference_loads_b200_actor_critic_checkpoint(tag):
    """ddpg.py:186-197 / td3.py:232-246 / sac.py:321-339 load() on a checkpoint written by the B200 agent after two learns."""
    d = os.path.join(CKPT, tag)
    kw = AC_CASES[tag]
    case = {"H": kw["hidden_size"], "D": kw["state_size"], "A": kw["action_size"], "agent": tag}
    ck = torch.load(os.path.join(d, "ckpt"), map_location="cpu", weights_only=False)
    actor = _load_module(ck["actor"], G.ac_shapes(case, "actor"))
    opts = [_load_optimizer(ck["actor_optimizer"], actor)]
    if tag == "ddpg":
        critic = _load_module(ck["critic"], G.ac_shapes(case, "critic"))
        opts.append(_load_optimizer(ck["critic_optimizer"], critic))
    else:       # the reference's load() puts critic2's weights into critic1 and never loads critic2
        critic = _load_module(ck["critic1"], G.ac_shapes(case, "critic"))
        critic = _load_module(ck["critic2"], G.ac_shapes(case, "critic"))
        critic2 = _load_module(ck["critic2"], G.ac_shapes(case, "critic"))
        opts += [_load_optimizer(ck["critic_optimizer1"], critic), _load_optimizer(ck["critic_optimizer2"], critic2)]
    exp = dict(np.load(os.path.join(d, "outputs.npz")))
    x, a = torch.from_numpy(exp["state"]), torch.from_numpy(exp["action"])
    if tag == "ddpg":
        act = oac.act_ddpg(actor, exp["state"], None, None, 0.0, 1e-3, 2e-3, training=False)[0]
    elif tag == "td3":
        act = oac.act_td3(actor, exp["state"], None, 0.1, training=False)
    else:
        act = oac.act_sac(actor, exp["state"], None, training=False)
    np.testing.assert_allclose(act, exp["action_eval"], rtol=0, atol=2e-6)
    with torch.no_grad():
        np.testing.assert_allclose(oac.continuous_q_network(critic, x, a).numpy(), exp["q1" if tag == "ddpg" else "q2"],
                                   rtol=2e-5, atol=2e-6)
    for i, o in enumerate(opts):
        st = o.state_dict()["state"]
        steps = 1.0 if (tag == "td3" and i == 0) else 2.0          # TD3's actor steps on every second learn (td3.py:174)
        assert len(st) == len(o.param_groups[0]["params"]) and all(float(v["step"]) == steps for v in st.values())
    if tag == "sac":
        np.testing.assert_allclose(ck["log_alpha"].detach().numpy(), exp["log_alpha"], rtol=0, atol=0)
        log_alpha = {"log_alpha": torch.nn.Parameter(ck["log_alpha"].detach().clone().reshape(1))}
        alpha_opt = _load_optimizer(ck["alpha_optimizer"], log_alpha)
        assert float(alpha_opt.state_dict()["state"][0]["step"]) == 2.0
