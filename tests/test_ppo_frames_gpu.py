"""PPO with the CNN head on uint8 frame stacks (config.ppo.atari), on the B200 (pytest -m gpu).

The CNN trunk, the PPO loss / GAE / Adam and the synthetic Atari env are each pinned elsewhere; here the whole agent runs
on [rows, 4, 84, 84] uint8 rollouts and is checked against oracle.ppo with CNN parameters (oracle.nets dispatches to
cnn_head when the parameters hold conv weights).  Tolerances are those of test_ppo_gpu.py:
  value / log_prob_old / adv / ret : rtol 1e-4, atol 2e-5
  first-minibatch gradients        : rtol 2e-3, atol 2e-6
  parameters after the whole learn(): atol 0.1*lr
  result dict                      : rtol/atol 2e-4
"""
from collections import OrderedDict

import numpy as np
import pytest
import torch

import gen_inputs as G
from oracle import collect as oc
from oracle import ppo as oppo
from oracle.frames import FramesBatch

pytestmark = pytest.mark.gpu
DEV = "cuda"
STACK = (4, 84, 84)
ROW_BYTES = 4 * 84 * 84          # 28 224

HP = dict(lr=2.5e-4, gamma=0.99, lam=0.95, eps_clip=0.1, vf_coef=1.0, ent_coef=0.01, clip_grad_norm=1.0, standardize=True)
CASES = {
    "n4_t16_b16": dict(HP, seed=41, N=4, T=16, A=4, H=64, batch_size=16, n_epoch=2),
    # 60 rows = 3 x 16 + a ragged tail of 12
    "tail_n3_t20_b16": dict(HP, seed=42, N=3, T=20, A=6, H=512, batch_size=16, n_epoch=2),
}


def _shapes(case):
    s = OrderedDict()
    feat = G._head_shapes(s, dict(case, head="cnn", D=list(STACK)))
    H, A = case["H"], case["A"]
    s["l.weight"] = (H, feat); s["l.bias"] = (H,)
    s["pi.weight"] = (A, H); s["pi.bias"] = (A,)
    s["v.weight"] = (1, H); s["v.bias"] = (1,)
    return s


def _params(case):
    return {k: torch.from_numpy(v) for k, v in G.make_params(_shapes(case), case["seed"]).items()}


def _inputs(case):
    rs = np.random.RandomState(case["seed"] + 1)
    NT = case["N"] * case["T"]
    return dict(state=rs.randint(0, 256, size=(NT,) + STACK, dtype=np.uint8),
                next_state=rs.randint(0, 256, size=(NT,) + STACK, dtype=np.uint8),
                action=rs.randint(0, case["A"], size=(NT, 1)).astype(np.int64),
                reward=rs.choice([0.0, 1.0, -1.0], size=(NT, 1)).astype(np.float32),
                done=(rs.uniform(size=(NT, 1)) < 0.07).astype(np.float32),
                perms=[rs.permutation(NT) for _ in range(case["n_epoch"])])


def _oracle(case, params, inp, **kw):
    batch = {"state": torch.from_numpy(inp["state"].astype(np.float32)),
             "next_state": torch.from_numpy(inp["next_state"].astype(np.float32)),
             "action": torch.from_numpy(inp["action"].astype(np.float32)),
             "reward": torch.from_numpy(inp["reward"]), "done": torch.from_numpy(inp["done"])}
    hp = {"continuous": False, "n_step": case["T"], "gamma": case["gamma"], "lambda": case["lam"],
          "standardize": case["standardize"], "batch_size": case["batch_size"], "n_epoch": case["n_epoch"],
          "eps_clip": case["eps_clip"], "vf_coef": case["vf_coef"], "ent_coef": case["ent_coef"],
          "clip_grad_norm": case["clip_grad_norm"]}
    return oppo.learn(params, batch, hp, inp["perms"], lr=case["lr"], **kw)


def _agent(case, **kw):
    from jorldy_b200.core import Agent
    return Agent("ppo", state_size=list(STACK), action_size=case["A"], hidden_size=case["H"],
                 network="discrete_policy_value", head="cnn", optim_config={"name": "adam", "lr": case["lr"]},
                 gamma=case["gamma"], use_standardization=case["standardize"], run_step=1000, lr_decay=False, device=DEV,
                 batch_size=case["batch_size"], n_step=case["T"], n_epoch=case["n_epoch"], _lambda=case["lam"],
                 epsilon_clip=case["eps_clip"], vf_coef=case["vf_coef"], ent_coef=case["ent_coef"],
                 clip_grad_norm=case["clip_grad_norm"], **kw)


def _learn(case, inp, **kw):
    agent = _agent(case, **kw)
    agent.network.load_state_dict(_params(case))
    agent._inject_perms = inp["perms"]
    t = lambda a: torch.from_numpy(a).to(DEV)
    res = agent._learn_tensors(t(inp["state"]), t(inp["action"]).reshape(-1).to(torch.int32), t(inp["reward"]).reshape(-1),
                               t(inp["done"]).reshape(-1), next_state=t(inp["next_state"]))
    torch.cuda.synchronize()
    return agent, res


def _call_im2col_rows(x_ptr, idx, B, col):
    from jorldy_b200._lib import C
    C.jb_im2col_u8_rows(x_ptr, idx.data_ptr() if idx is not None else 0, B, 4, 84, 84, 8, 8, 4, col.data_ptr(),
                        torch.cuda.current_stream().cuda_stream)


def _im2col_ref(xg):
    """jb_im2col_u8 on the rows gathered by torch."""
    from jorldy_b200._lib import C
    col = torch.empty(xg.shape[0] * 400, 256, device=DEV)
    C.jb_im2col_u8(xg.data_ptr(), xg.shape[0], 4, 84, 84, 8, 8, 4, col.data_ptr(), torch.cuda.current_stream().cuda_stream)
    return col


# ---------------------------------------------------------------------------------------------------- 1. im2col gather
@pytest.mark.parametrize("kernel", ["vec4", "scalar"])
def test_im2col_rows_equals_gathered_im2col(kernel):
    R = 37
    g = torch.Generator(device=DEV).manual_seed(7)
    # the scalar kernel is taken when the input is not 16-byte aligned: offset the stacks by one byte
    off = 0 if kernel == "vec4" else 1
    buf = torch.randint(0, 256, (R * ROW_BYTES + 16,), dtype=torch.uint8, device=DEV, generator=g)
    x = buf[off:off + R * ROW_BYTES].view(R, *STACK)
    for rows in ([3, 3, 0, 36, 3, 17], list(range(R - 1, -1, -1))):
        idx = torch.tensor(rows, dtype=torch.int32, device=DEV)
        col = torch.empty(len(rows) * 400, 256, device=DEV)
        _call_im2col_rows(x.data_ptr(), idx, len(rows), col)
        assert torch.equal(col, _im2col_ref(x.index_select(0, idx.long()).contiguous()))
    # idx = NULL reads rows in order
    col = torch.empty(R * 400, 256, device=DEV)
    _call_im2col_rows(x.data_ptr(), None, R, col)
    assert torch.equal(col, _im2col_ref(x.contiguous()))


def test_im2col_rows_past_2gb():
    """A 600 x 128-row uint8 rollout is 2.17 GB: rows from 76 088 on start past 2^31 bytes."""
    R = 600 * 128
    assert (R - 1) * ROW_BYTES >= 2 ** 31 and 76088 * ROW_BYTES >= 2 ** 31 > 76087 * ROW_BYTES
    x = torch.empty(R, *STACK, dtype=torch.uint8, device=DEV)
    g = torch.Generator(device=DEV).manual_seed(11)
    x[:64].random_(0, 256, generator=g)
    x[76000:].random_(0, 256, generator=g)
    idx = torch.tensor([R - 1, 76088, 76087, 5, R - 1, 76100, 0, 76799], dtype=torch.int32, device=DEV)
    col = torch.empty(idx.numel() * 400, 256, device=DEV)
    _call_im2col_rows(x.data_ptr(), idx, idx.numel(), col)
    torch.cuda.synchronize()
    assert torch.equal(col, _im2col_ref(x.index_select(0, idx.long()).contiguous()))
    del x
    torch.cuda.empty_cache()


def test_cnn_head_rejects_non_uint8_input():
    case = CASES["n4_t16_b16"]
    agent = _agent(case)
    out = torch.empty(2, agent.network.nout, device=DEV)
    with pytest.raises(ValueError, match="uint8"):
        agent.network.forward_rows(torch.zeros(2, *STACK, device=DEV), out)
    with pytest.raises(ValueError, match="contiguous"):
        agent.network.forward_rows(torch.zeros(2, 84, 84, 4, dtype=torch.uint8, device=DEV).permute(0, 3, 1, 2), out)


# --------------------------------------------------------------------------------------------------- 2. learn vs oracle
@pytest.mark.parametrize("name", list(CASES))
def test_learn_matches_oracle(name):
    case = CASES[name]
    inp = _inputs(case)
    ref = _oracle(case, _params(case), inp)
    agent, res = _learn(case, inp, use_cuda_graph=False)
    st = agent._st
    for mine, theirs in (("value", "value"), ("logp_old", "log_prob_old"), ("adv", "adv"), ("ret", "ret")):
        np.testing.assert_allclose(st[mine].cpu().numpy().reshape(-1), ref[theirs].numpy().reshape(-1), rtol=1e-4,
                                   atol=2e-5, err_msg=mine)
    for k, v in ref["params"].items():
        np.testing.assert_allclose(agent.network.p[k].cpu().numpy(), v.numpy(), rtol=1e-4, atol=0.1 * case["lr"], err_msg=k)
    for k, v in ref["result"].items():
        np.testing.assert_allclose(res[k], v, rtol=2e-4, atol=2e-4, err_msg=k)
    n_mb = -(-case["N"] * case["T"] // case["batch_size"])
    assert agent.n_launches == case["n_epoch"] * sum(
        agent._launches_per_minibatch(min(case["batch_size"], case["N"] * case["T"] - k * case["batch_size"]))
        for k in range(n_mb))


@pytest.mark.parametrize("name", list(CASES))
def test_first_minibatch_grads_match_oracle(name):
    case = CASES[name]
    inp = _inputs(case)
    params = _params(case)
    ref = _oracle(case, params, inp, max_minibatches=1)
    agent, _ = _learn(dict(case, n_epoch=0), inp, use_cuda_graph=False)       # pre-pass and GAE only
    B = case["batch_size"]
    idx = torch.as_tensor(inp["perms"][0][:B], dtype=torch.int32, device=DEV)
    agent._minibatch_step(agent._st, idx, B)
    torch.cuda.synchronize()
    for k, g in ref["first_grads"].items():
        np.testing.assert_allclose(agent.network.g[k].cpu().numpy(), g.numpy(), rtol=2e-3, atol=2e-6, err_msg=k)


# ------------------------------------------------------------------------------------------------ 3. eager vs graph
def test_graph_path_equals_eager(monkeypatch):
    import jorldy_b200.core.agent.ppo as ppo_mod
    monkeypatch.setattr(ppo_mod, "GRAPH_CHUNK", 2)
    case = CASES["tail_n3_t20_b16"]                  # 3 full minibatches: one graph replay, one eager step, the tail
    inp = _inputs(case)
    a_eager, r_eager = _learn(case, inp, use_cuda_graph=False)
    a_graph, r_graph = _learn(case, inp, use_cuda_graph=True)
    assert a_graph._graphs and not a_eager._graphs
    assert torch.equal(a_eager.network.flat, a_graph.network.flat)
    assert r_eager == r_graph


# ------------------------------------------------------------------------------------------------------------ 4. act
def test_act_matches_oracle():
    case = CASES["n4_t16_b16"]
    params = _params(case)
    agent = _agent(case)
    agent.network.load_state_dict(params)
    rs = np.random.RandomState(5)
    M = 48
    state = rs.randint(0, 256, size=(M,) + STACK, dtype=np.uint8)
    u = rs.uniform(size=M).astype(np.float32)
    s = torch.from_numpy(state).to(DEV)
    a = agent.act_device(s, True, noise=torch.from_numpy(u).to(DEV)).cpu().numpy()
    np.testing.assert_array_equal(a.reshape(-1, 1), oc.act_ppo(params, state.astype(np.float32), False, True, u=u))
    greedy = agent.act_device(s, False).cpu().numpy()
    np.testing.assert_array_equal(greedy.reshape(-1, 1), oc.act_ppo(params, state.astype(np.float32), False, False))
    # the numpy plugin call takes the uint8 stacks as they are
    out = agent.act(state, training=False)["action"]
    assert out.shape == (M, 1) and out.dtype == np.int64
    np.testing.assert_array_equal(out.reshape(-1), greedy)


# ------------------------------------------------------------------------------------------------ 5. resident path
def _frames_rollout(N, T, seed, case, **kw):
    from jorldy_b200.core import Env
    from jorldy_b200.core.collect import RolloutCollector
    env = Env("breakout", num_envs=N, seed=seed, device=DEV)
    agent = _agent(dict(case, T=T), **kw)
    return env, agent, RolloutCollector(env, agent, n_step=T, use_cuda_graph=False)


def test_rollout_holds_the_env_frames():
    """64 envs x 64 steps (8 auto-resets with this seed): the rollout's bytes are the observation sequence the oracle
    generator produces."""
    N, T, seed = 64, 64, 3
    case = dict(CASES["n4_t16_b16"], batch_size=512)
    env, agent, col = _frames_rollout(N, T, seed, case)
    ro = col.collect()
    torch.cuda.synchronize()
    assert ro.state.dtype == torch.uint8 and ro.state.shape == (N, T) + STACK
    assert ro.state.numel() * ro.state.element_size() == N * T * ROW_BYTES
    assert ro.last_next_state.dtype == torch.uint8 and ro.last_next_state.shape == (N,) + STACK
    ref = FramesBatch(N, seed=seed, stream_base=0, auto_reset=True)
    ref.reset()
    state = ro.state.cpu().numpy()
    dones = 0
    for t in range(T):
        assert np.array_equal(state[:, t], ref.obs), f"step {t}"
        nobs, r, d = ref.step()
        np.testing.assert_array_equal(ro.reward[:, t].cpu().numpy(), r)
        np.testing.assert_array_equal(ro.done[:, t].cpu().numpy() > 0.5, d)
        dones += int(d.sum())
    assert np.array_equal(ro.last_next_state.cpu().numpy(), nobs)
    assert dones > 0


def test_learn_rollout_equals_host_learn():
    """The resident path (rollout rows, V(s') by the value shift) and the numpy plugin path (host transitions, explicit
    next_state) on the same transitions and permutations."""
    N, T, seed = 16, 32, 3
    case = dict(CASES["n4_t16_b16"], batch_size=128, n_epoch=2)
    env, agent, col = _frames_rollout(N, T, seed, case)
    params = _params(case)
    agent.network.load_state_dict(params)
    ro = col.collect()
    torch.cuda.synchronize()
    st, act, rew, done, last = (x.cpu().numpy() for x in (ro.state, ro.action, ro.reward, ro.done, ro.last_next_state))
    perms = [np.random.RandomState(9 + e).permutation(N * T) for e in range(case["n_epoch"])]
    agent._inject_perms = perms
    r1 = agent.learn_rollout(ro)
    host = _agent(dict(case, T=T))
    host.network.load_state_dict(params)
    host._inject_perms = perms
    nxt = np.concatenate([st[:, 1:], last[:, None]], axis=1)
    host.memory.store([{"state": st[:, t], "action": act[:, t, None].astype(np.int64), "reward": rew[:, t, None],
                        "done": done[:, t, None], "next_state": nxt[:, t]} for t in range(T)])
    r2 = host.learn()
    torch.cuda.synchronize()
    assert host._host_in["state"].dtype == torch.uint8 and host._host_in["state"].shape == (N * T,) + STACK
    for k in agent.network.p:
        np.testing.assert_allclose(agent.network.p[k].cpu().numpy(), host.network.p[k].cpu().numpy(), rtol=1e-4,
                                   atol=0.1 * case["lr"], err_msg=k)
    for k in r1:
        np.testing.assert_allclose(r1[k], r2[k], rtol=2e-4, atol=2e-4, err_msg=k)


# ------------------------------------------------------------------------------------------------------ 6. checkpoint
def test_checkpoint_is_the_reference_layout(tmp_path):
    case = CASES["n4_t16_b16"]
    inp = _inputs(case)
    agent, _ = _learn(case, inp, use_cuda_graph=False)
    agent.save(str(tmp_path))
    ck = torch.load(str(tmp_path / "ckpt"), map_location="cpu", weights_only=False)
    H, A = case["H"], case["A"]
    want = OrderedDict([("head.conv1.weight", (32, 4, 8, 8)), ("head.conv1.bias", (32,)),
                        ("head.conv2.weight", (64, 32, 4, 4)), ("head.conv2.bias", (64,)),
                        ("head.conv3.weight", (64, 64, 3, 3)), ("head.conv3.bias", (64,)),
                        ("l.weight", (H, 3136)), ("l.bias", (H,)), ("pi.weight", (A, H)), ("pi.bias", (A,)),
                        ("v.weight", (1, H)), ("v.bias", (1,))])
    assert [(k, tuple(v.shape)) for k, v in ck["network"].items()] == list(want.items())
    other = _agent(case)
    other.load(str(tmp_path))
    assert torch.equal(other.network.flat, agent.network.flat)
    o1, o2 = agent.optimizer.state_dict(), other.optimizer.state_dict()
    assert o1["state"].keys() == o2["state"].keys()
    for i in o1["state"]:
        for k in ("exp_avg", "exp_avg_sq"):
            assert torch.equal(o1["state"][i][k].cpu(), o2["state"][i][k].cpu())


# -------------------------------------------------------------------------------------------------- 7. reproducibility
def test_seeded_runs_are_bit_identical():
    def run():
        torch.manual_seed(0)
        np.random.seed(0)
        from jorldy_b200.core import Env
        from jorldy_b200.core.collect import RolloutCollector
        case = dict(CASES["n4_t16_b16"], T=32, batch_size=128)
        env = Env("breakout", num_envs=16, seed=1, device=DEV)
        agent = _agent(case, seed=5)
        col = RolloutCollector(env, agent)
        for _ in range(2):
            agent.learn_rollout(col.collect())
        torch.cuda.synchronize()
        return agent.network.flat.clone()
    assert torch.equal(run(), run())
