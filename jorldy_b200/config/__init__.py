"""Built-in hot-path configs, generated from tables instead of one file per (agent, env) pair.

`load("config.<agent>.<env>")` returns a module-like namespace with the four dicts the reference's
config modules define (jorldy/config/<agent>/<env>.py: env / agent / optim / train).  Values follow the
reference's shipped configs for the agents on the north-star path (dqn, double, dueling, multistep,
per, noisy, c51, rainbow, ape_x, ppo, and ddpg / td3 / sac of SURVEY 8f-4) on cartpole / mountaincar / pendulum / atari(synthetic) /
mujoco(synthetic dims); an existing JORLDY config directory on sys.path takes precedence
(manager/config_manager.py).
"""
from types import SimpleNamespace

_TRAIN_SMALL = dict(training=True, load_path=None, run_step=100000, print_period=1000, save_period=10000)
_TRAIN_ATARI = dict(training=True, load_path=None, run_step=30000000, print_period=10000, save_period=100000,
                    eval_iteration=5, eval_time_limit=None, record=True, record_period=300000)
_EPS = dict(epsilon_init=1.0, epsilon_min=0.01, explore_ratio=0.2)
_REPLAY = dict(gamma=0.99, buffer_size=50000, batch_size=32, start_train_step=2000, target_update_period=500, lr_decay=True)
_REPLAY_ATARI = dict(gamma=0.99, buffer_size=1000000, batch_size=32, start_train_step=100000,
                     target_update_period=10000, lr_decay=True, head="cnn")
_ATARI_ENV = dict(render=False, gray_img=True, img_width=84, img_height=84, stack_frame=4, no_op=True, skip_frame=4,
                  reward_clip=True, episodic_life=True)

# agent name -> (network, extra agent keys, eval_iteration, update_period on cartpole)
_VALUE_AGENTS = {
    "dqn": ("discrete_q_network", dict(_EPS), 10, 32),
    "double": ("discrete_q_network", dict(_EPS), 5, 32),
    "dueling": ("dueling", dict(_EPS), 5, 32),
    "multistep": ("discrete_q_network", dict(_EPS, n_step=4), 5, 8),
    "per": ("discrete_q_network", dict(_EPS, alpha=0.6, beta=0.4, learn_period=2, uniform_sample_prob=1e-3), 5, 2),
    "noisy": ("noisy", dict(noise_type="factorized"), 5, 32),
    "c51": ("discrete_q_network", dict(_EPS, v_min=-1, v_max=10, num_support=51), 5, 32),
    "rainbow": ("rainbow", dict(n_step=3, alpha=0.5, beta=0.4, learn_period=2, uniform_sample_prob=1e-3,
                                noise_type="factorized", v_min=-1, v_max=10, num_support=51), 10, 8),
}


def _value_config(agent, env):
    net, extra, eval_it, upd = _VALUE_AGENTS[agent]
    if env == "atari":
        a = dict(name=agent, network=net, **_REPLAY_ATARI)
        a.update(extra)
        if "epsilon_min" in a:
            a.update(epsilon_min=0.1, explore_ratio=0.1)
        if agent == "rainbow":
            a.update(learn_period=4)
        lr = 2.5e-4 / 4 if agent == "rainbow" else 1e-4
        return dict(env=dict(_ATARI_ENV), agent=a, optim=dict(name="adam", lr=lr),
                    train=dict(_TRAIN_ATARI, run_step=30000000 if agent == "rainbow" else 10000000,
                               update_period=32, num_workers=16))
    a = dict(name=agent, network=net, **_REPLAY)
    a.update(extra)
    env_d = dict(name="cartpole", action_type="discrete", render=False) if env == "cartpole" else dict(name="mountain_car", render=False)
    return dict(env=env_d, agent=a, optim=dict(name="adam", lr=1e-4),
                train=dict(_TRAIN_SMALL, eval_iteration=eval_it, update_period=upd, num_workers=8))


def _ape_x_config(env):
    a = dict(name="ape_x", network="dueling", gamma=0.99, clip_grad_norm=40.0, lr_decay=True, n_step=3, alpha=0.6,
             beta=0.4, uniform_sample_prob=1e-3, batch_size=32)
    opt = dict(name="rmsprop", eps=1.5e-7, centered=True)
    if env == "atari":
        a.update(head="cnn", buffer_size=2000000, start_train_step=50000, target_update_period=2500)
        return dict(env=dict(_ATARI_ENV), agent=a, optim=dict(opt, lr=2.5e-4 / 4),
                    train=dict(_TRAIN_ATARI, distributed_batch_size=512, update_period=100, num_workers=128))
    a.update(buffer_size=50000, start_train_step=2000, target_update_period=1000)
    env_d = dict(name="cartpole", action_type="discrete", render=False) if env == "cartpole" else dict(name="mountain_car", render=False)
    return dict(env=env_d, agent=a, optim=dict(opt, lr=1e-4),
                train=dict(_TRAIN_SMALL, eval_iteration=10, distributed_batch_size=512, update_period=16, num_workers=32))


def _ppo_config(env):
    a = dict(name="ppo", gamma=0.99, _lambda=0.95, epsilon_clip=0.1, vf_coef=1.0, ent_coef=0.01, clip_grad_norm=1.0,
             lr_decay=True)
    if env == "mujoco":
        a.update(network="continuous_policy_value", batch_size=512, n_step=2048, n_epoch=10)
        return dict(env=dict(render=False), agent=a, optim=dict(name="adam", lr=3e-4),
                    train=dict(training=True, load_path=None, run_step=1000000, print_period=10000, save_period=100000,
                               eval_iteration=10, record=True, record_period=500000, distributed_batch_size=2048,
                               update_period=2048, num_workers=32))
    a.update(batch_size=32, n_step=128, n_epoch=3, use_standardization=True)
    if env == "atari":
        # Shaped after the reference's config/ppo/atari.py: the cartpole PPO agent keys plus head="cnn", with the Atari
        # env and train dicts the value agents use.  Not checked line by line against that file.
        a.update(network="discrete_policy_value", head="cnn")
        return dict(env=dict(_ATARI_ENV), agent=a, optim=dict(name="adam", lr=2.5e-4),
                    train=dict(_TRAIN_ATARI, run_step=30000000, distributed_batch_size=1024, update_period=128,
                               num_workers=32))
    if env == "pendulum":
        a.update(network="continuous_policy_value")
        env_d = dict(name="pendulum", render=False)
    elif env == "mountaincar":
        a.update(network="discrete_policy_value")
        env_d = dict(name="mountain_car", render=False)
    else:
        a.update(network="discrete_policy_value")
        env_d = dict(name="cartpole", action_type="discrete", render=False)
    return dict(env=env_d, agent=a, optim=dict(name="adam", lr=2.5e-4),
                train=dict(_TRAIN_SMALL, eval_iteration=10, distributed_batch_size=256, update_period=128, num_workers=8))


# ---- continuous off-policy family: jorldy/config/{ddpg,td3,sac}/{cartpole,pendulum,mujoco}.py --------------------------------
_TRAIN_MUJOCO = dict(training=True, load_path=None, run_step=1000000, print_period=10000, save_period=100000, eval_iteration=10)
_AC_ENVS = {"ddpg": ("cartpole", "pendulum", "mujoco"), "td3": ("cartpole", "mujoco"), "sac": ("cartpole", "pendulum", "mujoco")}


def _ac_config(agent, env):
    env_d = {"cartpole": dict(name="cartpole", action_type="continuous", render=False), "pendulum": dict(name="pendulum", render=False),
             "mujoco": dict(render=False)}[env]
    mj = env == "mujoco"
    if agent == "ddpg":
        a = dict(name="ddpg", actor="deterministic_policy", critic="continuous_q_network", gamma=0.99, buffer_size=50000,
                 batch_size=128, start_train_step=1000 if mj else 2000, tau=1e-3, lr_decay=True, mu=0, theta=1e-3, sigma=2e-3)
        opt = dict(actor="adam", critic="adam", actor_lr=5e-4, critic_lr=1e-3)
        tr = dict(_TRAIN_MUJOCO, distributed_batch_size=256, update_period=1, num_workers=8) if mj else \
            dict(_TRAIN_SMALL, eval_iteration=10, update_period=1, num_workers=8)
        if env == "pendulum":
            tr = dict(_TRAIN_SMALL, eval_iteration=10, distributed_batch_size=128, update_period=1, num_workers=8)
    elif agent == "td3":
        a = dict(name="td3", actor="deterministic_policy", critic="continuous_q_network")
        if mj:
            a.update(hidden_size=512, gamma=0.99, buffer_size=1000000, batch_size=128, start_train_step=25000,
                     initial_random_step=25000, tau=5e-3, update_delay=2, action_noise_std=0.1, target_noise_std=0.2,
                     target_noise_clip=0.5, lr_decay=True)
            opt = dict(actor="adam", critic="adam", actor_lr=3e-4, critic_lr=3e-4)
            tr = dict(_TRAIN_MUJOCO, distributed_batch_size=256, update_period=1, num_workers=8)
        else:       # td3/cartpole.py spells two keys differently from the constructor (actor_period, act_noise_std): kept as shipped
            a.update(gamma=0.99, buffer_size=50000, batch_size=128, start_train_step=1000, initial_random_step=0, tau=1e-3,
                     actor_period=2, act_noise_std=0.1, target_noise_std=0.2, target_noise_clip=0.5, lr_decay=True)
            opt = dict(actor="adam", critic="adam", actor_lr=1e-3, critic_lr=1e-3)
            tr = dict(_TRAIN_SMALL, eval_iteration=10, update_period=1, num_workers=8)
    else:
        a = dict(name="sac", actor="continuous_policy", critic="continuous_q_network", use_dynamic_alpha=True, gamma=0.99, tau=5e-3,
                 buffer_size=50000, batch_size=256 if mj else 64, start_train_step=25000 if mj else 5000, static_log_alpha=-2.0,
                 lr_decay=True)
        if env == "cartpole":
            a.update(target_update_period=500)
            a = {k: a[k] for k in ("name", "actor", "critic", "use_dynamic_alpha", "gamma", "tau", "buffer_size", "batch_size",
                                   "start_train_step", "static_log_alpha", "target_update_period", "lr_decay")}
        opt = dict(actor="adam", critic="adam", alpha="adam", actor_lr=5e-4, critic_lr=1e-3, alpha_lr=3e-4)
        if env == "cartpole":
            opt.update(actor_lr=1.5e-4, critic_lr=3e-4, alpha_lr=1e-5)
        tr = dict(_TRAIN_MUJOCO, record=False, record_period=500000, update_period=128, num_workers=16) if mj else \
            dict(_TRAIN_SMALL, eval_iteration=10, update_period=32, num_workers=8)
    return dict(env=env_d, agent=a, optim=opt, train=tr)


def available():
    out = []
    for ag, envs in _AC_ENVS.items():
        out += [f"config.{ag}.{e}" for e in envs]
    for ag in list(_VALUE_AGENTS) + ["ape_x"]:
        out += [f"config.{ag}.{e}" for e in ("cartpole", "mountaincar", "atari")]
    out += [f"config.ppo.{e}" for e in ("cartpole", "mountaincar", "pendulum", "mujoco", "atari")]
    return out


def load(config_path):
    parts = config_path.split(".")
    if len(parts) != 3 or parts[0] != "config":
        raise ImportError(f"no config '{config_path}' (built-ins: {available()})")
    _, agent, env = parts
    if agent in _VALUE_AGENTS and env in ("cartpole", "mountaincar", "atari"):
        d = _value_config(agent, env)
    elif agent == "ape_x" and env in ("cartpole", "mountaincar", "atari"):
        d = _ape_x_config(env)
    elif agent == "ppo" and env in ("cartpole", "mountaincar", "pendulum", "mujoco", "atari"):
        d = _ppo_config(env)
    elif agent in _AC_ENVS and env in _AC_ENVS[agent]:
        d = _ac_config(agent, env)
    else:
        raise ImportError(f"no config '{config_path}' (built-ins: {available()})")
    return SimpleNamespace(**d)
