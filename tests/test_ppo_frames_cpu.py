"""CPU checks of PPO on frame stacks: the built-in Atari config and the gathering im2col entry point of the C ABI."""
from jorldy_b200 import config as cfg


def test_ppo_atari_config():
    assert "config.ppo.atari" in cfg.available()
    c = cfg.load("config.ppo.atari")
    assert c.env["stack_frame"] == 4 and c.env["img_width"] == 84 and c.env["img_height"] == 84
    assert c.agent == dict(name="ppo", network="discrete_policy_value", head="cnn", gamma=0.99, batch_size=32, n_step=128,
                           n_epoch=3, _lambda=0.95, epsilon_clip=0.1, vf_coef=1.0, ent_coef=0.01, clip_grad_norm=1.0,
                           use_standardization=True, lr_decay=True)
    assert c.optim == dict(name="adam", lr=2.5e-4)
    assert c.train["run_step"] == 30_000_000 and c.train["distributed_batch_size"] == 1024
    assert c.train["update_period"] == 128 and c.train["num_workers"] == 32


def test_im2col_u8_rows_is_declared():
    import ctypes
    from jorldy_b200._lib import parse_header
    decls = parse_header()
    assert decls["jb_im2col_u8_rows"] == [ctypes.c_void_p, ctypes.c_void_p] + [ctypes.c_int] * 7 + [ctypes.c_void_p] * 2


def test_head_launch_counts():
    """The MLP head keeps PPO's 13-launch minibatch step; the CNN head counts its own convolution kernels."""
    from jorldy_b200.core.network.head import CNNHead, MLPHead
    mlp = MLPHead(4, 64)
    assert mlp.fwd_launches + mlp.bwd_launches(1024) == 2
    cnn = CNNHead([4, 84, 84], 512)
    assert cnn.fwd_launches == 7
    # B = 1024: every conv dW is split over the grid (gemm + weight fold + bias fold); B = 8: only conv1's; B = 1: none
    assert cnn.bwd_launches(1024) == 1 + 3 * 3 + 4
    assert cnn.bwd_launches(8) == 1 + 3 + 1 + 1 + 4
    assert cnn.bwd_launches(1) == 1 + 3 * 1 + 4
