"""CPU-only checks of the host side: C-ABI exports, config manager (the reference's
test/manager/test_config_manager.py behaviour), built-in configs, product path refusing to run without
CUDA, oracle env restatement bookkeeping, world_size-2 gloo test of the multi-GPU plumbing."""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_c_abi_exports_every_declared_symbol():
    from jorldy_b200._lib import LIB_PATH, declared_symbols, load
    assert os.path.exists(LIB_PATH), "build the library first (__graft_entry__.build())"
    lib = ctypes.CDLL(LIB_PATH)
    names = declared_symbols()
    assert len(names) >= 30
    for n in names:
        assert hasattr(lib, n), n
    load()


def test_fused_args_struct_matches_its_ctypes_mirror():
    """include/jorldy_b200_fused.h is mirrored field by field in core/agent/ppo_fused.py: sizes must agree (host-only call)."""
    from jorldy_b200._lib import C
    from jorldy_b200.core.agent.ppo_fused import FusedArgs
    assert ctypes.sizeof(FusedArgs) == C.jb_ppo_fused_args_size()
    names = [f[0] for f in FusedArgs._fields_]
    hdr = open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "include", "jorldy_b200_fused.h")).read()
    body = hdr[hdr.index("typedef struct jb_ppo_fused_args {") + len("typedef struct jb_ppo_fused_args {"):hdr.index("} jb_ppo_fused_args;")]
    import re
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    decl = []
    for stmt in body.split(";"):
        stmt = stmt.strip()
        if not stmt or stmt.startswith("typedef"):
            continue
        for part in stmt.split(","):
            m = re.search(r"\*?\s*([A-Za-z_][A-Za-z_0-9]*)\s*(\[\d+\])?\s*$", part.strip())
            if m:
                decl.append(m.group(1))
    assert decl == names, (decl, names)


def test_product_path_has_no_cpu_fallback():
    from jorldy_b200._lib import JbError
    from jorldy_b200.core import Agent
    with pytest.raises(JbError):
        Agent("ppo", state_size=4, action_size=2, device="cpu")
    if not torch.cuda.is_available():
        with pytest.raises(JbError):
            Agent("dqn", state_size=4, action_size=2)


def test_product_never_imports_oracle():
    for dirpath, _, files in os.walk(os.path.join(ROOT, "jorldy_b200")):
        for f in files:
            if f.endswith(".py"):
                src = open(os.path.join(dirpath, f)).read()
                assert "import oracle" not in src and "from oracle" not in src, f


def test_config_manager_overrides_and_typecast():
    from jorldy_b200.manager import ConfigManager, type_cast
    assert type_cast("3") == 3 and type_cast("1e-3") == 1e-3 and type_cast("True") is True
    assert type_cast("None") is None and type_cast("abc") == "abc"
    cm = ConfigManager("config.dqn.cartpole", ["--agent.batch_size", "64", "--optim.lr=0.5", "--env.render", "True",
                                               "--train.load_path", "None", "--agent.network", "dueling"])
    c = cm.config
    assert c.agent.batch_size == 64 and c.optim.lr == 0.5 and c.env.render is True and c.agent.network == "dueling"
    assert "load_path" not in c.train
    assert c.agent.name == "dqn" and c.agent.buffer_size == 50000 and c.agent.target_update_period == 500
    with pytest.raises(AssertionError):
        ConfigManager("config.dqn.cartpole", ["--foo.bar", "1"])


def test_builtin_configs_match_reference_headline_values():
    from jorldy_b200 import config as cfg
    ppo = cfg.load("config.ppo.cartpole")
    assert ppo.agent["n_step"] == 128 and ppo.agent["n_epoch"] == 3 and ppo.optim["lr"] == 2.5e-4
    assert ppo.train["distributed_batch_size"] == 256 and ppo.train["num_workers"] == 8
    rb = cfg.load("config.rainbow.atari")
    assert rb.agent["buffer_size"] == 1000000 and rb.agent["learn_period"] == 4 and rb.agent["head"] == "cnn"
    ax = cfg.load("config.ape_x.atari")
    assert ax.agent["buffer_size"] == 2000000 and ax.optim["eps"] == 1.5e-7 and ax.train["num_workers"] == 128
    mj = cfg.load("config.ppo.mujoco")
    assert mj.agent["n_step"] == 2048 and mj.train["distributed_batch_size"] == 2048
    for p in cfg.available():
        cfg.load(p)


def test_oracle_cartpole_wrapper_semantics():
    from oracle.classic_control import CartPoleBatch
    env = CartPoleBatch(3, seed=5, auto_reset=True)
    obs = env.reset()
    assert obs.shape == (3, 4) and obs.dtype == np.float32 and np.all(np.abs(obs) <= 0.05)
    total_done = 0
    for t in range(600):
        ns, r, d = env.step(np.ones(3, dtype=np.int64))
        assert np.all(np.where(d, r == -1.0, np.isclose(r, 0.1)))
        total_done += int(d.sum())
    assert total_done > 0 and np.all(env.elapsed < 500)


_GLOO_SCRIPT = r'''
import os, sys, torch, torch.distributed as dist
sys.path.insert(0, sys.argv[1])
from jorldy_b200.core import parallel
dist.init_process_group("gloo")
rank = dist.get_rank()
class Net: pass
class Ag: pass
a = Ag(); a.network = Net(); a.network.flat = torch.full((10,), float(rank + 1)); a.network.grad = torch.full((10,), float(rank))
a.allreduce = None; a.world_size = 1
parallel.attach(a, dist.get_world_size(), average_with="sum_div")
assert torch.all(a.network.flat == 1.0), a.network.flat
a.allreduce(a.network.grad)
assert torch.allclose(a.network.grad, torch.full((10,), 0.5)), a.network.grad
dist.barrier()
print("rank", rank, "ok")
'''


def test_parallel_attach_gloo_world2(tmp_path):
    script = tmp_path / "gloo_test.py"
    script.write_text(_GLOO_SCRIPT)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
           "--master-port", "29511", str(script), ROOT]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=240)
    assert r.returncode == 0, r.stdout + r.stderr
    assert r.stdout.count("ok") == 2


def test_exchange_layout_satisfies_the_kernel_checks():
    """jb_ppo_fused_run (csrc/ppo_fused.cu) rejects an exchange buffer whose regions are not 32-byte aligned or overlap;
    the PPO obs-11/act-3 network (num_flat % 8 == 4) was the case that tripped it."""
    from jorldy_b200.core.parallel import exchange_layout, P2P_FLAG_WORDS

    def num_flat(shapes):
        return sum((int(np.prod(s)) + 3) // 4 * 4 for s in shapes)

    H = 512
    nets = {"cartpole": [(H, 4), (H,), (H, H), (H,), (2, H), (2,), (1, H), (1,)],
            "hopper": [(H, 11), (H,), (H, H), (H,), (3, H), (3,), (3, H), (3,), (1, H), (1,)],
            "tiny": [(32, 3), (32,), (32, 32), (32,), (1, 32), (1,)]}
    for name, shapes in nets.items():
        nf = num_flat(shapes)
        for world in (2, 3, 4, 8):
            lay = exchange_layout(nf, world)
            P4 = nf // 4
            q4 = (P4 + world - 1) // world
            assert lay["llin_off"] >= P4 * 4, name
            assert lay["gred_off"] >= lay["llin_off"] + 8 * world * q4, name
            assert lay["flag_off"] >= lay["gred_off"] + 8 * P4, name
            assert lay["llin_off"] % 8 == 0 and lay["gred_off"] % 8 == 0 and lay["flag_off"] % 4 == 0, (name, world, lay)
            assert lay["n"] == lay["flag_off"] + P2P_FLAG_WORDS


def test_actor_critic_configs_equal_the_reference_files():
    """config.{ddpg,td3,sac}.* (SURVEY 8f-4) are generated from tables; where the reference is present they must equal its
    shipped config modules key for key (including td3/cartpole.py's two keys the constructor silently ignores)."""
    from jorldy_b200 import config as cfg
    paths = [p for p in cfg.available() if p.split(".")[1] in ("ddpg", "td3", "sac")]
    assert len(paths) == 8
    for p in paths:
        mine = cfg.load(p)
        assert mine.agent["name"] == p.split(".")[1] and mine.optim["actor"] == "adam"
        ref_file = os.path.join("/root/reference/jorldy", *p.split(".")) + ".py"
        if os.path.exists(ref_file):
            ref = {}
            exec(open(ref_file).read(), ref)
            for sec in ("env", "agent", "optim", "train"):
                assert getattr(mine, sec) == ref[sec], (p, sec)


def test_public_headers_are_plain_c99(tmp_path):
    """The drop-in boundary is a C ABI: both public headers must compile as C99 (-pedantic -Werror) — no C++ types, no torch
    types, plain pointers and sizes — and the fused-args struct must have the size its ctypes mirror assumes."""
    import shutil
    import subprocess
    gcc = shutil.which("gcc")
    if gcc is None:
        pytest.skip("no gcc")
    src = tmp_path / "hdr.c"
    src.write_text('#include <stdio.h>\n#include "jorldy_b200.h"\n#include "jorldy_b200_fused.h"\n'
                   'int main(void) { printf("%zu\\n", sizeof(jb_ppo_fused_args)); return 0; }\n')
    exe = tmp_path / "hdr"
    r = subprocess.run([gcc, "-std=c99", "-Wall", "-Werror", "-pedantic", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    size = int(subprocess.run([str(exe)], capture_output=True, text=True).stdout)
    import ctypes
    from jorldy_b200.core.agent.ppo_fused import FusedArgs
    assert size == ctypes.sizeof(FusedArgs)


def test_bench_dump_outputs_files(tmp_path, monkeypatch):
    """bench.py --dump-outputs: floating data as float32, integers and scalar results as float64, an array above
    DUMP_MAX_ELEMS replaced by the same seeded sample on every call, and the byte budget enforced."""
    import bench
    arrays = {"net.big": torch.arange(bench.DUMP_MAX_ELEMS + 5, dtype=torch.float32),
              "rollout.action": torch.arange(6, dtype=torch.int32).view(2, 3)}
    result = {"loss": 0.5, "note": "not a number"}
    for d in ("d1", "d2"):
        bench.dump_outputs(str(tmp_path / d), arrays, result)
    assert sorted(os.listdir(tmp_path / "d1")) == ["net.big.npy", "result.loss.npy", "rollout.action.npy"]
    big1, big2 = np.load(tmp_path / "d1" / "net.big.npy"), np.load(tmp_path / "d2" / "net.big.npy")
    assert big1.dtype == np.float32 and big1.shape == (bench.DUMP_MAX_ELEMS,) and np.array_equal(big1, big2)
    assert np.all(np.diff(big1) >= 0)
    act = np.load(tmp_path / "d1" / "rollout.action.npy")
    assert act.dtype == np.float64 and np.array_equal(act, np.arange(6).reshape(2, 3))
    assert np.load(tmp_path / "d1" / "result.loss.npy") == 0.5
    monkeypatch.setattr(bench, "DUMP_MAX_BYTES", 1024)
    with pytest.raises(ValueError):
        bench.dump_outputs(str(tmp_path / "d3"), arrays, result)
