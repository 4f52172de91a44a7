"""CPU-only checks of the drop-in boundary: C-ABI exports, Python surface, host-side block cutting."""
import ctypes
import os
import re

import numpy as np

from oracle import synth
from helpers import build_oracle_replay, crc

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

REFERENCE_CONFIG_NAMES = [  # config.py:1-37 upstream
    "game_name", "obs_shape", "lr", "eps", "grad_norm", "batch_size", "learning_starts", "save_interval",
    "target_net_update_interval", "gamma", "prio_exponent", "importance_sampling_exponent", "training_steps",
    "buffer_capacity", "max_episode_steps", "actor_update_interval", "block_length", "num_actors", "base_eps", "alpha",
    "log_interval", "burn_in_steps", "learning_steps", "forward_steps", "seq_len", "hidden_dim", "render", "save_plot",
    "test_epsilon"]


def test_header_symbols_are_exported_and_bound():
    from r2d2_b200 import _lib
    header = open(os.path.join(ROOT, "include", "r2d2_b200.h")).read()
    declared = set(re.findall(r"\b(r2d2_[a-z0-9_]+)\s*\(", header))
    declared -= {"r2d2_tree", "r2d2_net", "r2d2_replay"}
    assert len(declared) >= 25
    lib = ctypes.CDLL(_lib.LIB_PATH)             # loads without a GPU; no compute call is made
    for name in sorted(declared):
        assert hasattr(lib, name), f"{name} declared in include/r2d2_b200.h but not exported"
        assert name in _lib.SIGNATURES, f"{name} has no ctypes signature in r2d2_b200/_lib.py"
    assert set(_lib.SIGNATURES) <= declared, set(_lib.SIGNATURES) - declared
    assert _lib.lib().r2d2_abi_version() >= 1


def test_config_surface_matches_reference():
    from r2d2_b200 import config
    for name in REFERENCE_CONFIG_NAMES:
        assert hasattr(config, name), name
    assert (config.batch_size, config.burn_in_steps, config.learning_steps, config.forward_steps) == (64, 40, 40, 5)
    assert config.seq_len == 85 and config.buffer_capacity == 2_000_000 and config.block_length == 400


def test_network_state_dict_surface():
    import torch
    from r2d2_b200.learner_core import PARAM_NAMES, param_shapes
    from r2d2_b200.model import AgentState, Network
    net = Network(9)
    sd = net.state_dict()
    assert list(sd.keys()) == PARAM_NAMES                          # model.py:39-63 order and names
    for k, shape in param_shapes(9).items():
        assert tuple(sd[k].shape) == shape
    st = AgentState(torch.zeros(1, 1, 84, 84, dtype=torch.uint8), 9)
    with torch.no_grad():
        q, (h, c) = net(st)
    assert q.shape == (1, 9) and h.shape[-1] == 512
    try:
        net.calculate_q(torch.zeros(1, 2, 1, 84, 84), torch.zeros(1, 2, 9), torch.zeros(1, 2), (h, c),
                        torch.tensor([0], dtype=torch.uint8), torch.tensor([1], dtype=torch.uint8))
    except RuntimeError as e:
        assert "no CPU fallback" in str(e)                          # the learner path refuses to run without CUDA
    else:
        raise AssertionError("calculate_q must not silently run on the CPU")


def test_dropin_modules_alias_the_package():
    import importlib
    import sys
    sys.path.insert(0, os.path.join(ROOT, "dropin"))
    try:
        for name in ("config", "model", "worker", "priority_tree", "environment"):
            sys.modules.pop(name, None)
            mod = importlib.import_module(name)
            assert mod is importlib.import_module(f"r2d2_b200.{name}")
        import worker
        for cls in ("Learner", "Actor", "ReplayBuffer"):
            assert hasattr(worker, cls)
    finally:
        sys.path.remove(os.path.join(ROOT, "dropin"))
        for name in ("config", "model", "worker", "priority_tree", "environment"):
            sys.modules.pop(name, None)


def test_dropin_config_overrides_in_a_fresh_process(tmp_path):
    """With dropin/ on PYTHONPATH, a script's `import config` binds this package's config with R2D2_CONFIG_OVERRIDES
    applied before `worker` captures its def-time defaults; an unknown name is an error."""
    import json
    import subprocess
    import sys
    code = ("import config, worker, r2d2_b200.config as pkg\n"
            "from worker import Learner, Actor, ReplayBuffer\n"
            "assert config is pkg\n"
            "print(config.training_steps, config.batch_size, config.seq_len, worker.Learner.__init__.__defaults__[3])\n")
    env = dict(os.environ)
    env["PYTHONPATH"] = os.pathsep.join([os.path.join(ROOT, "dropin"), ROOT, env.get("PYTHONPATH", "")])
    env["R2D2_CONFIG_OVERRIDES"] = json.dumps({"training_steps": 6, "batch_size": 8, "learning_steps": 10, "game_name": "Pong"})
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=300, cwd=str(tmp_path), env=env)
    assert r.returncode == 0, r.stderr[-3000:]
    assert r.stdout.split() == ["6", "8", "55", "Pong"], r.stdout
    env["R2D2_CONFIG_OVERRIDES"] = json.dumps({"trainig_steps": 6})
    r = subprocess.run([sys.executable, "-c", "import config"], capture_output=True, text=True, timeout=300, cwd=str(tmp_path), env=env)
    assert r.returncode != 0 and "unknown config name 'trainig_steps'" in r.stderr, r.stderr[-3000:]


def test_local_buffer_blocks_match_reference_golden(golden_dir):
    """The product's host-side block cutter (worker.LocalBuffer) against the reference's recorded blocks."""
    from r2d2_b200.worker import LocalBuffer
    g = np.load(os.path.join(golden_dir, "replay_ragged.npz"))
    _, blocks = build_oracle_replay(synth.RAGGED_SCRIPT, 8, 8, actor_cls=LocalBuffer)
    for i, (blk, prio, ep) in enumerate(blocks):
        assert crc(blk.obs) == int(g[f"blk{i}_obs_crc"])
        assert crc(blk.last_action) == int(g[f"blk{i}_last_action_crc"])
        assert crc(blk.hidden) == int(g[f"blk{i}_hidden_crc"])
        np.testing.assert_array_equal(blk.last_reward, g[f"blk{i}_last_reward"])
        np.testing.assert_array_equal(blk.action, g[f"blk{i}_action"])
        np.testing.assert_array_equal(blk.n_step_reward, g[f"blk{i}_n_step_reward"])
        np.testing.assert_array_equal(blk.gamma, g[f"blk{i}_gamma"])
        np.testing.assert_array_equal(np.stack([blk.burn_in_steps, blk.learning_steps, blk.forward_steps]), g[f"blk{i}_steps"])
        np.testing.assert_array_equal(prio, g[f"blk{i}_prio"])
        assert (-1.0 if ep is None else ep) == float(g[f"blk{i}_ep"])


def test_vector_actor_block_logic_with_stub_policy():
    """Host logic of worker.VectorActor (block cuts, bootstrap from the next step, resets, shipping) against N
    reference-style CPU `Actor`s, with the batched policy replaced by a stub that loops the CPU Network -- the GPU parity of
    the real policy is tests/test_gpu_worker.py."""
    import queue
    import numpy as np
    import torch
    from r2d2_b200 import config
    from r2d2_b200.environment import SyntheticAtariEnv
    from r2d2_b200.model import AgentState, Network
    from r2d2_b200.worker import Actor, LocalBuffer, VectorActor
    from oracle.learner import init_params
    A, C, N, STEPS, BL = 9, 1, 2, 130, 80            # A = 9: `Actor` builds its own env (MsPacman action count)
    config.obs_shape = (C, 84, 84)
    torch.set_num_threads(4)
    shared = Network(A, obs_shape=(C, 84, 84))
    shared.load_state_dict(init_params(A, in_channels=C, seed=9))
    shared.eval()
    mk = lambda i: SyntheticAtariEnv(A, (C, 84, 84), mean_episode_len=100, seed=700 + i)

    class StubPolicy:
        def load_state_dict(self, sd):
            pass

        def step(self, obs, last_action, last_reward, hidden):
            qs, hs = [], []
            for i in range(N):
                st = AgentState(torch.from_numpy(obs[i]).unsqueeze(0).float(), A)
                st.last_action = torch.from_numpy(last_action[i]).float().unsqueeze(0)
                st.last_reward = torch.tensor([[float(last_reward[i])]])
                h = hidden[i]
                st.hidden_state = (h[0].reshape(1, -1).contiguous(), h[1].reshape(1, -1).contiguous())
                with torch.no_grad():
                    q, (hn, cn) = shared(st)
                qs.append(q[0])
                hs.append(torch.stack([hn.reshape(-1), cn.reshape(-1)]))
            return torch.stack(qs), torch.stack(hs)

    shipped = [[] for _ in range(N)]
    va = VectorActor([0.0] * N, shared, queue.Queue(), obs_shape=(C, 84, 84), max_episode_steps=10 ** 6, block_length=BL,
                     envs=[mk(i) for i in range(N)], policy=StubPolicy())
    va._ship = lambda i, triple, over: shipped[i].append(triple)
    for _ in range(STEPS):
        va.step()
    for i in range(N):
        ac = Actor(0.0, shared, queue.Queue(), obs_shape=(C, 84, 84), max_episode_steps=10 ** 6, block_length=BL)
        ac.env = mk(i)
        ac.model.load_state_dict(shared.state_dict())
        ac.local_buffer = LocalBuffer(A, block_length=BL)
        ref = []
        ac._ship = lambda triple, over, ref=ref: ref.append(triple)
        while ac.actor_steps < STEPS + 60:
            ac.play_episode()
        assert len(shipped[i]) >= 1
        for (blk, prio, ret), (rblk, rprio, rret) in zip(shipped[i], ref):
            for f in ("obs", "last_action", "last_reward", "action", "n_step_reward", "gamma", "burn_in_steps",
                      "learning_steps", "forward_steps"):
                assert np.array_equal(getattr(blk, f), getattr(rblk, f)), f
            assert np.allclose(blk.hidden, rblk.hidden, atol=1e-6) and np.allclose(prio, rprio, atol=1e-5)
            assert (ret is None) == (rret is None)
