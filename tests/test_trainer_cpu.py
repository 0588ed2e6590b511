"""SURVEY.md 8 (f-2): the trainer loop mirror against the call trace of the unmodified reference trainer
(tests/golden/trainer_calls.json, made by tests/golden/make_trainer_golden.py) and the rollout memory semantics."""
import json
import os
import sys

import pytest
import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from trainer_fakes import FakeAgent, FakeEnv  # noqa: E402

from isaac_rover_orbit_b200.trainer import RolloutAgent, RolloutMemory, SkrlSequentialLogTrainer  # noqa: E402


@pytest.fixture(scope="module")
def golden_calls(golden_dir):
    return json.load(open(os.path.join(golden_dir, "trainer_calls.json")))


@pytest.mark.parametrize("name, mode, steps, headless", [("train_5", "train", 5, True), ("eval_4_headless", "eval", 4, True),
                                                          ("eval_3_render", "eval", 3, False)])
def test_trainer_call_trace_equals_reference(golden_calls, name, mode, steps, headless):
    log = []
    trainer = SkrlSequentialLogTrainer(env=FakeEnv(log), agents=FakeAgent(log),
                                       cfg={"timesteps": steps, "disable_progressbar": True, "headless": headless})
    getattr(trainer, mode)()
    assert json.loads(json.dumps(log)) == golden_calls[name]  # same calls, order, arguments and tensor checksums


def test_log_episode_info_can_be_skipped():
    log = []
    SkrlSequentialLogTrainer(env=FakeEnv(log), agents=FakeAgent(log), cfg={"timesteps": 4}, log_episode_info=False).train()
    assert not [c for c in log if c[0] == "track_data"]


def test_rollout_memory_wraps_like_skrl():
    mem = RolloutMemory(memory_size=3, num_envs=2, device="cpu")
    assert mem.create_tensor("states", 4) and not mem.create_tensor("states", 4)
    mem.create_tensor("rewards", 1)
    mem.create_tensor("terminated", 1, dtype=torch.bool)
    with pytest.raises(ValueError):
        mem.create_tensor("states", 5)
    with pytest.raises(ValueError):
        mem.add_samples()
    for t in range(4):
        mem.add_samples(states=torch.full((2, 4), float(t)), rewards=torch.full((2,), 0.5 * t),
                        terminated=torch.tensor([t == 3, False]), unknown=torch.zeros(2, 9))
        assert len(mem) == (min(t + 1, 3) * 2)
    assert mem.filled and mem.memory_index == 1
    assert mem.get_tensor_by_name("states")[:, 0, 0].tolist() == [3.0, 1.0, 2.0]  # row 0 overwritten by t = 3
    assert mem.get_tensor_by_name("rewards", keepdim=False).shape == (6, 1)
    assert mem.get_tensor_by_name("terminated")[0, :, 0].tolist() == [True, False]
    mem.reset()
    assert len(mem) == 0 and not mem.filled


def test_rollout_agent_writes_what_the_env_returned():
    class Policy:
        def act(self, inputs, role=""):
            s = inputs["states"]
            return s[:, :2] * 2.0, s[:, :1] * -1.0, {}

    log = []
    env = FakeEnv(log, num_envs=3)
    mem = RolloutMemory(memory_size=8, num_envs=3, device="cpu")
    agent = RolloutAgent(Policy(), mem, observation_size=4, action_size=2)
    SkrlSequentialLogTrainer(env=env, agents=agent, cfg={"timesteps": 5}).train()
    assert agent._initialised == 2  # the reference initialises the agent in __init__ and again in train()
    assert mem.memory_index == 5 and agent.training
    st = mem.get_tensor_by_name("states")
    assert torch.equal(st[0], torch.ones(3, 4))  # the reset observation
    assert torch.allclose(mem.get_tensor_by_name("actions")[:5], st[:5, :, :2] * 2.0)
    assert torch.allclose(mem.get_tensor_by_name("log_prob")[:5], st[:5, :, :1] * -1.0)
    assert torch.allclose(mem.get_tensor_by_name("rewards")[:5, 0, 0], torch.tensor([0.1, 0.2, 0.3, 0.4, 0.5]))
    assert agent.tracking_data["EpisodeInfo / Episode Reward/collision"] == [-0.5, -1.0]
