"""The caller of the hot path: ``SkrlSequentialLogTrainer`` (reference rover_envs/utils/skrl_utils.py:42-206), the
rollout storage it writes through the agent (skrl 1.1.0 ``Memory.add_samples``) and a small agent that samples
actions with the tcgen05 policy -- SURVEY.md 8 (f-2) -- and, for PPO, the returns and advantages skrl computes at the
end of every rollout (``compute_gae``, ``PPORolloutAgent``; one CUDA pass over the memory, DESIGN.md 3.8).

The trainer mirrors the reference call for call (same order, same keyword arguments, the double ``agents.init`` of
``__init__`` + ``train`` included), so that a maintainer can swap the import.  It is host-side glue: every tensor
stays on the GPU, nothing here synchronises except the ``.item()`` calls the reference itself makes when it logs
episode information (``log_episode_info=False`` skips them; ``RoverEnv`` keeps those statistics on the device anyway).
PPO's optimisation step (minibatches, clipped surrogate, backward pass) is outside the hot path and is not provided.

``capture_steps`` records a step function into CUDA graphs (one per input variant) -- how ``bench.py`` runs
act -> step -> record without per-launch host overhead.
"""
from __future__ import annotations

import copy

import torch

from . import torch_ops  # noqa: F401  (registers torch.ops.rover_b200.*, which the agents and compute_gae call)

# skrl 1.1.0, skrl/trainers/torch/sequential.py (third-party, pinned by the reference's environment; restated)
SEQUENTIAL_TRAINER_DEFAULT_CONFIG = {
    "timesteps": 100000,
    "headless": False,
    "disable_progressbar": False,
    "close_environment_at_exit": True,
}


class RolloutMemory:
    """Tensor storage of skrl 1.1.0 ``Memory`` (memories/torch/base.py) as ``RandomMemory`` is used by the reference
    (rover_envs/learning/train/agents.py:17-18): tensors ``[memory_size, num_envs, size]``, ``add_samples`` writes
    row ``memory_index`` and wraps, ``filled`` turns true on the first wrap."""

    def __init__(self, memory_size: int, num_envs: int = 1, device="cuda:0"):
        self.memory_size = int(memory_size)
        self.num_envs = int(num_envs)
        self.device = torch.device(device)
        self.filled = False
        self.memory_index = 0
        self.tensors: dict[str, torch.Tensor] = {}

    def __len__(self) -> int:
        return self.memory_size * self.num_envs if self.filled else self.memory_index * self.num_envs

    def create_tensor(self, name: str, size: int, dtype=torch.float32, keep_dimensions: bool = True) -> bool:
        if name in self.tensors:
            t = self.tensors[name]
            if t.shape[-1] != size or t.dtype != dtype:
                raise ValueError(f"tensor {name} exists with another size / dtype")
            return False
        self.tensors[name] = torch.zeros(self.memory_size, self.num_envs, int(size), dtype=dtype, device=self.device)
        return True

    def get_tensor_names(self):
        return sorted(self.tensors)

    def get_tensor_by_name(self, name: str, keepdim: bool = True) -> torch.Tensor:
        t = self.tensors[name]
        return t if keepdim else t.view(-1, t.shape[-1])

    def reset(self) -> None:
        self.filled = False
        self.memory_index = 0

    def add_samples(self, **tensors: torch.Tensor) -> None:
        """One transition per environment: every tensor is ``[num_envs, size]`` (or ``[num_envs]``); unknown names
        are ignored, as skrl does.  No host synchronisation (plain ``copy_`` into row ``memory_index``)."""
        if not tensors:
            raise ValueError("No samples to be recorded in memory")
        for name, value in tensors.items():
            if name in self.tensors and value is not None:
                dst = self.tensors[name][self.memory_index]
                dst.copy_(value.reshape(dst.shape))
        self.memory_index += 1
        if self.memory_index >= self.memory_size:
            self.memory_index = 0
            self.filled = True


class BaseAgent:
    """What skrl 1.1.0's base ``Agent`` (agents/torch/base.py) does in the hooks the trainer calls: tracking only.
    ``record_transition`` keeps per-env running returns / lengths and folds finished episodes into device-side totals
    (skrl reads them back with ``.item()`` at its write interval; ``finished_episode_stats`` does that on demand --
    nothing here synchronises per step).  The evaluation loop records through THIS method, bypassing the subclass
    (``super(type(agent), agent).record_transition``, skrl ``Trainer.single_agent_eval``)."""

    def __init__(self):
        self.training = False
        self.tracking_data: dict[str, list] = {}
        self._initialised = 0
        self._cum_rewards = None
        self._cum_steps = None
        self._finished = None  # [episodes, return sum, length sum]

    def init(self, trainer_cfg=None) -> None:
        self._initialised += 1

    def set_running_mode(self, mode: str) -> None:
        self.training = mode == "train"

    def pre_interaction(self, timestep: int, timesteps: int) -> None:
        pass

    def post_interaction(self, timestep: int, timesteps: int) -> None:
        pass

    def track_data(self, tag: str, value: float) -> None:
        self.tracking_data.setdefault(tag, []).append(value)

    def record_transition(self, states, actions, rewards, next_states, terminated, truncated, infos, timestep,
                          timesteps) -> None:
        r = rewards.reshape(-1).float()
        if self._cum_rewards is None:
            self._cum_rewards = torch.zeros_like(r)
            self._cum_steps = torch.zeros_like(r)
            self._finished = torch.zeros(3, device=r.device)
        self._cum_rewards += r
        self._cum_steps += 1
        done = (terminated.reshape(-1) | truncated.reshape(-1)).float()
        self._finished += torch.stack([done.sum(), (self._cum_rewards * done).sum(), (self._cum_steps * done).sum()])
        self._cum_rewards *= 1.0 - done
        self._cum_steps *= 1.0 - done

    def finished_episode_stats(self) -> dict:
        """Mean return / length of the episodes that finished so far (synchronises)."""
        if self._finished is None:
            return {"episodes": 0, "mean_return": 0.0, "mean_length": 0.0}
        k, ret, length = (float(v) for v in self._finished.cpu())
        return {"episodes": int(k), "mean_return": ret / max(k, 1.0), "mean_length": length / max(k, 1.0)}


class RolloutAgent(BaseAgent):
    """The part of the reference's skrl agent that sits on the hot path: ``act`` = ``GaussianMixin.act`` of the policy
    (sampling + log-prob, SURVEY.md A.4) and ``record_transition`` = the ``RandomMemory`` rollout write.  The
    hooks the trainer calls around them exist and do what skrl's base ``Agent`` does (tracking), nothing more."""

    def __init__(self, policy, memory: RolloutMemory | None = None, observation_size: int | None = None,
                 action_size: int = 2, value=None, action_out: torch.Tensor | None = None, action_rng=None):
        """``value``: the PPO value network (``DeterministicNeuralNetwork``).  skrl's PPO evaluates it in
        ``record_transition`` on the states ``act`` just saw; here both networks run in ONE pass over the observation
        (``policy.policy_value_forward``) and the values are written to the memory's ``values`` tensor.
        ``action_rng`` (an ``ops.ActionRng``): the policy samples inside its forward pass with noise keyed on
        (seed, step, env) instead of ``torch.randn`` -- one launch per ``act``, policy and value together
        (``policy.policy_value_act``); without it ``act`` draws ``torch.randn`` as before.  fp32 states and the bf16 mirror
        (``alloc_obs_bf16`` layout, what ``RoverEnv(observation_dtype=torch.bfloat16)`` returns) take the same routes.
        ``observation_size``: the width of the memory's ``states``; by default ``4 + policy.encoder_input_size`` for a
        policy that has one (965 for the shipped 961-ray scan), else 965."""
        super().__init__()
        if observation_size is None:
            r = getattr(policy, "encoder_input_size", None)
            observation_size = 965 if r is None else 4 + int(r)
        self.policy = policy
        self.value = value
        self.action_rng = action_rng
        self.action_out = action_out  # e.g. ``env.action_input``: the sampled actions land where the env's step reads them
        self.memory = memory
        self._log_prob = None
        self._values = None
        if memory is not None and value is not None:
            memory.create_tensor("values", 1)
        if memory is not None:
            memory.create_tensor("states", observation_size)
            memory.create_tensor("actions", action_size)
            memory.create_tensor("rewards", 1)
            memory.create_tensor("terminated", 1, dtype=torch.bool)
            memory.create_tensor("log_prob", 1)

    def act(self, states: torch.Tensor, timestep: int, timesteps: int):
        if self.action_rng is not None and self.value is not None:
            from .policy import policy_value_act

            actions, log_prob, self._values, mean = policy_value_act(self.policy, self.value, states, self.action_rng,
                                                                     out_actions=self.action_out)
            self._log_prob = log_prob
            return actions, log_prob, {"mean_actions": mean}
        if self.value is None:
            extra = {"out_actions": self.action_out} if self.action_out is not None else {}  # (any skrl-style policy works)
            if self.action_rng is not None:
                extra["rng"] = self.action_rng
            actions, log_prob, outputs = self.policy.act({"states": states}, role="policy", **extra)
            if self.value is not None:
                self._values = self.value.act({"states": states}, role="value")[0]
        else:
            from .policy import policy_value_forward

            mean, self._values = policy_value_forward(self.policy, self.value, states)
            eps = torch.randn(mean.shape[0], 2, device=mean.device)  # (the same draw GaussianNeuralNetwork.act makes)
            if self.action_out is not None:
                actions, log_prob = self.action_out, torch.empty(mean.shape[0], device=mean.device)
                torch.ops.rover_b200.gaussian_act_out(mean, self.policy.log_std_parameter, eps, actions, log_prob)
            else:
                actions, log_prob = torch.ops.rover_b200.gaussian_act(mean, self.policy.log_std_parameter, eps)
            log_prob = log_prob.unsqueeze(-1)
            outputs = {"mean_actions": mean}
        self._log_prob = log_prob
        return actions, log_prob, outputs

    def record_transition(self, states, actions, rewards, next_states, terminated, truncated, infos, timestep,
                          timesteps) -> None:
        super().record_transition(states, actions, rewards, next_states, terminated, truncated, infos, timestep, timesteps)
        if self.memory is not None:
            self.memory.add_samples(states=states, actions=actions, rewards=rewards, terminated=terminated,
                                    log_prob=self._log_prob, **({"values": self._values} if self.value is not None else {}))


def compute_gae(rewards: torch.Tensor, dones: torch.Tensor, values: torch.Tensor, next_values: torch.Tensor,
                discount_factor: float = 0.99, lambda_coefficient: float = 0.95):
    """skrl 1.1.0 ``PPO._update.compute_gae`` (restated in DESIGN.md 2): ``(returns, advantages)`` of the memory's
    ``[T, N, 1]`` (or ``[T, N]``) rewards / dones / values and the last values ``[N, 1]``, advantages normalised over all
    ``T * N`` entries.  One ``rover_b200::ppo_gae`` call (three launches, no host synchronisation); returns bit-identical
    to skrl's loop, the normalisation as DESIGN.md 2 states it."""
    returns = torch.empty_like(rewards, memory_format=torch.contiguous_format)
    advantages = torch.empty_like(rewards, memory_format=torch.contiguous_format)
    torch.ops.rover_b200.ppo_gae(rewards.contiguous(), dones.contiguous(), values.contiguous(), next_values.contiguous(),
                                 float(discount_factor), float(lambda_coefficient), returns, advantages)
    return returns, advantages


class PPORolloutAgent(RolloutAgent):
    """``RolloutAgent`` plus what skrl 1.1.0's PPO does with the rollout before its optimisation epochs: it creates the
    memory's ``returns`` / ``advantages`` (``PPO.init``), keeps the last ``next_states`` (``record_transition``) and, on
    every ``memory_size``-th ``post_interaction`` (``_rollout % _rollouts``), evaluates the value network on them and
    writes ``compute_gae`` of the memory into those tensors (``PPO._update``).  ``dones`` is the memory's ``terminated``,
    as in skrl 1.1.0: a truncated step bootstraps from the next row's value.  The optimisation epochs are not provided."""

    def __init__(self, policy, value, memory: RolloutMemory, discount_factor: float = 0.99, lambda_: float = 0.95,
                 action_out: torch.Tensor | None = None, action_rng=None, observation_size: int | None = None):
        if value is None or memory is None:
            raise ValueError("PPORolloutAgent needs a value network and a memory")
        super().__init__(policy, memory, observation_size=observation_size, value=value, action_out=action_out,
                         action_rng=action_rng)
        self.discount_factor = float(discount_factor)
        self.lambda_ = float(lambda_)
        self._rollout = 0
        self._current_next_states = None
        memory.create_tensor("returns", 1)
        memory.create_tensor("advantages", 1)

    def record_transition(self, states, actions, rewards, next_states, terminated, truncated, infos, timestep,
                          timesteps) -> None:
        super().record_transition(states, actions, rewards, next_states, terminated, truncated, infos, timestep, timesteps)
        self._current_next_states = next_states

    def post_interaction(self, timestep: int, timesteps: int) -> None:
        self._rollout += 1
        if self._rollout % self.memory.memory_size == 0:
            self._update_returns()
        super().post_interaction(timestep, timesteps)

    def _update_returns(self) -> None:
        mem = self.memory
        with torch.no_grad():
            # skrl passes next_states.float(); the value network gives the same values on bf16 and fp32 states
            last_values = self.value.act({"states": self._current_next_states}, role="value")[0]
            torch.ops.rover_b200.ppo_gae(mem.get_tensor_by_name("rewards"), mem.get_tensor_by_name("terminated"),
                                         mem.get_tensor_by_name("values"), last_values.contiguous(), self.discount_factor,
                                         self.lambda_, mem.get_tensor_by_name("returns"),
                                         mem.get_tensor_by_name("advantages"))


class SkrlSequentialLogTrainer:
    """rover_envs/utils/skrl_utils.py:42-206 over skrl 1.1.0 ``Trainer`` (trainers/torch/base.py)."""

    def __init__(self, env, agents, agents_scope: list | None = None, cfg: dict | None = None,
                 log_episode_info: bool = True):
        _cfg = copy.deepcopy(SEQUENTIAL_TRAINER_DEFAULT_CONFIG)  # skrl_utils.py:87-88
        _cfg.update(cfg if cfg is not None else {})
        self.cfg = _cfg
        self.env = env
        self.agents = agents
        self.agents_scope = agents_scope if agents_scope is not None else []
        self.timesteps = _cfg.get("timesteps", 0)
        self.headless = _cfg.get("headless", False)
        self.disable_progressbar = _cfg.get("disable_progressbar", False)
        self.close_environment_at_exit = _cfg.get("close_environment_at_exit", True)
        self.initial_timestep = 0
        self.num_simultaneous_agents = len(agents) if isinstance(agents, (list, tuple)) else 1
        self.log_episode_info = log_episode_info
        if getattr(self.env, "num_agents", 1) > 1:  # skrl_utils.py:94-98
            for agent in self.agents:
                agent.init(trainer_cfg=self.cfg)
        else:
            self.agents.init(trainer_cfg=self.cfg)

    def _log_episode(self, agent, infos) -> None:
        # skrl_utils.py:139-142 -- one host read per scalar, exactly as the reference does it
        if self.log_episode_info and "episode" in infos:
            for k, v in infos["episode"].items():
                if isinstance(v, torch.Tensor) and v.numel() == 1:
                    agent.track_data(f"EpisodeInfo / {k}", v.item())

    def train(self) -> None:
        """skrl_utils.py:100-148."""
        self.agents.init(trainer_cfg=self.cfg)
        self.agents.set_running_mode("train")
        states, infos = self.env.reset()
        for timestep in range(self.timesteps):
            self.agents.pre_interaction(timestep=timestep, timesteps=self.timesteps)
            with torch.no_grad():
                actions = self.agents.act(states, timestep=timestep, timesteps=self.timesteps)[0]
            next_states, rewards, terminated, truncated, infos = self.env.step(actions)
            with torch.no_grad():
                self.agents.record_transition(states=states, actions=actions, rewards=rewards, next_states=next_states,
                                              terminated=terminated, truncated=truncated, infos=infos,
                                              timestep=timestep, timesteps=self.timesteps)
            self._log_episode(self.agents, infos)
            self.agents.post_interaction(timestep=timestep, timesteps=self.timesteps)
            states.copy_(next_states)  # skrl_utils.py:148: in place -- the env may hand out its own buffer

    def eval(self) -> None:
        """skrl_utils.py:150-206; one agent -> skrl 1.1.0 ``Trainer.single_agent_eval``."""
        if self.num_simultaneous_agents > 1:
            for agent in self.agents:
                agent.set_running_mode("eval")
        else:
            self.agents.set_running_mode("eval")
        if self.num_simultaneous_agents == 1:
            self._single_agent_eval()
            return
        states, infos = self.env.reset()
        for timestep in range(self.initial_timestep, self.timesteps):
            with torch.no_grad():
                actions = torch.vstack([agent.act(states[scope[0]:scope[1]], timestep=timestep, timesteps=self.timesteps)[0]
                                        for agent, scope in zip(self.agents, self.agents_scope)])
            next_states, rewards, terminated, truncated, infos = self.env.step(actions)
            with torch.no_grad():
                for agent, scope in zip(self.agents, self.agents_scope):
                    agent.record_transition(states=states[scope[0]:scope[1]], actions=actions[scope[0]:scope[1]],
                                            rewards=rewards[scope[0]:scope[1]], next_states=next_states[scope[0]:scope[1]],
                                            terminated=terminated[scope[0]:scope[1]],
                                            truncated=truncated[scope[0]:scope[1]], infos=infos, timestep=timestep,
                                            timesteps=self.timesteps)
                    self._log_episode(agent, infos)
            states.copy_(next_states)

    def _single_agent_eval(self) -> None:
        states, infos = self.env.reset()
        for timestep in range(self.initial_timestep, self.timesteps):
            with torch.no_grad():
                actions = self.agents.act(states, timestep=timestep, timesteps=self.timesteps)[0]
            next_states, rewards, terminated, truncated, infos = self.env.step(actions)
            if not self.headless:
                self.env.render()  # skrl renders unless headless; RoverEnv.render is a no-op (no viewport without the simulator)
            with torch.no_grad():
                # evaluation records through the base class of the agent (tracking only), as skrl does
                super(type(self.agents), self.agents).record_transition(
                    states=states, actions=actions, rewards=rewards, next_states=next_states, terminated=terminated,
                    truncated=truncated, infos=infos, timestep=timestep, timesteps=self.timesteps)
            if self.env.num_envs > 1:
                states = next_states
            elif terminated.any() or truncated.any():
                with torch.no_grad():
                    states, infos = self.env.reset()
            else:
                states = next_states


def capture_steps(step_fn, n_variants: int = 1, warmup: int = 1):
    """Record ``step_fn(i)`` for ``i in range(n_variants)`` into CUDA graphs and return ``replay(i)``.
    ``step_fn`` must only enqueue work on the current stream (our operators do); it is run ``warmup`` times per
    variant before capture so that one-time driver calls happen outside the graph."""
    for _ in range(warmup):
        for i in range(n_variants):
            step_fn(i)
    torch.cuda.synchronize()
    graphs = []
    for i in range(n_variants):
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            step_fn(i)
        graphs.append(g)
    return lambda i: graphs[i % n_variants].replay()
