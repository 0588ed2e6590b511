"""``GaussianNeuralNetwork`` -- the skrl Gaussian policy of the reference over the tcgen05 kernel.

Mirrors rover_envs/envs/navigation/learning/skrl/models.py:39-102 (+ ``HeightmapEncoder`` :24-36): same constructor
arguments, same ``state_dict`` keys as ``best_agent.pt`` (``dense_encoder.encoder_layers.{0,2}``, ``mlp.{0,2,4,6}``,
``log_std_parameter``), ``compute(inputs, role) -> (mean [N,2], log_std [2], {})``, and ``act`` with skrl 1.1.0
``GaussianMixin`` semantics (clamp log_std to [-20, 2], reparameterised sample, clip to the action box, summed
log-prob).  The forward pass is inference-only (no autograd): bf16 operands, fp32 accumulation on the tensor cores.
"""
from __future__ import annotations

import torch

from . import _lib, torch_ops

WEIGHT_KEYS = ("dense_encoder.encoder_layers.0", "dense_encoder.encoder_layers.2", "mlp.0", "mlp.2", "mlp.4", "mlp.6")
OBS_COLS = 965


def alloc_obs(num_envs: int, device, cols: int = OBS_COLS) -> torch.Tensor:
    """Observation buffer ``[N, cols]`` whose rows start on 16-byte boundaries (row stride padded to a multiple of
    4 floats), as the policy kernel's TMA tensor map requires.  Returns the ``[:, :cols]`` view."""
    stride = (cols + 3) // 4 * 4
    return torch.zeros(num_envs, stride, dtype=torch.float32, device=device)[:, :cols]


def alloc_obs_bf16(num_envs: int, device, cols: int = OBS_COLS) -> torch.Tensor:
    """bf16 mirror of the observation buffer (``ops.height_scan(..., obs_bf16=...)`` fills it): rows padded to a
    multiple of 8 elements so that they start on 16-byte boundaries.  Returns the ``[:, :cols]`` view."""
    stride = (cols + 7) // 8 * 8
    return torch.zeros(num_envs, stride, dtype=torch.bfloat16, device=device)[:, :cols]


class _RoverNetwork:
    """Encoder + MLP of both reference networks (models.py:24-36, 39-162) over the packed tcgen05 weights."""

    _OUT_DIM = 2
    _HAS_LOG_STD = True

    def __init__(self, observation_space=None, action_space=None, device="cuda:0", mlp_input_size=4,
                 mlp_layers=(256, 160, 128), mlp_activation="leaky_relu", encoder_input_size=961,
                 encoder_layers=(80, 60), encoder_activation="leaky_relu", **kwargs):
        if mlp_activation != "leaky_relu" or encoder_activation != "leaky_relu":
            raise ValueError(f"Activation function {mlp_activation}/{encoder_activation} not supported.")
        if (mlp_input_size, tuple(mlp_layers), encoder_input_size, tuple(encoder_layers)) != (4, (256, 160, 128), 961, (80, 60)):
            raise ValueError("the tcgen05 policy kernel is built for the AAURoverEnv-v0 policy shape "
                             "(961->80->60 (+4) ->256->160->128->2, configure_models.py:41-53)")
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise RuntimeError("GaussianNeuralNetwork needs a CUDA device; there is no CPU fallback")
        self.mlp_input_size, self.encoder_input_size = mlp_input_size, encoder_input_size
        dims = [(80, 961), (60, 80), (256, 64), (160, 256), (128, 160), (self._OUT_DIM, 128)]
        self._params = {}
        for key, (o, i) in zip(WEIGHT_KEYS, dims):
            self._params[key + ".weight"] = torch.zeros(o, i, device=self.device)
            self._params[key + ".bias"] = torch.zeros(o, device=self.device)
        self.log_std_parameter = torch.zeros(2, device=self.device)
        self._clip_log_std, self._log_std_min, self._log_std_max = True, -20.0, 2.0  # models.py:65-67
        n_bytes = torch_ops.policy_packed_bytes()
        self._packed = torch.zeros(n_bytes + 128, dtype=torch.uint8, device=self.device)
        off = (-self._packed.data_ptr()) % 128
        self._packed = self._packed[off: off + n_bytes]
        self._dirty = True

    # ---- state dict with the reference's keys
    def state_dict(self) -> dict:
        sd = {"log_std_parameter": self.log_std_parameter} if self._HAS_LOG_STD else {}
        sd.update(self._params)
        return sd

    def load_state_dict(self, sd: dict, strict: bool = True):
        want = set(self._params) | ({"log_std_parameter"} if self._HAS_LOG_STD else set())
        if strict and set(sd) != want:
            raise KeyError(f"unexpected / missing keys: {sorted(set(sd) ^ want)}")
        for k in want & set(sd):
            dst = self.log_std_parameter if k == "log_std_parameter" else self._params[k]
            src = torch.as_tensor(sd[k]).to(self.device, torch.float32)
            if src.shape != dst.shape:
                raise RuntimeError(f"size mismatch for {k}: {tuple(src.shape)} vs {tuple(dst.shape)}")
            dst.copy_(src)
        self._dirty = True
        self._fused_dirty = True

    def _pack(self):
        torch.ops.rover_b200.policy_pack([self._params[k + ".weight"] for k in WEIGHT_KEYS],
                                         [self._params[k + ".bias"] for k in WEIGHT_KEYS], self._packed)
        # the forward kernels start under programmatic dependent launch and read the blob BEFORE they wait for the kernel
        # in front of them (csrc/common.cuh): launch-invariant data must be complete before that kernel is launched
        torch.cuda.current_stream(self.device).synchronize()
        self._dirty = False

    def packed(self) -> torch.Tensor:
        """The packed weight blob of ``rover_policy_pack`` (re-packed after ``load_state_dict``)."""
        if self._dirty:
            self._pack()
        return self._packed

    def packed_fused(self) -> torch.Tensor:
        """The encoder weights as the fused scan + encoder kernel reads them (``rover_policy_pack_fused``: W0 as the
        tensor-memory image of a transposed MMA's A operand, W1 as a shared-memory A operand); packed on first use and
        after ``load_state_dict``."""
        if self.__dict__.get("_packed_fused") is None or self.__dict__.get("_fused_dirty", True):
            n_bytes = torch_ops.policy_packed_fused_bytes()
            buf = self.__dict__.get("_packed_fused")
            if buf is None:
                raw = torch.zeros(n_bytes + 128, dtype=torch.uint8, device=self.device)
                off = (-raw.data_ptr()) % 128
                buf = self._packed_fused = raw[off: off + n_bytes]
            torch.ops.rover_b200.policy_pack_fused([self._params[k + ".weight"] for k in WEIGHT_KEYS],
                                                   [self._params[k + ".bias"] for k in WEIGHT_KEYS], buf)
            torch.cuda.current_stream(self.device).synchronize()  # (see _pack)
            self._fused_dirty = False
        return self._packed_fused

    def _forward(self, states: torch.Tensor, value_head: bool) -> torch.Tensor:
        if not states.is_cuda or states.dtype != torch.float32 or states.dim() != 2 or states.shape[1] != OBS_COLS:
            raise RuntimeError("compute: states must be a CUDA fp32 [N,965] tensor")
        if states.stride(1) != 1 or states.stride(0) % 4 != 0 or states.data_ptr() % 16 != 0:
            # the reference accepts any tensor; re-home it once into an aligned buffer (one copy kernel)
            buf = alloc_obs(states.shape[0], states.device)
            buf.copy_(states)
            states = buf
        if self._dirty:
            self._pack()
        return torch.ops.rover_b200.policy_forward(states, self._packed, value_head)

    def _forward_bf16(self, states: torch.Tensor, value_head: bool) -> torch.Tensor:
        """bf16 observations ``[N, 965]`` (``alloc_obs_bf16`` layout): the TMA tile is the MMA operand, no conversion."""
        _check_bf16_states(states, "compute_bf16")
        if self._dirty:
            self._pack()
        return torch.ops.rover_b200.policy_forward(states, self._packed, value_head)


class GaussianNeuralNetwork(_RoverNetwork):
    """models.py:39-102."""

    # ---- skrl Model API
    def compute(self, inputs: dict, role: str = "actor"):
        """models.py:89-102: ``(mean [N,2], log_std_parameter [2], {})`` for ``inputs["states"] [N,965]``.
        A bf16 observation (``alloc_obs_bf16`` layout) is routed to ``compute_bf16``."""
        if inputs["states"].dtype == torch.bfloat16:
            return self.compute_bf16(inputs, role)
        return self._forward(inputs["states"], False), self.log_std_parameter, {}

    def compute_bf16(self, inputs: dict, role: str = "actor"):
        """``compute`` on the bf16 observation mirror; identical means (the fp32 path rounds to the same bf16)."""
        return self._forward_bf16(inputs["states"], False), self.log_std_parameter, {}

    def act(self, inputs: dict, role: str = "actor", eps: torch.Tensor | None = None,
            out_actions: torch.Tensor | None = None, rng=None):
        """skrl 1.1.0 ``GaussianMixin.act`` (SURVEY.md A.4): returns ``(actions [N,2], log_prob [N,1], outputs)``.
        ``eps`` (standard-normal draws) may be supplied for reproducible parity checks; ``out_actions`` (fp32 ``[N,2]``,
        e.g. the env's action input buffer) receives the actions in place of a new tensor (no copy on the way to the env).
        ``rng`` (an ``ops.ActionRng``) and no ``eps``: the forward pass samples in its last epilogue -- ONE launch, noise
        keyed on (seed, step, env) instead of ``torch.randn`` (``rover_policy_act``); fp32 or bf16 states."""
        if rng is not None and eps is None:
            return self._act_sampled(inputs["states"], out_actions, rng)
        mean, log_std, outputs = self.compute(inputs, role)
        n = mean.shape[0]
        if eps is None:
            eps = torch.randn(n, 2, device=mean.device)
        if out_actions is not None:
            log_prob = torch.empty(n, dtype=torch.float32, device=mean.device)
            torch.ops.rover_b200.gaussian_act_out(mean, log_std, eps.contiguous(), out_actions, log_prob)
            actions = out_actions
        else:
            actions, log_prob = torch.ops.rover_b200.gaussian_act(mean, log_std, eps.contiguous())
        outputs["mean_actions"] = mean
        return actions, log_prob.unsqueeze(-1), outputs

    def _act_sampled(self, states: torch.Tensor, out_actions: torch.Tensor | None, rng):
        if states.dtype != torch.bfloat16:
            states = _aligned_states(states, "act")
        if self._dirty:
            self._pack()
        n = states.shape[0]
        mean = torch.empty(n, 2, dtype=torch.float32, device=states.device)
        actions = out_actions if out_actions is not None else torch.empty_like(mean)
        log_prob = torch.empty(n, 1, dtype=torch.float32, device=states.device)
        torch.ops.rover_b200.policy_act(states, self._packed, self.log_std_parameter, rng.state, 0, mean, actions, log_prob)
        return actions, log_prob, {"mean_actions": mean}


def _check_bf16_states(states: torch.Tensor, what: str) -> None:
    """bf16 states must already be in the ``alloc_obs_bf16`` layout (a copy into it would cost what the mirror saves)."""
    if (not states.is_cuda or states.dtype != torch.bfloat16 or states.dim() != 2 or states.shape[1] != OBS_COLS
            or states.stride(1) != 1 or states.stride(0) % 8 != 0 or states.data_ptr() % 16 != 0):
        raise RuntimeError(f"{what}: states must be a CUDA bf16 [N,965] view from alloc_obs_bf16()")


def _aligned_states(states: torch.Tensor, what: str) -> torch.Tensor:
    """fp32 ``[N,965]`` CUDA states with 16-byte aligned rows: the tensor itself, or one copy into ``alloc_obs``."""
    if not states.is_cuda or states.dtype != torch.float32 or states.dim() != 2 or states.shape[1] != OBS_COLS:
        raise RuntimeError(f"{what}: states must be a CUDA fp32 [N,965] tensor")
    if states.stride(1) != 1 or states.stride(0) % 4 != 0 or states.data_ptr() % 16 != 0:
        buf = alloc_obs(states.shape[0], states.device)
        buf.copy_(states)
        states = buf
    return states


def policy_value_act(policy: "GaussianNeuralNetwork", value: "DeterministicNeuralNetwork", states: torch.Tensor, rng,
                     out_actions: torch.Tensor | None = None):
    """``policy.act`` (sampled with ``rng``, an ``ops.ActionRng``) and the value network on ``states [N,965]`` in ONE
    launch (``rover_policy_value_act``): ``(actions [N,2], log_prob [N,1], value [N,1], mean [N,2])``, each bit-identical
    to ``policy_value_forward`` followed by ``gaussian_act`` with ``rng.noise(N)``.  bf16 states (``alloc_obs_bf16``
    layout) take ``rover_policy_value_act_bf16``."""
    bf16 = states.dtype == torch.bfloat16
    if bf16:
        _check_bf16_states(states, "policy_value_act")
    else:
        states = _aligned_states(states, "policy_value_act")
    for net in (policy, value):
        if net._dirty:
            net._pack()
    n = states.shape[0]
    mean = torch.empty(n, 2, dtype=torch.float32, device=states.device)
    val = torch.empty(n, 1, dtype=torch.float32, device=states.device)
    actions = out_actions if out_actions is not None else torch.empty_like(mean)
    log_prob = torch.empty(n, 1, dtype=torch.float32, device=states.device)
    op = torch.ops.rover_b200.policy_value_act_bf16 if bf16 else torch.ops.rover_b200.policy_value_act
    op(states, policy._packed, value._packed, policy.log_std_parameter, rng.state, 0, mean, val, actions, log_prob)
    return actions, log_prob, val, mean


def policy_value_forward(policy: "GaussianNeuralNetwork", value: "DeterministicNeuralNetwork", states: torch.Tensor):
    """Policy mean ``[N,2]`` and value ``[N,1]`` of ``states [N,965]`` (fp32) in ONE pass over the observation
    (``rover_policy_value_forward``): what a PPO rollout evaluates every step -- ``policy.act`` in the trainer loop
    (skrl_utils.py:139-142) and ``value.act`` in ``record_transition`` (models.py:89-102 + :151-162).  Bit-identical to
    ``policy.compute`` / ``value.compute``.  bf16 states (``alloc_obs_bf16`` layout) take
    ``rover_policy_value_forward_bf16``: one pass over the bf16 mirror, bit-identical to ``compute_bf16`` of both."""
    bf16 = states.dtype == torch.bfloat16
    if bf16:
        _check_bf16_states(states, "policy_value_forward")
    else:
        if not states.is_cuda or states.dtype != torch.float32 or states.dim() != 2 or states.shape[1] != OBS_COLS:
            raise RuntimeError("policy_value_forward: states must be a CUDA fp32 [N,965] tensor")
        if states.stride(1) != 1 or states.stride(0) % 4 != 0 or states.data_ptr() % 16 != 0:
            buf = alloc_obs(states.shape[0], states.device)
            buf.copy_(states)
            states = buf
    for net in (policy, value):
        if net._dirty:
            net._pack()
    op = torch.ops.rover_b200.policy_value_forward_bf16 if bf16 else torch.ops.rover_b200.policy_value_forward
    return op(states, policy._packed, value._packed)


class DeterministicNeuralNetwork(_RoverNetwork):
    """The value network: rover_envs/envs/navigation/learning/skrl/models.py:105-162 (same encoder + MLP with its own
    weights -- the ``value`` entry of ``best_agent.pt`` -- one linear output, no tanh), ``compute -> (value [N,1], {})``
    and skrl 1.1.0 ``DeterministicMixin.act`` (``clip_actions=False``): ``(value, None, outputs)``."""

    _OUT_DIM = 1
    _HAS_LOG_STD = False

    def compute(self, inputs: dict, role: str = "actor"):
        if inputs["states"].dtype == torch.bfloat16:
            return self.compute_bf16(inputs, role)
        return self._forward(inputs["states"], True), {}

    def compute_bf16(self, inputs: dict, role: str = "actor"):
        return self._forward_bf16(inputs["states"], True), {}

    def act(self, inputs: dict, role: str = "actor"):
        value, outputs = self.compute(inputs, role)
        return value, None, outputs
