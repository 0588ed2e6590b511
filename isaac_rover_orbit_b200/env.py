"""``RoverEnv``: the reference's environment entry point over the fused CUDA kernels.

Mirrors ``rover_envs/envs/navigation/entrypoints/rover_env.py`` (``RoverEnv(RLTaskEnv)``: ``step`` :42-102,
``_reset_idx`` :27-39) and the slice of ORBIT's ``RLTaskEnv`` / manager objects that the reference's term functions
read (SURVEY.md 8b "What env must expose to terms"):

    env.num_envs, env.device, env.max_episode_length, env.episode_length_buf (int64),
    env.command_manager.get_command(name), env.action_manager.action / prev_action,
    env.scene.sensors[name].data.{pos_w, ray_hits_w, force_matrix_w},
    env.scene[asset].data.{root_pos_w, root_quat_w, heading_w, default_root_state}, env.scene.terrain

The step keeps the reference's order (process actions -> physics x decimation -> counters -> terminations ->
rewards -> reset -> command update -> observations) but runs it as three launches -- ``rover_mdp_pre_step``
(ACTIONS | TERMS), ``rover_mdp_post_step_v3`` (variates drawn in the kernel, episode log written by the kernel) and
``rover_height_scan`` -- or four when the physics callable must see this step's joint targets (ACTIONS and TERMS then
sit on either side of it).  Nothing else is launched per step.
PhysX is out of scope: ``physics`` is any callable ``(env) -> None`` that updates ``robot.data.root_pos_w /
root_quat_w`` and ``contact_sensor.data.force_matrix_w`` in place (default: synthetic state, see synthetic.py).
"""
from __future__ import annotations

import types

import torch

from . import _lib, ops
from .config import REWARD_TERMS, TERMINATION_TERMS, RoverEnvCfg
from .terrain import TerrainTables


class _Data(types.SimpleNamespace):
    pass


class RobotArticulation:
    """The slice of ORBIT ``Articulation`` the terms touch (``scene["robot"]``)."""

    def __init__(self, n, device):
        self.data = _Data(
            root_pos_w=torch.zeros(n, 3, device=device), root_quat_w=torch.zeros(n, 4, device=device),
            default_root_state=torch.zeros(n, 13, device=device))
        self.data.root_quat_w[:, 0] = 1.0
        self.joint_pos_target = None
        self.joint_vel_target = None
        self._drive_ids, self._steer_ids = list(range(6)), list(range(6, 10))

    def find_joints(self, names):
        if any("Drive" in n for n in names):
            return self._drive_ids, [f"{p}_Drive_Continuous" for p in ("ML", "FL", "RL", "RR", "MR", "FR")]
        return self._steer_ids, [f"{p}_Steer_Revolute" for p in ("FL", "RL", "RR", "FR")]

    def set_joint_velocity_target(self, target, joint_ids=None):
        self.joint_vel_target = target

    def set_joint_position_target(self, target, joint_ids=None):
        self.joint_pos_target = target

    def write_root_pose_to_sim(self, pose, env_ids=None):
        self.data.root_pos_w[env_ids] = pose[:, :3]
        self.data.root_quat_w[env_ids] = pose[:, 3:]


class RayCaster:
    """ORBIT ``RayCaster`` facade: ``data.pos_w`` is the body pose, ``data.ray_hits_w`` is produced on demand by the
    CUDA raycaster (the fused path never materialises it: 12 B/ray of traffic the reference pays, SURVEY.md a-7/a-8)."""

    def __init__(self, env, cfg):
        self.cfg = cfg
        self._env = env
        self.ray_pattern = ops.RayPattern.grid(env.device, cfg.pattern_cfg.resolution, cfg.pattern_cfg.size, cfg.offset_pos,
                                               direction=cfg.pattern_cfg.direction, offset_rot=cfg.offset_rot)
        self.ray_starts = self.ray_pattern.starts
        outer = self

        class _SensorData:
            @property
            def pos_w(self):
                return outer._env.scene["robot"].data.root_pos_w

            @property
            def quat_w(self):
                return outer._env.scene["robot"].data.root_quat_w

            @property
            def ray_hits_w(self):
                robot = outer._env.scene["robot"].data
                _, hits = ops.height_scan(robot.root_pos_w, robot.root_quat_w, outer.ray_pattern, outer._env.scan_grid,
                                          outer.cfg.max_distance, outer._env.cfg.height_scan_base_offset,
                                          return_hits=True, attach_yaw_only=outer.cfg.attach_yaw_only)
                return hits

        self.data = _SensorData()


class ContactSensor:
    def __init__(self, n, num_bodies, device):
        self.data = _Data(force_matrix_w=torch.zeros(n, num_bodies, 1, 3, device=device))


class RoverTerrainImporter:
    """``RoverTerrainImporter`` (utils/terrains/terrain_importer.py:127-184) over the device tables."""

    def __init__(self, env, tables: TerrainTables):
        self._env = env
        self.tables = tables
        self.handle = ops.TerrainTablesHandle(tables.heightmap, tables.safe_mask, tables.offset_xy, tables.spawn_table,
                                              tables.resolution, env.device)
        self.target_distance = env.cfg.commands.target_distance

    @property
    def env_origins(self):
        return self._env._buf.env_origins

    def get_spawn_locations(self):
        """terrain_importer.py:177-184."""
        return self.handle.spawn_table

    def sample_new_targets(self, env_ids):
        """terrain_importer.py:134-157: rejection-sampled targets 9 m around the env origins -> ``[K,3]``."""
        cmd = self._env.command_manager.get_term("target_pose")
        saved = cmd.pos_command_w[env_ids].clone(), cmd.heading_command_w[env_ids].clone(), \
            cmd.time_left[env_ids].clone(), cmd.command_counter[env_ids].clone()
        self._env._run_post(env_ids, _lib.PHASE_RESAMPLE)
        out = cmd.pos_command_w[env_ids].clone()
        cmd.pos_command_w[env_ids], cmd.heading_command_w[env_ids] = saved[0], saved[1]
        cmd.time_left[env_ids], cmd.command_counter[env_ids] = saved[2], saved[3]
        return out


class Scene:
    def __init__(self, assets: dict, sensors: dict, terrain):
        self._assets = assets
        self.sensors = sensors
        self.terrain = terrain

    def __getitem__(self, name):
        return self._assets[name]


class ActionManager:
    """ORBIT ``ActionManager`` with one term (A.2): ``process_action`` shifts prev <- action <- new."""

    def __init__(self, env, term):
        self._env = env
        self._term = term

    @property
    def action(self):
        return self._env._buf.action

    @property
    def prev_action(self):
        return self._env._buf.prev_action

    def get_term(self, name="actions"):
        return self._term

    def process_action(self, action):
        self._term.process_actions(action)

    def apply_action(self):
        self._term.apply_actions()


class CommandManager:
    def __init__(self, env, terms: dict):
        self._env = env
        self._terms = terms

    def get_command(self, name):
        return self._terms[name].command

    def get_term(self, name):
        return self._terms[name]

    def compute(self, dt):
        for t in self._terms.values():
            t.compute(dt)


class RoverEnv:
    """Drop-in for ``RoverEnv.step`` on synthetic physics (see the module docstring).

    ``physics``: callable ``(env) -> None``, the stand-in for the PhysX stepping of rover_env.py:64-75.
    ``physics_needs_targets`` (default True): the callable reads the joint targets of this step, so the action term must
    have run before it -- ``step`` is then pre_step(ACTIONS), physics, pre_step(TERMS), post_step, scan (4 launches).
    With ``False`` (a replayed / synthetic state source) or without physics everything but the scan runs as ONE launch
    after the state update (``rover_mdp_step_v3``): 2 launches per step.
    Random variates of the reset path come from the in-kernel counter-based generator keyed on ``seed`` (no torch
    generator call per step); ``set_variates`` feeds explicit arrays instead (parity tests).
    ``enable_cuda_graph()`` captures the whole step once; ``step`` then costs one action copy + one graph launch.
    ``observation_dtype=torch.bfloat16``: the height scan also writes a bf16 mirror of the observation (same launch,
    ``ops.height_scan_obs``), and ``reset`` / ``step`` return that mirror (``policy.alloc_obs_bf16`` layout) -- the operand
    the policy and value networks read in place at half the bytes.  ``obs_buf`` stays fp32 and is written as before.
    """

    def __init__(self, cfg: RoverEnvCfg, terrain: TerrainTables, device="cuda:0", physics=None, seed: int = 0,
                 physics_needs_targets: bool = True, scan_grid: "ops.ScanGridHandle | None" = None,
                 observation_dtype: torch.dtype = torch.float32):
        from .mdp.actions import AckermannAction2
        from .mdp.commands import TerrainBasedPositionCommand
        from .policy import alloc_obs, alloc_obs_bf16

        if observation_dtype not in (torch.float32, torch.bfloat16):
            raise ValueError(f"observation_dtype must be torch.float32 or torch.bfloat16, not {observation_dtype}")

        self.cfg = cfg
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise RuntimeError("RoverEnv needs a CUDA device; there is no CPU fallback")
        self.num_envs = n = cfg.num_envs
        self.step_dt = cfg.step_dt
        self.max_episode_length = cfg.max_episode_length
        self.max_episode_length_s = cfg.episode_length_s
        self.common_step_counter = 0
        self._buf = ops.MdpBuffers.allocate(n, self.device)
        self._params = ops.mdp_params(cfg)
        self.episode_length_buf = self._buf.episode_length_buf
        # the raycaster's acceleration structure (built from the mesh unless the caller shares one already on the device)
        self.scan_grid = scan_grid if scan_grid is not None else ops.ScanGridHandle.from_mesh(
            terrain.vertices, terrain.faces, self.device)
        robot = RobotArticulation(n, self.device)
        self.scene = Scene({"robot": robot}, {}, None)
        self.scene.terrain = RoverTerrainImporter(self, terrain)
        if self.scene.terrain.handle.n_spawns < n:
            # randomizations.py:22 draws randperm(len(spawn_locations))[:K] with K up to num_envs
            raise ValueError(f"spawn table has {self.scene.terrain.handle.n_spawns} rows for {n} envs: build the terrain "
                             f"tables for at least num_envs environments")
        self.scene.sensors["height_scanner"] = RayCaster(self, cfg.height_scanner)
        self.scene.sensors["contact_sensor"] = ContactSensor(n, cfg.num_contact_bodies, self.device)
        self.action_manager = ActionManager(self, AckermannAction2(cfg.actions, self))
        self.command_manager = CommandManager(self, {"target_pose": TerrainBasedPositionCommand(cfg.commands, self)})
        # rows padded to 16 bytes: the policy kernel's TMA tensor map reads the buffer in place (no re-homing copy)
        self.obs_buf = alloc_obs(n, self.device, 4 + self.scene.sensors["height_scanner"].ray_pattern.n_rays)
        self.observation_dtype = observation_dtype
        # bf16: the mirror of obs_buf that the scan writes beside it (rows padded to 16 bytes, as the policy reads it)
        self.obs_buf_bf16 = alloc_obs_bf16(n, self.device, self.obs_buf.shape[1]) if observation_dtype == torch.bfloat16 else None
        self._obs_out = self.obs_buf if self.obs_buf_bf16 is None else self.obs_buf_bf16
        self.reward_buf = self._buf.reward
        self.reset_buf = self._buf.reset_flags
        # the kernels write 0 / 1 bytes: the bool tensors the reference returns are views, not per-step conversions
        self.reset_terminated = self._buf.terminated.view(torch.bool)
        self.reset_time_outs = self._buf.truncated.view(torch.bool)
        # extras["log"]: 0-dim views of the vector the post-step kernel refreshes whenever an env reset (ORBIT
        # manager.reset() semantics, A.2; the values of the last reset persist in between, as in the reference)
        lg = self._buf.log
        self._log = {f"Episode Reward/{name}": lg[i] for i, name in enumerate(REWARD_TERMS)}
        self._log.update({f"Episode Termination/{name}": lg[7 + i] for i, name in enumerate(TERMINATION_TERMS)})
        self._log["Metrics/target_pose/error_pos"] = lg[11]
        self._log["Metrics/target_pose/error_heading"] = lg[12]
        self.extras = {"log": self._log, "episode": self._log}
        self._rng = ops.ResetRng(seed, self.device)
        self._physics = physics
        self._physics_needs_targets = bool(physics_needs_targets) and physics is not None
        self._variates = None
        self._terms_current = False   # term columns (rewards / terminations) belong to the current state
        self._graph = None
        # input buffer of the captured step = the action term's raw_actions (the reference's ``_raw_actions[:] = actions``
        # is then the one copy a step makes)
        self._action_in = self.action_manager.get_term().raw_actions
        # rover_env.py:18-25: env origins are shifted by +100 m in x and y
        self._buf.env_origins[:, 0] += 100.0
        self._buf.env_origins[:, 1] += 100.0
        self._buf.time_left.fill_(cfg.commands.resampling_time_range[0])

    # ---------------------------------------------------------------------------------------------- helpers
    def seed(self, seed: int = -1) -> int:
        """``RLTaskEnv.seed``: re-key the variate generator (step counter back to 0)."""
        self._rng.state.copy_(torch.tensor([int(seed), 0], dtype=torch.int64))
        return seed

    def set_variates(self, spawn_perm, yaw_u, heading_u, theta_u):
        """Parity hook: feed the random variates of the next post-step explicitly (oracle and kernel share them)."""
        if self._graph is not None:
            raise RuntimeError("set_variates: the captured step draws its variates in the kernel")
        self._variates = (spawn_perm, yaw_u, heading_u, theta_u)

    def _post(self, phases, obs):
        robot = self.scene["robot"].data
        v, self._variates = self._variates, None
        if v is not None:
            ops.mdp_post_step(self._buf, self._params, self.scene.terrain.handle, robot.root_pos_w, robot.root_quat_w, *v,
                              obs=obs, phases=phases)
        else:
            ops.mdp_post_step(self._buf, self._params, self.scene.terrain.handle, robot.root_pos_w, robot.root_quat_w,
                              obs=obs, phases=phases, rng=self._rng, n_rounds=self.cfg.target_rounds)

    def _run_post(self, env_ids, phases, obs=None):
        """Single-purpose use of the post-step kernel for the envs in ``env_ids`` (the reference's per-term calls)."""
        b = self._buf
        b.reset_flags.zero_()
        b.reset_flags[env_ids] = 1
        blocks = b.block_reset_counts.numel()
        padded = torch.zeros(blocks * _lib.MDP_BLOCK, dtype=torch.int32, device=self.device)
        padded[: self.num_envs] = b.reset_flags
        b.block_reset_counts.copy_(padded.view(blocks, _lib.MDP_BLOCK).sum(dim=1))
        self._post(phases, obs)

    # ---------------------------------------------------------------------------------------------- API
    def reset(self):
        """Reset every env (spawn, targets), then compute the first observation."""
        ids = torch.arange(self.num_envs, device=self.device)
        self._reset_idx(ids)
        self._run_post(ids[:0], _lib.PHASE_METRICS | _lib.PHASE_COMMAND | _lib.PHASE_OBS, obs=self.obs_buf)
        self._scan()
        # a private copy: ``step`` refreshes ``obs_buf`` in place, and the reference's trainer keeps the tensor it got
        # from ``reset`` as its ``states`` buffer (``states.copy_(next_states)``, skrl_utils.py:148).  The bf16 copy keeps
        # the padded rows of alloc_obs_bf16 (a .clone() of the view comes back dense, a layout the bf16 kernels reject).
        if self.obs_buf_bf16 is None:
            return self.obs_buf.clone(), self.extras
        from .policy import alloc_obs_bf16

        states = alloc_obs_bf16(self.num_envs, self.device, self.obs_buf_bf16.shape[1])
        states.copy_(self.obs_buf_bf16)
        return states, self.extras

    def _reset_idx(self, idx):
        """rover_env.py:27-39 / ORBIT ``RLTaskEnv._reset_idx`` (A.2) for explicit ids."""
        self._run_post(idx, _lib.PHASE_SPAWN | _lib.PHASE_MANAGERS | _lib.PHASE_RESAMPLE)

    def _scan(self):
        robot = self.scene["robot"].data
        sensor = self.scene.sensors["height_scanner"]
        if self.obs_buf_bf16 is not None:
            # one launch: the fp32 heights (the term functions read obs_buf) and the bf16 mirror of columns 0..4+R-1
            general = not sensor.cfg.attach_yaw_only or not sensor.ray_pattern.vertical_down
            ops.height_scan_obs(robot.root_pos_w, robot.root_quat_w, sensor.ray_pattern, self.scan_grid, obs=self.obs_buf,
                                obs_bf16=self.obs_buf_bf16, head_cols=4, max_distance=sensor.cfg.max_distance,
                                base_offset=self.cfg.height_scan_base_offset, variant=ops.RAY_CAST_VARIANT if general else None,
                                attach_yaw_only=sensor.cfg.attach_yaw_only)
            return
        ops.height_scan(robot.root_pos_w, robot.root_quat_w, sensor.ray_pattern, self.scan_grid,
                        sensor.cfg.max_distance, self.cfg.height_scan_base_offset, out=self.obs_buf[:, 4:],
                        attach_yaw_only=sensor.cfg.attach_yaw_only)

    def episode_log(self) -> dict:
        """Host-side copy of the last episode log (synchronises): the values of ``extras["log"]`` + ``num_resets``."""
        s = self._buf.log.detach().double().cpu()
        log = {k: float(v) for k, v in zip(self._log, s[:13])}
        for name in TERMINATION_TERMS:
            log[f"Episode Termination/{name}"] = int(round(log[f"Episode Termination/{name}"]))
        log["num_resets"] = int(round(float(s[13])))
        return log

    def render(self, *args, **kwargs):
        """No viewport without Isaac Sim; the reference's eval loop calls it unless ``headless`` (skrl_utils.py:150-206)."""
        return None

    def close(self):
        self._graph = None

    def _step_body(self, action):
        b, robot = self._buf, self.scene["robot"].data
        contact = self.scene.sensors["contact_sensor"].data
        if self._physics_needs_targets:
            # -- process actions; physics stepping (decimation x: identical joint targets, ackermann_actions.py:231-236)
            self.action_manager.process_action(action)
            self.action_manager.apply_action()
            self._physics(self)
            # -- counters, terminations, rewards (one launch; reads the PREVIOUS command like the reference)
            ops.mdp_pre_step(b, self._params, None, contact.force_matrix_w, phases=_lib.PRE_TERMS)
        else:
            # the state source does not read the joint targets: nothing has to run between the action term and the rest
            if self._physics is not None:
                self._physics(self)
            term = self.action_manager.get_term()
            if self._variates is None:
                # ONE launch: action term + counters + terminations + rewards + reset + command update + observation
                # head + episode log.  The in-kernel spawn draw needs no reset rank, so nothing crosses blocks in front
                # of the reset chain (rover_mdp_step_v3).
                term.stage_actions(action)
                ops.mdp_step(b, term._params, self.scene.terrain.handle, term.raw_actions, contact.force_matrix_w,
                             robot.root_pos_w, robot.root_quat_w, obs=self.obs_buf, rng=self._rng,
                             n_rounds=self.cfg.target_rounds)
                self.action_manager.apply_action()
                self._scan()
                return
            term.process_actions(action, fused_terms_force=contact.force_matrix_w)  # explicit variates: rank by pre-step
            self.action_manager.apply_action()
        # -- reset, command update, observation head, episode log (one launch; variates drawn in the kernel)
        self._post(_lib.PHASE_ALL, self.obs_buf)
        # -- height scan straight into the observation buffer (one launch)
        self._scan()

    def enable_cuda_graph(self, warmup: int = 2):
        """Capture the step (all launches + a graph-safe ``physics``) into one CUDA graph.  The warm-up steps are real
        steps (they advance the env); afterwards ``step(action)`` = copy of the action into the captured input + one
        ``cudaGraphLaunch``."""
        if self._variates is not None:
            raise RuntimeError("enable_cuda_graph: explicit variates are pending (set_variates)")
        side = torch.cuda.Stream(self.device)
        side.wait_stream(torch.cuda.current_stream(self.device))
        with torch.cuda.stream(side):
            for _ in range(max(warmup, 1)):
                self._step_body(self._action_in)
                self.common_step_counter += 1
        torch.cuda.current_stream(self.device).wait_stream(side)
        torch.cuda.synchronize(self.device)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            self._step_body(self._action_in)
        self._graph = g  # (capturing does not execute: the first replay is the next step)
        return self

    @property
    def action_input(self) -> torch.Tensor:
        """The buffer the step reads its actions from (the action term's ``raw_actions``, ``[N, 2]`` fp32).  A producer that
        writes its actions straight into it (``policy.act(..., out_actions=env.action_input)``) and then calls
        ``env.step(env.action_input)`` saves the copy of the action tensor, also under ``enable_cuda_graph()``."""
        return self._action_in

    def step(self, action: torch.Tensor):
        """rover_env.py:42-102."""
        if self._graph is not None:
            if action.data_ptr() != self._action_in.data_ptr():
                self._action_in.copy_(action)
            self._graph.replay()
        else:
            self._step_body(action)
        self.common_step_counter += 1
        self._terms_current = True
        return self._obs_out, self.reward_buf, self.reset_terminated, self.reset_time_outs, self.extras
