"""Constants and declarative configuration of AAURoverEnv-v0, mirroring the reference's config classes.

Names follow the reference (paths relative to its root):
``AckermannActionCfg`` rover_envs/mdp/actions/actions_cfg.py:9-51,
``AAURoverEnvCfg`` values rover_envs/envs/navigation/robots/aau_rover/env_cfg.py:21-31,
``RoverEnvCfg`` wiring rover_envs/envs/navigation/rover_env_cfg.py:78-278.
"""
from __future__ import annotations

import math
from dataclasses import dataclass, field

REWARD_TERMS = ("distance_to_target", "reached_target", "oscillation", "angle_to_target", "heading_soft_contraint",
                "collision", "far_from_target")
TERMINATION_TERMS = ("time_limit", "is_success", "far_from_target", "collision")


@dataclass
class AckermannActionCfg:
    """rover_envs/mdp/actions/actions_cfg.py:9-51 (``class_type`` = AckermannAction2, :17)."""

    asset_name: str = "robot"
    scale: tuple = (1.0, 1.0)
    offset: float | tuple = 0.0
    wheelbase_length: float = 0.849
    middle_wheel_distance: float = 0.894
    rear_and_front_wheel_distance: float = 0.77
    wheel_radius: float = 0.1
    min_steering_radius: float = 0.8
    steering_joint_names: list = field(default_factory=lambda: [".*Steer_Revolute"])
    drive_joint_names: list = field(default_factory=lambda: [".*Drive_Continuous"])
    steering_order: list = field(default_factory=lambda: ["FL", "FR", "RL", "RR"])
    drive_order: list = field(default_factory=lambda: ["FL", "FR", "CL", "CR", "RL", "RR"])
    variant: int = 2  # which reference class backs ``class_type``: 1 AckermannAction, 2 AckermannAction2, 3 AckermannAction3

    def offsets(self) -> tuple:
        return tuple(self.offset) if isinstance(self.offset, (tuple, list)) else (self.offset, self.offset)


def aau_rover_action_cfg() -> AckermannActionCfg:
    """robots/aau_rover/env_cfg.py:21-31."""
    return AckermannActionCfg(offset=-0.0135)


def exomy_action_cfg() -> AckermannActionCfg:
    """robots/exomy/env_cfg.py:21-30 (Exomy-v0; same kernels, other constants)."""
    return AckermannActionCfg(wheelbase_length=0.29778, middle_wheel_distance=0.1548,
                              rear_and_front_wheel_distance=0.1548, wheel_radius=0.1, min_steering_radius=0.4,
                              steering_joint_names=["FL_Steer_Joint", "RL_Steer_Joint", "RR_Steer_Joint",
                                                    "FR_Steer_Joint"],
                              drive_joint_names=[".*Drive_Joint"])


@dataclass
class GridPatternCfg:
    """ORBIT ``patterns.GridPatternCfg`` as wired at rover_env_cfg.py:82."""

    resolution: float = 0.1
    size: tuple = (3.0, 3.0)
    direction: tuple = (0.0, 0.0, -1.0)


@dataclass
class RayCasterCfg:
    """ORBIT ``RayCasterCfg`` as wired at rover_env_cfg.py:78-86."""

    offset_pos: tuple = (0.0, 0.0, 10.0)
    # RayCasterCfg.offset.rot (w, x, y, z): rotates the pattern's directions, not its starts (RayPattern.grid)
    offset_rot: tuple = (1.0, 0.0, 0.0, 0.0)
    attach_yaw_only: bool = True
    pattern_cfg: GridPatternCfg = field(default_factory=GridPatternCfg)
    max_distance: float = 100.0


@dataclass
class RewardsCfg:
    """rover_env_cfg.py:127-163 -- weights in declaration order of REWARD_TERMS."""

    weights: tuple = (5.0, 5.0, -0.1, -1.5, -0.5, -2.0, -2.0)
    reached_threshold: float = 0.18
    far_threshold: float = 11.0


@dataclass
class CommandsCfg:
    """rover_env_cfg.py:188-200 + terrain_importer.py:132."""

    resampling_time_range: tuple = (150.0, 150.0)
    heading_range: tuple = (-math.pi, math.pi)
    simple_heading: bool = False
    target_distance: float = 9.0


@dataclass
class RoverEnvCfg:
    """rover_env_cfg.py:228-278."""

    num_envs: int = 256
    sim_dt: float = 1.0 / 30.0
    decimation: int = 6
    episode_length_s: float = 150.0
    actions: AckermannActionCfg = field(default_factory=aau_rover_action_cfg)
    height_scanner: RayCasterCfg = field(default_factory=RayCasterCfg)
    rewards: RewardsCfg = field(default_factory=RewardsCfg)
    commands: CommandsCfg = field(default_factory=CommandsCfg)
    obs_distance_scale: float = 0.11  # rover_env_cfg.py:104-105
    obs_heading_scale: float = 1.0 / math.pi  # :106-112
    height_scan_base_offset: float = 0.26878  # mdp/observations.py:45
    spawn_z_offset: float = 0.5  # mdp/randomizations.py:12
    num_contact_bodies: int = 14  # contact_sensor regex .*_(Drive|Steer|Boogie|Body), rover_env_cfg.py:73
    target_rounds: int = 16  # bound of the rejection loop (terrain_importer.py:143-151 is unbounded)

    @property
    def step_dt(self) -> float:
        return self.sim_dt * self.decimation

    @property
    def max_episode_length(self) -> int:
        return math.ceil(self.episode_length_s / self.step_dt)
