"""Environment configuration: the reference's ``env_config`` keyword surface.

Mirrors the constructor keywords of the reference env stack (``SafeMotionsBase.__init__`` safe_motions_base.py:85-207,
``AccelerationPredictionBoundedJerkAccVelPos.__init__`` actions.py:29-44, ``RewardBase`` / ``CollisionAvoidanceReward``
rewards.py:40-54, :409-417, ``SafeObservation`` observations.py:46-49) with the same names and defaults, so a
``params.json`` of a reference checkpoint can be passed unchanged.  Unknown keys are swallowed exactly like the
reference's ``**kwargs`` (safe_motions_base.py:207; SURVEY Appendix A, Q13).  Keys that select parts of the reference
this package does not implement raise ``NotImplementedError`` as soon as their value differs from the reference
default, instead of being silently ignored (``_UNSUPPORTED_UNLESS``).
"""
import json

# name -> default, taken from the reference signatures cited above
_DEFAULTS = dict(
    experiment_name="smenv",
    # limits / timing
    pos_limit_factor=1.0, vel_limit_factor=1.0, acc_limit_factor=1.0, jerk_limit_factor=1.0, torque_limit_factor=1.0,
    acceleration_after_max_vel_limit_factor=0.01,
    trajectory_duration=8.0, trajectory_time_step=0.1,
    limit_velocity=True, limit_position=True, set_velocity_after_max_pos_to_zero=True,
    action_preprocessing_function=None, action_mapping_factor=1.0,
    # scene
    robot_scene=0, obstacle_scene=0, ball_machine_mode=False, use_controller_target_velocities=False,
    collision_check_time=None, closest_point_safety_distance=0.1, starting_point_cartesian_range_scene=0,
    target_link_name=None, target_link_offset=None, no_self_collision=False,
    # planets
    planet_mode=False, planet_one_center=None, planet_one_radius_xy=None, planet_one_euler_angles=None,
    planet_one_period=None, planet_two_center=None, planet_two_radius_xy=None, planet_two_euler_angles=None,
    planet_two_period=None, planet_two_time_shift=None, obs_planet_size_per_planet=1,
    # balls
    use_moving_objects=False, moving_object_sequence=0, moving_object_area_center=None,
    moving_object_area_width_height=None, moving_object_sphere_center=None, moving_object_sphere_radius=None,
    moving_object_sphere_height_min_max=None, moving_object_sphere_angle_min_max=None,
    moving_object_speed_meter_per_second=1.0, moving_object_aim_at_current_robot_position=False,
    moving_object_check_invalid_target_link_point_positions=False, moving_object_active_number_single=1,
    moving_object_random_initial_position=False, moving_object_high_launch_angle_probability=1.0,
    # human (robot_scene_base.py:96-99, ctlp.py:4647-4959)
    human_network_checkpoint=None, human_network_use_full_observation=False,
    human_network_use_collision_avoidance_starting_point_sampling=False,
    human_network_collision_avoidance_kinematic_state_sampling_probability=0.3,
    human_network_collision_avoidance_stay_in_state_probability=0.3,
    # termination / collision avoidance mode
    terminate_on_self_collision=False, terminate_on_collision_with_static_obstacle=False,
    terminate_on_collision_with_moving_obstacle=False,
    collision_avoidance_mode=False, collision_avoidance_kinematic_state_sampling_mode=False,
    collision_avoidance_kinematic_state_sampling_probability=1.0, collision_avoidance_stay_in_state_probability=0.3,
    # rewards
    punish_action=False, action_punishment_min_threshold=0.9, action_max_punishment=1.0,
    collision_avoidance_self_collision_max_reward=0.0, collision_avoidance_self_collision_max_reward_distance=0.05,
    collision_avoidance_static_obstacles_max_reward=0.0,
    collision_avoidance_static_obstacles_max_reward_distance=0.1,
    collision_avoidance_moving_obstacles_max_reward=0.0,
    collision_avoidance_moving_obstacles_max_reward_distance=0.30,
    collision_avoidance_low_acceleration_max_reward=1.0, collision_avoidance_low_acceleration_threshold=0.1,
    collision_avoidance_low_velocity_max_reward=1.0, collision_avoidance_low_velocity_threshold=0.1,
    collision_avoidance_episode_termination_bonus=0.0, collision_avoidance_episode_early_termination_punishment=-0.0,
    normalize_reward_to_frequency=False,
    # braking-trajectory method and target points: not part of the hot path this package implements
    check_braking_trajectory_collisions=False, check_braking_trajectory_torque_limits=False,
    risk_config_dir=None, risk_config=None, risk_threshold=None, risk_state_config=0,
    risk_state_backup_trajectory_steps=None, risk_check_initial_backup_trajectory=False,
    risk_state_initial_backup_trajectory_steps=None, risk_use_backup_agent_for_initial_backup_trajectory_only=False,
    risk_state_deterministic_backup_trajectory=False, risk_store_ground_truth=False,
    risk_ignore_estimation_probability=0.0,
    # reward terms of TargetPointReachingReward that belong to the braking-trajectory / torque machinery
    # (rewards.py:231-266, :316-375)
    punish_adaptation=False, punish_end_min_distance=False, punish_end_max_torque=False,
    punish_braking_trajectory_min_distance=False, punish_braking_trajectory_max_torque=False,
    # other keys of the reference constructor that change the behaviour of the path (safe_motions_base.py:85-207)
    obstacle_use_computed_actual_values=False, distance_calculation_check_observed_points=False,
    collision_avoidance_new_state_sample_time_range=None, always_use_collision_avoidance_starting_point_sampling=False,
    terminate_on_robot_stop=False, max_resampling_attempts=0, static_robot=False, activate_obstacle_collisions=False,
    observed_link_point_scene=0, control_time_step=None,
    # target points of the reaching task (safe_motions_base.py:131-137, rewards.py:231-266)
    use_target_points=False, target_point_cartesian_range_scene=0, target_point_relative_pos_scene=0,
    target_point_radius=0.05, target_point_sequence=0, target_point_reached_reward_bonus=0.0,
    target_point_use_actual_position=False, target_point_reward_factor=1.0,
    normalize_reward_to_initial_target_point_distance=False, obs_add_target_point_pos=False,
    obs_add_target_point_relative_pos=False,
    # misc accepted-and-ignored (rendering, logging, real robot; SURVEY section 2 rows 12-15)
    use_gui=False, render_video=False, use_real_robot=False, seed=None, random_agent=False, logging_level="WARNING",
    solver_iterations=None, episodes_per_simulation_reset=None, log_obstacle_data=False,
    # extension of this package: test contacts every n-th 1/240 s sub-step (1 = reference behaviour)
    contact_check_stride=1,
)

# Keys that select parts of the reference this package does not implement: any value other than the listed
# (reference default) one raises instead of being silently ignored.  A key whose non-default value is a no-op for the
# path (rendering, logging, file output) is not listed.
_UNSUPPORTED_UNLESS = dict(
    check_braking_trajectory_collisions=False, check_braking_trajectory_torque_limits=False, use_real_robot=False,
    moving_object_aim_at_current_robot_position=False,
    # klimits constructor arguments (actions.py:97-106) that the range model here does not have a knob for: the range is
    # the exact set of accelerations from which the limits stay satisfiable (DESIGN.md section 2, deviation 1)
    acceleration_after_max_vel_limit_factor=0.01, set_velocity_after_max_pos_to_zero=True,
    action_preprocessing_function=None,   # "tanh" is computed and discarded by the reference (SURVEY Q1); others unknown
    punish_adaptation=False, punish_end_min_distance=False, punish_end_max_torque=False,
    punish_braking_trajectory_min_distance=False, punish_braking_trajectory_max_torque=False,
    obstacle_use_computed_actual_values=False, distance_calculation_check_observed_points=False,
    collision_avoidance_new_state_sample_time_range=None, always_use_collision_avoidance_starting_point_sampling=False,
    terminate_on_robot_stop=False, max_resampling_attempts=0, static_robot=False, activate_obstacle_collisions=False,
    observed_link_point_scene=0, control_time_step=None,
    human_network_use_full_observation=False,
    risk_state_config=0, risk_use_backup_agent_for_initial_backup_trajectory_only=False,
    risk_state_deterministic_backup_trajectory=False, risk_store_ground_truth=False,
    risk_ignore_estimation_probability=0.0, risk_config=None,
)
# values besides the default that are implemented: "tanh" is equivalent to the default (SURVEY Appendix A, Q1);
# risk_state_config 3 (RISK_CHECK_NEXT_STATE_SIMULATE_NEXT_STEP) rates the simulated next state with a state risk network
# inside the step (smenv_set_risk_next_state); risk_state_config 4 (RISK_CHECK_NEXT_STATE_SIMULATE_NEXT_STEP_AND_BACKUP_
# TRAJECTORY) is the backup-trajectory look-ahead inside the step (smenv_set_risk_lookahead)
_ALSO_ACCEPTED = dict(action_preprocessing_function=("tanh",), risk_state_config=(3, 4))


def _names_state_action_network(path):
    """True if a component of `path` is state_action (the shipped networks, risk_networks/state_action/<scene>) or
    state_action_risk (the state-action outputs of risk_train)."""
    parts = str(path).replace("\\", "/").split("/")
    return any(p in ("state_action", "state_action_risk") for p in parts)


class EnvConfig(dict):
    """Dict of the recognised env_config keys with reference defaults filled in (attribute access allowed)."""

    def __init__(self, **kwargs):
        super().__init__(_DEFAULTS)
        self.ignored = {}
        for key, value in kwargs.items():
            if key in _DEFAULTS:
                self[key] = value
            else:
                self.ignored[key] = value  # swallowed like the reference's **kwargs
        for key, default in _UNSUPPORTED_UNLESS.items():
            if self[key] != default and self[key] not in _ALSO_ACCEPTED.get(key, ()):
                raise NotImplementedError("env_config key '{}' = {!r} selects a part of the reference this package does "
                                          "not implement (only {!r} is supported; see DESIGN.md)".format(
                                              key, self[key], default))
        if (self["risk_config_dir"] is None) != (self["risk_threshold"] is None) and self["risk_config_dir"] is not None:
            raise ValueError("risk_config_dir needs risk_threshold (safe_motions_base.py:527-579, README.md:223-235)")
        if self["risk_state_config"] == 4 and self["risk_config_dir"] is None:
            raise ValueError("risk_state_config=4 (the backup-trajectory look-ahead) needs risk_config_dir, which supplies "
                             "the backup policy, and risk_threshold")
        if self["risk_state_config"] == 3:
            if self["risk_config_dir"] is None or self["risk_threshold"] is None:
                raise ValueError("risk_state_config=3 (rate the simulated next state) needs risk_config_dir, which supplies "
                                 "the state risk network, and risk_threshold")
            if _names_state_action_network(self["risk_config_dir"]):
                raise NotImplementedError("risk_state_config=3 rates the simulated next state with a state risk network "
                                          "(risk_train on state_risk data); rating it with the state-action network of "
                                          "{!r} is not implemented".format(self["risk_config_dir"]))
        if self["robot_scene"] != 0:
            raise NotImplementedError("only robot_scene=0 (one iiwa7) is implemented; the reference itself defines "
                                      "only robot_scene 0 and 9 (robot_scene_base.py:169-183)")
        if self["moving_object_sequence"] != 0 and self["use_moving_objects"]:
            raise NotImplementedError("moving_object_sequence != 0 is not implemented")
        if self["use_target_points"] and (self["target_point_sequence"] != 0 or self["target_point_use_actual_position"]):
            raise NotImplementedError("target points: only target_point_sequence=0 on the setpoint pose is implemented")
        if self["trajectory_time_step"] <= 0:
            raise ValueError("trajectory_time_step must be positive")

    def __getattr__(self, name):
        try:
            return self[name]
        except KeyError:
            raise AttributeError(name)

    @classmethod
    def from_params_json(cls, path, **overrides):
        """Loads the ``env_config`` of a reference checkpoint's params.json (evaluate.py:452-639)."""
        with open(path) as f:
            params = json.load(f)
        cfg = dict(params.get("env_config", params))
        cfg.update(overrides)
        return cls(**cfg)


# README.md:74 / :81 training commands and trained_networks/backup_networks/*/params.json
_BACKUP_COMMON = dict(
    acc_limit_factor=1.0, action_max_punishment=0.4, action_punishment_min_threshold=0.95,
    closest_point_safety_distance=0.01, collision_avoidance_episode_early_termination_punishment=-15.0,
    collision_avoidance_episode_termination_bonus=15.0, collision_avoidance_kinematic_state_sampling_mode=True,
    collision_avoidance_kinematic_state_sampling_probability=0.7,
    collision_avoidance_low_acceleration_max_reward=0.0, collision_avoidance_low_acceleration_threshold=1.0,
    collision_avoidance_low_velocity_max_reward=0.0, collision_avoidance_low_velocity_threshold=1.0,
    collision_avoidance_mode=True, collision_avoidance_moving_obstacles_max_reward_distance=0.6,
    collision_avoidance_moving_obstacles_max_reward=3.0, collision_avoidance_self_collision_max_reward_distance=0.05,
    collision_avoidance_self_collision_max_reward=1.0, collision_avoidance_static_obstacles_max_reward_distance=0.1,
    collision_avoidance_static_obstacles_max_reward=1.0, collision_avoidance_stay_in_state_probability=0.3,
    collision_check_time=0.033, jerk_limit_factor=1.0, obstacle_scene=5, pos_limit_factor=1.0, punish_action=True,
    robot_scene=0, solver_iterations=50, starting_point_cartesian_range_scene=1,
    terminate_on_collision_with_moving_obstacle=True, terminate_on_collision_with_static_obstacle=True,
    terminate_on_self_collision=True, trajectory_duration=2.0, trajectory_time_step=0.1,
    use_controller_target_velocities=True, vel_limit_factor=1.0,
)


def space_backup_config(**overrides):
    """The Space backup-policy env of README.md:74 (BASELINE.json configs[0])."""
    cfg = dict(_BACKUP_COMMON, experiment_name="backup_space", obs_planet_size_per_planet=2, planet_mode=True,
               planet_one_center=[-0.1, 0.0, 0.8], planet_one_euler_angles=[0.35, 0, 0], planet_one_period=5.0,
               planet_one_radius_xy=[0.65, 0.8], planet_two_center=[-0.1, 0, 0.8],
               planet_two_euler_angles=[-0.35, 0, 0], planet_two_radius_xy=[0.75, 0.8], planet_two_time_shift=-2.0)
    cfg.update(overrides)
    return EnvConfig(**cfg)


def ball_backup_config(**overrides):
    """The Ball backup-policy env of README.md:81 (BASELINE.json configs[1])."""
    cfg = dict(_BACKUP_COMMON, experiment_name="backup_ball", moving_object_sphere_center=[0, 0, 0.5],
               moving_object_sphere_radius=2.5, moving_object_sphere_height_min_max=[-0.5, 0.5],
               moving_object_sphere_angle_min_max=[0, 6.2831], moving_object_speed_meter_per_second=6.0,
               moving_object_check_invalid_target_link_point_positions=True,
               moving_object_random_initial_position=True, use_moving_objects=True)
    cfg.update(overrides)
    return EnvConfig(**cfg)


def space_task_config(**overrides):
    """The Space reaching task of README.md:223 (SafeMotionsEnv with target points; the env the risk gate wraps)."""
    cfg = dict(acc_limit_factor=1.0, action_max_punishment=0.4, action_punishment_min_threshold=0.95,
               closest_point_safety_distance=0.01, collision_check_time=0.033, jerk_limit_factor=1.0,
               normalize_reward_to_initial_target_point_distance=True, obs_add_target_point_pos=True,
               obs_add_target_point_relative_pos=True, obstacle_scene=5, pos_limit_factor=1.0, punish_action=True,
               robot_scene=0, solver_iterations=50, starting_point_cartesian_range_scene=1,
               target_point_cartesian_range_scene=0, target_point_radius=0.065, target_point_reached_reward_bonus=5,
               target_point_relative_pos_scene=0, target_point_sequence=0,
               terminate_on_collision_with_moving_obstacle=True, terminate_on_collision_with_static_obstacle=True,
               terminate_on_self_collision=True, trajectory_duration=8.0, trajectory_time_step=0.1,
               use_controller_target_velocities=True, use_target_points=True, vel_limit_factor=1.0,
               experiment_name="reaching_task_space", obs_planet_size_per_planet=2, planet_mode=True,
               planet_one_center=[-0.1, 0.0, 0.8], planet_one_euler_angles=[0.35, 0, 0], planet_one_period=5.0,
               planet_one_radius_xy=[0.65, 0.8], planet_two_center=[-0.1, 0, 0.8],
               planet_two_euler_angles=[-0.35, 0, 0], planet_two_radius_xy=[0.75, 0.8], planet_two_time_shift=-2.0)
    cfg.update(overrides)
    return EnvConfig(**cfg)


def human_backup_config(**overrides):
    """The Human backup-policy env (trained_networks/backup_networks/human/params.json; BASELINE.json configs[2]): the
    iiwa next to a human whose arms are moved by the shipped human policy."""
    cfg = dict(_BACKUP_COMMON, experiment_name="Backup_Human", trajectory_duration=3.0,
               human_network_checkpoint="human_network/checkpoint/checkpoint",
               human_network_use_collision_avoidance_starting_point_sampling=True,
               human_network_collision_avoidance_kinematic_state_sampling_probability=0.3,
               human_network_collision_avoidance_stay_in_state_probability=0.3,
               human_network_use_full_observation=False)
    cfg.update(overrides)
    return EnvConfig(**cfg)
