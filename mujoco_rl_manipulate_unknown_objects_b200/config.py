"""Environment constructor contract: the fields RobotEnv reads from the reference's argparse Namespace
(reference config/base_config.py:13-43, same names and defaults)."""
import argparse
import os

ASSETS = os.path.join(os.path.dirname(os.path.abspath(__file__)), "assets")

DEFAULTS = dict(sim_env="/xmls/acorn_env.xml", width_capture=64, height_capture=64, full_observation=True, camera_id=3,
                show_obs=False, max_rotation=0.15, max_translation=0.05, grasp_tolerance=0.03, pos_tolerance=0.002,
                include_roll=True, max_steps=400, im_reward=False, her_buffer=False, direction=0, time_horizon=400,
                rendering_zoom_width=10, rendering_zoom_height=7.5,
                # not in the reference (its resets are deterministic): object pose jitter at reset, SURVEY.md §8f N4
                reset_noise_xy=0.0, reset_noise_yaw=0.0, seed=0)


def make_config(**overrides):
    """Namespace with the reference defaults; keyword arguments override (unknown names are rejected).  `sim_env` may be a list or
    tuple of scenes: a mixed simulator whose environments each run one of them per episode (GripperSim.next_object_ids)."""
    unknown = set(overrides) - set(DEFAULTS)
    if unknown:
        raise TypeError("unknown config field(s): %s" % ", ".join(sorted(unknown)))
    d = dict(DEFAULTS)
    d.update(overrides)
    return argparse.Namespace(**d)


def scene_path(sim_env):
    """Resolve `config.sim_env` ('/xmls/<name>_env.xml', robot_env.py:26) against the packaged scenes; absolute
    paths to existing files are used as they are."""
    if os.path.isabs(sim_env) and os.path.exists(sim_env):
        return sim_env
    p = os.path.join(ASSETS, sim_env.lstrip("/"))
    if not os.path.exists(p):
        raise FileNotFoundError("scene file %r not found (looked in %s)" % (sim_env, ASSETS))
    return p


def scene_paths(sim_env):
    """`config.sim_env` as a list of resolved scene files: one for a string, one per entry for a list or tuple."""
    if isinstance(sim_env, (list, tuple)):
        return [scene_path(e) for e in sim_env]
    return [scene_path(sim_env)]
