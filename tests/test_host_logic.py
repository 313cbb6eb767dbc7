"""CPU: host-side logic of the VecEnv mirror (no GPU, no native calls): the lazily built `infos` (robot_env.py:226-241
keys, SB3's terminal_observation / TimeLimit.truncated / Monitor episode record), the spaces (sensor.py:12-54,
actuator.py:217-247), the target direction (robot_env.py:30-33, 46-54) and compute_reward (robot_env.py:243-273,
reward.py:18-41) against stored outputs of the reference's own Reward class."""
import numpy as np
import pytest

from mujoco_rl_manipulate_unknown_objects_b200._native import INFO as I
from mujoco_rl_manipulate_unknown_objects_b200.config import make_config
from mujoco_rl_manipulate_unknown_objects_b200.vec_env import LazyInfos, STATUS_NAMES, make_spaces, target_direction, BatchedRobotVecEnv


def _rows(n):
    r = np.zeros((n, I["STRIDE"]), np.float32)
    r[:, I["STATUS"]] = [0, 2, 1][:n] if n <= 3 else 0
    r[:, I["INIT_OBJ_POS"]:I["INIT_OBJ_POS"] + 3] = [0.06, 0.0, 0.0]
    r[:, I["FINAL_OBJ_POS"]:I["FINAL_OBJ_POS"] + 3] = [0.09, 0.01, 0.0]
    r[:, I["GRIPPER_POS"]:I["GRIPPER_POS"] + 3] = [-0.4, 0.0, 0.15]
    r[:, I["NSUB_A"]] = 74; r[:, I["NSUB_C"]] = 120
    r[:, I["EPISODE_STEP"]] = 400; r[:, I["EPISODE_RETURN"]] = 1.5
    r[:, I["GRIPPER_OPEN"]] = 1
    r[:, I["ACHIEVED"]:I["ACHIEVED"] + 2] = [0.09, 0.01]; r[:, I["DESIRED"]:I["DESIRED"] + 2] = [1, 0]
    return r


def test_lazy_infos_follow_the_reference_keys_and_sb3_conventions():
    from mujoco_rl_manipulate_unknown_objects_b200.vec_env import Status, intrinsic_reward
    rows, dones = _rows(3), np.array([False, True, True])
    obs = np.arange(3 * 5 * 4 * 4, dtype=np.uint8).reshape(3, 5, 4, 4)
    prev = obs[::-1].copy()
    tobs = {1: obs[1] + 7, 2: obs[2] + 9}            # terminal observations exist for finished episodes only
    ep = np.arange(3 * 6, dtype=np.float64).reshape(3, 6)
    fin = {1: np.ones(6), 2: np.full(6, 2.0)}
    infos = LazyInfos(rows, dones, tobs, np.array([1, 0]), t_start=0.0, obs=obs, prev_obs=prev, episode_rewards=ep, finished_rewards=fin,
                      truncation_key=True)
    assert len(infos) == 3 and len(infos[:]) == 3 and infos[-1] is infos[2]
    a = infos[0]
    # robot_env.py:226-241: the sixteen keys, in the reference's order
    assert list(a)[:16] == ["old_obs", "new_obs", "init_obj_pos", "final_obj_pos", "target_dir", "gripper_open", "controls", "object_grasped",
                            "episode_step", "episode_rewards", "status", "gripper_position", "object_position", "position_reached",
                            "total_distance", "line_distance"]
    assert a["status"] is Status.RUNNING and a["status"].value == 0 and a["gripper_open"] is True and a["substeps"] == 194
    assert "episode" not in a and "terminal_observation" not in a and "TimeLimit.truncated" not in a
    np.testing.assert_array_equal(a["old_obs"], prev[0]); np.testing.assert_array_equal(a["new_obs"], obs[0])
    np.testing.assert_array_equal(a["episode_rewards"], ep[0])
    np.testing.assert_array_equal(a["controls"], np.zeros(2))  # robot_env.py:149,168: ctrl[5:7] is zero when step() returns
    b, c = infos[1], infos[2]
    assert b["status"] is Status.TIME_LIMIT and b["TimeLimit.truncated"] is True and c["status"] is Status.FAIL and c["TimeLimit.truncated"] is False
    assert b["episode"]["l"] == 400 and abs(b["episode"]["r"] - 1.5) < 1e-6 and b["episode"]["t"] > 0
    np.testing.assert_array_equal(b["terminal_observation"]["observation"], tobs[1])
    np.testing.assert_array_equal(b["new_obs"], tobs[1])          # the finished episode's last image, not the next episode's first
    np.testing.assert_array_equal(b["episode_rewards"], fin[1])
    # default: no TimeLimit.truncated key (the reference has no TimeLimit wrapper, train_agent.py:17-23)
    assert "TimeLimit.truncated" not in LazyInfos(rows, dones, tobs, np.array([1, 0]), t_start=0.0)[1]
    # the host-side intrinsic term against the reference's own IntrinsicReward outputs (tests/golden/unit_vectors.npz)
    u = np.load(__import__("os").path.join(__import__("os").path.dirname(__file__), "golden", "unit_vectors.npz"))
    for i in range(len(u["ir_full"])):
        assert abs(intrinsic_reward(u["ir_a"][i], u["ir_b"][i], True) - u["ir_full"][i]) < 1e-6
        assert abs(intrinsic_reward(u["ir_a"][i][[0, 1, 2, 4]], u["ir_b"][i][[0, 1, 2, 4]], False) - u["ir_rgb"][i]) < 1e-6
    assert STATUS_NAMES == ("RUNNING", "FAIL", "TIME_LIMIT")  # RobotEnv.Status, robot_env.py:19-22


def test_spaces_and_direction():
    obs, act = make_spaces(make_config())
    assert obs["observation"].shape == (5, 64, 64) and obs["observation"].dtype == np.uint8 and act.shape == (6,) and act.dtype == np.float32
    obs, act = make_spaces(make_config(full_observation=False, include_roll=False))
    assert obs["observation"].shape == (4, 64, 64) and act.shape == (5,)
    assert obs["achieved_goal"].shape == (2,) and obs["desired_goal"].dtype == np.float32
    np.testing.assert_array_equal(target_direction(0), [1, 0])
    np.testing.assert_array_equal(target_direction(45), [1, 1])  # robot_env.py:33: not normalised
    d = target_direction(120)
    assert abs(np.linalg.norm(d) - 1) < 1e-12 and abs(np.arctan2(d[1], d[0]) - np.round(np.deg2rad(120), 2)) < 1e-12
    with pytest.raises(TypeError):
        make_config(no_such_field=1)


def test_compute_reward_matches_the_reference_reward_class():
    env = BatchedRobotVecEnv.__new__(BatchedRobotVecEnv)  # host logic only: no simulator behind it
    env.config = make_config()
    env.target_direction = np.array([1, 0])
    info = LazyInfos(_rows(1), np.array([False]), None, env.target_direction, 0.0)[0]
    r = env.compute_reward(info["achieved_goal"], info["desired_goal"], info)
    assert abs(r - 30 * 0.03) < 1e-6  # 3 cm along the direction, lateral error 1 cm < 10 cm: 30 x progress (reward.py:30-33)
    many = env.compute_reward(np.tile(info["achieved_goal"], (2, 1)), np.tile(info["desired_goal"], (2, 1)), np.array([info, info], dtype=object))
    assert many.shape == (2,) and np.allclose(many, r)
    env.config = make_config(her_buffer=True)
    rh = env.compute_reward(info["achieved_goal"], info["desired_goal"], info)
    assert abs(rh - (r + np.exp(-np.linalg.norm(info["desired_goal"] - info["achieved_goal"])))) < 1e-6  # robot_env.py:268-271
    backwards = dict(info, final_obj_pos=np.array([0.03, 0.0, 0.0]))
    env.config = make_config()
    assert env.compute_reward(info["achieved_goal"], info["desired_goal"], backwards) == 0.0
    # the reference's own Reward.agent_reward outputs on 64 seeded inputs (tests/golden/unit_vectors.npz, tools/gen_golden.py)
    u = np.load(__import__("os").path.join(__import__("os").path.dirname(__file__), "golden", "unit_vectors.npz"))
    for i in range(len(u["rw_out"])):
        env.target_direction = u["rw_dir"][i]
        row = dict(info, init_obj_pos=u["rw_init"][i], final_obj_pos=u["rw_final"][i], gripper_open=bool(u["rw_open"][i]),
                   controls=u["rw_ctrl"][i], object_grasped=int(u["rw_grasp"][i]))
        assert abs(env.compute_reward(info["achieved_goal"], info["desired_goal"], row) - u["rw_out"][i]) < 1e-9, i
