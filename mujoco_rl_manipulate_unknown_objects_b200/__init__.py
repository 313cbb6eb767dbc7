"""B200-native batched simulator for the two-finger-gripper manipulation environment.

Public surface:
  GripperSim           thin object over the C-ABI (include/b200_gripper_sim.h); device buffers as torch tensors
  BatchedRobotVecEnv   stable-baselines3-style VecEnv over GripperSim (drop-in for DummyVecEnv([RobotEnv]))
  AsyncGripperEnv      EnvPool-style asynchronous send / recv over GripperSim
  make_config          Namespace with the reference's config/base_config.py defaults
  compile_model        model compiler only (no GPU needed)
"""
from .config import make_config, scene_path  # noqa: F401
from .sim import GripperSim, CompiledModel, compile_model  # noqa: F401
from .vec_env import BatchedRobotVecEnv  # noqa: F401
from .async_env import AsyncGripperEnv  # noqa: F401

__all__ = ["GripperSim", "CompiledModel", "compile_model", "BatchedRobotVecEnv", "AsyncGripperEnv", "make_config", "scene_path"]
