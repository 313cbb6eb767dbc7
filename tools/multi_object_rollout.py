"""One mixed simulator of several objects against separate single-scene simulators, in one process.

  python tools/multi_object_rollout.py [--envs 8192] [--pool-batch 4096] [--steps 20] [--rounds 2] [--warm 100] [--out FILE]

Modes (uniform random actions):
  mixed       one GripperSim over all four scenes, N environments (variant n % 4)
  single_X    one GripperSim of scene X, N environments
  split       four single-scene simulators of N / 4 environments each, stepped one after another (what a user without
              mixed simulators would run)
  mixed_pool  AsyncGripperEnv over the mixed simulator, batch --pool-batch

Every simulator first takes --warm agent steps from reset (untimed, every environment of the pool as well), then the modes are
timed in turn, --rounds times: --steps synchronous steps, or steps x N / batch recvs.  Reported per mode and round: physics
substeps/s (NSUB_A + NSUB_B + NSUB_C of the info rows of the window), transitions/s, and the step kernel's shared-memory layout
(bytes per block, whether the hull vertices are staged in shared memory).  The card's name, power limit and max SM clock are
read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

SCENES = ("sugar_cube", "sand_ball", "bread_crumb", "acorn")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=8192)
    ap.add_argument("--pool-batch", type=int, default=4096)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--warm", type=int, default=100)
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    a = ap.parse_args()
    import torch
    from mujoco_rl_manipulate_unknown_objects_b200 import AsyncGripperEnv, GripperSim, make_config
    from mujoco_rl_manipulate_unknown_objects_b200._native import INFO
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: nothing to measure")
    lines = []

    def emit(d):
        s = json.dumps(d)
        print(s, flush=True)
        lines.append(s)

    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True)
    emit({"device": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip() or q.stderr.strip(), "envs": a.envs, "pool_batch": a.pool_batch,
          "steps": a.steps, "rounds": a.rounds, "warm": a.warm, "scenes": SCENES})
    N, B = a.envs, a.pool_batch
    gen = torch.Generator(device="cuda").manual_seed(0)
    nsub = slice(INFO["NSUB_A"], INFO["NSUB_C"] + 1)
    rand = lambda n: torch.rand((n, 6), device="cuda", generator=gen) * 2 - 1  # noqa: E731

    def sim(scenes, n):
        env = ["/xmls/%s_env.xml" % s for s in scenes]
        return GripperSim(make_config(sim_env=env if len(env) > 1 else env[0]), num_envs=n, auto_reset=True)

    def layout(s):
        smem, hull_smem, hull_count, warps = (int(x) for x in s.get("step_smem"))
        return dict(smem_per_block=smem, hull_in_smem=bool(hull_smem), hull_vertices=hull_count, warps=warps)

    class Sync:
        def __init__(self, name, sims):
            self.name, self.sims = name, sims

        def warm(self):
            for _ in range(a.warm):
                for s in self.sims:
                    s.step(rand(s.num_envs))

        def window(self):
            sub = torch.zeros((), dtype=torch.float64, device="cuda")
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(a.steps):
                for s in self.sims:
                    s.step(rand(s.num_envs))
                    sub += s.info[:, nsub].sum(dtype=torch.float64)
            torch.cuda.synchronize()
            return float(sub), sum(s.num_envs for s in self.sims) * a.steps, time.perf_counter() - t0

    class Pool:
        def __init__(self):
            self.name, self.sims = "mixed_pool", [sim(SCENES, N)]
            self.pool = AsyncGripperEnv(self.sims[0], B)
            self.pool.async_reset()

        def one(self):
            r = self.pool.recv()
            self.pool.send(rand(B), r["env_id"])
            return r

        def warm(self):
            for _ in range(a.warm * N // B + N // B):
                self.one()
            self.pool.status()

        def window(self):
            R = a.steps * N // B
            sub = torch.zeros((), dtype=torch.float64, device="cuda")
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(R):
                sub += self.one()["info"][:, nsub].sum(dtype=torch.float64)
            torch.cuda.synchronize()
            return float(sub), R * B, time.perf_counter() - t0

    modes = [Sync("mixed", [sim(SCENES, N)])] + [Sync("single_" + s, [sim((s,), N)]) for s in SCENES]
    modes += [Sync("split", [sim((s,), N // len(SCENES)) for s in SCENES]), Pool()]
    for m in modes:
        m.warm()
        emit({"mode": m.name, "layout": [layout(s) for s in m.sims]})
    for rnd in range(a.rounds):
        for m in modes:
            sub, tr, dt = m.window()
            emit({"mode": m.name, "round": rnd, "substeps_per_s": round(sub / dt), "transitions_per_s": round(tr / dt), "seconds": round(dt, 3)})
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "a") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
