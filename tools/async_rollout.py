"""Synchronous vs asynchronous stepping of one scene, in one process, alternating.

  python tools/async_rollout.py [--scene acorn] [--batch 4096] [--steps 40] [--rounds 2] [--policy] [--out FILE]

Modes:
  sync_B    GripperSim.step over N = B environments
  sync_2B   GripperSim.step over N = 2B environments
  async     AsyncGripperEnv with N = 2B in the pool and batch B (recv, then send for the returned batch)

Actions are uniform random, or with --policy the tensor-core policy forward (GripperPolicy) on the observations just
returned.  Protocol as bench.py: every environment of every mode first takes >= 150 agent steps from reset (untimed), then
the modes are timed in turn, `--rounds` times: `--steps` synchronous steps, or 2 x steps x N / (2B) recvs in async mode (the
same number of transitions per environment).  Reported per mode and round: substeps/s (sum of the phase substep counts
NSUB_A + NSUB_B + NSUB_C of the info rows handed out in the window), transitions/s, kernel launches per step or recv.  A
last, separate pass runs torch.profiler over a few async recvs for the per-kernel device times (step kernel, indexed
observation kernel, queue kernels, the gather of the returned batch) and counts parked environments per recv.  The card's
name and power limit are read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

STEADY_STATE_STEP = 150


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--scene", default="acorn")
    ap.add_argument("--batch", type=int, default=4096)
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--policy", action="store_true")
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
    emit({"device": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip() or q.stderr.strip(), "scene": a.scene, "batch": a.batch,
          "policy": a.policy, "steps": a.steps, "rounds": a.rounds})
    B = a.batch
    cfg = make_config(sim_env="/xmls/%s_env.xml" % a.scene)
    gen = torch.Generator(device="cuda").manual_seed(0)
    pol = None
    if a.policy:
        from mujoco_rl_manipulate_unknown_objects_b200.policy import GripperPolicy
        pol = GripperPolicy(max_envs=2 * B, seed=1)

    def actions(obs):
        n = obs.shape[0]
        if pol is not None:
            return pol(obs)
        return torch.rand((n, 6), device="cuda", generator=gen) * 2 - 1

    nsub = slice(INFO["NSUB_A"], INFO["NSUB_C"] + 1)

    class Sync:
        def __init__(self, n):
            self.name, self.n = "sync_%s" % ("B" if n == B else "2B"), n
            self.sim = GripperSim(cfg, num_envs=n, auto_reset=True)

        def warm(self):
            for _ in range(STEADY_STATE_STEP):
                self.sim.step(actions(self.sim.obs))

        def window(self):
            sim, sub = self.sim, torch.zeros((), dtype=torch.float64, device="cuda")
            l0 = sim.launch_count
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(a.steps):
                sim.step(actions(sim.obs))
                sub += sim.info[:, nsub].sum(dtype=torch.float64)
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
            return dict(substeps=float(sub), transitions=self.n * a.steps, seconds=dt, calls=a.steps, launches=sim.launch_count - l0)

    class Async:
        def __init__(self):
            self.name, self.n = "async", 2 * B
            self.sim = GripperSim(cfg, num_envs=2 * B, auto_reset=True)
            self.pool = AsyncGripperEnv(self.sim, B)
            self.pool.async_reset()

        def one(self):
            r = self.pool.recv()
            self.pool.send(actions(r["obs"]), r["env_id"])
            return r

        def warm(self):
            # every environment >= 150 agent steps: each recv returns B of the 2B, FIFO, so 2 x 150 recvs (+ the reset batches)
            for _ in range(2 * STEADY_STATE_STEP + 2):
                self.one()
            self.pool.status()  # raises on any error the device recorded

        def window(self):
            R = 2 * a.steps
            sub = torch.zeros((), dtype=torch.float64, device="cuda")
            l0 = self.sim.launch_count
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(R):
                r = self.one()
                sub += r["info"][:, nsub].sum(dtype=torch.float64)
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
            self.pool.status()
            return dict(substeps=float(sub), transitions=B * R, seconds=dt, calls=R, launches=self.sim.launch_count - l0)

    modes = [Sync(B), Sync(2 * B), Async()]
    for m in modes:
        t0 = time.perf_counter()
        m.warm()
        torch.cuda.synchronize()
        emit({"warm": m.name, "seconds": round(time.perf_counter() - t0, 2)})
    for rnd in range(a.rounds):
        for m in modes:
            w = m.window()
            emit({"mode": m.name, "round": rnd, "envs": m.n, "batch": B, "substeps_per_s": w["substeps"] / w["seconds"],
                  "transitions_per_s": w["transitions"] / w["seconds"], "ms_per_call": 1e3 * w["seconds"] / w["calls"],
                  "launches_per_call": w["launches"] / w["calls"], "calls": w["calls"]})

    # per-kernel device times of the async mode, and how many environments each recv parks
    am = modes[-1]
    parked = []
    for _ in range(8):
        am.one()
        parked.append(am.pool.status()["parked"])
    from torch.profiler import ProfilerActivity, profile
    R = 16
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(R):
            am.one()
        torch.cuda.synchronize()
    per = {}
    for e in prof.key_averages():
        t = getattr(e, "device_time_total", None)
        if t is None:
            t = e.cuda_time_total
        if t > 0 and e.count > 0:
            per[e.key[:90]] = dict(ms_per_recv=round(t / 1e3 / R, 4), calls_per_recv=round(e.count / R, 2))
    emit({"async_kernels": dict(sorted(per.items(), key=lambda kv: -kv[1]["ms_per_recv"])[:14]), "parked_after_recv": parked})
    am.pool.status()
    if pol is not None:
        pol.close()
    for m in modes:
        m.sim.close()
    if a.out:
        with open(a.out, "a") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
