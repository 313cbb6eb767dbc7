#!/usr/bin/env python
"""bench.py — env-steps/sec of the batched gripper environment (BASELINE.json metric) on N B200s of one node.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--config 2|3|4|5] [--scene acorn] [--envs 4096]
                   [--dump-outputs DIR]

Workload (BASELINE.json configs[1], `--config 2`): acorn_env (stand-in mesh, see DESIGN.md), 4 096 environments per GPU,
actions U(-1,1)^6 from a seeded generator, physics + reward + observation, auto-reset on.  One "step" = one VecEnv.step over
the whole batch (one pass of the hot path).  Environments shard across ranks with no data-path collective ("weak" scaling);
NCCL carries only the rollout statistics.

Where in the rollout the timed window sits matters: from reset it takes ~100 agent steps until the batch reaches its steady
state (grippers in contact, a fifth of the environments running a 400-substep timed-out gripper phase), and the early steps
are up to twice as fast.  Both arms therefore roll `--preroll` untimed agent steps from reset first (default: whatever
brings the start of the timed window to agent step 150), then W warm-up steps, then K timed steps — so a short window
(the driver's 20/5) measures the same regime as the default 200/50.

Unit: the headline `value` is S = physics substeps/s (one substep == one MuJoCo `mj_step`, 2 ms of simulated time in one
environment; BASELINE.md §3 reads the 1e7/s target in this unit).  T = agent transitions/s (VecEnv.step rows) and the
mean substeps per transition that links the two are printed beside it.

The reference arm (--impl reference) times the CPU implementation of the same path on the host cores: the oracle's
fp64 C restatement (oracle/engine.c on a model compiled by oracle/mjcf.py, kind "port" — MuJoCo itself cannot be installed
here, SURVEY.md §8c) with one environment per thread, on a bounded sample of the same workload, same protocol
(pre-roll, W warm-up and K timed transitions per environment).  It never loads the product library.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

UNIT = "physics substeps/s (one substep = one mj_step of one env)"
BYTES_PER_SUBSTEP = 428 + 64  # SURVEY.md §8(d): 56 f32 read + 51 f32 written + ~64 B contact summary, if state round-tripped HBM
BYTES_PER_TRANSITION = 21100  # SURVEY.md §8(d): state in/out + action + obs write (20 480 B) + goals/reward/done
STEADY_STATE_STEP = 150       # agent step (from reset) at which the timed window starts by default
XMLS = os.path.join(ROOT, "mujoco_rl_manipulate_unknown_objects_b200", "assets", "xmls")

# BASELINE.json configs[1..4] (configs[0], the single-env trained-policy rollout, is blocked: SURVEY.md F1-F3)
CONFIGS = {2: dict(scene="acorn", envs=4096, direction=0, actions="uniform", policy=False),
           3: dict(scene="sugar_cube", envs=8192, direction=45, actions="uniform", policy=False),
           4: dict(scene="bread_crumb", envs=4096, direction=0, actions="uniform", policy=True),
           5: dict(scene="sand_ball", envs=16384, direction=0, actions="contact", policy=False)}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)  # SURVEY.md §8d: >= 200 timed agent steps after >= 50 warm-up
    ap.add_argument("--warmup", type=int, default=50)
    ap.add_argument("--preroll", type=int, default=None, help="untimed agent steps from reset before the warm-up (default: max(0, %d - warmup))" % STEADY_STATE_STEP)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=int, default=None, choices=sorted(CONFIGS), help="BASELINE.json configs[i-1] preset (scene, envs, direction, actions)")
    ap.add_argument("--scene", default=None)
    ap.add_argument("--envs", type=int, default=None, help="environments per GPU")
    ap.add_argument("--direction", type=int, default=None)
    ap.add_argument("--actions", default=None, choices=["uniform", "contact"],
                    help="uniform: U(-1,1)^6.  contact: biased towards +x / close (SURVEY.md §8d cfg5) so that grippers stay in finger-object-floor contact")
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-vecenv", action="store_true", help="skip the e2e_vecenv leg (BatchedRobotVecEnv.step)")
    ap.add_argument("--policy", action="store_true", default=None, help="actions from the tensor-core policy forward on the previous observation "
                    "(device-resident rollout loop, BASELINE.json configs[3]) instead of a random tape")
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="target wall time of the CPU sample")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step returned (rank 0's environments) as DIR/<name>.npy")
    a = ap.parse_args()
    if a.steps < 1 or a.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    preset = CONFIGS[a.config or 2]
    for k, v in preset.items():
        if getattr(a, k) is None:
            setattr(a, k, v)
    a.policy = bool(a.policy)
    if a.preroll is None:
        a.preroll = max(0, STEADY_STATE_STEP - a.warmup)
    return a


def metric_name(a):
    return "env-steps/sec (%s_env, %d envs/GPU)" % (a.scene, a.envs)


def shape_actions(u, mode):
    """u: uniform(-1,1) samples [..., 6] (numpy or torch) -> the action tape of `mode` (in place)."""
    if mode == "contact":
        u[..., 0] = 0.6 + 0.4 * u[..., 0]      # +x: towards / along the object, U(0.2, 1)
        u[..., 1:5] *= 0.3                      # little lateral / vertical / rotational wander
        u[..., 5] = -0.5 - 0.5 * u[..., 5]      # close, U(-1, 0)
    return u


# ----------------------------------------------------------------------------------------------- clocks
class ClockSampler:
    """nvidia-smi sampling DURING the timed region (B200_PROFILING.md clocks line)."""

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
            "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q, "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons), "samples": len(sm)}


# ----------------------------------------------------------------------------------------------- CPU arm (oracle port)
def cpu_rollout(args, seconds, threads=None):
    """The oracle's C restatement on the oracle's own compiled model, one environment per host thread, same action
    distribution, auto-reset, same protocol: every environment rolls preroll + warmup transitions from reset (neither counted
    nor timed), then `steps` timed ones.  Nothing of the product is imported or loaded.
    Returns dict(value substeps/s, transitions/s, cores, sample, seconds = time inside the timed windows)."""
    from oracle import engine, mjcf
    om = engine.Model(mjcf.compile_mjcf(os.path.join(XMLS, "%s_env.xml" % args.scene)))
    cores = threads or os.cpu_count() or 1
    skip, K = args.preroll + args.warmup, max(1, args.steps)
    rng = np.random.default_rng(args.seed)
    # calibration: two envs per core through the whole protocol, then size the sample to `seconds` of wall time
    a = shape_actions(rng.uniform(-1, 1, (2 * cores, skip + K, 6)), args.actions)
    t = time.perf_counter()
    engine.rollout_window(om, a, cores, skip, direction=args.direction)
    per_env = max(time.perf_counter() - t, 1e-3) / 2  # wall seconds per environment and core
    per_core = int(max(2, min(256, seconds / per_env)))
    nenv = cores * per_core
    a = shape_actions(rng.uniform(-1, 1, (nenv, skip + K, 6)), args.actions)
    t = time.perf_counter()
    r = engine.rollout_window(om, a, cores, skip, direction=args.direction)
    wall = time.perf_counter() - t
    sub, tr, dt = r["substeps"], r["transitions"], max(r["seconds"], 1e-9)
    return dict(value=sub / dt, unit=UNIT, cores=cores, kind="port",
                sample="%d envs x %d timed transitions (after %d untimed from reset) of %s_env, %s actions, on %d host threads (%d substeps in %.2f s of timed "
                       "windows, %.1f s wall), oracle/engine.c fp64 restatement on the oracle/mjcf.py model, not MuJoCo" % (
                           nenv, K, skip, args.scene, args.actions, cores, sub, dt, wall),
                transitions_per_s=tr / dt, substeps_per_transition=sub / max(tr, 1), seconds=dt, ncon_mean=r["ncon_sum"] / max(tr, 1), envs=nenv)


def workload_text(args, N, ours):
    mesh = "synthetic stand-in mesh: acorn.stl is absent from the reference tree" if args.scene == "acorn" else "reference mesh"
    if args.policy and ours:
        act = "actions from the tcgen05 policy forward on the previous observation (random-init weights, stochastic)"
    else:
        act = "U(-1,1)^6 actions" if args.actions == "uniform" else "contact-biased actions (+x / close, SURVEY.md §8d cfg5)"
    what = "physics + progress reward + RGB-D observation, auto-reset" if ours else "physics + progress reward + scalar obs channels (no image render on the CPU arm), auto-reset"
    return "%s_env (%s), %s, %s, %s; timed window = agent steps %d..%d from reset" % (
        args.scene, mesh, "%d envs/GPU" % N if ours else "bounded sample of the %d-env batch" % N, act, what,
        args.preroll + args.warmup, args.preroll + args.warmup + args.steps)


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    r = cpu_rollout(args, max(2.0, args.cpu_seconds))
    K = max(1, args.steps)
    line = {"impl": "reference", "metric": metric_name(args), "value": r["value"], "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "preroll": args.preroll, "ms_per_step": r["seconds"] * 1e3 / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic",
            "config": {"workload": workload_text(args, args.envs, False), "direction": args.direction, "envs_per_step": r["envs"],
                       "step": "one transition of every environment of the sample (%d envs on %d threads)" % (r["envs"], r["cores"])},
            "cpu_baseline": {k: r[k] for k in ("value", "unit", "cores", "kind", "sample")},
            "transitions_per_s": r["transitions_per_s"], "substeps_per_transition": r["substeps_per_transition"], "ncon_mean": r["ncon_mean"],
            "e2e": {"value": r["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))
    return 0


# ----------------------------------------------------------------------------------------------- our arm
DUMP_ROWS, DUMP_IMAGES = 65536, 256  # environments whose records / images --dump-outputs writes: <= 14 + 2 x 21 MB as float32


def dump_outputs(out_dir, sim, action):
    """Writes what the last sim.step returned to its caller as float32 / float64 DIR/<name>.npy: the per-environment records
    of up to DUMP_ROWS environments, the observations of up to DUMP_IMAGES, and the terminal observations of up to
    DUMP_IMAGES of the environments that finished in that step (terminal_obs_env: their indices), each a fixed seeded
    sample when there are more.  `action` is the policy's action of that step (None when the actions came from the tape,
    which is an input)."""
    import torch
    N = sim.num_envs
    rng = np.random.default_rng(0)

    def sample(idx, n):
        return np.sort(rng.choice(idx, n, replace=False)) if len(idx) > n else idx

    rows, imgs = sample(np.arange(N), DUMP_ROWS), sample(np.arange(N), DUMP_IMAGES)
    fin = sample(np.nonzero(sim.done.cpu().numpy())[0], DUMP_IMAGES)
    rows, imgs, fin_t = [torch.as_tensor(i, device=sim.device) for i in (rows, imgs, fin)]
    out = {"obs": sim.obs[imgs], "terminal_obs": sim.terminal_obs[fin_t], "reward": sim.reward[rows], "done": sim.done[rows],
           "achieved_goal": sim.achieved_goal[rows], "desired_goal": sim.desired_goal[rows], "info": sim.info[rows]}
    if action is not None:
        out["action"] = action[rows]
    os.makedirs(out_dir, exist_ok=True)
    for name, t in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.float().cpu().numpy())
    np.save(os.path.join(out_dir, "terminal_obs_env.npy"), fin.astype(np.float64))


def run_ours(args):
    import torch
    import torch.distributed as dist
    from mujoco_rl_manipulate_unknown_objects_b200 import BatchedRobotVecEnv, GripperSim, make_config
    from mujoco_rl_manipulate_unknown_objects_b200._native import INFO

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: there is no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    N, K, W, P = args.envs, args.steps, args.warmup, args.preroll
    cfg = make_config(sim_env="/xmls/%s_env.xml" % args.scene, direction=args.direction)
    sim = GripperSim(cfg, num_envs=N, device=local, auto_reset=True)
    gen = torch.Generator(device=dev).manual_seed(args.seed + rank)  # per-rank seed (SURVEY.md §8e)
    actions = shape_actions(torch.rand((P + W + K, N, sim.action_dim), device=dev, generator=gen) * 2 - 1, args.actions)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2
    c0, c1 = INFO["NSUB_A"], INFO["NSUB_A"] + 3
    sub_k = torch.zeros(K, device=dev, dtype=torch.float64)    # substeps of every timed step
    chain_k = torch.zeros(K, device=dev, dtype=torch.float64)  # longest substep chain of the batch, per timed step
    acc = torch.zeros(4, device=dev, dtype=torch.float64)      # episodes finished, reward sum, sum of ncon_max, transitions with >= 400 substeps
    from mujoco_rl_manipulate_unknown_objects_b200.policy import GripperPolicy
    policy = GripperPolicy(max_envs=N, obs_shape=sim.obs_shape, action_dim=sim.action_dim, device=local, seed=args.seed)
    noise = torch.randn((P + W + K, N, sim.action_dim), device=dev, generator=gen) if args.policy else None
    pol_act = torch.empty((N, sim.action_dim), device=dev)

    def one_step(i):
        if args.policy:
            policy.forward(sim.obs, deterministic=False, noise=noise[i], out=pol_act)
            sim.step(pol_act)
        else:
            sim.step(actions[i])

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    sim.reset()
    for i in range(P + W):
        one_step(i)
    barrier()
    sim.step_kernel_ms(reset=True)
    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
    launches0 = sim.launch_count + policy.launch_count
    barrier()
    wall0 = time.perf_counter()
    for i in range(K):
        flush.zero_()  # L2 flush between timed iterations (outside the event pair)
        ev[i][0].record()
        one_step(P + W + i)
        ev[i][1].record()
        nsub = sim.info[:, c0:c1].sum(1)
        sub_k[i] = nsub.sum()
        chain_k[i] = nsub.max()
        acc[0] += sim.done.sum()
        acc[1] += sim.reward.sum()
        acc[2] += sim.info[:, INFO["NCON_MAX"]].sum()
        acc[3] += (nsub >= 400).sum()
    barrier()
    wall = time.perf_counter() - wall0
    launches = sim.launch_count + policy.launch_count - launches0
    step_ms = np.array([a.elapsed_time(b) for a, b in ev])
    dev_ms = float(step_ms.sum())
    kernel_ms = sim.step_kernel_ms(reset=True)
    clk = clocks.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, sim, pol_act if args.policy else None)
    sub_k_h, chain_k_h = sub_k.cpu().numpy(), chain_k.cpu().numpy()
    q = max(1, K // 4)  # the last quarter of the timed window
    # ---- policy forward alone on the last observation (tensor roofline): CUDA events on the launching stream, L2 flushed
    pol_ms = []
    for i in range(3 + 10):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        policy.forward(sim.obs, out=pol_act)
        e1.record()
        torch.cuda.synchronize(dev)
        if i >= 3:
            pol_ms.append(e0.elapsed_time(e1))
    pol_ms = float(np.median(pol_ms))
    # ---- end to end with HOST buffers.  Two legs, both replaying the very trajectories of the device-timed region (same reset
    # state, same pre-roll / warm-up / timed action tapes), so they differ from `value` only by what the host path adds:
    #   e2e        : the C-ABI call grs_step_host with pinned host arrays (H2D actions, step, observations stored into the pinned
    #                arrays by the kernel as environments finish, D2H of the small records)
    #   e2e_vecenv : BatchedRobotVecEnv.step — the stable-baselines3 drop-in a user calls (numpy in, numpy + lazy infos out)
    Cc, H, Wd = sim.obs_shape
    pin = lambda shape, dt: torch.empty(shape, dtype=dt).pin_memory().numpy()  # noqa: E731
    h_act = pin((N, sim.action_dim), torch.float32)
    h_obs, h_rew, h_done = pin((N, Cc, H, Wd), torch.uint8), pin((N,), torch.float32), pin((N,), torch.uint8)
    h_ag, h_dg, h_info = pin((N, 2), torch.float32), pin((N, 2), torch.float32), pin((N, INFO["STRIDE"]), torch.float32)
    h_tobs = pin((N, Cc, H, Wd), torch.uint8)
    acts_host = actions.cpu().numpy() if not args.policy else None
    e2e_sub, e2e_s, vec_sub, vec_s = 0.0, 0.0, 0.0, 0.0
    if not args.policy:
        sim.reset()
        for i in range(P + W):
            one_step(i)
        barrier()
        t0 = time.perf_counter()
        for i in range(K):
            h_act[...] = acts_host[P + W + i]
            sim.step_host(h_act, obs=h_obs, achieved=h_ag, desired=h_dg, reward=h_rew, done=h_done, info=h_info, terminal_obs=h_tobs)
            e2e_sub += float(h_info[:, c0:c1].sum())
        barrier()
        e2e_s = time.perf_counter() - t0
        if not args.no_vecenv:
            venv = BatchedRobotVecEnv(cfg, num_envs=N, device=local, _sim=sim)
            venv.reset()
            for i in range(P + W):
                venv.step(acts_host[i])
            barrier()
            t0 = time.perf_counter()
            for i in range(K):
                obs, rew, dones, infos = venv.step(acts_host[P + W + i])
                vec_sub += float(venv.last_info_rows[:, c0:c1].sum())
            barrier()
            vec_s = time.perf_counter() - t0
    else:
        # the policy loop keeps observations and actions on the device; its host-facing cost is the read of the step's rewards
        t0 = time.perf_counter()
        for i in range(K):
            one_step(P + W + i)
            h_rew[...] = sim.reward.cpu().numpy()
            e2e_sub += float(sim.info[:, c0:c1].sum().item())
        barrier()
        e2e_s = time.perf_counter() - t0
    h2d = h_act.nbytes if not args.policy else 0
    d2h = (h_obs.nbytes + h_rew.nbytes + h_done.nbytes + h_ag.nbytes + h_dg.nbytes + h_info.nbytes) if not args.policy else h_rew.nbytes
    # ---- aggregate over ranks: units summed, time = max
    stats = torch.tensor([sub_k_h.sum(), float(N * K), acc[0].item(), acc[1].item(), e2e_sub, float(launches), chain_k_h.sum(), acc[2].item(), acc[3].item(),
                          sub_k_h[-q:].sum(), vec_sub], device=dev, dtype=torch.float64)
    tmax = torch.tensor([dev_ms, wall * 1e3, e2e_s * 1e3, kernel_ms, pol_ms, float(step_ms[-q:].sum()), vec_s * 1e3], device=dev, dtype=torch.float64)
    per_rank = torch.tensor([kernel_ms, float(chain_k_h.max()), float(chain_k_h.mean()), dev_ms / K], device=dev, dtype=torch.float64)
    ranks = [per_rank.clone() for _ in range(world)]
    if world > 1:
        dist.all_reduce(stats, op=dist.ReduceOp.SUM)  # rollout-statistics reduction: the only collective on this path
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        dist.all_gather(ranks, per_rank)
    stats, tmax = stats.cpu().numpy(), tmax.cpu().numpy()
    ranks = np.stack([r.cpu().numpy() for r in ranks])
    if rank == 0:
        substeps, transitions = stats[0], stats[1]
        dev_s = tmax[0] / 1e3
        value = substeps / dev_s
        line = {"metric": metric_name(args), "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W, "preroll": P, "ms_per_step": tmax[0] / K,
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": {"workload": workload_text(args, N, True), "direction": args.direction, "envs_per_gpu": N, "actions": "policy" if args.policy else args.actions,
                           "l2": "256 MiB buffer written between timed steps (outside the event pairs)",
                           "parallelism": "env-sharded x%d, no data-path collective" % world},
                # the same metric over the LAST QUARTER of the timed window: equal to `value` when the window sits in the steady state
                "value_late": stats[9] / (tmax[5] / 1e3), "ncon_mean": stats[7] / transitions, "frac_transitions_ge_400_substeps": stats[8] / transitions,
                "transitions_per_s": transitions / dev_s, "substeps_per_transition": substeps / transitions, "episodes_finished": stats[2],
                "mean_reward_per_transition": stats[3] / transitions, "wall_ms_per_step": tmax[1] / K,
                "e2e": {"value": stats[4] / (tmax[2] / 1e3), "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "steps": K,
                        "transitions_per_s": N * K * world / (tmax[2] / 1e3),
                        "api": "grs_step_host (C-ABI, pinned host buffers; observations are stored into them by the kernel as environments finish)"
                        if not args.policy else "device-resident policy loop; the step's rewards are read back to the host"},
                "gpu_launches": int(stats[5] // world), "clocks": clk,
                # an agent step is a chain of dependent substeps; the synchronous VecEnv step lasts as long as the batch's longest chain
                "longest_chain_substeps": stats[6] / world / K, "us_per_substep_of_longest_chain": tmax[3] * 1e3 / max(stats[6] / world / K, 1.0)}
        if vec_s > 0:
            line["e2e_vecenv"] = {"value": stats[10] / (tmax[6] / 1e3), "unit": UNIT, "transitions_per_s": N * K * world / (tmax[6] / 1e3), "steps": K,
                                  "api": "BatchedRobotVecEnv.step (numpy actions in; numpy views of the pinned observation / reward / done arrays and lazy infos out)"}
        if world > 1:
            # weak-scaling loss is the max over ranks of per-rank times: show each rank's numbers so it is attributable
            line["per_rank"] = {"kernel_ms": {"min": float(ranks[:, 0].min()), "median": float(np.median(ranks[:, 0])), "max": float(ranks[:, 0].max())},
                                "ms_per_step": {"min": float(ranks[:, 3].min()), "median": float(np.median(ranks[:, 3])), "max": float(ranks[:, 3].max())},
                                "longest_chain_substeps_max": [float(x) for x in ranks[:, 1]], "longest_chain_substeps_mean": [float(x) for x in ranks[:, 2]]}
        per_launch_sub = substeps / world / K
        kms = tmax[3]
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0))
        achieved = per_launch_sub * BYTES_PER_SUBSTEP / (kms / 1e3) / 1e9 if kms > 0 else None
        prof = {}
        try:
            prof = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
        except Exception:
            pass
        line["roofline"] = {"bound": "hbm", "kernel": "k_env_step_ls, physics phase (fused agent step: controller + <=1200 substeps + reward, state on chip; "
                                                      "device-timed: first block start -> last block leaving the substep loop)",
                            "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak if achieved else None,
                            "traffic": prof.get("k_env_step_bytes_per_launch"),
                            "peak_source": "MEASURED_PEAKS.json hbm_gbs" if peaks else "fallback 6650 GB/s (B200_PROFILING.md)",
                            "kernel_ms": kms, "bytes_per_substep": BYTES_PER_SUBSTEP, "substeps_per_launch": per_launch_sub,
                            # what actually limits this kernel (SURVEY.md §8d asks for it beside the HBM figure): from the committed ncu capture
                            "issue_active_pct": prof.get("k_env_step_issue_active_pct"), "fma_pipe_pct": prof.get("k_env_step_fma_pipe_pct"),
                            "achieved_occupancy_pct": prof.get("k_env_step_achieved_occupancy_pct"), "ncu_source": prof.get("source"),
                            "note": "fused kernel keeps state on chip: it is bound by instruction latency along the batch's chains of dependent substeps, not by HBM "
                                    "(SURVEY.md §8d, DESIGN.md §3.1; traffic = physics + observation phases of one launch); "
                                    "per-transition accounting (%d B incl. the 20 480 B observation) gives %.1f GB/s over the whole step" % (
                                        BYTES_PER_TRANSITION, transitions / world / K * BYTES_PER_TRANSITION / (tmax[0] / K / 1e3) / 1e9)}
        flop = 2 * (225 * 64 * (sim.obs_shape[0] - 1) * 32 + 36 * 512 * 64 + 16 * 576 * 64 + 1024 * 512 + 514 * 256 + 256 * 256 + 256 * 2 * sim.action_dim)
        tpeak = float(peaks.get("bf16_tflops", 1667.5))  # the forward is timed alone: the burst figure applies
        tfl = N * flop / (tmax[4] / 1e3) / 1e12 if tmax[4] > 0 else None
        line["policy"] = {"kernel": "policy forward (tcgen05.mma kind::f16, TMEM accumulators): NatureCNN + actor MLP for %d observations" % N,
                          "ms": tmax[4], "in_timed_region": bool(args.policy), "flop_per_obs": flop,
                          "roofline": {"bound": "tensor", "achieved": tfl, "peak": tpeak, "unit": "TFLOP/s", "frac": tfl / tpeak if tfl else None,
                                       "peak_source": "MEASURED_PEAKS.json bf16_tflops (burst: kernel timed alone)" if peaks else "fallback"}}
        if world == 1 and not args.no_cpu_baseline:
            try:
                cb = cpu_rollout(args, args.cpu_seconds)
                line["cpu_baseline"] = {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample")}
                line["cpu_baseline"]["transitions_per_s"] = cb["transitions_per_s"]
            except Exception as e:  # noqa: BLE001
                line["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": 0, "kind": "port", "sample": "failed: %r" % (e,)}
        print(json.dumps(line))
    policy.close()
    sim.close()
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    a = parse()
    sys.exit(run_reference(a) if a.impl == "reference" else run_ours(a))
