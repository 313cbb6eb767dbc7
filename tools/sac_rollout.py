#!/usr/bin/env python
"""SAC on the device-resident HER replay buffer: rollouts feed DeviceReplayBuffer (k_replay_add), SACLearner trains on batches
from it (k_replay_sample + torch autograd + one flat-bucket Adam per optimiser, gradients all-reduced over NCCL).

  python tools/sac_rollout.py [--envs 4096] [--capacity 128] [--steps 16] [--iters 3] [--gradient-steps 16]   # one GPU
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P tools/sac_rollout.py
  python tools/sac_rollout.py --pool-batch B [...]   # the asynchronous pool: N = --envs environments, batch B

Per iteration, rank 0 prints one JSON line: rollout substeps/s over all ranks with and without replay= (two workers built with the
same seeds and weights, so both step the same trajectories), the gradient-step time, the replay ratio (gradient steps per
collected transition), the buffer's bytes, and every rank's parameter checksum.  A last line gives the k_replay_add /
k_replay_sample times (CUDA events over many launches) with the bytes they move, computed from the shapes, and the card's name
and power limit.

With --pool-batch B the workers run an AsyncGripperEnv pool (RolloutWorker.start_async / collect_async) and the buffer is in
indexed write mode.  An iteration is steps x N / B recvs, the same number of transitions per environment as the synchronous
mode; the "plain" worker runs the same pool without the buffer (its completion order is scheduling-dependent, so
same_trajectories is not expected).  The kernel line times k_replay_add_indexed at B ids and the indexed sample (k_replay_scan +
k_replay_sample<true>) at batch 256 and 4 096, each next to the lock-step kernel at the same size (k_replay_add over B
environments, k_replay_sample<false> on a filled lock-step buffer of the training buffer's shape)."""
import argparse, json, os, subprocess, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import torch.distributed as dist
from mujoco_rl_manipulate_unknown_objects_b200 import make_config
from mujoco_rl_manipulate_unknown_objects_b200._native import INFO
from mujoco_rl_manipulate_unknown_objects_b200.replay import DeviceReplayBuffer
from mujoco_rl_manipulate_unknown_objects_b200.rollout import RolloutWorker, dist_info, rank_seed
from mujoco_rl_manipulate_unknown_objects_b200.sac import SACLearner

ap = argparse.ArgumentParser()
ap.add_argument("--scene", default="sugar_cube"); ap.add_argument("--envs", type=int, default=4096); ap.add_argument("--capacity", type=int, default=128)
ap.add_argument("--steps", type=int, default=16); ap.add_argument("--iters", type=int, default=3); ap.add_argument("--gradient-steps", type=int, default=16)
ap.add_argument("--batch", type=int, default=256); ap.add_argument("--her-ratio", type=float, default=0.8); ap.add_argument("--launches", type=int, default=50)
ap.add_argument("--pool-batch", type=int, default=0, help="run the asynchronous pool with this batch size (0: the synchronous step)")
a = ap.parse_args()
pool = a.pool_batch > 0
rank, world, local = dist_info()
local %= torch.cuda.device_count()  # more ranks than GPUs (a functional check on one card) share them over gloo instead of NCCL
torch.cuda.set_device(local)
if world > 1:
    if world <= torch.cuda.device_count():
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    else:
        dist.init_process_group("gloo")
cfg = make_config(sim_env="/xmls/%s_env.xml" % a.scene, her_buffer=True)
plain = RolloutWorker(cfg, envs_per_gpu=a.envs, device=local, seed=0)
w = RolloutWorker(cfg, envs_per_gpu=a.envs, device=local, seed=0)
N, obs_shape, A = a.envs, w.sim.obs_shape, w.sim.action_dim
rb = DeviceReplayBuffer(a.capacity, N, obs_shape, A, her_reward=True, seed=rank_seed(0, rank), device=local)
learner = SACLearner(w, rb, batch_size=a.batch, her_ratio=a.her_ratio, seed=1)
plain.policy.load_state_dict(learner.actor.state_dict())
if pool:
    recvs = a.steps * N // a.pool_batch
    plain.start_async(a.pool_batch)
    w.start_async(a.pool_batch, replay=rb)
    collect_plain = lambda: plain.collect_async(recvs)  # noqa: E731
    collect_replay = lambda: w.collect_async(recvs, replay=rb)  # noqa: E731
else:
    collect_plain = lambda: plain.collect(a.steps)  # noqa: E731
    collect_replay = lambda: w.collect(a.steps, replay=rb)  # noqa: E731


def timed(fn):
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return time.perf_counter() - t0, out


def max_over_ranks(*xs):
    t = torch.tensor(xs, device=w.device, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return t.tolist()


def gather(x):
    t = torch.zeros(world, device=w.device, dtype=torch.float64)
    t[rank] = x
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
    return t.tolist()


collected = 0
for it in range(a.iters):
    t_plain, s_plain = timed(lambda: collect_plain().all_reduce())
    t_replay, s_replay = timed(lambda: collect_replay().all_reduce())
    collected += s_replay.as_dict()["transitions"]
    t_update, losses = timed(lambda: learner.update(a.gradient_steps))
    plain.policy.load_state_dict(learner.actor.state_dict())  # both workers keep stepping the same trajectories
    t_plain, t_replay, t_update = max_over_ranks(t_plain, t_replay, t_update)
    sums = gather(learner.checksum())
    dp, dr = s_plain.as_dict(), s_replay.as_dict()
    if rank == 0:
        print(json.dumps({"iter": it, "n_gpus": world, "envs_per_gpu": N, "rollout_steps": a.steps, "capacity": a.capacity,
                          "mode": "pool" if pool else "sync", "pool_batch": a.pool_batch if pool else None,
                          "substeps_per_s_plain": dp["substeps"] / t_plain, "substeps_per_s_replay": dr["substeps"] / t_replay,
                          "transitions_per_s_plain": dp["transitions"] / t_plain, "transitions_per_s_replay": dr["transitions"] / t_replay,
                          "same_trajectories": None if pool else dp["substeps"] == dr["substeps"] and dp["reward_sum"] == dr["reward_sum"],
                          "replay_overhead": t_replay / t_plain - 1.0, "gradient_steps": a.gradient_steps, "batch": a.batch,
                          "gradient_step_ms": 1e3 * t_update / a.gradient_steps, "replay_ratio": learner.actor_opt.step_count * world / collected,
                          "buffer_bytes_per_gpu": rb.nbytes, "stored_transitions_per_gpu": len(rb), "losses": losses,
                          "added_min_max": [int(rb.added.min()), int(rb.added.max())] if pool else None,
                          "param_checksum_per_rank": sums, "checksums_equal": len(set(sums)) == 1}), flush=True)

# kernel times: CUDA events over many launches.  The add kernel runs on a second, small buffer (its cost does not depend on the
# capacity), the sample kernel on the training buffer (>> L2, and every launch draws new rows).
img = int(torch.tensor(obs_shape).prod())
small = 4 * (A + 1 + INFO["STRIDE"]) + 1
add_bytes = {"read": N * (img + small), "written": N * (2 * img + small + 8)}
s = w.sim
args = (w.actions, s.reward, s.done, s.info, s.obs, s.terminal_obs)


def events(fn, n):
    for _ in range(3):
        fn()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda._sleep(50_000_000)  # keeps the GPU busy while the host enqueues: the events time back-to-back kernels, not launches
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n * 1e3  # us


def sample_bytes(B):
    return {"read": B * (2 * img + small + 16), "written": B * (2 * img + small + 16 + 16)}


def rate(d):
    d["GB_per_s"] = (d["read"] + d["written"]) / d["us"] / 1e3
    return d


if not pool:
    bench = DeviceReplayBuffer(16, N, obs_shape, A, device=local)
    bench.begin(w.sim.obs)
    res = {"k_replay_add": rate({"envs": N, "us": events(lambda: bench.add(*args), a.launches), **add_bytes})}
    res["k_replay_sample"] = []
    for B in (256, 4096, 16384):
        draws = iter(range(10 ** 6, 2 * 10 ** 6))
        us = events(lambda: rb.sample(B, a.her_ratio, draw=next(draws)), a.launches)
        res["k_replay_sample"].append(rate({"batch": B, "us": us, **sample_bytes(B)}))
    bench.close()
else:
    # k_replay_add_indexed at B ids (an indexed buffer over all N environments, armed once) next to k_replay_add over B environments
    Bp = a.pool_batch
    ix = DeviceReplayBuffer(16, N, obs_shape, A, device=local)
    ix.begin_indexed()
    ids = torch.randperm(N, device=w.device, generator=torch.Generator(device=w.device).manual_seed(0)).int()
    ix.add_indexed(ids, *args)
    ids = ids[:Bp].contiguous()
    ls = DeviceReplayBuffer(16, Bp, obs_shape, A, device=local)
    ls.begin(s.obs[:Bp])
    ls_args = tuple(x[:Bp] for x in args)
    rows = {"read": Bp * (img + small) + 4 * Bp, "written": Bp * (2 * img + small + 8)}
    res = {"k_replay_add_indexed": rate({"ids": Bp, "us": events(lambda: ix.add_indexed(ids, *args), a.launches), **rows}),
           "k_replay_add": rate({"envs": Bp, "us": events(lambda: ls.add(*ls_args), a.launches), **dict(rows, read=Bp * (img + small))})}
    ix.close()
    ls.close()
    # the indexed sample (scan + gather) on the training buffer, the lock-step sample on a filled buffer of the same shape
    ref = DeviceReplayBuffer(a.capacity, N, obs_shape, A, her_reward=True, device=local)
    ref.begin(s.obs)
    for _ in range(a.capacity + 1):
        ref.add(*args)
    res["sample"] = []
    for B in (256, 4096):
        draws = iter(range(10 ** 6, 2 * 10 ** 6))
        us_ix = events(lambda: rb.sample(B, a.her_ratio, draw=next(draws)), a.launches)
        us_ls = events(lambda: ref.sample(B, a.her_ratio, draw=next(draws)), a.launches)
        res["sample"].append({"batch": B, "indexed": rate({"us": us_ix, **sample_bytes(B), "scan_read": 8 * N, "scan_written": 8 * N}),
                              "lock_step": rate({"us": us_ls, **sample_bytes(B)})})
    ref.close()
    rb.status()  # raises on a bad id or an empty sample recorded on the device
if rank == 0:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", str(local)],
                       stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True).stdout.strip()
    print(json.dumps({"kernels": res, "device": torch.cuda.get_device_name(local), "nvidia_smi": q,
                      "note": "sample bytes include the output writes; the add kernel reads terminal_obs instead of obs on done rows"}), flush=True)
plain.close()
w.close()
rb.close()
if world > 1:
    dist.destroy_process_group()
