"""GPU: the replay buffer's indexed write mode (DeviceReplayBuffer.begin_indexed / add_indexed, csrc/replay_kernels.cu), which
takes the environments of an asynchronous pool (AsyncGripperEnv) at their own rates, and SAC trained from the pool
(RolloutWorker.start_async / collect_async).

* equivalence: fed every environment in every call (in a random order), an indexed buffer holds the same bytes as a lock-step
  buffer fed the same rollout and samples the same batches, indices included;
* pool storage: every environment's stored transitions equal its returns recorded in torch, however ragged the counts;
* pool sampling: environments in proportion to their complete transitions, transitions uniform within an environment,
  goals from the same episode, rewards equal to compute_reward;
* protocol: mode mixing, bad ids, an empty sample and a second async_reset.
"""
import math

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _bits(x):
    import torch
    return x.view(torch.int32) if x.dtype == torch.float32 else x


def _same(a, b):
    import torch
    return torch.equal(_bits(a), _bits(b))


def _chi2_ok(counts, expected):
    chi2, dof = float(((counts - expected) ** 2 / expected).sum()), len(counts) - 1
    return chi2 < dof + 8 * math.sqrt(2 * dof), (chi2, dof)


# ------------------------------------------------------------------------------------------------------- lock-step equivalence
def test_indexed_buffer_fed_in_lock_step_equals_the_lock_step_buffer():
    import torch
    from mujoco_rl_manipulate_unknown_objects_b200 import make_config
    from mujoco_rl_manipulate_unknown_objects_b200.replay import DeviceReplayBuffer
    from mujoco_rl_manipulate_unknown_objects_b200.rollout import RolloutWorker
    N, CAP, STEPS = 64, 16, 40
    cfg = make_config(sim_env="/xmls/sugar_cube_env.xml", time_horizon=6, her_buffer=True, reset_noise_xy=0.02, reset_noise_yaw=0.3, seed=3)
    w = RolloutWorker(cfg, envs_per_gpu=N, seed=3)
    s = w.sim
    ls = DeviceReplayBuffer(CAP, N, s.obs_shape, s.action_dim, her_reward=True, seed=7)
    ix = DeviceReplayBuffer(CAP, N, s.obs_shape, s.action_dim, her_reward=True, seed=7)
    gen = torch.Generator(device="cuda").manual_seed(0)

    def add_indexed():  # the synchronous step need not write the simulator's action buffer: pass the worker's actions
        ix.add_indexed(torch.randperm(N, device="cuda", generator=gen).int(), w.actions, s.reward, s.done, s.info, s.obs, s.terminal_obs)

    ix.begin_indexed()
    add_indexed()  # arms every environment with its reset observation
    assert len(ix) == 0 and int(ix.added.sum()) == 0
    for k in range(1, STEPS + 1):
        w.collect(1, random_actions=True, replay=ls)
        add_indexed()
        if k in (10, STEPS):  # before and after the ring wraps
            assert torch.equal(ix.added, torch.full((N,), k, dtype=torch.int64, device="cuda"))
            assert len(ix) == len(ls) == min(k, CAP) * N and ix.status() == len(ls)
            for d in (0, 1, 7, 123456789):
                a, b = ls.sample(4096, 0.8, draw=d), ix.sample(4096, 0.8, draw=d)
                for key in a:
                    assert _same(a[key], b[key]), (k, d, key)
                assert (a["goal_index"] >= 0).any()
    assert int(ls.done.sum()) > 0
    for key in ("obs", "next_obs", "actions", "reward", "done", "info"):
        assert _same(getattr(ls, key), getattr(ix, key)), key
    with pytest.raises(RuntimeError, match="grl_replay_status"):
        ix.transitions_per_env
    w.close()
    ls.close()
    ix.close()


# ------------------------------------------------------------------------------------------------------- the pool
N_POOL, B_POOL, CAP_POOL = 512, 64, 8


def _pool_run(her_buffer=True, im_reward=False, seed=2):
    """sugar_cube pool (N 512, batch 64, time_horizon 2) feeding an indexed buffer of capacity 8.  Environment e's j-th send
    is tape[j, e].  Every return is recorded in torch.  Runs until some environment holds more than CAP + 2 transitions."""
    import torch
    from mujoco_rl_manipulate_unknown_objects_b200 import AsyncGripperEnv, GripperSim, make_config
    from mujoco_rl_manipulate_unknown_objects_b200.replay import DeviceReplayBuffer
    N, B = N_POOL, B_POOL
    cfg = make_config(sim_env="/xmls/sugar_cube_env.xml", time_horizon=2, her_buffer=her_buffer, im_reward=im_reward, reset_noise_xy=0.02,
                      reset_noise_yaw=0.3, seed=seed)
    sim = GripperSim(cfg, num_envs=N, auto_reset=True)
    rb = DeviceReplayBuffer(CAP_POOL, N, sim.obs_shape, sim.action_dim, her_reward=her_buffer, seed=9)
    T = 64
    tape = torch.rand((T, N, sim.action_dim), device="cuda", generator=torch.Generator(device="cuda").manual_seed(seed)) * 2 - 1
    pool = AsyncGripperEnv(sim, B)
    pool.async_reset()
    rb.begin_indexed()
    seen = np.zeros(N, np.int64)  # returns per environment
    rec = {k: [] for k in ("env", "seq", "obs", "reward", "done", "info", "next_obs")}
    while seen.max() <= CAP_POOL + 3:
        assert len(rec["env"]) < 400
        r = pool.recv()
        ids = r["env_id"]
        rb.add_indexed(ids, sim.actions, sim.reward, sim.done, sim.info, sim.obs, sim.terminal_obs)
        ids_h = ids.cpu().numpy().astype(np.int64)
        assert ids_h.min() >= 0
        rec["env"].append(ids_h)
        rec["seq"].append(seen[ids_h].copy())
        rec["obs"].append(r["obs"])
        rec["reward"].append(r["reward"])
        rec["done"].append(r["done"])
        rec["info"].append(r["info"])
        rec["next_obs"].append(torch.where(r["done"].bool()[:, None, None, None], r["terminal_obs"], r["obs"]))
        k = torch.as_tensor(seen[ids_h], device="cuda").clamp(max=T - 1)
        seen[ids_h] += 1
        pool.send(tape[k, ids.long()], ids)
    pool.status()
    flat = {k: (np.concatenate(v) if k in ("env", "seq") else torch.cat(v)) for k, v in rec.items()}
    pos = np.full((N, seen.max()), -1, np.int64)  # pos[e, j]: row of flat holding environment e's j-th return
    pos[flat["env"], flat["seq"]] = np.arange(len(flat["env"]))
    return dict(sim=sim, pool=pool, rb=rb, tape=tape, seen=seen, flat=flat, pos=pos)


@pytest.fixture(scope="module")
def pool_run():
    run = _pool_run()
    yield run
    run["rb"].close()
    run["sim"].close()


def _stored(run):
    """(env, j) of every complete transition the buffer holds: j in [added - min(added, CAP), added)."""
    added = run["seen"] - 1
    env, j = [], []
    for e in range(N_POOL):
        js = np.arange(max(0, added[e] - CAP_POOL), added[e])
        env.append(np.full(len(js), e))
        j.append(js)
    return np.concatenate(env), np.concatenate(j)


def test_pool_storage_equals_the_recorded_returns(pool_run):
    import torch
    rb, f, pos, seen, tape = pool_run["rb"], pool_run["flat"], pool_run["pos"], pool_run["seen"], pool_run["tape"]
    S = CAP_POOL + 1
    added = seen - 1
    assert np.array_equal(rb.added.cpu().numpy(), added)
    assert added.min() < CAP_POOL < added.max(), "the counts are not ragged: %d .. %d" % (added.min(), added.max())
    assert rb.status() == len(rb) == int(np.minimum(added, CAP_POOL).sum())
    env, j = _stored(pool_run)
    slot = torch.as_tensor(j % S, device="cuda")
    e = torch.as_tensor(env, device="cuda")
    src, dst = torch.as_tensor(pos[env, j], device="cuda"), torch.as_tensor(pos[env, j + 1], device="cuda")
    assert bool((src >= 0).all()) and bool((dst >= 0).all())
    assert _same(rb.obs[slot, e], f["obs"][src])
    assert _same(rb.actions[slot, e], tape[torch.as_tensor(j, device="cuda"), e])
    for key in ("reward", "done", "info", "next_obs"):
        assert _same(getattr(rb, key)[slot, e], f[key][dst]), key
    assert int(rb.done[slot, e].sum()) > 0
    # the pending slot holds each environment's last returned observation
    last = torch.as_tensor(pos[np.arange(N_POOL), seen - 1], device="cuda")
    ar = torch.arange(N_POOL, device="cuda")
    assert _same(rb.obs[torch.as_tensor(added % S, device="cuda"), ar], f["obs"][last])


def test_pool_sampling_follows_the_transition_counts(pool_run):
    import torch
    rb, seen = pool_run["rb"], pool_run["seen"]
    N, S = N_POOL, CAP_POOL + 1
    added = torch.as_tensor(seen - 1, device="cuda")
    size = added.clamp(max=CAP_POOL)
    first = added - size  # the oldest complete transition of each environment
    draws = [rb.sample(16384, 0.8, draw=d) for d in range(4)]
    b = {k: torch.cat([x[k] for x in draws]) for k in draws[0]}
    idx, gi = b["index"], b["goal_index"]
    assert bool((idx >= 0).all())
    env, slot = idx % N, idx // N

    def t_of(slot, env):
        return first[env] + (slot - first[env] % S) % S

    t = t_of(slot, env)
    off = t - first[env]
    assert bool((off < size[env]).all()), "a sample returned the pending slot or a slot not written yet"
    assert not bool((slot == added[env] % S).any())
    # environments in proportion to their complete transitions
    M, counts, has = idx.numel(), torch.bincount(env, minlength=N).double(), size > 0
    assert not bool(counts[~has].any())
    ok, stat = _chi2_ok(counts[has], M * size[has].double() / float(size.sum()))
    assert ok, stat
    # the transition uniform within its environment: one chi-square over (size, offset) cells
    cells = torch.bincount(size[env] * (CAP_POOL + 1) + off, minlength=(CAP_POOL + 1) ** 2).double().reshape(CAP_POOL + 1, CAP_POOL + 1)
    per_size = torch.bincount(size[env], minlength=CAP_POOL + 1).double()
    chi2, dof = 0.0, 0
    for s in range(1, CAP_POOL + 1):
        if per_size[s] >= 50 * s:
            e = per_size[s] / s
            chi2 += float(((cells[s, :s] - e) ** 2 / e).sum())
            dof += s - 1
    assert dof > 0 and chi2 < dof + 8 * math.sqrt(2 * dof), (chi2, dof)
    # HER goals: same environment, at or after the sample, stored, in the same episode
    rel = gi >= 0
    assert rel.any()
    assert torch.equal(gi[rel] % N, env[rel])
    tg = t_of(gi[rel] // N, env[rel])
    assert bool((tg >= t[rel]).all()) and bool((tg < added[env[rel]]).all()) and bool((tg > t[rel]).any())
    f, pos = pool_run["flat"], torch.as_tensor(pool_run["pos"], device="cuda")
    dn = f["done"].long()
    # no done in [t, tg): the return after transition j is row pos[e, j + 1]
    for k in range(CAP_POOL):
        m = (t[rel] + k < tg)
        if m.any():
            assert not bool(dn[pos[env[rel][m], t[rel][m] + k + 1]].any())
    # reproducible from (seed, draw)
    again = rb.sample(16384, 0.8, draw=2)
    assert all(_same(again[k], draws[2][k]) for k in again)
    assert not torch.equal(rb.sample(16384, 0.8, draw=5)["index"], draws[2]["index"])
    rb.status()


@pytest.mark.parametrize("her_buffer,im_reward", [(0, 0), (1, 0), (0, 1), (1, 1)])
def test_pool_sampled_reward_equals_compute_reward(her_buffer, im_reward):
    from mujoco_rl_manipulate_unknown_objects_b200 import BatchedRobotVecEnv
    from mujoco_rl_manipulate_unknown_objects_b200._native import INFO
    from mujoco_rl_manipulate_unknown_objects_b200.vec_env import LazyInfos
    run = _pool_run(her_buffer=bool(her_buffer), im_reward=bool(im_reward), seed=4)
    sim, rb = run["sim"], run["rb"]
    env = BatchedRobotVecEnv(sim.config, num_envs=N_POOL, _sim=sim)
    b = {k: v.cpu().numpy() for k, v in rb.sample(1024, 0.8, draw=3).items()}
    infos = LazyInfos(b["info"], b["done"].astype(bool), None, env.target_direction, 0.0, obs=b["next_obs"], prev_obs=b["obs"])
    ref = env.compute_reward(b["achieved_goal"], b["desired_goal"], infos)
    bad = (b["info"][:, INFO["FLAGS"]].astype(np.int32) & 2) != 0
    assert (b["reward"][bad] == 0).all()
    err = np.abs(ref - b["reward"])[~bad] / np.maximum(1.0, np.abs(ref[~bad]))
    assert err.max() <= 1e-5, (err.max(), int(np.argmax(err)))
    if her_buffer:
        rel = b["goal_index"] >= 0
        assert (b["desired_goal"][rel] != b["info"][rel, INFO["DESIRED"]:INFO["DESIRED"] + 2]).any()
    env.close()
    rb.close()
    sim.close()


# ------------------------------------------------------------------------------------------------------- protocol
def test_indexed_protocol_and_errors():
    import torch
    from mujoco_rl_manipulate_unknown_objects_b200.replay import DeviceReplayBuffer
    from mujoco_rl_manipulate_unknown_objects_b200.sim import NativeError
    N, CAP, A = 8, 4, 6
    g = torch.Generator(device="cuda").manual_seed(0)
    obs = torch.randint(0, 256, (N, 5, 64, 64), dtype=torch.uint8, device="cuda", generator=g)
    tobs = torch.randint(0, 256, (N, 5, 64, 64), dtype=torch.uint8, device="cuda", generator=g)
    act = torch.rand((N, A), device="cuda", generator=g)
    rew = torch.rand(N, device="cuda", generator=g)
    done = torch.zeros(N, dtype=torch.uint8, device="cuda")
    info = torch.rand((N, 40), device="cuda", generator=g)
    ids = lambda *v: torch.tensor(v, dtype=torch.int32, device="cuda")  # noqa: E731
    args = (act, rew, done, info, obs, tobs)

    # the two modes do not mix; add_indexed needs begin_indexed
    ls = DeviceReplayBuffer(CAP, N)
    with pytest.raises(NativeError, match="begin_indexed"):
        ls.add_indexed(ids(0), *args)
    ls.begin(obs)
    with pytest.raises(NativeError, match="cannot be mixed"):
        ls.begin_indexed()
    with pytest.raises(NativeError, match="lock-step"):
        ls.add_indexed(ids(0), *args)
    ls.add(*args)
    assert len(ls) == N and ls.status() == N
    ls.close()

    rb = DeviceReplayBuffer(CAP, N)
    rb.begin_indexed()
    with pytest.raises(NativeError, match="cannot be mixed"):
        rb.begin(obs)
    with pytest.raises(NativeError, match="indexed"):
        rb.add(*args)
    # nothing stored: the sample reports it and returns -1 indices
    s = rb.sample(16, 0.5)
    assert bool((s["index"] == -1).all()) and bool((s["goal_index"] == -1).all())
    with pytest.raises(NativeError, match="no complete transition"):
        rb.status()
    assert rb.status() == 0  # reporting cleared the error
    # arming: records the observation, adds no transition; -1 entries are skipped
    rb.add_indexed(ids(*range(N), -1, -1), *args)
    assert rb.status() == 0 and torch.equal(rb.obs[0], obs)
    rb.add_indexed(ids(-1, -1), *args)
    assert rb.status() == 0
    # an id out of range and an id listed twice: reported, the duplicate written once
    rb.add_indexed(ids(3, N, 3, -1, 5), *args)
    with pytest.raises(NativeError, match="num_envs") as e:
        rb.status()
    assert "twice" in str(e.value)
    expect = torch.zeros(N, dtype=torch.int64, device="cuda")
    expect[3] = expect[5] = 1
    assert torch.equal(rb.added, expect) and rb.status() == 2 and len(rb) == 2
    assert torch.equal(rb.next_obs[0, 3], obs[3]) and torch.equal(rb.obs[1, 3], obs[3]) and torch.equal(rb.actions[0, 3], act[3])
    s = rb.sample(256, 0.0, draw=1)
    assert set((s["index"] % N).tolist()) == {3, 5} and set((s["index"] // N).tolist()) == {0}
    rb.status()
    rb.close()


def test_second_async_reset_closes_the_open_episodes():
    import torch
    from mujoco_rl_manipulate_unknown_objects_b200 import make_config
    from mujoco_rl_manipulate_unknown_objects_b200.replay import DeviceReplayBuffer
    from mujoco_rl_manipulate_unknown_objects_b200.rollout import RolloutWorker
    N, B, CAP = 64, 16, 64
    cfg = make_config(sim_env="/xmls/sugar_cube_env.xml", time_horizon=100, her_buffer=True, reset_noise_xy=0.02, reset_noise_yaw=0.3, seed=1)
    w = RolloutWorker(cfg, envs_per_gpu=N, seed=1)
    rb = DeviceReplayBuffer(CAP, N, w.sim.obs_shape, w.sim.action_dim, her_reward=True, seed=3)
    w.start_async(B, replay=rb)
    w.collect_async(16, replay=rb)
    pool, s = w.pool, w.sim
    while True:  # drain: receive without sending until nothing is in flight
        c = pool.status()
        if c["pending"] + c["parked"] + c["ready"] == 0:
            break
        rb.add_indexed(pool.recv()["env_id"], s.actions, s.reward, s.done, s.info, s.obs, s.terminal_obs)
    a0 = rb.added.clone()
    assert int(a0.min()) >= 1
    w.start_async(B, replay=rb)
    w.collect_async(12, replay=rb)
    rb.status()
    a1 = rb.added
    assert bool((a1 > a0).any()) and int(a1.max()) < CAP
    b = rb.sample(16384, 1.0, draw=5)
    idx, gi = b["index"], b["goal_index"]
    env = idx % N
    t, tg = idx // N, gi // N  # the ring has not wrapped: slot == transition number
    rel = gi >= 0
    old = t < a0[env]
    assert bool((old & rel).any()) and bool((~old & rel).any())
    assert bool((tg[old & rel] < a0[env[old & rel]]).all()), "an episode cut by the reset must end before it"
    assert bool((tg[~old & rel] >= a0[env[~old & rel]]).all())
    w.close()
    rb.close()


# ------------------------------------------------------------------------------------------------------- SAC from the pool
def test_sac_trains_from_the_pool():
    from mujoco_rl_manipulate_unknown_objects_b200 import make_config
    from mujoco_rl_manipulate_unknown_objects_b200.replay import DeviceReplayBuffer
    from mujoco_rl_manipulate_unknown_objects_b200.rollout import RolloutWorker
    from mujoco_rl_manipulate_unknown_objects_b200.sac import SACLearner
    N, B, CAP, R = 512, 128, 64, 8
    cfg = make_config(sim_env="/xmls/sugar_cube_env.xml", her_buffer=True)
    w = RolloutWorker(cfg, envs_per_gpu=N, seed=0)
    rb = DeviceReplayBuffer(CAP, N, w.sim.obs_shape, w.sim.action_dim, her_reward=True, seed=0)
    learner = SACLearner(w, rb, batch_size=64, seed=1)
    w.start_async(B, replay=rb)
    transitions, recvs = 0.0, 0
    for _ in range(3):
        st = w.collect_async(R, replay=rb)
        recvs += R
        transitions += st.as_dict()["transitions"]
        losses = learner.update(2)
        assert all(np.isfinite(v) for v in losses.values()), losses
    assert int(rb.added.max()) < CAP  # nothing overwritten, so every complete transition is still stored
    assert len(rb) == rb.status() == recvs * B - N == int(transitions)
    w.pool.status()
    w.close()
    rb.close()
