"""GPU: mixed simulators (grs_create_scenes) — several object scenes in one simulator, one variant per environment and episode.

* bit-identity: environment n of a mixed simulator computes exactly what environment n of the single-scene simulator of its
  variant computes (step outputs with auto-resets and reset noise, renders of every camera, a substep); the mixed simulator
  reads the convex hulls from global memory and the single-scene ones from shared memory, so this also holds the two hull
  placements of the step kernel against each other;
* next_object: a written variant takes effect at that environment's next auto-reset or explicit reset, and nowhere else;
* the asynchronous pool and SAC work over a mixed simulator unchanged;
* create errors: no scenes, too many scenes, a scene that differs in a shared field.
"""
import re

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

SCENES = ("sugar_cube", "sand_ball", "bread_crumb", "acorn")
OBJ = 39  # GRS_INFO_OBJECT


def _path(scene):
    return "/xmls/%s_env.xml" % scene


def _sim(scenes, n, **cfg):
    from mujoco_rl_manipulate_unknown_objects_b200 import GripperSim, make_config
    env = [_path(s) for s in scenes] if isinstance(scenes, (list, tuple)) else _path(scenes)
    return GripperSim(make_config(sim_env=env, **cfg), num_envs=n, auto_reset=True)


def _bits(x):
    import torch
    return x.view(torch.int32) if x.dtype == torch.float32 else x


def _rows_equal(a, b):
    """per-row bit equality of two [n, ...] tensors"""
    return (_bits(a) == _bits(b)).reshape(a.shape[0], -1).all(1)


# ------------------------------------------------------------------------------------------------ bit-identity with single scenes
def test_mixed_rows_equal_single_scene_rows():
    import torch
    N, T = 256, 5
    cfg = dict(time_horizon=2, reset_noise_xy=0.02, reset_noise_yaw=0.4, im_reward=True, seed=11)
    mixed = _sim(SCENES, N, **cfg)
    singles = [_sim(s, N, **cfg) for s in SCENES]
    assert mixed.scenes[2].endswith("bread_crumb_env.xml") and len(mixed.scenes) == 4
    assert tuple(mixed.reset_obs.shape) == (4,) + mixed.obs_shape and tuple(singles[0].reset_obs.shape) == singles[0].obs_shape
    # step_smem[1]: hull vertices staged in shared memory (DESIGN.md §3.6: the four hulls together do not fit beside the models)
    assert mixed.get("step_smem")[1] == 0, "the mixed simulator no longer reads the hull from global memory"
    assert all(s.get("step_smem")[1] == 1 for s in singles), "a single-scene simulator no longer stages the hull in shared memory"
    obj = mixed.object_ids.long()
    assert torch.equal(obj.cpu(), torch.arange(N) % 4) and torch.equal(mixed.next_object_ids.long(), obj)
    rows = torch.arange(N, device="cuda")
    gen = torch.Generator(device="cuda").manual_seed(3)

    def pick(get):  # row n of the single-scene simulator of variant object[n]
        return torch.stack([get(s) for s in singles])[obj, rows]

    def compare(what, get_m, get_s, mask=None):
        ok = _rows_equal(get_m(mixed), pick(get_s))
        if mask is not None:
            ok = ok | ~mask
        assert bool(ok.all()), "%s differs in environments %s" % (what, torch.flatnonzero(~ok)[:8].tolist())

    for name, f in (("obs", lambda s: s.obs), ("state", lambda s: s.state), ("info", lambda s: s.info[:, :OBJ])):
        compare("reset " + name, f, f)
    assert torch.equal(mixed.info[:, OBJ], obj.float())
    dones = 0
    for t in range(T):
        a = torch.rand((N, 6), device="cuda", generator=gen) * 2 - 1
        for s in (mixed,) + tuple(singles):
            s.step(a)
        for name in ("obs", "reward", "done", "achieved_goal", "desired_goal", "state"):
            compare("step %d %s" % (t, name), lambda s, k=name: getattr(s, k), lambda s, k=name: getattr(s, k))
        compare("step %d info" % t, lambda s: s.info[:, :OBJ], lambda s: s.info[:, :OBJ])
        assert torch.equal(mixed.info[:, OBJ], obj.float()), "info slot 39 is not the environment's variant"
        done = mixed.done != 0
        compare("step %d terminal_obs" % t, lambda s: s.terminal_obs, lambda s: s.terminal_obs, mask=done)
        dones += int(done.sum())
    assert dones >= N, "the tape did not reach the auto-resets"
    for cam in range(3):  # the world cameras' poses differ in bread_crumb
        rgb_m, depth_m = mixed.render(camera_id=cam, width=48, height=40)
        ref = [s.render(camera_id=cam, width=48, height=40) for s in singles]
        assert bool(_rows_equal(rgb_m, torch.stack([r[0] for r in ref])[obj, rows]).all()), "render camera %d rgb" % cam
        assert bool(_rows_equal(depth_m, torch.stack([r[1] for r in ref])[obj, rows]).all()), "render camera %d depth" % cam
    for s in (mixed,) + tuple(singles):
        s.substep(1)
    compare("substep state", lambda s: s.state, lambda s: s.state)
    for s in (mixed,) + tuple(singles):
        s.close()


# ------------------------------------------------------------------------------------------------ next_object
def test_next_object_takes_effect_at_the_next_reset():
    import torch
    N, K = 128, 3
    mixed = _sim(SCENES[:K], N, time_horizon=2)
    gen = torch.Generator(device="cuda").manual_seed(4)
    act = lambda: torch.rand((N, 6), device="cuda", generator=gen) * 2 - 1  # noqa: E731
    mixed.step(act())
    obj0 = mixed.object_ids.clone()
    nxt = (obj0 + 1 + torch.arange(N, device="cuda", dtype=torch.int32) // K % 2) % K  # a permutation of the variants
    mixed.next_object_ids.copy_(nxt)
    cur = obj0.clone()
    switched = 0
    for _ in range(3):
        mixed.step(act())
        done = mixed.done != 0
        assert torch.equal(mixed.info[:, OBJ], cur.float()), "slot 39 must name the variant of the episode the step belongs to"
        now = mixed.object_ids
        assert torch.equal(now[done], nxt[done]) and torch.equal(now[~done], cur[~done])
        if bool(done.any()):
            ref = mixed.reset_obs[now[done].long()]
            assert torch.equal(mixed.obs[done], ref), "the first observation of an episode is the reset image of its variant"
        switched += int((done & (cur != nxt)).sum())
        cur = now.clone()
    assert switched > 0
    # a value that names no variant: set_next_objects refuses it, a raw write is ignored by the reset
    with pytest.raises(ValueError):
        mixed.set_next_objects(torch.full((N,), K, dtype=torch.int32))
    mixed.next_object_ids.fill_(K)
    mixed.reset()
    assert torch.equal(mixed.object_ids, cur)
    # an explicit reset applies next_object to the masked environments only
    again = (cur + 1) % K
    mixed.set_next_objects(again)
    mask = torch.arange(N, device="cuda") % 2 == 0
    mixed.reset(mask)
    assert torch.equal(mixed.object_ids[mask], again[mask]) and torch.equal(mixed.object_ids[~mask], cur[~mask])
    assert torch.equal(mixed.obs[mask], mixed.reset_obs[again[mask].long()])
    assert torch.equal(mixed.info[mask, OBJ], again[mask].float())
    mixed.close()


# ------------------------------------------------------------------------------------------------ asynchronous pool
def test_async_pool_over_a_mixed_simulator_equals_synchronous_steps():
    """environment e's k-th transition from the pool equals row e of the k-th synchronous step of a second mixed simulator"""
    import torch
    from mujoco_rl_manipulate_unknown_objects_b200 import AsyncGripperEnv
    N, B, K = 512, 64, 4
    cfg = dict(time_horizon=2, reset_noise_xy=0.02, reset_noise_yaw=0.4, seed=11)
    gen = torch.Generator(device="cuda").manual_seed(5)
    tape = torch.rand((K + 1, N, 6), device="cuda", generator=gen) * 2 - 1
    ref_sim = _sim(SCENES, N, **cfg)
    ref_sim.reset()  # AsyncGripperEnv.async_reset resets once more: the episode counter of the reset noise must match
    fields = ("obs", "reward", "done", "info", "achieved_goal", "desired_goal")
    ref = {f: [] for f in fields + ("terminal_obs",)}
    for k in range(K):
        ref_sim.step(tape[k])
        for f in ref:
            ref[f].append(getattr(ref_sim, f).clone())
    ref = {f: torch.stack(v) for f, v in ref.items()}
    ref_sim.close()
    sim = _sim(SCENES, N, **cfg)
    pool = AsyncGripperEnv(sim, B)
    pool.async_reset()
    seen = np.zeros(N, np.int64)
    bad = {f: 0 for f in ref}
    recvs = 0
    while seen.min() <= K:
        assert recvs < 4 * N * (K + 1) // B + 50
        r = pool.recv()
        ids = r["env_id"].long()
        ids_h = ids.cpu().numpy()
        recvs += 1
        k = torch.as_tensor(seen[ids_h], device="cuda")
        m = (k >= 1) & (k <= K)
        if bool(m.any()):
            ks, es = k[m] - 1, ids[m]
            for f in fields:
                bad[f] += int((~_rows_equal(r[f][m], ref[f][ks, es])).sum())
            d = ref["done"][ks, es] != 0
            if bool(d.any()):
                bad["terminal_obs"] += int((~_rows_equal(r["terminal_obs"][m][d], ref["terminal_obs"][ks, es][d])).sum())
        seen[ids_h] += 1
        pool.send(tape[torch.clamp(k, max=K), ids], ids)
    pool.status()
    assert all(v == 0 for v in bad.values()), bad
    assert int(ref["done"].sum()) > 0 and sorted(set(ref["info"][..., OBJ].flatten().tolist())) == [0.0, 1.0, 2.0, 3.0]
    sim.close()


# ------------------------------------------------------------------------------------------------ SAC from a mixed pool
def test_sac_from_a_mixed_pool():
    import torch
    from mujoco_rl_manipulate_unknown_objects_b200 import make_config
    from mujoco_rl_manipulate_unknown_objects_b200.replay import DeviceReplayBuffer
    from mujoco_rl_manipulate_unknown_objects_b200.rollout import RolloutWorker
    from mujoco_rl_manipulate_unknown_objects_b200.sac import SACLearner
    N, B, CAP, R, K = 512, 128, 64, 8, len(SCENES)
    cfg = make_config(sim_env=[_path(s) for s in SCENES], her_buffer=True, time_horizon=4)
    w = RolloutWorker(cfg, envs_per_gpu=N, seed=0)
    rb = DeviceReplayBuffer(CAP, N, w.sim.obs_shape, w.sim.action_dim, her_reward=True, seed=0)
    learner = SACLearner(w, rb, batch_size=64, seed=1)
    w.start_async(B, replay=rb)
    first = torch.arange(N, device="cuda") % K
    w.collect_async(R, replay=rb)
    w.sim.set_next_objects((first + 1) % K)  # mid-collection: every environment switches at its next episode boundary
    for _ in range(3):
        w.collect_async(R, replay=rb)
    losses = learner.update(1)
    assert all(np.isfinite(v) for v in losses.values()), losses
    # every stored transition carries the variant of its own episode: n % K up to an episode end, (n + 1) % K after it
    rb.status()
    added = rb.added.cpu().numpy()
    assert int(added.max()) < CAP  # the ring has not wrapped: slot t holds transition t
    v = rb.info[..., OBJ].long().cpu().numpy()
    done = rb.done.cpu().numpy()
    switched = 0
    for n in range(N):
        a, b_ = n % K, (n + 1) % K
        seq = v[:added[n], n]
        assert set(seq.tolist()) <= {a, b_}, (n, seq)
        for t in range(1, len(seq)):
            if seq[t] != seq[t - 1]:
                assert (seq[t - 1], seq[t]) == (a, b_) and done[t - 1, n], (n, seq, done[:added[n], n])
                switched += 1
    assert switched > N // 2
    b = rb.sample(4096, 0.8, draw=1)
    assert bool((b["index"] >= 0).all())
    assert torch.equal(b["info"][:, OBJ].long(), rb.info[b["index"] // N, b["index"] % N, OBJ].long())
    w.pool.status()
    w.close()
    rb.close()


# ------------------------------------------------------------------------------------------------ create errors
def test_create_refuses_bad_scene_lists():
    import ctypes as C
    from mujoco_rl_manipulate_unknown_objects_b200 import _native
    from mujoco_rl_manipulate_unknown_objects_b200.config import scene_path
    from mujoco_rl_manipulate_unknown_objects_b200 import make_config
    from mujoco_rl_manipulate_unknown_objects_b200.sim import NativeError, _grs_config
    lib = _native.load()
    cfg = _grs_config(make_config(), True)
    paths = [scene_path(_path(s)) for s in SCENES] * 3

    def create(ps):
        arr = (C.c_char_p * max(1, len(ps)))(*[p.encode() for p in ps])
        return lib.grs_create_scenes(arr, len(ps), 8, C.byref(cfg), 0)

    assert create([]) is None and b"1..8 scenes" in lib.grs_last_error()
    assert create(paths[:9]) is None and b"1..8 scenes" in lib.grs_last_error()
    h = create(paths[:8])  # MAXOBJ variants (repeats allowed)
    assert h, _native.last_error()
    assert lib.grs_num_scenes(h) == 8
    lib.grs_destroy(h)
    box = scene_path("/xmls/gripper_two_fingers.xml")
    assert create([paths[0], box]) is None
    msg = _native.last_error()
    m = re.search(r"gripper_two_fingers\.xml cannot share a simulator with .*sugar_cube_env\.xml: ([\w:]+) differs", msg)
    assert m, msg
    from mujoco_rl_manipulate_unknown_objects_b200 import GripperSim
    with pytest.raises(NativeError, match="differs"):  # the same through the Python constructor
        GripperSim(make_config(sim_env=[_path("sugar_cube"), "/xmls/gripper_two_fingers.xml"]), num_envs=8)


# ------------------------------------------------------------------------------------------------ VecEnv info key
def test_vecenv_object_id_info_key():
    from mujoco_rl_manipulate_unknown_objects_b200 import BatchedRobotVecEnv, make_config
    N = 16
    for scenes in (list(SCENES[:2]), SCENES[0]):
        env_cfg = [_path(s) for s in scenes] if isinstance(scenes, list) else _path(scenes)
        env = BatchedRobotVecEnv(make_config(sim_env=env_cfg, time_horizon=2), num_envs=N)
        env.reset()
        rng = np.random.default_rng(0)
        for _ in range(3):
            _, _, _, infos = env.step(rng.uniform(-1, 1, (N, 6)).astype(np.float32))
            rows = env.last_info_rows
            for i in range(N):
                if isinstance(scenes, list):
                    assert infos[i]["object_id"] == int(rows[i, OBJ]) == i % 2
                else:
                    assert "object_id" not in infos[i]
        env.close()
