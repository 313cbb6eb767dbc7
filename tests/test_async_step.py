"""GPU: the asynchronous step (AsyncGripperEnv, C-ABI grs_async_*).

* bit-exactness per environment: environment e's k-th transition from the pool equals row e of the k-th synchronous step
  with the same action, in every output, however often the pool parked and resumed it;
* protocol: recv returns `batch` distinct returned ids, the state counts always cover the pool, no environment starves,
  a recv with enough ready environments steps nothing, invalid sends are reported, synchronous calls are refused while
  environments are in flight and work again after draining.
"""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

FIELDS = ("obs", "reward", "done", "info", "achieved_goal", "desired_goal")


def _sim(scene, n, **cfg):
    from mujoco_rl_manipulate_unknown_objects_b200 import GripperSim, make_config
    return GripperSim(make_config(sim_env="/xmls/%s_env.xml" % scene, **cfg), num_envs=n, auto_reset=True)


def _bits(x):
    import torch
    return x.view(torch.int32) if x.dtype == torch.float32 else x


def _sync_reference(scene, n, tape, cfg):
    sim = _sim(scene, n, **cfg)
    sim.reset()  # AsyncGripperEnv.async_reset resets once more: with reset noise the episode counter must match
    ref = {k: [] for k in FIELDS + ("terminal_obs",)}
    for k in range(tape.shape[0] - 1):
        sim.step(tape[k])
        for f, x in (("obs", sim.obs), ("reward", sim.reward), ("done", sim.done), ("info", sim.info), ("achieved_goal", sim.achieved_goal),
                     ("desired_goal", sim.desired_goal), ("terminal_obs", sim.terminal_obs)):
            ref[f].append(x.clone())
    sim.close()
    return {f: __import__("torch").stack(v) for f, v in ref.items()}


CASES = [("acorn", 4096, 1024, {}), ("acorn", 512, 64, {}), ("acorn", 512, 1, {}), ("acorn", 512, 512, {}), ("sugar_cube", 512, 64, {}),
         ("sugar_cube", 512, 16, dict(im_reward=True, reset_noise_xy=0.02, reset_noise_yaw=0.4, direction=45, seed=11))]


@pytest.mark.parametrize("scene,n,batch,extra", CASES, ids=["%s-%d-%d%s" % (c[0], c[1], c[2], "-im-noise-45" if c[3] else "") for c in CASES])
def test_async_transitions_equal_synchronous_steps(scene, n, batch, extra):
    """A fixed action tape tape[k, e]; environment e's k-th send uses tape[k, e].  Its first K returned transitions must be
    bit-equal to row e of the synchronous steps 1..K (time_horizon=2, so auto-resets and terminal observations are covered).
    The synchronous step builds its observations in the step kernel's fused observation phase, the pool with the standalone
    observation kernel (k_render_obs_indexed), so this also holds the two observation paths against each other, terminal_obs
    included."""
    import torch
    from mujoco_rl_manipulate_unknown_objects_b200 import AsyncGripperEnv
    K = 4
    cfg = dict(time_horizon=2, **extra)
    gen = torch.Generator(device="cuda").manual_seed(5)
    tape = torch.rand((K + 1, n, 6), device="cuda", generator=gen) * 2 - 1
    ref = _sync_reference(scene, n, tape, cfg)
    sim = _sim(scene, n, **cfg)
    pool = AsyncGripperEnv(sim, batch)
    pool.async_reset()
    seen = np.zeros(n, np.int64)  # transitions received per environment (the first one is the reset observation)
    bad = {f: 0 for f in FIELDS + ("terminal_obs",)}
    parked_max = 0
    recvs = 0
    limit = 4 * n * (K + 1) // batch + 50  # FIFO: every environment's K + 1 transitions arrive within a small multiple of the minimum
    while seen.min() <= K:
        assert recvs < limit, "environments %s still have fewer than %d transitions after %d recvs" % (np.flatnonzero(seen <= K)[:8], K + 1, recvs)
        r = pool.recv()
        ids = r["env_id"].long()
        ids_h = ids.cpu().numpy()
        recvs += 1
        assert len(set(ids_h.tolist())) == batch and ids_h.min() >= 0
        parked_max = max(parked_max, int((pool.async_state == 2).sum()))
        k = torch.as_tensor(seen[ids_h], device="cuda")
        m = (k >= 1) & (k <= K)
        if bool(m.any()):
            ks, es = k[m] - 1, ids[m]
            for f in FIELDS:
                bad[f] += int((~(_bits(r[f][m]) == _bits(ref[f][ks, es])).reshape(int(m.sum()), -1).all(1)).sum())
            d = ref["done"][ks, es] != 0
            if bool(d.any()):
                bad["terminal_obs"] += int((~(r["terminal_obs"][m][d] == ref["terminal_obs"][ks, es][d]).reshape(int(d.sum()), -1).all(1)).sum())
        seen[ids_h] += 1
        pool.send(tape[torch.clamp(k, max=K), ids], ids)
    pool.status()  # raises on any error the device recorded
    assert all(v == 0 for v in bad.values()), "rows that differ from the synchronous step: %s (after %d recvs)" % (bad, recvs)
    assert int(ref["done"].sum()) > 0
    if batch < n:
        assert parked_max > 0, "no environment was ever parked: the test did not exercise resuming"
    sim.close()


def test_async_protocol():
    import torch
    from mujoco_rl_manipulate_unknown_objects_b200 import AsyncGripperEnv
    from mujoco_rl_manipulate_unknown_objects_b200.sim import NativeError
    N, B, max_steps = 256, 32, 50
    sim = _sim("sugar_cube", N, max_steps=max_steps, time_horizon=20)
    with pytest.raises(ValueError):
        AsyncGripperEnv(sim, N + 1)
    assert sim._lib.grs_async_begin(sim._h, N + 1, None) != 0
    pool = AsyncGripperEnv(sim, B)
    pool.async_reset()
    gen = torch.Generator(device="cuda").manual_seed(1)
    act = lambda m: torch.rand((m, sim.action_dim), device="cuda", generator=gen) * 2 - 1  # noqa: E731

    # the first N / B recvs hand out the reset environments in id order; with B ready, a recv steps nothing
    r0 = pool.recv()["env_id"]
    assert torch.equal(r0.cpu(), torch.arange(B, dtype=torch.int32))
    pool.send(act(B), r0)
    assert pool.status() == dict(returned=0, pending=B, parked=0, ready=N - B)
    r1 = pool.recv()["env_id"]
    assert torch.equal(r1.cpu(), torch.arange(B, 2 * B, dtype=torch.int32))
    assert pool.status() == dict(returned=B, pending=B, parked=0, ready=N - 2 * B), "a recv with B ready environments stepped"

    # invalid sends: a pending id, a duplicated id, an id out of range -> reported by the next synchronising call
    pool.send(act(1), r0[:1])
    with pytest.raises(NativeError, match="not in the returned state"):
        pool.status()
    pool.send(act(2), torch.stack([r1[0], r1[0]]))
    with pytest.raises(NativeError, match="not in the returned state"):
        pool.status()
    pool.send(act(1), torch.tensor([N], dtype=torch.int32))
    with pytest.raises(NativeError, match="out of range"):
        pool.status()
    assert pool.status()["pending"] == B + 1  # r1[0] went through once
    pool.send(act(B - 1), r1[1:])

    # synchronous calls are refused while the pool is in use
    with pytest.raises(NativeError, match="asynchronous mode"):
        sim.step(act(N))
    with pytest.raises(NativeError, match="asynchronous mode"):
        sim.reset()
    with pytest.raises(NativeError, match="asynchronous mode"):
        sim.substep(1)
    with pytest.raises(NativeError, match="receive them all first"):
        pool.async_end()

    # steady state: B distinct returned ids per recv, counts cover the pool, nobody starves
    last = np.full(N, -1)
    last[:2 * B] = [0] * B + [1] * B
    gap = 0
    parked = 0
    for j in range(2, 400):
        ids = pool.recv()["env_id"]
        ids_h = ids.cpu().numpy()
        assert len(set(ids_h.tolist())) == B and ids_h.min() >= 0
        st = pool.async_state.cpu().numpy()
        assert np.all(st[ids_h] == 0), "a returned id is not in the returned state"
        counts = pool.status()
        assert sum(counts.values()) == N and counts["returned"] == B
        parked = max(parked, counts["parked"])
        gap = max(gap, int((j - last[ids_h]).max()))
        last[ids_h] = j
        pool.send(act(B), ids)
    # an environment in flight gains >= 1 substep in every launch that steps (all of them fit on the grid at once) and its
    # agent step has <= 3 x max_steps substeps; after that it waits behind at most N / B batches of the FIFO
    bound = 4 * max_steps + 2 * N // B
    assert last.min() >= 0 and (399 - last).max() <= bound, "an environment starved"
    assert gap <= bound, gap
    assert parked > 0

    # drain: receive without sending until nothing is in flight, then the synchronous calls work again
    while True:
        c = pool.status()
        if c["pending"] + c["parked"] + c["ready"] == 0:
            break
        pool.recv()
    pool.async_end()
    sim.step(act(N))
    sim.reset()
    sim.synchronize()
    sim.close()
