"""GPU: size-independent properties at BASELINE.json's full batch sizes (4 096 and 8 192 environments per GPU), where
the fp64 oracle is too slow to follow.

* scheduling independence: which warp / block / wave integrates an environment and in which order environments leave the
  work queue (longest-first order; a permutation of the environments moves each to another queue position, warp and
  block) must not change a single bit of any output;
* determinism: two runs of the same action tape are bit-identical; identical environments stay identical;
* host path: grs_step_host into pageable and into pinned host arrays returns what the device step computes, bit for bit;
* conservation-style sanity: every environment takes between 1 and 3 x max_steps substeps, finite state, rewards in
  the progress reward's range [0, 3] (reward.py:18-41 with the unreachable bonus gate), done only on the time limit
  or FAIL.
"""
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _run(n, scene, steps, env=None, seed=0, perm=None):
    """`steps` agent steps of a seeded action tape; with `perm`, environment j takes the actions of environment perm[j]"""
    import torch
    from mujoco_rl_manipulate_unknown_objects_b200 import GripperSim, make_config
    old = {k: os.environ.get(k) for k in (env or {})}
    os.environ.update(env or {})
    try:
        sim = GripperSim(make_config(sim_env="/xmls/%s_env.xml" % scene), num_envs=n, auto_reset=True)
    finally:
        for k, v in old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v
    gen = torch.Generator(device="cuda").manual_seed(seed)
    out = []
    for _ in range(steps):
        a = torch.rand((n, 6), device="cuda", generator=gen) * 2 - 1
        sim.step(a if perm is None else a[perm])
        out.append(dict(obs=sim.obs.clone(), reward=sim.reward.clone(), done=sim.done.clone(), info=sim.info.clone(), state=sim.state.clone(),
                        ag=sim.achieved_goal.clone(), tobs=sim.terminal_obs.clone()))
    sim.close()
    return out


@pytest.mark.parametrize("n,scene", [(4096, "acorn"), (8192, "sugar_cube"), (16384, "sand_ball")])  # BASELINE.json configs[1], [2], [4]
def test_results_do_not_depend_on_scheduling(n, scene):
    import torch
    steps = 4 if n <= 8192 else 3
    base = _run(n, scene, steps)
    # permuted environments: with the default (zero) reset noise a reset does not depend on the environment id, so environment
    # j of the second run is environment perm[j] of the first, now at another queue position and in another warp and block
    perm = torch.randperm(n, generator=torch.Generator().manual_seed(7)).cuda()
    other = _run(n, scene, steps, perm=perm)
    for t in range(steps):
        for k in base[t]:
            assert torch.equal(base[t][k][perm], other[t][k]), "%s differs at step %d with the environments permuted" % (k, t)
    # GRS_GAP_SKIP=0 evaluates every cached separating axis instead of skipping those whose separation budget is still positive
    # (sim_kernels.cuh : collision) — the skip is exact, so not a bit may change
    other = _run(n, scene, steps, dict(GRS_GAP_SKIP="0"))
    for t in range(steps):
        for k in base[t]:
            assert torch.equal(base[t][k], other[t][k]), "%s differs at step %d with GRS_GAP_SKIP=0" % (k, t)
    again = _run(n, scene, steps)
    for t in range(steps):
        for k in base[t]:
            assert torch.equal(base[t][k], again[t][k]), "run-to-run difference in %s at step %d" % (k, t)


def test_host_step_equals_device_step():
    """grs_step_host copies the outputs into pageable host arrays after the step kernel, while into pinned arrays the
    observation phase stores each image itself as it finishes.  Both must return what the device step leaves in its buffers.
    The copy of the terminal observations takes the done rows one by one when at most N/8 environments are done and the
    whole array otherwise; the tape reaches both (time_horizon=2, every 16th environment starts one step before it)."""
    import torch
    from mujoco_rl_manipulate_unknown_objects_b200 import GripperSim, make_config
    from mujoco_rl_manipulate_unknown_objects_b200._native import INFO as I
    n, th = 4096, 2
    sims = [GripperSim(make_config(sim_env="/xmls/acorn_env.xml", time_horizon=th), num_envs=n, auto_reset=True) for _ in range(3)]
    for s in sims:
        flags = s.get_state()["flags"]
        flags[::16, 1] = th - 1  # episode step
        s.set_state(flags=flags)
    Cc, H, W = sims[0].obs_shape

    def host_arrays(alloc):
        return dict(obs=alloc((n, Cc, H, W), np.uint8), achieved=alloc((n, 2), np.float32), desired=alloc((n, 2), np.float32),
                    reward=alloc((n,), np.float32), done=alloc((n,), np.uint8), info=alloc((n, I["STRIDE"]), np.float32),
                    terminal_obs=alloc((n, Cc, H, W), np.uint8))
    pageable = host_arrays(np.zeros)
    pinned = host_arrays(lambda shape, dt: torch.from_numpy(np.zeros(shape, dt)).pin_memory().numpy())
    rng = np.random.default_rng(5)
    ndone = []
    for t in range(2):
        a = (rng.random((n, 6), dtype=np.float32) * 2 - 1) * 0.3
        sims[0].step_host(a, **pageable)
        sims[1].step_host(a, **pinned)
        dev = sims[2]
        dev.step(torch.from_numpy(a).cuda())
        ref = dict(obs=dev.obs, achieved=dev.achieved_goal, desired=dev.desired_goal, reward=dev.reward, done=dev.done, info=dev.info)
        ref = {k: v.cpu().numpy() for k, v in ref.items()}
        done = ref["done"] != 0
        ndone.append(int(done.sum()))
        tobs = dev.terminal_obs.cpu().numpy()
        for name, h in (("pageable", pageable), ("pinned", pinned)):
            for k, v in ref.items():
                assert h[k].tobytes() == v.tobytes(), "%s differs at step %d (%s host arrays)" % (k, t, name)
            assert np.array_equal(h["terminal_obs"][done], tobs[done]), "terminal_obs differs at step %d (%s host arrays)" % (t, name)
    assert ndone[0] <= n // 8 < ndone[1], "the tape missed a terminal-observation copy branch: %s environments done" % ndone
    for s in sims:
        s.close()


def test_separation_budget_skip_is_exact():
    """sim_kernels.cuh : collision skips a convex pair while the separation measured along its cached axis, minus how far the two
    geoms can have moved since, stays positive.  That is a proof that the axis still separates them, so the contact sets — and
    with them every bit of the trajectory — must equal those of the kernel that evaluates the axis every substep.  40 agent
    steps of contact-seeking actions (grippers push and squeeze the objects, fingers press against each other)."""
    import torch
    from mujoco_rl_manipulate_unknown_objects_b200 import GripperSim, make_config
    n, steps = 2048, 40
    res = []
    for skip in ("1", "0"):
        os.environ["GRS_GAP_SKIP"] = skip
        try:
            sim = GripperSim(make_config(sim_env="/xmls/bread_crumb_env.xml"), num_envs=n, auto_reset=True)
        finally:
            os.environ.pop("GRS_GAP_SKIP", None)
        gen = torch.Generator(device="cuda").manual_seed(3)
        snap = []
        for t in range(steps):
            a = torch.rand((n, 6), device="cuda", generator=gen) * 2 - 1
            a[:, 0] = 0.6 + 0.4 * a[:, 0]
            a[:, 5] = torch.where(torch.arange(n, device="cuda") % 3 == 0, a[:, 5], -a[:, 5].abs())
            sim.step(a)
            if t % 8 == 7:
                snap.append((sim.state.clone(), sim.info.clone(), sim.reward.clone(), sim.obs[::64].clone()))
        res.append(snap)
        sim.close()
    from mujoco_rl_manipulate_unknown_objects_b200._native import INFO as I
    assert float(res[0][-1][1][:, I["NCON_MAX"]].mean()) > 2.5, "the tape did not bring the batch into contact"
    for a, b in zip(*res):
        for x, y in zip(a, b):
            assert torch.equal(x, y)


def test_full_batch_sanity():
    import torch
    from mujoco_rl_manipulate_unknown_objects_b200._native import INFO as I
    n = 4096
    out = _run(n, "acorn", 6, seed=5)
    for t, o in enumerate(out):
        info = o["info"].cpu().numpy()
        ns = info[:, I["NSUB_A"]:I["NSUB_A"] + 3]
        assert (ns.sum(1) >= 1).all() and (ns <= 400).all()  # robot_env.py:97-168: each phase is capped by max_steps
        assert np.isfinite(o["state"].cpu().numpy()).all()
        r = o["reward"].cpu().numpy()
        assert (r >= 0).all() and (r <= 3.0 + 1e-5).all()
        done = o["done"].cpu().numpy().astype(bool)
        status = info[:, I["STATUS"]].astype(int)
        assert ((status != 0) == done).all()  # RUNNING <=> not done
        pad = o["obs"][:, 4].cpu().numpy()
        assert (pad[:, 0, 2:] == 0).all() and (pad[:, 1:] == 0).all() and (pad[:, 0, :2] <= 3).all()  # robot_env.py:283-288
    # identical environments (same reset, same action) stay bit-identical: tile one action over the batch
    from mujoco_rl_manipulate_unknown_objects_b200 import GripperSim, make_config
    sim = GripperSim(make_config(sim_env="/xmls/acorn_env.xml"), num_envs=n)
    a = torch.tensor([[0.9, 0.1, -0.2, 0.3, -0.4, -1.0]], device="cuda").repeat(n, 1)
    for _ in range(3):
        sim.step(a)
    assert bool((sim.state == sim.state[0]).all()) and bool((sim.obs == sim.obs[0]).all()) and bool((sim.reward == sim.reward[0]).all())
    sim.close()
