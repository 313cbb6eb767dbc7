"""AsyncGripperEnv — EnvPool-style asynchronous stepping (`async_reset` / `send` / `recv`) over a GripperSim.

A synchronous step over N environments lasts as long as its longest chain of substeps.  Here the pool holds N environments
and `recv()` returns the first B (the batch size) whose agent steps have completed; environments still mid-step are parked
at a substep boundary and continue in a later `recv()` (DESIGN.md §3.1 "Asynchronous step").  Results are bit-identical to
the synchronous step of the same environment with the same actions.

All of it runs on the device, on torch's current stream, without host synchronisation: `send` and `recv` only enqueue work.
Invalid ids in `send` (not returned, duplicated, out of range) and a `recv` with fewer than B environments in flight set a
sticky error on the device that the next `status()` or `async_end()` raises.  While asynchronous mode is on, the simulator's
synchronous calls (step, reset, substep, set_state) raise.
"""
import ctypes as C

from .sim import NativeError, _check

STATES = ("returned", "pending", "parked", "ready")


class AsyncGripperEnv:
    """EnvPool's asynchronous interface over `sim` (a GripperSim created with auto_reset=True), batch size `batch_size`."""

    def __init__(self, sim, batch_size):
        if not 1 <= int(batch_size) <= sim.num_envs:
            raise ValueError("batch_size must be within 1..%d" % sim.num_envs)
        self.sim = sim
        self.batch_size = int(batch_size)
        self.num_envs = sim.num_envs
        self.action_dim = sim.action_dim
        self._lib, self._h, self._torch = sim._lib, sim._h, sim._torch
        self._on = False

    def async_reset(self):
        """Resets every environment (EnvPool async_reset); the first num_envs / batch_size recv() calls return them in id
        order, with their reset observations."""
        if self._on:
            self.async_end()
        self.sim.reset()
        _check(self._lib.grs_async_begin(self._h, self.batch_size, self.sim._stream()))
        self._on = True

    def send(self, actions, env_ids):
        """actions [n, action_dim] float32 and env_ids [n] (ids from earlier recv() calls) on the simulator's device."""
        t = self._torch
        actions = actions.to(device=self.sim.device, dtype=t.float32).contiguous()
        env_ids = env_ids.to(device=self.sim.device, dtype=t.int32).contiguous()
        n = env_ids.numel()
        if tuple(actions.shape) != (n, self.action_dim):
            raise ValueError("actions must have shape (%d, %d), got %s" % (n, self.action_dim, tuple(actions.shape)))
        _check(self._lib.grs_async_send(self._h, C.c_void_p(actions.data_ptr()), C.c_void_p(env_ids.data_ptr()), n, self.sim._stream()))

    def recv(self):
        """The next batch_size finished environments: a dict of device tensors with a leading dimension of batch_size,
        `env_id` (int32, completion order), `obs`, `reward`, `done`, `info`, `achieved_goal`, `desired_goal` and
        `terminal_obs` (meaningful where done).  They are copies, gathered from the simulator's per-environment buffers by
        id with torch indexing: one index_select per field, which moves 2 x batch_size observations (20 KB each at
        5 x 64 x 64) plus 181 bytes of the other fields per environment and costs a few kernel launches."""
        s = self.sim
        ids = self._torch.empty(self.batch_size, dtype=self._torch.int32, device=s.device)
        _check(self._lib.grs_async_recv(self._h, C.c_void_p(ids.data_ptr()), s._stream()))
        gi = ids.clamp(min=0)  # -1 marks a missing entry (reported by status()); it must not index out of bounds
        g = lambda x: x.index_select(0, gi)  # noqa: E731
        return dict(env_id=ids, obs=g(s.obs), reward=g(s.reward), done=g(s.done), info=g(s.info), achieved_goal=g(s.achieved_goal),
                    desired_goal=g(s.desired_goal), terminal_obs=g(s.terminal_obs))

    def status(self):
        """Synchronises and returns the number of environments in each state; raises NativeError if an earlier send or
        recv was invalid (the error is cleared by reporting it)."""
        counts = (C.c_int64 * 5)()
        _check(self._lib.grs_async_status(self._h, counts))
        return dict(zip(STATES, (int(c) for c in counts[:4])))

    def async_end(self):
        """Leaves asynchronous mode; every environment must have been received (none pending, parked or ready)."""
        _check(self._lib.grs_async_end(self._h))
        self._on = False

    @property
    def async_state(self):
        """int32 [num_envs] view of the per-environment state (0 returned, 1 pending, 2 parked, 3 ready)."""
        return self.sim._tensor("async_state", (self.num_envs,), "<i4")


__all__ = ["AsyncGripperEnv", "NativeError", "STATES"]
