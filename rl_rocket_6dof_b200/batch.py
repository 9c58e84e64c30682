"""Rocket6DOFBatch — N independent Rocket6DOF environments resident on one B200.

Mirrors the reference's gym contract (`reset()` / `step(a)` / observation / reward / done,
/root/reference/my_environment/envs/rocket_env.py:180-231) for a whole batch: state lives in HBM
as component-major float64 [14][N]; every call enqueues one hand-written CUDA kernel through the
C ABI (include/r6dof.h) on the current torch stream.  torch is plumbing only (allocation, streams).
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional

import numpy as np
import torch

from . import _lib
from ._lib import R6Buffers, R6Mlp
from .params import EnvParams, derive_params, load_config

ACT_PHILOX, ACT_MLP, ACT_BUFFER, ACT_MLP_TC = 0, 1, 2, 3
F_EVENT, F_OOB, F_TRUNCATED = 0x01, 0x02, 0x04
F_LANDING_ALL = 0xF8
FLAG_NAMES = ["zero_height", "velocity_limit", "landing_radius", "attitude_limit", "omega_limit"]
SPLIT_MIN_ENVS = 65536
MULTIPASS_MIN_ENVS = 1 << 18   # smallest batch the multi-pass integrator is the default for (float64; float32: twice that)
#                                (profiles/r02_sweep_dispatch.json: 2^18 envs, two lanes: 120 vs 129 us per step)
STAT_NAMES = ["episodes", "return_sum", "length_sum", "landed", "ground", "out_of_bounds", "truncated", "steps"]


class Rocket6DOFBatch:
    """Batched env.  All tensors are CUDA tensors on `device`; nothing is computed on the host."""

    def __init__(self, num_envs: int, env_config: Optional[dict] = None, sb3_config: Optional[dict] = None, *,
                 device: str | torch.device = "cuda", seed: Optional[int] = None, auto_reset: bool = True,
                 clip_reward: bool = True, time_limit: bool = True, env_offset: int = 0,
                 num_envs_global: Optional[int] = None, debug_buffers: bool = False, record_attempts: bool = False,
                 ic_table: Optional[np.ndarray] = None, params: Optional[EnvParams] = None,
                 precision: str = "fp64", reward_annealing: bool = False, vertical_attitude_reward=None,
                 split_step: Optional[bool] = None, lanes: int = 1, multipass: Optional[bool] = None):
        if not torch.cuda.is_available():
            raise RuntimeError("Rocket6DOFBatch needs a CUDA device (no CPU fallback)")
        self.lib = _lib.load()
        if params is None:
            if env_config is None:
                sb3_config, env_config = load_config()
            params = derive_params(env_config, sb3_config)
        self.params = params
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise RuntimeError("Rocket6DOFBatch needs a CUDA device (no CPU fallback)")
        self.num_envs = int(num_envs)
        self.env_offset = int(env_offset)
        self.num_envs_global = int(num_envs_global if num_envs_global is not None else env_offset + num_envs)
        self.seed_value = int(params.seed if seed is None else seed)
        self.auto_reset = auto_reset
        if precision not in ("fp64", "fp32"):
            raise ValueError("precision must be 'fp64' (parity path) or 'fp32' (throughput path)")
        self.precision = precision
        self._struct_kw = dict(auto_reset=auto_reset, clip_reward=clip_reward, time_limit=time_limit,
                               precision=1 if precision == "fp32" else 0, reward_annealing=reward_annealing,
                               vertical_attitude_reward=vertical_attitude_reward)
        self._p = params.to_struct(**self._struct_kw)
        n, dev = self.num_envs, self.device
        f64, f32 = torch.float64, torch.float32
        sdt = f32 if precision == "fp32" else f64      # dtype of state / terminal_state (R6_PREC_*)
        with torch.cuda.device(dev):
            self.state = torch.zeros(14, n, dtype=sdt, device=dev)
            self.m0 = torch.zeros(n, dtype=f32, device=dev)
            self.v0 = torch.zeros(n, dtype=f32, device=dev)
            self.step_count = torch.zeros(n, dtype=torch.int32, device=dev)
            self.episode_id = torch.zeros(n, dtype=torch.int32, device=dev)     # uint32 on the device side
            self.ep_return = torch.zeros(n, dtype=f64, device=dev)
            self.obs = torch.zeros(14, n, dtype=f32, device=dev)
            self.reward = torch.zeros(n, dtype=f64, device=dev)
            self.reward_f32 = torch.zeros(n, dtype=f32, device=dev)
            self.done = torch.zeros(n, dtype=torch.uint8, device=dev)
            self.flags = torch.zeros(n, dtype=torch.uint8, device=dev)
            self.terminal_obs = torch.zeros(14, n, dtype=f32, device=dev)
            self.terminal_state = torch.zeros(14, n, dtype=sdt, device=dev)
            self.ep_info = torch.zeros(2, n, dtype=f64, device=dev)       # (return, length) of the finished episode
            self.tgo = torch.zeros(n, dtype=f32, device=dev)              # warm start of the t_go root iteration
            self.stats = torch.zeros(8, dtype=f64, device=dev)
            # r6_step as two kernels (integrator | post-step) needs 2 bytes of device scratch per env; two launches
            # only pay off once the grid fills the machine several times over (measured cross-over: 2^16..2^17 envs)
            if split_step is None:
                env_flag = os.environ.get("R6_SPLIT_STEP")
                split_step = (n > SPLIT_MIN_ENVS) if env_flag is None else (env_flag != "0")
            # stream lanes: `step` / `step_random` run the kernel pair on `lanes` contiguous env sub-ranges, each on
            # its own stream, so one range's kernel tails (the integrator grid is ~18 waves of one-warp CTAs of
            # uneven length) are covered by the next range's work: 0.468 -> 0.430 ms per 2^20-env step free-running,
            # 0.454 ms when every step is joined back into the caller's stream (profiles/two_stream_shards.py)
            self.lanes = max(int(lanes), 1)
            if self.lanes > 1:
                if n < self.lanes or self.lanes > 32:          # R6_MAX_LANES
                    raise ValueError("lanes must be <= min(num_envs, 32)")
                split_step = True
                self._lane_streams = [torch.cuda.Stream(device=dev) for _ in range(self.lanes)]
                self._lane_fork = torch.cuda.Event()
            base, rem = divmod(n, self.lanes)           # one contiguous env sub-range (first, count) per lane
            self._lane_ranges = [(r * base + min(r, rem), base + (1 if r < rem else 0)) for r in range(self.lanes)]
            self._lanes_pending = False
            self.scratch = torch.zeros(2, n, dtype=torch.uint8, device=dev) if split_step else None
            # multi-pass integrator (R6Buffers.work): one RK attempt per pass, unfinished envs compacted into work
            # lists for the next pass; on with the kernel pair for large batches unless asked otherwise (below 2^19 envs
            # the four small launches cost more than the idle lanes did).  Round 2: with the one-attempt pass kernels it
            # also pays on the float32 path (0.263 -> 0.236 ms per 2^20-env step) — profiles/r02_fp32_multipass.txt
            if multipass is None:
                env_flag = os.environ.get("R6_MULTIPASS")
                multipass = ((split_step and n >= MULTIPASS_MIN_ENVS * (2 if precision == "fp32" else 1)) if env_flag is None
                             else (env_flag != "0" and split_step))
            if multipass and not split_step:
                raise ValueError("multipass needs the split step (split_step=True)")
            self.work = None
            if multipass:                  # 544 B per env of work records; only the list counters (first 256 B) start at zero
                self.work = torch.empty(int(self.lib.r6_work_bytes(n)), dtype=torch.uint8, device=dev)
                self.work[:256].zero_()
            self.t_table = torch.from_numpy(np.ascontiguousarray(params.t_table)).to(dev)
            self.reward_terms = torch.zeros(7, n, dtype=f64, device=dev) if debug_buffers else None
            self.nattempts = torch.zeros(n, dtype=torch.uint8, device=dev) if (debug_buffers or record_attempts) else None
            self.status = torch.zeros(n, dtype=torch.int8, device=dev) if debug_buffers else None
            self.ic_table = None
            if ic_table is not None:
                self.ic_table = torch.from_numpy(np.ascontiguousarray(ic_table, np.float32).reshape(-1, 14)).to(dev)
        self._b = self._make_buffers()
        self.steps_done = 0          # global step counter (Philox action stream)

    # ------------------------------------------------------------------ plumbing
    def _make_buffers(self) -> R6Buffers:
        def ptr(t):
            return 0 if t is None else t.data_ptr()
        b = R6Buffers()
        b.state, b.m0, b.v0 = ptr(self.state), ptr(self.m0), ptr(self.v0)
        b.step_count, b.episode_id, b.ep_return = ptr(self.step_count), ptr(self.episode_id), ptr(self.ep_return)
        b.obs, b.reward, b.done, b.flags = ptr(self.obs), ptr(self.reward), ptr(self.done), ptr(self.flags)
        b.terminal_obs, b.terminal_state = ptr(self.terminal_obs), ptr(self.terminal_state)
        b.reward_terms, b.nattempts, b.status = ptr(self.reward_terms), ptr(self.nattempts), ptr(self.status)
        b.ep_info = ptr(self.ep_info)
        b.reward_f32 = ptr(self.reward_f32)
        b.t_table = ptr(self.t_table)
        b.ic_table = ptr(self.ic_table)
        b.ic_table_len = 0 if self.ic_table is None else self.ic_table.shape[0]
        b.n_global = self.num_envs_global
        b.stats = ptr(self.stats)
        b.scratch = ptr(self.scratch)
        b.work = ptr(self.work)
        b.tgo = ptr(self.tgo)
        return b

    def _stream(self) -> int:
        return torch.cuda.current_stream(self.device).cuda_stream

    # ------------------------------------------------------------------ stream lanes
    def _fork(self, actions: Optional[torch.Tensor] = None, mlp: Optional[dict] = None) -> list:
        """(lane, first, count, stream) for every lane; with one lane the whole batch on the caller's stream.  With lanes,
        every lane stream first waits for what the caller's stream has enqueued so far (the producer of `actions`, the
        previous joined step), and the caller's tensors the lanes read (`actions`, the weights in `mlp`) are recorded on
        every lane stream, so that the allocator does not hand their memory out again before the lanes are done with it
        (the caller may drop them before `join()`)."""
        streams = [torch.cuda.current_stream(self.device)]
        if self.lanes > 1:
            self._lane_fork.record(streams[0])
            streams = self._lane_streams
            reads = [t for t in [actions, *(mlp or {}).values()] if isinstance(t, torch.Tensor)]
            for st in streams:
                st.wait_event(self._lane_fork)
                for t in reads:
                    t.record_stream(st)
        return [(ln, first, count, st) for ln, ((first, count), st) in enumerate(zip(self._lane_ranges, streams))]

    def _advance(self, k: int, join: bool = True):
        """Counts k env-steps issued by `_fork`'s schedule; with lanes they are pending until `join()`."""
        self.steps_done += k
        if self.lanes > 1:
            self._lanes_pending = True
            if join:
                self.join()

    def _env_step(self, lane: int, first: int, count: int, actions: int, step_index: int, stream: torch.cuda.Stream):
        """One env-step of envs [first, first + count) on `stream`; `actions` is a device pointer, 0 for in-kernel Philox
        actions of step `step_index`.  With lanes, the kernel pair on the lane's sub-range; on one stream, r6_step (which
        picks the fused kernel, the kernel pair or the multi-pass integrator) or the random-action kernel pair."""
        L, p, b, s = self.lib, C.byref(self._p), C.byref(self._b), stream.cuda_stream
        if self.lanes > 1:
            rc = L.r6_step_range(p, b, self.num_envs, first, count, lane, self.env_offset, actions, self.seed_value,
                                 step_index, s)
        elif actions:
            rc = L.r6_step(p, b, self.num_envs, self.env_offset, actions, self.seed_value, s)
        else:
            rc = L.r6_step_random(p, b, self.num_envs, self.env_offset, self.seed_value, step_index, s)
        _lib.check(rc, L)

    def _policy(self, m: R6Mlp, obs: int, first: int, count: int, tensor_cores, stochastic: bool, step_index: int,
                act: int, raw: Optional[int], val: Optional[int], logp: Optional[int], stream: torch.cuda.Stream):
        """The policy network over envs [first, first + count) of the component-major observations at device pointer
        `obs` (r6_policy_range); the output pointers raw / val / logp may be None (not written)."""
        _lib.check(self.lib.r6_policy_range(C.byref(m), obs, self.num_envs, first, count, int(tensor_cores),
                                            int(bool(stochastic)), self.seed_value, self.env_offset, step_index, act, raw,
                                            val, logp, stream.cuda_stream), self.lib)

    def join(self):
        """Orders everything the lanes have been given before whatever the caller's current stream does next.  A no-op
        without lanes or when nothing is pending; every method other than `step(..., join=False)`,
        `step_random(..., join=False)` and `step_policy(..., join=False)` joins by itself."""
        if self._lanes_pending:
            cur = torch.cuda.current_stream(self.device)
            for st in self._lane_streams:
                cur.wait_stream(st)
            self._lanes_pending = False

    # ------------------------------------------------------------------ gym-like API (batched)
    def seed(self, seed: int):
        self.seed_value = int(seed)
        return [seed]

    def reset(self, mask: Optional[torch.Tensor] = None) -> torch.Tensor:
        """Rocket6DOF.reset for every env (or those with mask != 0). Returns obs [14, N] (view)."""
        self.join()
        mp = 0
        if mask is not None:
            mask = mask.to(device=self.device, dtype=torch.uint8).contiguous()
            mp = mask.data_ptr()
        with torch.cuda.device(self.device):
            _lib.check(self.lib.r6_reset(C.byref(self._p), C.byref(self._b), self.num_envs, self.env_offset, mp,
                                         self.seed_value, self._stream()), self.lib)
        return self.obs

    def step(self, actions: torch.Tensor, *, join: bool = True):
        """actions: float32 CUDA tensor [N, 3] in [-1, 1].  Returns (obs[14,N], reward[N], done[N], flags[N])
        as views of the persistent output tensors (valid until the next call).  With stream lanes, join=False leaves
        the step running on the lane streams (the outputs are ordered on the caller's stream only after `join()`), so
        consecutive steps pipeline; the default joins every step."""
        if actions.dtype != torch.float32 or not actions.is_cuda or actions.shape != (self.num_envs, 3):
            raise ValueError("actions must be a float32 CUDA tensor of shape [num_envs, 3]")
        actions = actions.contiguous()
        with torch.cuda.device(self.device):
            for ln, first, count, st in self._fork(actions):
                self._env_step(ln, first, count, actions.data_ptr(), self.steps_done, st)
        self._advance(1, join)
        return self.obs, self.reward, self.done, self.flags

    def rollout(self, k: int, mode: int = ACT_PHILOX, *, actions: Optional[torch.Tensor] = None,
                mlp: Optional[dict] = None, record: bool = False, fused: Optional[bool] = None):
        """k env-steps without a host round trip.  fused=True: one launch, state in registers for all k steps
        (`r6_rollout`).  For the random policy on large auto-reset batches the integrator | post-step kernel pair
        is faster than the fused kernel, so fused=None picks `step_random` there (same action stream, results equal to
        round-off); recording, other action sources and one-episode semantics always use the fused kernel."""
        self.join()
        if fused is None:
            fused = not (mode == ACT_PHILOX and not record and self.auto_reset and self.num_envs > SPLIT_MIN_ENVS)
        if not fused:
            if mode != ACT_PHILOX or record:
                raise ValueError("the split rollout exists for the random policy without recording")
            self.step_random(k)
            return None
        n = self.num_envs
        traj = None
        po = pa = pr = pd = 0
        if record:
            dev = self.device
            traj = dict(obs=torch.empty(k, 13, n, dtype=torch.float32, device=dev),
                        act=torch.empty(k, n, 3, dtype=torch.float32, device=dev),
                        rew=torch.empty(k, n, dtype=torch.float32, device=dev),
                        done=torch.empty(k, n, dtype=torch.uint8, device=dev))
            po, pa, pr, pd = (traj[x].data_ptr() for x in ("obs", "act", "rew", "done"))
        ab = 0
        if mode == ACT_BUFFER:
            if actions is None or actions.shape != (k, n, 3) or actions.dtype != torch.float32:
                raise ValueError("ACT_BUFFER needs float32 actions [k, N, 3]")
            actions = actions.contiguous()
            ab = actions.data_ptr()
        m = None
        if mode in (ACT_MLP, ACT_MLP_TC):
            if mlp is None:
                raise ValueError("ACT_MLP needs the policy weights")
            m = _lib.make_mlp(mlp)
        with torch.cuda.device(self.device):
            _lib.check(self.lib.r6_rollout(C.byref(self._p), C.byref(self._b), n, self.env_offset, int(k), int(mode),
                                           C.byref(m) if m is not None else None, ab, self.seed_value,
                                           self.steps_done, po, pa, pr, pd, self._stream()), self.lib)
        self.steps_done += int(k)
        return traj

    def step_random(self, k: int = 1, *, join: bool = True):
        """k env-steps with in-kernel Philox actions through the integrator | post-step kernel pair (2k launches).
        Same action stream and results as `rollout(k)`; faster for large batches, where the two specialised kernels
        beat the single fused one.  With stream lanes the k steps run free on the lanes and are joined at the end."""
        if self.scratch is None:                       # the random-action step exists only as the kernel pair
            self.scratch = torch.zeros(2, self.num_envs, dtype=torch.uint8, device=self.device)
            self._b.scratch = self.scratch.data_ptr()
        k = int(k)
        with torch.cuda.device(self.device):
            lanes = self._fork()
            for j in range(k):
                for ln, first, count, st in lanes:
                    self._env_step(ln, first, count, 0, self.steps_done + j, st)
        self._advance(k, join)
        return self.obs, self.reward, self.done, self.flags

    def policy_actions(self, mlp: dict, *, tensor_cores=False, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """Deterministic policy actions [N, 3] for the current observations (one policy launch).
        tensor_cores: False / 0 = float32 FMA network; True / 1 = mma.sync 3xTF32 tiles (faithful to 2e-6);
        2 = tcgen05 + TMEM single-pass TF32 (fast mode, ~1e-3); 3 = tcgen05 + TMEM 3xTF32 (faithful to 3e-6)."""
        self.join()
        if out is None:
            out = torch.empty(self.num_envs, 3, dtype=torch.float32, device=self.device)
        with torch.cuda.device(self.device):
            self._policy(_lib.make_mlp(mlp), self.obs.data_ptr(), 0, self.num_envs, tensor_cores, False, self.steps_done,
                         out.data_ptr(), None, None, None, torch.cuda.current_stream(self.device))
        return out

    def policy_forward(self, mlp: dict, *, stochastic: bool = False, tensor_cores=False, step_index: Optional[int] = None,
                       out: Optional[tuple] = None):
        """SB3 `ActorCriticPolicy.forward` for the current observations in one launch: returns
        (env_actions [N,3] clipped, raw_actions [N,3], values [N], log_prob [N]).  `mlp` may carry the critic head
        ("wv", "bv") and the Gaussian "log_std"; stochastic=True samples mean + exp(log_std) eps with Philox noise
        keyed by (seed, global env id, step_index) — reproducible and independent of the shard count."""
        self.join()
        n, dev = self.num_envs, self.device
        if out is not None:                      # (act, raw, val, logp) contiguous float32 CUDA tensors to write into
            act, raw, val, logp = out
        else:
            act = torch.empty(n, 3, dtype=torch.float32, device=dev)
            raw = torch.empty(n, 3, dtype=torch.float32, device=dev)
            val = torch.empty(n, dtype=torch.float32, device=dev)
            logp = torch.empty(n, dtype=torch.float32, device=dev)
        step = self.steps_done if step_index is None else int(step_index)
        with torch.cuda.device(dev):
            self._policy(_lib.make_mlp(mlp), self.obs.data_ptr(), 0, n, tensor_cores, stochastic, step, act.data_ptr(),
                         raw.data_ptr(), val.data_ptr(), logp.data_ptr(), torch.cuda.current_stream(dev))
        return act, raw, val, logp

    def collect_rollout(self, k: int, mlp: dict, *, gamma: float = 0.99, gae_lambda: float = 0.95,
                        stochastic: bool = True, tensor_cores=3, bootstrap_truncated: bool = False) -> dict:
        """What SB3's `PPO.collect_rollouts` + `RolloutBuffer.compute_returns_and_advantage` produce for k steps of
        this VecEnv, entirely on the device: per step one policy launch (action, value, log-prob; by default the
        faithful tcgen05 3xTF32 kernel, tensor_cores=3) and one env step, then the GAE scan.  Returns tensors shaped
        [k, N, ...]: obs (13), actions (raw Gaussian samples), values, log_probs, rewards, dones, advantages, returns.

        bootstrap_truncated=True adds SB3's timeout handling: the reward of a step that ended its episode by the TimeLimit
        (flag F_TRUNCATED) becomes fl32(r + fl32(gamma * V(terminal observation))), V from the same policy kernel and
        `tensor_cores` mode as `values`, before the GAE scan; `dones` stays as it is.  Each truncation is filed after its
        step (`r6_trunc_record`), the critic runs once per slot layer after the rollout and `r6_trunc_bootstrap` adds the
        values, all without a host synchronise.  Needs auto-reset (ValueError otherwise).  The default False leaves the
        rewards as the env returned them.

        The trajectory is written in place: the env step of step j writes its observations straight into slice j + 1 of
        a component-major buffer [k + 1, 14, N] (the layout the kernels read and write), its reward and done flags into
        row j of `rewards` / `dones`, and the policy of step j + 1 reads that slice — no per-step copies (with auto-reset,
        the training configuration; one-episode batches keep the copies).  `obs` is therefore a strided [k, N, 13] view of
        that buffer (`.contiguous()` gives dense rows if a consumer needs them)."""
        from .gae import compute_gae
        k = int(k)
        n, dev = self.num_envs, self.device
        if bootstrap_truncated and not self.auto_reset:
            raise ValueError("bootstrap_truncated needs auto_reset=True (a frozen one-episode env keeps its flags)")
        self.join()
        # one slot per truncation an env can have in k steps: two of them are at least max_episode_steps apart
        limit = int(self._p.max_episode_steps)
        slots = -(-k // limit) if bootstrap_truncated and limit > 0 else 0
        if slots:                                    # filled before the lanes fork, so that they see the -1
            slot_step = torch.full((slots, n), -1, dtype=torch.int32, device=dev)
            slot_obs = torch.empty(slots, 13, n, dtype=torch.float32, device=dev)
        obs_cm = torch.empty(k + 1, 14, n, dtype=torch.float32, device=dev)
        obs_cm[0].copy_(self.obs)
        acts = torch.empty(k, n, 3, dtype=torch.float32, device=dev)
        vals = torch.empty(k, n, dtype=torch.float32, device=dev)
        logp = torch.empty(k, n, dtype=torch.float32, device=dev)
        rews = torch.empty(k, n, dtype=torch.float32, device=dev)
        dones = torch.empty(k, n, dtype=torch.uint8, device=dev)
        a_env = torch.empty(n, 3, dtype=torch.float32, device=dev)
        m = _lib.make_mlp(mlp)
        # Without auto-reset a finished env is frozen: the step reads its done flag and writes NOTHING for it, so its
        # obs / reward / done must carry over from the previous step — that mode keeps the per-step copies.
        in_place = bool(self.auto_reset)
        saved = (self._b.obs, self._b.reward_f32, self._b.done)
        lanes = self._fork(mlp=mlp)                  # every lane runs [policy, env step] x k over its env range on its stream
        try:
            with torch.cuda.device(dev):
                for j in range(k):
                    if in_place:
                        self._b.obs, self._b.reward_f32, self._b.done = (obs_cm[j + 1].data_ptr(), rews[j].data_ptr(),
                                                                        dones[j].data_ptr())
                    for ln, first, count, st in lanes:
                        if not in_place and j > 0:
                            with torch.cuda.stream(st):
                                obs_cm[j, :, first:first + count] = self.obs[:, first:first + count]
                        self._policy(m, obs_cm[j].data_ptr(), first, count, tensor_cores, stochastic, self.steps_done + j,
                                     a_env.data_ptr(), acts[j].data_ptr(), vals[j].data_ptr(), logp[j].data_ptr(), st)
                        self._env_step(ln, first, count, a_env.data_ptr(), self.steps_done + j, st)
                        if slots:
                            _lib.check(self.lib.r6_trunc_record(self.flags.data_ptr(), self.terminal_obs.data_ptr(), n, first,
                                                                count, j, slots, slot_step.data_ptr(), slot_obs.data_ptr(),
                                                                st.cuda_stream), self.lib)
                        if not in_place:
                            with torch.cuda.stream(st):
                                rews[j, first:first + count] = self.reward_f32[first:first + count]
                                dones[j, first:first + count] = self.done[first:first + count]
        finally:
            self._b.obs, self._b.reward_f32, self._b.done = saved
        self._advance(k)
        if k > 0 and in_place:                       # the batch's own output tensors end up as after k calls of step()
            self.obs.copy_(obs_cm[k])
            self.reward_f32.copy_(rews[k - 1])
            self.done.copy_(dones[k - 1])
        _, _, last_v, _ = self.policy_forward(mlp, stochastic=False, tensor_cores=tensor_cores)
        if slots:
            cur = torch.cuda.current_stream(dev)
            slot_v = torch.empty(slots, n, dtype=torch.float32, device=dev)
            with torch.cuda.device(dev):
                for s in range(slots):
                    self._policy(m, slot_obs[s].data_ptr(), 0, n, tensor_cores, False, 0, a_env.data_ptr(), None,
                                 slot_v[s].data_ptr(), None, cur)
                _lib.check(self.lib.r6_trunc_bootstrap(rews.data_ptr(), k, n, slots, slot_step.data_ptr(), slot_v.data_ptr(),
                                                       float(gamma), cur.cuda_stream), self.lib)
        adv, ret = compute_gae(rews, vals, dones, last_v, gamma, gae_lambda)
        return dict(obs=obs_cm[:k, :13].permute(0, 2, 1), actions=acts, values=vals, log_probs=logp, rewards=rews, dones=dones,
                    advantages=adv, returns=ret, last_values=last_v)

    def step_policy(self, k: int, mlp: dict, *, tensor_cores=3, join: bool = True):
        """k closed-loop env-steps as 2k launches: the policy kernel (a uniform GEMM chain at high occupancy) writes
        the actions, the step kernel consumes them — VecEnv semantics (auto-reset as configured).  Faster than the
        single fused rollout kernel for large batches; `rollout(k, ACT_MLP)` remains for one-episode semantics.
        With stream lanes every lane runs its own policy -> step chain (r6_policy_range, r6_step_range) for the k
        steps and the lanes are joined at the end (join=False leaves them running, as in `step`)."""
        act = getattr(self, "_policy_act", None)
        if act is None:
            act = self._policy_act = torch.empty(self.num_envs, 3, dtype=torch.float32, device=self.device)
        k, m = int(k), _lib.make_mlp(mlp)
        with torch.cuda.device(self.device):
            lanes = self._fork(mlp=mlp)
            for j in range(k):
                for ln, first, count, st in lanes:
                    self._policy(m, self.obs.data_ptr(), first, count, tensor_cores, False, self.steps_done + j,
                                 act.data_ptr(), None, None, None, st)
                    self._env_step(ln, first, count, act.data_ptr(), self.steps_done + j, st)
        self._advance(k, join)
        return self.obs, self.reward, self.done, self.flags

    # ------------------------------------------------------------------ state injection / inspection
    def set_state(self, state: torch.Tensor, idx: Optional[torch.Tensor] = None, *, step_count: int = 0):
        """Starts new episodes from given float32 initial conditions [M,14] (already normalised
        quaternion), as `reset()` would after sampling them (parity runs inject the oracle's ICs)."""
        self.join()
        ic = torch.as_tensor(state, dtype=torch.float32, device=self.device).reshape(-1, 14)
        if idx is None:
            idx = torch.arange(self.num_envs, device=self.device)
        idx = torch.as_tensor(idx, device=self.device, dtype=torch.long).reshape(-1)
        self.state[:, idx] = ic.t().to(self.state.dtype)
        self.m0[idx] = ic[:, 13]
        # ||v|| float32 with the sdot rule: f32 products, f64 accumulation, one rounding
        v = ic[:, 3:6]
        acc = (v * v).to(torch.float64).sum(1)          # products are rounded to f32 before widening
        self.v0[idx] = acc.to(torch.float32).sqrt()
        self.step_count[idx] = step_count
        self.ep_return[idx] = 0
        self.tgo[idx] = 0
        self.done[idx] = 0          # a new episode: un-freezes the env under one-episode semantics (auto_reset=False)
        self.obs[:, idx] = (self.state[:, idx].to(torch.float64) / torch.as_tensor(self.params.state_normalizer, device=self.device)[:, None]).to(torch.float32)

    def get_state(self) -> torch.Tensor:
        return self.state

    def reset_stats(self):
        self.join()
        with torch.cuda.device(self.device):
            _lib.check(self.lib.r6_stats_reset(self.stats.data_ptr(), self._stream()), self.lib)

    def stats_dict(self, stats: Optional[torch.Tensor] = None) -> dict:
        self.join()
        s = (self.stats if stats is None else stats).detach().cpu().numpy()
        d = dict(zip(STAT_NAMES, (float(x) for x in s)))
        ep = max(d["episodes"], 1.0)
        d["mean_return"] = d["return_sum"] / ep
        d["mean_length"] = d["length_sum"] / ep
        d["landing_rate"] = d["landed"] / ep
        return d
