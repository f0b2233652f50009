"""TennisBatch: N lock-step envs on one B200, stepped by the CUDA kernels behind the C ABI.

PyTorch is used for device memory and streams only; all arithmetic of the env step happens in
libtennisbot_b200.so (csrc/tb_kernels.cu).  Replaces, for a batch, what one reference env object does with
p.connect / loadURDF / stepSimulation / getContactPoints (tennisbot/envs/*.py, tennisbot/resources/*.py).
"""
import ctypes as C
import functools

import numpy as np
import torch

from . import _lib

ENV_IDS = {"SwingRacket-v0": _lib.ENV_SWING, "Tennisbot-v0": _lib.ENV_HIT, "swing": _lib.ENV_SWING, "hit": _lib.ENV_HIT}
PRECISIONS = {"f32": _lib.F32, "f64": _lib.F64, "float32": _lib.F32, "float64": _lib.F64}


def _dptr(t):
    return None if t is None else C.c_void_p(t.data_ptr())


def _hptr(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


class TennisBatch:
    def __init__(self, env_id="SwingRacket-v0", num_envs=4096, device=0, seed=0, precision="f64", auto_reset=True,
                 env_id_offset=0):
        if not torch.cuda.is_available():
            raise _lib.TennisbotLibraryError("TennisBatch needs a CUDA device: the env step has no CPU fallback")
        self.lib = _lib.load()
        self.kind = ENV_IDS[env_id] if isinstance(env_id, str) else int(env_id)
        self.precision = PRECISIONS[precision] if isinstance(precision, str) else int(precision)
        self.device = torch.device("cuda", device if isinstance(device, int) else torch.device(device).index or 0)
        self.num_envs = int(num_envs)
        self.obs_dim = self.lib.tb_obs_dim(self.kind)
        self.act_dim = self.lib.tb_act_dim(self.kind)
        torch.cuda.init()
        with torch.cuda.device(self.device):
            torch.zeros(1, device=self.device)  # make sure the primary context exists before the library uses it
        cfg = _lib.TbConfig(C.sizeof(_lib.TbConfig), self.kind, self.precision, self.device.index, self.num_envs,
                            int(env_id_offset), int(seed) & (2 ** 64 - 1), int(bool(auto_reset)), 0)
        h = C.c_void_p()
        _lib.check(self.lib.tb_create(C.byref(cfg), C.byref(h)))
        self.h = h
        n, od = self.num_envs, self.obs_dim
        dev = self.device
        self.obs = torch.zeros((n, od), dtype=torch.float32, device=dev)
        self.reward = torch.zeros(n, dtype=torch.float32, device=dev)
        self.done = torch.zeros(n, dtype=torch.uint8, device=dev)
        self.terminal_obs = torch.zeros((n, od), dtype=torch.float32, device=dev)
        self.events = torch.zeros(n, dtype=torch.uint8, device=dev)
        self._host = None

    # ------------------------------------------------------------------ lifetime
    def close(self):
        if getattr(self, "h", None):
            self.lib.tb_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    # ------------------------------------------------------------------ parameters
    def set_param(self, name, value):
        _lib.check(self.lib.tb_set_param(self.h, name.encode(), float(value)))

    def set_control_mode(self, mode):
        """'force' (both gym envs) or 'pid' (Racket.apply_action: the action is a target position)."""
        m = {"force": _lib.CONTROL_FORCE, "pid": _lib.CONTROL_PID}.get(mode, mode)
        _lib.check(self.lib.tb_set_control_mode(self.h, int(m)))

    def get_param(self, name):
        v = C.c_double()
        _lib.check(self.lib.tb_get_param(self.h, name.encode(), C.byref(v)))
        return v.value

    # ------------------------------------------------------------------ device-resident API (zero copy)
    def reset(self, mask=None, init=None):
        """New episode for masked envs (all if None). `init`: [N, 8] explicit placement. Returns obs (device)."""
        m = None if mask is None else torch.as_tensor(mask, device=self.device).to(torch.uint8).contiguous()
        if init is None:
            _lib.check(self.lib.tb_reset(self.h, _dptr(m), _dptr(self.obs), self._stream()))
        else:
            i = torch.as_tensor(init, dtype=torch.float64, device=self.device).reshape(self.num_envs, _lib.INIT_WORDS).contiguous()
            _lib.check(self.lib.tb_reset_from(self.h, _dptr(i), _dptr(m), _dptr(self.obs), self._stream()))
        return self.obs

    def step(self, actions, obs=None, reward=None, done=None, terminal_obs=None, events=None):
        """One env step for all N envs (step_kernel + ff_kernel on the current stream). actions: float32 CUDA tensor [N, act_dim].
        Returns (obs, reward, done, terminal_obs, events) device tensors (the caller's, or reused internal ones)."""
        if actions.dtype != torch.float32 or not actions.is_cuda or not actions.is_contiguous():
            actions = actions.to(device=self.device, dtype=torch.float32).contiguous()
        if actions.numel() != self.num_envs * self.act_dim:
            raise ValueError(f"actions must have shape ({self.num_envs}, {self.act_dim})")
        obs = self.obs if obs is None else obs
        reward = self.reward if reward is None else reward
        done = self.done if done is None else done
        terminal_obs = self.terminal_obs if terminal_obs is None else terminal_obs
        events = self.events if events is None else events
        _lib.check(self.lib.tb_step(self.h, _dptr(actions), _dptr(obs), _dptr(reward), _dptr(done), _dptr(terminal_obs),
                                    _dptr(events), self._stream()))
        return obs, reward, done, terminal_obs, events

    def rollout(self, k_steps, action_mode=_lib.ACT_RANDOM, want_outputs=True):
        """K env steps fused in one launch with in-kernel actions. Returns (obs, reward_sum, done_count)."""
        if want_outputs:
            if not hasattr(self, "_rsum"):
                self._rsum = torch.zeros(self.num_envs, dtype=torch.float32, device=self.device)
                self._dcount = torch.zeros(self.num_envs, dtype=torch.int32, device=self.device)
            args = (_dptr(self.obs), _dptr(self._rsum), _dptr(self._dcount))
        else:
            args = (None, None, None)
        _lib.check(self.lib.tb_rollout(self.h, int(action_mode), int(k_steps), *args, self._stream()))
        return (self.obs, self._rsum, self._dcount) if want_outputs else None

    def _need(self, who, t, name, shape, dtype=torch.float32, optional=False):
        """The library writes through raw pointers: a buffer must be a contiguous tensor of this shape and dtype on this device."""
        if t is None and optional:
            return
        if t is None or t.dtype != dtype or t.device != self.device or not t.is_contiguous() or tuple(t.shape) != shape:
            got = None if t is None else (tuple(t.shape), t.dtype, str(t.device), t.is_contiguous())
            raise ValueError(f"{who}: {name} must be a contiguous {dtype} tensor of shape {shape} on {self.device}, got {got}")

    # ------------------------------------------------------------------ policy rollout (tb_set_policy / tb_policy_rollout)
    def set_policy(self, params):
        """params: float32 CUDA tensor [policy_floats] in the layout of include/tennisbot_b200.h for this batch's env
        (POLICY_FLOATS for SwingRacket-v0, POLICY_FLOATS_HIT for Tennisbot-v0; pack_policy builds it)."""
        p = params.to(device=self.device, dtype=torch.float32).contiguous()
        want = _lib.POLICY_FLOATS if self.kind == _lib.ENV_SWING else _lib.POLICY_FLOATS_HIT
        if p.numel() != want:
            raise ValueError(f"policy parameter vector must have {want} floats for this env, got {p.numel()}")
        _lib.check(self.lib.tb_set_policy(self.h, _dptr(p), p.numel(), self._stream()))

    def set_policies(self, params):
        """A population: params float32 CUDA tensor [P, policy_floats] on this batch's device, rows in set_policy's layout, P
        dividing num_envs.  Env i acts with row i // (num_envs // P) in the next policy_rollout; set_policy returns to one
        policy.  A stream-ordered copy, capturable once the library's buffer holds P rows (tb_set_policies)."""
        want = _lib.POLICY_FLOATS if self.kind == _lib.ENV_SWING else _lib.POLICY_FLOATS_HIT
        agents = int(params.shape[0]) if torch.is_tensor(params) and params.dim() == 2 else -1
        if agents < 1 or self.num_envs % agents:
            raise ValueError(f"set_policies: params must have shape (P, {want}) with P dividing {self.num_envs}, got "
                             f"{tuple(params.shape) if torch.is_tensor(params) else type(params).__name__}")
        self._need("set_policies", params, "params", (agents, want))
        _lib.check(self.lib.tb_set_policies(self.h, _dptr(params), agents, agents * want, self._stream()))

    def policy_rollout(self, obs, reward, done, last_obs, actions=None, logp=None, value=None, last_value=None,
                       deterministic=False, noise_seed=0, raw_reward=None):
        """K = obs.shape[0] env steps with actions sampled in-kernel from the policy set by set_policy (or, after
        set_policies, env i from row i // (num_envs // P)).  obs[0] must hold
        the current observation.  obs [K, N, obs_dim], actions [K, N, act_dim], reward / logp / value [K, N], last_obs
        [N, obs_dim], last_value [N]: contiguous float32 tensors on this batch's device; done [K, N] uint8.  raw_reward
        [K, N] (optional) receives the env's reward before normalisation (tb_policy_rollout_raw; reward itself without a
        normaliser).  The library writes through raw pointers, so every buffer is checked here."""
        k, n = int(obs.shape[0]) if obs.dim() == 3 else -1, self.num_envs
        if k < 1:
            raise ValueError(f"policy_rollout: obs must have shape (K >= 1, {n}, {self.obs_dim}), got {tuple(obs.shape)}")
        need = functools.partial(self._need, "policy_rollout")
        need(obs, "obs", (k, n, self.obs_dim))
        need(actions, "actions", (k, n, self.act_dim), optional=True)
        need(logp, "logp", (k, n), optional=True)
        need(value, "value", (k, n), optional=True)
        need(reward, "reward", (k, n))
        need(done, "done", (k, n), dtype=torch.uint8)
        need(last_obs, "last_obs", (n, self.obs_dim))
        need(last_value, "last_value", (n,), optional=True)
        need(raw_reward, "raw_reward", (k, n), optional=True)
        _lib.check(self.lib.tb_policy_rollout_raw(self.h, k, int(bool(deterministic)), int(noise_seed) & (2 ** 64 - 1), _dptr(obs),
                                                  _dptr(actions), _dptr(logp), _dptr(value), _dptr(reward), _dptr(raw_reward),
                                                  _dptr(done), _dptr(last_obs), _dptr(last_value), self._stream()))

    # ------------------------------------------------------------------ normaliser of the policy rollout (tb_set_vecnorm)
    def set_vecnorm(self, training=True, norm_obs=True, norm_reward=True, clip_obs=10.0, clip_reward=10.0, gamma=0.99,
                    epsilon=1e-8, agents=1, stats=None):
        """Attach SB3 VecNormalize's observation / reward normalisation to policy_rollout (semantics in the header at
        tb_set_vecnorm).  stats: float64 [2 obs_dim + 4] to start from (obs mean, obs var, obs count, ret mean, ret var, ret
        count), None = fresh; a given record is checked on the host, which synchronises the stream.  agents > 1: one record
        per agent of a population (tb_set_vecnorms; env i uses record i // (num_envs // agents)), all with this
        configuration, and stats is [agents, 2 obs_dim + 4]."""
        words, agents = _lib.vecnorm_words(self.obs_dim), int(agents)
        cfg = _lib.TbVecNorm(C.sizeof(_lib.TbVecNorm), int(bool(training)), int(bool(norm_obs)), int(bool(norm_reward)),
                             float(clip_obs), float(clip_reward), float(gamma), float(epsilon))
        if agents == 1:
            self._need("set_vecnorm", stats, "stats", (words,), torch.float64, optional=True)
            _lib.check(self.lib.tb_set_vecnorm(self.h, C.byref(cfg), _dptr(stats), self._stream()))
            return
        if agents < 1 or self.num_envs % agents:
            raise ValueError(f"set_vecnorm: agents must be >= 1 and divide {self.num_envs}, got {agents}")
        self._need("set_vecnorm", stats, "stats", (agents, words), torch.float64, optional=True)
        _lib.check(self.lib.tb_set_vecnorms(self.h, C.byref(cfg), agents, _dptr(stats), self._stream()))

    def clear_vecnorm(self):
        """Detach the normaliser: policy_rollout behaves as if none had been attached."""
        _lib.check(self.lib.tb_set_vecnorm(self.h, None, None, self._stream()))

    def _vecnorm_buffer(self):
        """(device address, records) of the library's record buffer; (None, 1) when no normaliser is attached."""
        p, agents = C.c_void_p(), C.c_int64()
        if self.lib.tb_vecnorm_device_ptr(self.h, C.byref(p), C.byref(agents)) != 0:
            return None, 1
        return p.value, agents.value

    def vecnorm_stats(self, out=None):
        """float64 device tensor [2 obs_dim + 4]: the normaliser's current record (stream-ordered copy); [A, 2 obs_dim + 4]
        with A > 1 records (set_vecnorm(agents=A))."""
        agents = self._vecnorm_buffer()[1]
        shape = (_lib.vecnorm_words(self.obs_dim),) if agents == 1 else (agents, _lib.vecnorm_words(self.obs_dim))
        if out is None:
            out = torch.empty(shape, dtype=torch.float64, device=self.device)
        self._need("vecnorm_stats", out, "out", shape, torch.float64)
        if agents == 1:
            _lib.check(self.lib.tb_get_vecnorm(self.h, _dptr(out), self._stream()))
        else:
            _lib.check(self.lib.tb_get_vecnorms(self.h, _dptr(out), agents, self._stream()))
        return out

    def vecnorm_records(self):
        """float64 [A, 2 obs_dim + 4] view of the library's record buffer (tb_vecnorm_device_ptr): the kernels read a record
        when they run, so an in-place write to a row (copying one agent's record over another's) is seen by the next
        policy_rollout, a replayed graph included, without zeroing returns or arming the reset fold.  Valid until a
        set_vecnorm call with more records than before, or close()."""
        ptr, agents = self._vecnorm_buffer()
        if ptr is None:
            raise _lib.TennisbotLibraryError("vecnorm_records: no normaliser attached (set_vecnorm)")
        return _wrap_device(ptr, (agents, _lib.vecnorm_words(self.obs_dim)), "<f8", self.device, owner=self)

    def vecnorm_apply(self, x, what="obs", out=None):
        """The normaliser's formula on a batch of raw values (tb_vecnorm_apply), with the record as it stands when the kernel
        runs: what 'obs' (VECNORM_OBS), x float32 [rows, obs_dim]; 'reward' (VECNORM_REWARD), x float32 [rows].  out: None (a
        new tensor) or a tensor of x's shape, x itself included.  One launch on the current stream; returns out."""
        what = {"obs": _lib.VECNORM_OBS, "reward": _lib.VECNORM_REWARD}.get(what, what)
        if what not in (_lib.VECNORM_OBS, _lib.VECNORM_REWARD):
            raise ValueError(f"vecnorm_apply: what must be 'obs' or 'reward', got {what!r}")
        obs = what == _lib.VECNORM_OBS
        rows = int(x.shape[0]) if torch.is_tensor(x) and x.dim() == (2 if obs else 1) else -1
        shape = (rows, self.obs_dim) if obs else (rows,)
        if rows < 0:
            raise ValueError(f"vecnorm_apply: x must have shape {('rows', self.obs_dim) if obs else ('rows',)}, got "
                             f"{None if x is None else tuple(x.shape)}")
        self._need("vecnorm_apply", x, "x", shape)
        if out is None:
            out = torch.empty_like(x)
        self._need("vecnorm_apply", out, "out", shape)
        _lib.check(self.lib.tb_vecnorm_apply(self.h, _dptr(x), rows, int(what), _dptr(out), self._stream()))
        return out

    # ------------------------------------------------------------------ ES fitness rollout (tb_es_begin / tb_es_rollout)
    def es_begin(self, weights, normalizer=None):
        """Start an ES generation: weights float32 [individuals, es_floats] (individuals divides num_envs; env i evaluates
        individual i // (num_envs // individuals)), normalizer float64 [3, obs_dim] = the master (n, mean, mean_diff) or None.
        Resets every env, so a generation always starts new episodes."""
        floats = self._es_floats()
        if weights.dim() != 2 or weights.shape[1] != floats or weights.shape[0] < 1 or self.num_envs % weights.shape[0]:
            raise ValueError(f"es_begin: weights must have shape (individuals, {floats}) with individuals dividing {self.num_envs}, "
                             f"got {tuple(weights.shape)}")
        self._need("es_begin", weights, "weights", tuple(weights.shape), torch.float32)
        self._need("es_begin", normalizer, "normalizer", (3, self.obs_dim), torch.float64, optional=True)
        _lib.check(self.lib.tb_es_begin(self.h, _dptr(weights), int(weights.shape[0]), floats, _dptr(normalizer), self._stream()))

    def es_rollout(self, k_steps, ret, alive, obs=None, actions=None, reward=None, done=None):
        """k_steps env steps of the generation with in-kernel GatedCNN actions.  ret float64 [N] and alive uint8 [N] receive the
        state after the last step.  Optional traces: obs float32 [K+1, N, obs_dim] (the raw observation each normaliser update
        consumed, [0] the one before this call), actions float32 [K, N, act_dim] (clipped), reward float32 [K, N], done uint8
        [K, N].  The library writes through raw pointers, so every buffer is checked here."""
        k, n = int(k_steps), self.num_envs
        if k < 1:
            raise ValueError(f"es_rollout: k_steps must be >= 1, got {k}")
        self._need("es_rollout", ret, "ret", (n,), torch.float64)
        self._need("es_rollout", alive, "alive", (n,), torch.uint8)
        self._need("es_rollout", obs, "obs", (k + 1, n, self.obs_dim), torch.float32, optional=True)
        self._need("es_rollout", actions, "actions", (k, n, self.act_dim), torch.float32, optional=True)
        self._need("es_rollout", reward, "reward", (k, n), torch.float32, optional=True)
        self._need("es_rollout", done, "done", (k, n), torch.uint8, optional=True)
        _lib.check(self.lib.tb_es_rollout(self.h, k, _dptr(ret), _dptr(alive), _dptr(obs), _dptr(actions), _dptr(reward),
                                          _dptr(done), self._stream()))

    # ------------------------------------------------------------------ ES population and update (seeded perturbations)
    def _es_floats(self):
        return _lib.ES_FLOATS if self.kind == _lib.ENV_SWING else _lib.ES_FLOATS_HIT

    def es_begin_noise(self, theta, individuals, sigma, noise_seed, generation, normalizer=None):
        """es_begin with the antithetic population drawn in the library: global individual g = env_id_offset // repeats + p is
        theta + sigma * eps_{g // 2} for even g and theta - sigma * eps_{g // 2} for odd g (tb_es_begin_noise documents eps).
        theta float32 [es_floats]; individuals even and dividing num_envs; env_id_offset a multiple of 2 x repeats."""
        floats, individuals = self._es_floats(), int(individuals)
        if individuals < 2 or individuals % 2 or self.num_envs % individuals:
            raise ValueError(f"es_begin_noise: individuals must be even and divide {self.num_envs}, got {individuals}")
        self._need("es_begin_noise", theta, "theta", (floats,), torch.float32)
        self._need("es_begin_noise", normalizer, "normalizer", (3, self.obs_dim), torch.float64, optional=True)
        _lib.check(self.lib.tb_es_begin_noise(self.h, _dptr(theta), individuals, floats, float(sigma), int(noise_seed) & (2 ** 64 - 1),
                                              int(generation) & (2 ** 32 - 1), _dptr(normalizer), self._stream()))

    def es_noise_combine(self, dirs, coef, noise_seed, generation, out=None):
        """out float32 [es_floats] = sum_k coef[k] * eps_{dirs[k]} of `generation` (float64 sum in order k), regenerated from the
        seed.  dirs int64 [count] (global direction indices), coef float32 [count]."""
        count = int(dirs.shape[0]) if dirs is not None and dirs.dim() == 1 else -1
        if count < 0:
            raise ValueError(f"es_noise_combine: dirs must be a 1-d int64 tensor, got {None if dirs is None else tuple(dirs.shape)}")
        self._need("es_noise_combine", dirs, "dirs", (count,), torch.int64)
        self._need("es_noise_combine", coef, "coef", (count,), torch.float32)
        if out is None:
            out = torch.empty(self._es_floats(), dtype=torch.float32, device=self.device)
        self._need("es_noise_combine", out, "out", (self._es_floats(),), torch.float32)
        _lib.check(self.lib.tb_es_noise_combine(self.h, _dptr(dirs), _dptr(coef), count, int(noise_seed) & (2 ** 64 - 1),
                                                int(generation) & (2 ** 32 - 1), _dptr(out), self._stream()))
        return out

    def es_normalizer_stats(self, out=None):
        """float64 [3, obs_dim] = (count, mean, M2) of the observations this batch's normalisers took since the last
        es_begin*, without the master's share.  Merge with the master (and other shards) by Chan's formula."""
        if out is None:
            out = torch.empty((3, self.obs_dim), dtype=torch.float64, device=self.device)
        self._need("es_normalizer_stats", out, "out", (3, self.obs_dim), torch.float64)
        _lib.check(self.lib.tb_es_normalizer_stats(self.h, _dptr(out), self._stream()))
        return out

    # ------------------------------------------------------------------ SAC actor and replay ring (tb_set_sac_actor / tb_sac_*)
    def set_sac_actor(self, params):
        """params: float32 CUDA tensor [sac_floats] in the layout of include/tennisbot_b200.h for this batch's env
        (SAC_FLOATS for SwingRacket-v0, SAC_FLOATS_HIT for Tennisbot-v0; sac.pack_sac_actor builds it)."""
        want = _lib.SAC_FLOATS if self.kind == _lib.ENV_SWING else _lib.SAC_FLOATS_HIT
        self._need("set_sac_actor", params, "params", (want,))
        _lib.check(self.lib.tb_set_sac_actor(self.h, _dptr(params), want, self._stream()))

    def set_sac_actors(self, params):
        """A population: params float32 CUDA tensor [P, sac_floats] on this batch's device, rows in set_sac_actor's layout, P
        dividing num_envs and, for P > 1, num_envs // P a multiple of 128.  Env i acts with row i // (num_envs // P) in the
        next sac_rollout; set_sac_actor returns to one actor.  One capturable launch once the library's image buffer holds P
        actors (tb_set_sac_actors)."""
        want = _lib.SAC_FLOATS if self.kind == _lib.ENV_SWING else _lib.SAC_FLOATS_HIT
        agents = int(params.shape[0]) if torch.is_tensor(params) and params.dim() == 2 else -1
        if agents < 1 or self.num_envs % agents:
            raise ValueError(f"set_sac_actors: params must have shape (P, {want}) with P dividing {self.num_envs}, got "
                             f"{tuple(params.shape) if torch.is_tensor(params) else type(params).__name__}")
        if agents > 1 and (self.num_envs // agents) % 128:
            raise ValueError(f"set_sac_actors: with P > 1, envs per agent ({self.num_envs} / {agents}) must be a multiple of "
                             f"128: a 128-env tile multiplies against one actor's W2 image in shared memory")
        self._need("set_sac_actors", params, "params", (agents, want))
        _lib.check(self.lib.tb_set_sac_actors(self.h, _dptr(params), agents, agents * want, self._stream()))

    def sac_begin(self):
        """Reset every env and start the ring at slot 0 (needs force control and auto_reset)."""
        _lib.check(self.lib.tb_sac_begin(self.h, self._stream()))

    def sac_rollout(self, k, mode=_lib.SAC_SAMPLE, ring=None, noise_seed=0, last_obs=None, normalize=False):
        """k env steps with in-kernel SAC actions.  mode: SAC_SAMPLE, SAC_MEAN or SAC_UNIFORM (or 'sample', 'mean', 'uniform').
        ring: None or a dict of tensors obs / next_obs float32 [slots, N, obs_dim], act float32 [slots, N, act_dim], reward
        float32 [slots, N], done uint8 [slots, N]; step j since sac_begin goes to slot j % slots.  last_obs float32 [N, obs_dim]
        receives the observation after the last step.  normalize: the normaliser of set_vecnorm applies (TB_SAC_VECNORM: the
        actor acts on normalised observations, a training normaliser folds every step; ring and last_obs stay raw).  The
        library writes through raw pointers, so every buffer is checked here."""
        k, n = int(k), self.num_envs
        if k < 1:
            raise ValueError(f"sac_rollout: k must be >= 1, got {k}")
        mode = {"sample": _lib.SAC_SAMPLE, "mean": _lib.SAC_MEAN, "uniform": _lib.SAC_UNIFORM}.get(mode, mode)
        need = functools.partial(self._need, "sac_rollout")
        need(last_obs, "last_obs", (n, self.obs_dim), optional=True)
        r = None
        if ring is not None:
            slots = int(ring["obs"].shape[0]) if torch.is_tensor(ring.get("obs")) and ring["obs"].dim() == 3 else -1
            if slots < 1:
                raise ValueError(f"sac_rollout: ring['obs'] must have shape (slots >= 1, {n}, {self.obs_dim})")
            need(ring.get("obs"), "ring['obs']", (slots, n, self.obs_dim))
            need(ring.get("next_obs"), "ring['next_obs']", (slots, n, self.obs_dim))
            need(ring.get("act"), "ring['act']", (slots, n, self.act_dim))
            need(ring.get("reward"), "ring['reward']", (slots, n))
            need(ring.get("done"), "ring['done']", (slots, n), dtype=torch.uint8)
            r = _lib.TbSacRing(C.sizeof(_lib.TbSacRing), 0, slots, *(ring[key].data_ptr() for key in
                                                                     ("obs", "act", "reward", "next_obs", "done")))
        mode = int(mode) | (_lib.SAC_VECNORM if normalize else 0)
        _lib.check(self.lib.tb_sac_rollout(self.h, k, mode, int(noise_seed) & (2 ** 64 - 1), None if r is None else C.byref(r),
                                           _dptr(last_obs), self._stream()))

    # ------------------------------------------------------------------ frames (tb_render)
    def render(self, camera, states=None, depth=False, body=False):
        """Frames of canonical state records through `camera` (render.Camera), one kernel launch on the current stream.
        states: None renders every env of this batch from a fresh get_state(); else a float64 [M, 32] tensor on this batch's
        device.  Returns (rgb uint8 [M, H, W, 3], depth float32 [M, H, W] or None, body uint8 [M, H, W] or None): device
        tensors, row 0 at the top; depth is the distance from the eye (+inf: sky), body holds _lib.BODY_*."""
        if states is None:
            states = self.get_state()
        m = int(states.shape[0]) if states.dim() == 2 else -1
        if m < 1:
            raise ValueError(f"render: states must have shape (M >= 1, {_lib.STATE_WORDS}), got {tuple(states.shape)}")
        self._need("render", states, "states", (m, _lib.STATE_WORDS), torch.float64)
        h, w = int(camera.height), int(camera.width)
        rgb = torch.empty((m, h, w, 3), dtype=torch.uint8, device=self.device)
        dep = torch.empty((m, h, w), dtype=torch.float32, device=self.device) if depth else None
        bod = torch.empty((m, h, w), dtype=torch.uint8, device=self.device) if body else None
        _lib.check(self.lib.tb_render(self.h, C.byref(camera.to_c()), _dptr(states), m, _dptr(rgb), _dptr(dep), _dptr(bod),
                                      self._stream()))
        return rgb, dep, bod

    # ------------------------------------------------------------------ substep trace (tb_trace_step)
    def trace_step(self, actions, states=None, max_substeps=None):
        """One env step of canonical state records taken substep by substep, one kernel launch on the current stream; the
        batch's own envs are not stepped.  actions: float32 [M, act_dim] on this batch's device, as step() receives them
        (clip them to the Box yourself).  states: None traces every env of this batch from a fresh get_state(); else a
        float64 [M, 32] tensor on this batch's device.  max_substeps: records kept per env (None: the env's bound,
        _lib.TRACE_MAX_SUBSTEPS for SwingRacket-v0, 1 for Tennisbot-v0).  Returns device tensors (trace float64 [S, M, 32],
        bits uint8 [S, M], substeps int32 [M], reward float32 [M], done uint8 [M], events uint8 [M]): trace[k, i] is record i
        after substep k + 1, padded with the final record; bits are the contacts of that substep alone.  Frames of the
        flight: render(camera, states=trace[::k].reshape(-1, 32))."""
        if states is None:
            states = self.get_state()
        m = int(states.shape[0]) if states.dim() == 2 else -1
        if m < 1:
            raise ValueError(f"trace_step: states must have shape (M >= 1, {_lib.STATE_WORDS}), got {tuple(states.shape)}")
        need = functools.partial(self._need, "trace_step")
        need(states, "states", (m, _lib.STATE_WORDS), torch.float64)
        need(actions, "actions", (m, self.act_dim))
        bound = self.lib.tb_trace_max_substeps(self.kind)
        s = bound if max_substeps is None else int(max_substeps)
        if not 1 <= s <= bound:
            raise ValueError(f"trace_step: max_substeps must be in 1 .. {bound} for this env, got {s}")
        dev = self.device
        trace = torch.empty((s, m, _lib.STATE_WORDS), dtype=torch.float64, device=dev)
        bits = torch.empty((s, m), dtype=torch.uint8, device=dev)
        substeps = torch.empty(m, dtype=torch.int32, device=dev)
        reward = torch.empty(m, dtype=torch.float32, device=dev)
        done = torch.empty(m, dtype=torch.uint8, device=dev)
        events = torch.empty(m, dtype=torch.uint8, device=dev)
        _lib.check(self.lib.tb_trace_step(self.h, _dptr(states), _dptr(actions), m, s, _dptr(trace), _dptr(bits), _dptr(substeps),
                                          _dptr(reward), _dptr(done), _dptr(events), self._stream()))
        return trace, bits, substeps, reward, done, events

    def get_state(self):
        s = torch.empty((self.num_envs, _lib.STATE_WORDS), dtype=torch.float64, device=self.device)
        _lib.check(self.lib.tb_get_state(self.h, _dptr(s), self._stream()))
        return s

    def set_state(self, state):
        s = torch.as_tensor(state, dtype=torch.float64, device=self.device).reshape(self.num_envs, _lib.STATE_WORDS).contiguous()
        _lib.check(self.lib.tb_set_state(self.h, _dptr(s), self._stream()))

    def stats_tensor(self):
        """int64[10] statistics vector living in HBM, as a torch view (all-reduce it over NCCL)."""
        p = C.c_void_p()
        _lib.check(self.lib.tb_stats_device_ptr(self.h, C.byref(p)))
        return _wrap_device(p.value, (_lib.NUM_STATS,), "<i8", self.device, owner=self)

    def read_stats(self, clear=False):
        out = np.zeros(_lib.NUM_STATS, np.int64)
        _lib.check(self.lib.tb_read_stats(self.h, _hptr(out), int(clear), self._stream()))
        return out

    def launch_count(self):
        v = C.c_int64()
        _lib.check(self.lib.tb_launch_count(self.h, C.byref(v)))
        return v.value

    def ff_diagnostics(self):
        """int64[16] record of the most recent fast-forward launch (see tb_ff_diagnostics)."""
        import numpy as np

        out = np.zeros(16, np.int64)
        _lib.check(self.lib.tb_ff_diagnostics(self.h, out.ctypes.data_as(C.POINTER(C.c_int64))))
        return out

    def set_kernel_timing(self, enabled):
        _lib.check(self.lib.tb_set_kernel_timing(self.h, int(bool(enabled))))

    def kernel_timing(self):
        """(ms in step_kernel, ms in ff_kernel, steps covered) accumulated since the last call."""
        a, b, n = C.c_double(), C.c_double(), C.c_int64()
        _lib.check(self.lib.tb_get_kernel_timing(self.h, C.byref(a), C.byref(b), C.byref(n)))
        return a.value, b.value, n.value

    # ------------------------------------------------------------------ host-buffer API (pinned numpy in/out)
    def host_buffers(self):
        """Pinned host arrays reused by reset_host/step_host (views of torch pinned tensors)."""
        if self._host is None:
            n, od, ad = self.num_envs, self.obs_dim, self.act_dim

            def pin(shape, dt):
                return torch.zeros(shape, dtype=dt).pin_memory()

            t = dict(actions=pin((n, ad), torch.float32), obs=pin((n, od), torch.float32), reward=pin((n,), torch.float32),
                     done=pin((n,), torch.uint8), terminal_obs=pin((n, od), torch.float32), events=pin((n,), torch.uint8))
            self._host_t = t
            self._host = {k: v.numpy() for k, v in t.items()}
        return self._host

    def reset_host(self, mask=None):
        hb = self.host_buffers()
        m = None if mask is None else np.ascontiguousarray(mask, np.uint8)
        _lib.check(self.lib.tb_reset_host(self.h, _hptr(m), _hptr(hb["obs"])))
        return hb["obs"]

    def step_host(self, actions=None, want_terminal=True, want_events=True):
        """actions: float32 [N, act_dim] host array (None = already written into host_buffers()['actions']).
        One env step inside the C call, synchronised on return.  The buffers are pinned, so by default the kernels read the
        actions from and write the results to host memory themselves (zero copy; TB_HOST_MODE=staging copies them through
        device buffers instead).  Returns the pinned result arrays (overwritten by the next call)."""
        hb = self.host_buffers()
        if actions is not None:
            np.copyto(hb["actions"], np.asarray(actions, np.float32).reshape(self.num_envs, self.act_dim))
        _lib.check(self.lib.tb_step_host(self.h, _hptr(hb["actions"]), _hptr(hb["obs"]), _hptr(hb["reward"]),
                                         _hptr(hb["done"]), _hptr(hb["terminal_obs"]) if want_terminal else None,
                                         _hptr(hb["events"]) if want_events else None))
        return hb


def _wrap_device(ptr, shape, typestr, device, owner):
    """View a C-contiguous array of `shape` and numpy `typestr` at raw device address `ptr` as a torch tensor through
    __cuda_array_interface__."""

    class _Holder:
        pass

    h = _Holder()
    h.__cuda_array_interface__ = {"shape": tuple(shape), "typestr": typestr, "data": (int(ptr), False), "version": 3}
    h._owner = owner
    return torch.as_tensor(h, device=device)
