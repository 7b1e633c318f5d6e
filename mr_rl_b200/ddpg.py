"""DDPG learner on the device — the other caller of the env (RL/MR_ddpg.py; SURVEY §8f rank 3).

Mirrors the reference's pieces with the same names and arguments where they exist:
``ReplayBuffer`` (:16-56) as a ring in HBM, ``OUNoise`` (:58-78) with one process per env, ``DDPGLearner`` = the
ActorNetwork / CriticNetwork pair (:80-231) with their Adam optimisers and target networks, and ``train`` (:233-323)
as a vectorised acting / learning loop.  One learner update (:285-305) is ONE kernel launch (csrc/mr_ddpg.cu).
``DDPGPopulation`` / ``PopulationReplay`` / ``train_population`` train many independent learners (seeds, sweeps) with one
update launch and one collect launch for all of them; ``evaluate_population`` plays every member's greedy policy on fresh
episodes in one launch, and ``pbt_population`` runs population-based training on top of it.
Everything here fails without the CUDA library: there is no CPU path.
"""
from __future__ import annotations

import ctypes as C
import dataclasses
import math

import numpy as np
import torch

from . import _lib as L
from .actor import ORDER as ACTOR_ORDER, SHAPES as ACTOR_SHAPES, actor_forward, init_actor, pack_actor
from .vec_env import raise_for_status

CRITIC_ORDER = ("wc1", "bc1", "gc", "bec", "mc", "vc", "t1", "t1b", "t2", "t2b", "wo", "bo")
CRITIC_SHAPES = {"wc1": (5, 64), "bc1": (64,), "gc": (64,), "bec": (64,), "mc": (64,), "vc": (64,),
                 "t1": (64, 32), "t1b": (32,), "t2": (2, 32), "t2b": (32,), "wo": (32,), "bo": (1,)}


def init_critic(seed=1):
    """tflearn defaults as in create_critic_network (:202-222): truncated-normal(0.02) FC weights, zero biases,
    BN gamma ~ N(1, 0.002), moving mean 0 / variance 1, output layer U[-3e-3, 3e-3]."""
    g = torch.Generator().manual_seed(seed)

    def tn(*shape):
        w = torch.empty(*shape)
        torch.nn.init.trunc_normal_(w, mean=0.0, std=0.02, a=-0.04, b=0.04, generator=g)
        return w

    return {"wc1": tn(5, 64), "bc1": torch.zeros(64), "gc": 1 + 0.002 * torch.randn(64, generator=g), "bec": torch.zeros(64),
            "mc": torch.zeros(64), "vc": torch.ones(64), "t1": tn(64, 32), "t1b": torch.zeros(32), "t2": tn(2, 32),
            "t2b": torch.zeros(32), "wo": (torch.rand(32, generator=g) * 2 - 1) * 0.003, "bo": torch.zeros(1)}


def pack_critic(params, device="cuda"):
    flat = []
    for k in CRITIC_ORDER:
        v = torch.as_tensor(np.asarray(params[k]) if not torch.is_tensor(params[k]) else params[k]).float()
        if tuple(v.shape) != CRITIC_SHAPES[k]:
            raise ValueError(f"{k}: expected {CRITIC_SHAPES[k]}, got {tuple(v.shape)}")
        flat.append(v.reshape(-1))
    w = torch.cat(flat).to(device)
    assert w.numel() == L.load().mr_critic_param_count()
    return w


def _unpack(flat, order, shapes):
    out, o = {}, 0
    flat = flat.detach().cpu()
    for k in order:
        n = int(np.prod(shapes[k]))
        out[k] = flat[o:o + n].reshape(shapes[k]).clone()
        o += n
    return out


def _stream(device):
    return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def _cuda_device(device):
    dev = torch.device(device)
    if dev.type != "cuda":
        raise L.MRLibraryError("the DDPG learner needs a CUDA device: there is no CPU fallback")
    return torch.device("cuda", torch.cuda.current_device()) if dev.index is None else dev


class ReplayBuffer:
    """ReplayBuffer (:16-56) as a ring of float32 rows in HBM.  ``add`` takes the whole vectorised step."""

    def __init__(self, buffer_size, random_seed=123, device="cuda"):
        self.lib = L.load()
        self.device = _cuda_device(device)
        self.buffer_size = int(buffer_size)
        self.random_seed = int(random_seed)
        self.count = 0
        self.head = 0
        z = lambda *s: torch.zeros(*s, dtype=torch.float32, device=self.device)
        self.s, self.a, self.r, self.d, self.s2 = z(buffer_size, 5), z(buffer_size, 2), z(buffer_size), z(buffer_size), z(buffer_size, 5)
        self._c = L.Replay(self.s.data_ptr(), self.a.data_ptr(), self.r.data_ptr(), self.d.data_ptr(), self.s2.data_ptr(),
                           self.buffer_size)

    def add(self, obs_soa, actions, rew, done, obs_next_soa, n=None):
        """obs_soa / obs_next_soa: [5, stride] SoA rows (VecMREnv buffers), actions [n, 2], rew [n], done [n] uint8."""
        n = int(actions.shape[0] if n is None else n)
        if n > self.buffer_size:
            raise ValueError("more transitions in one step than the buffer holds")
        dt = {torch.float64: L.MR_F64, torch.float32: L.MR_F32}[obs_soa.dtype]
        with torch.cuda.device(self.device):
            rc = self.lib.mr_replay_add(C.byref(self._c), self.head, obs_soa.data_ptr(), obs_soa.stride(0), actions.data_ptr(),
                                        rew.data_ptr(), done.data_ptr(), obs_next_soa.data_ptr(), obs_next_soa.stride(0), n, dt,
                                        _stream(self.device))
        L.check(rc, "mr_replay_add")
        self.head = (self.head + n) % self.buffer_size
        self.count = min(self.count + n, self.buffer_size)

    def size(self):
        return self.count

    def sample_indices(self, batch_size, update_index=1):
        """``batch_size`` distinct rows of the filled part of the ring (random.sample, :43-46) as a device int64 tensor."""
        idx = torch.empty(int(batch_size), dtype=torch.int64, device=self.device)
        with torch.cuda.device(self.device):
            rc = self.lib.mr_replay_sample(self.count, int(batch_size), self.random_seed, int(update_index), idx.data_ptr(),
                                           _stream(self.device))
        L.check(rc, "mr_replay_sample")
        return idx

    def clear(self):
        self.count = 0
        self.head = 0


class OUNoise:
    """OUNoise (:58-78), one independent process per env and action dimension, state in HBM (float64)."""

    def __init__(self, num_envs, mu=0.0, sigma=0.3, theta=0.15, dt=1e-2, seed=0, env_base=0, device="cuda"):
        self.lib = L.load()
        self.device = _cuda_device(device)
        self.mu, self.sigma, self.theta, self.dt = float(mu), float(sigma), float(theta), float(dt)
        self.seed, self.env_base, self.calls = int(seed), int(env_base), 0
        self.x_prev = torch.zeros(num_envs, 2, dtype=torch.float64, device=self.device)

    def add_to(self, actions, reset_mask=None):
        """actions [n, 2] (float64 / float32 device tensor) += the next OU sample, in place."""
        dt = {torch.float64: L.MR_F64, torch.float32: L.MR_F32}[actions.dtype]
        with torch.cuda.device(self.device):
            rc = self.lib.mr_ou_noise_add(self.x_prev.data_ptr(), actions.data_ptr(),
                                          reset_mask.data_ptr() if reset_mask is not None else None, actions.shape[0], dt,
                                          self.theta, self.mu, self.sigma, self.dt, self.seed, self.calls, self.env_base,
                                          _stream(self.device))
        L.check(rc, "mr_ou_noise_add")
        self.calls += 1
        return actions

    def reset(self):
        self.x_prev.zero_()


class DDPGLearner:
    """ActorNetwork + CriticNetwork (:80-231): online and target parameters, Adam moments, one-launch update."""

    def __init__(self, actor=None, critic=None, action_bound=(20.0, 2 * math.pi), actor_lr=1e-3, critic_lr=1e-2, tau=1e-3,
                 gamma=0.99, seed=0, device="cuda", actor_target_init=None, critic_target_init=None, target_init="independent"):
        self.lib = L.load()
        self.device = _cuda_device(device)
        self.actor = pack_actor(actor if actor is not None else init_actor(seed), self.device)
        self.critic = pack_critic(critic if critic is not None else init_critic(seed + 1), self.device)
        # The reference initialises the target graphs independently (tf.global_variables_initializer) and then calls
        # update_target_network() once (:237-241), i.e. theta' = tau * theta + (1 - tau) * theta'_init — NOT a copy.
        # target_init="independent" reproduces that (with *_target_init dicts, or fresh draws); "copy" starts the
        # targets at the online values.
        if target_init == "copy":
            self.actor_target = self.actor.clone()
            self.critic_target = self.critic.clone()
        elif target_init == "independent":
            at = pack_actor(actor_target_init if actor_target_init is not None else init_actor(seed + 2), self.device)
            ct = pack_critic(critic_target_init if critic_target_init is not None else init_critic(seed + 3), self.device)
            self.actor_target = tau * self.actor + (1 - tau) * at
            self.critic_target = tau * self.critic + (1 - tau) * ct
        else:
            raise ValueError("target_init must be 'independent' or 'copy'")
        self._moments = [torch.zeros_like(self.actor), torch.zeros_like(self.actor), torch.zeros_like(self.critic),
                         torch.zeros_like(self.critic)]
        self._grads = [torch.zeros_like(self.actor), torch.zeros_like(self.critic)]
        self._c = L.DDPGState(self.actor.data_ptr(), self.actor_target.data_ptr(), self.critic.data_ptr(),
                              self.critic_target.data_ptr(), *[m.data_ptr() for m in self._moments],
                              *[g.data_ptr() for g in self._grads])
        self.hyper = L.DDPGHyper(gamma, tau, actor_lr, critic_lr, (C.c_double * 2)(*map(float, action_bound)), 0.9, 0.999, 1e-8)
        self.action_bound = tuple(map(float, action_bound))
        self.seed = int(seed)
        self.updates = 0
        self._info = torch.zeros(2, dtype=torch.float32, device=self.device)
        self._ws = None
        self.kernel_launches = 0

    def predict(self, obs_soa, n=None):
        """ActorNetwork.predict (:146-149) for the env's SoA observation rows -> actions [n, 2] (obs dtype)."""
        self.kernel_launches += 1
        return actor_forward(self.actor, obs_soa, n, self.action_bound, env_obs=True)

    def update(self, replay, batch_size=64, indices=None):
        """The update block of train() (:285-305).  ``indices`` (int64 device tensor) pins the minibatch; by default the
        kernel samples it without replacement like random.sample.  Returns the device tensor [critic loss, mean Q]."""
        idx_ptr = None
        if indices is not None:
            indices = torch.as_tensor(indices, dtype=torch.int64, device=self.device).contiguous()
            batch_size = int(indices.numel())
            idx_ptr = indices.data_ptr()
        self.updates += 1
        ws_ptr, ws_bytes = None, 0
        if batch_size > 64:                        # data-parallel kernels (one CTA per SM) need per-CTA gradient slabs
            ws_bytes = int(self.lib.mr_ddpg_workspace_bytes(int(batch_size)))
            if self._ws is None or self._ws.numel() * 8 < ws_bytes:
                self._ws = torch.empty((ws_bytes + 7) // 8, dtype=torch.float64, device=self.device)
            ws_ptr = self._ws.data_ptr()
        with torch.cuda.device(self.device):
            rc = self.lib.mr_ddpg_update(C.byref(self._c), C.byref(replay._c), replay.count, int(batch_size), idx_ptr,
                                         self.seed ^ replay.random_seed, self.updates, C.byref(self.hyper), self._info.data_ptr(),
                                         ws_ptr, ws_bytes, _stream(self.device))
        if rc:
            self.updates -= 1
        L.check(rc, "mr_ddpg_update")
        self.kernel_launches += 1
        return self._info

    def update_distributed(self, replay, batch_size=64, indices=None, group=None):
        """The same update with the gradient exchange of a data-parallel learner (one process per GPU, each with its own
        replay shard and the same parameters): every rank computes the gradients of ITS minibatch, the gradient vectors
        are summed over the ranks (torch.distributed all_reduce, NCCL) and every rank applies the mean — the effective
        minibatch is world_size * batch_size.  Without an initialised process group this is the single-rank split path.
        Returns the device tensor [critic loss, mean Q] over the global minibatch."""
        import torch.distributed as dist
        world = dist.get_world_size(group) if dist.is_available() and dist.is_initialized() else 1
        idx_ptr = None
        if indices is not None:
            indices = torch.as_tensor(indices, dtype=torch.int64, device=self.device).contiguous()
            batch_size = int(indices.numel())
            idx_ptr = indices.data_ptr()
        ws_bytes = int(self.lib.mr_ddpg_workspace_bytes(int(batch_size)))
        if self._ws is None or self._ws.numel() * 8 < ws_bytes:
            self._ws = torch.empty((ws_bytes + 7) // 8, dtype=torch.float64, device=self.device)
        if getattr(self, "_gbuf", None) is None:
            self._gbuf = torch.zeros(self.actor.numel() + 8, dtype=torch.float32, device=self.device)
        g = self._gbuf
        self.updates += 1
        n_c, n_a = self.critic.numel(), self.actor.numel()
        seed = self.seed ^ replay.random_seed
        with torch.cuda.device(self.device):
            for which, n in ((0, n_c + 2), (1, n_a)):
                rc = self.lib.mr_ddpg_gradients(C.byref(self._c), C.byref(replay._c), replay.count, int(batch_size), idx_ptr, seed,
                                                self.updates, C.byref(self.hyper), which, g.data_ptr(), self._ws.data_ptr(),
                                                ws_bytes, _stream(self.device))
                L.check(rc, "mr_ddpg_gradients")
                if world > 1:
                    dist.all_reduce(g[:n], group=group)
                if which == 0:
                    self._info.copy_(g[n_c:n_c + 2] / float(batch_size * world))
                rc = self.lib.mr_ddpg_apply(C.byref(self._c), which, g.data_ptr(), 1.0 / world, self.updates, C.byref(self.hyper),
                                            _stream(self.device))
                L.check(rc, "mr_ddpg_apply")
        self.kernel_launches += 8
        return self._info

    def actor_params(self, target=False):
        return _unpack(self.actor_target if target else self.actor, ACTOR_ORDER, ACTOR_SHAPES)

    def critic_params(self, target=False):
        return _unpack(self.critic_target if target else self.critic, CRITIC_ORDER, CRITIC_SHAPES)


def collect(env, learner, actor_noise, replay, k_steps, **rollout_kw):
    """K iterations of train()'s acting loop in ONE launch: per step, every env acts with mu(s) + the next OU sample, steps,
    and its transition (s, a, r, done, s2) enters the replay ring.  Uses the online actor ``learner.actor`` as it is at
    launch time, the noise's state / call count / seed / env base and the ring's head.  Afterwards ``replay.head`` /
    ``replay.count`` and ``actor_noise.calls`` have advanced exactly as K ``add`` / ``add_to`` calls advance them; the stream
    is not synchronised.  On the 3xTF32 actor path (``_lib.set_actor_path("tf32")``) the ring, the noise state and the env
    equal K rounds of predict -> add_to -> step -> add bit for bit; the default 3xFP16 path agrees to ~1e-4 of the action
    range.  ``rollout_kw`` go to ``env.rollout`` (recording rows, statistics, reset_init), whose result is returned."""
    k = int(k_steps)
    n = env.num_envs
    if k < 1:
        raise ValueError("k_steps must be at least 1")
    if n > replay.buffer_size:
        raise ValueError(f"{n} envs add more transitions per step than the replay buffer holds ({replay.buffer_size})")
    if actor_noise.x_prev.shape[0] < n:
        raise ValueError(f"the OU noise has {actor_noise.x_prev.shape[0]} processes for {n} envs")
    if tuple(learner.action_bound) != (env.params.action_high[0], env.params.action_high[1]):
        raise ValueError("learner.action_bound must equal the env's action_space.high (the in-kernel actor scales by it)")
    c = L.DDPGCollect(actor_noise.x_prev.data_ptr(), actor_noise.theta, actor_noise.mu, actor_noise.sigma, actor_noise.dt,
                      actor_noise.seed & (2**64 - 1), actor_noise.calls, actor_noise.env_base, replay._c, replay.head)
    res = env.rollout(policy=learner.actor, k_steps=k, ddpg_collect=c, **rollout_kw)
    replay.head = (replay.head + k * n) % replay.buffer_size
    replay.count = min(replay.count + k * n, replay.buffer_size)
    actor_noise.calls += k
    return res


def train(env, learner, actor_noise, buffer_size=10000, min_batch=64, steps=1000, updates_per_step=1, replay=None,
          noise_var=1, a0=1, log_every=0, stale_state_warmup=False, collect_steps=None):
    """train() (:233-323) for a vectorised env: every iteration all N envs act with mu(s) + OU noise, the N transitions
    enter the ring, and once it holds ``min_batch`` transitions the learner takes ``updates_per_step`` updates.  ``env``
    is a VecMREnv built with auto_reset=True (an env that ends starts its next episode inside the same launch, the
    reference's ``break`` + ``env.reset()``).  Returns per-iteration (mean reward, critic loss, mean Q) as a numpy array.
    Forced by vectorisation: N transitions per iteration instead of one.
    ``stale_state_warmup=True`` reproduces the scalar loop's warm-up quirk: while the buffer holds fewer than
    ``min_batch`` transitions the loop ``continue``s before ``state = next_state`` (:281-284), so the policy keeps seeing —
    and the buffer keeps storing as ``s`` — the observation of the last reset, while the env itself moves on.  With
    N >= min_batch envs the buffer is full after the first iteration and the flag changes nothing.
    ``collect_steps=K`` fuses the acting: an iteration is one ``collect`` of K env steps (the last one shorter if K does
    not divide ``steps``), then K * ``updates_per_step`` updates once the ring holds ``min_batch`` transitions — the same
    ratio of updates to env steps, with a policy up to K steps stale.  The log then has one row per launch: the mean
    reward over its transitions (from the env's statistics vector, which these launches accumulate) and the loss and
    mean Q of its last update.  ``collect_steps=1`` on the 3xTF32 actor path reproduces the default loop bit for bit."""
    n = env.num_envs
    if collect_steps is not None:
        if stale_state_warmup:
            raise ValueError("stale_state_warmup reproduces the per-step loop; it cannot be combined with collect_steps")
        return _train_collect(env, learner, actor_noise, buffer_size, min_batch, steps, updates_per_step, replay,
                              noise_var, a0, log_every, int(collect_steps))
    replay = replay if replay is not None else ReplayBuffer(buffer_size, 0, device=env.device)
    obs_rows = env._obs
    env.reset(noise_var=noise_var, a0=a0)
    state = obs_rows.clone()                       # the loop's `state`: policy input and the stored s
    log = torch.zeros(steps, 3, dtype=torch.float64, device=env.device)
    for it in range(steps):
        actions = learner.predict(state, n)
        actor_noise.add_to(actions)
        _, rew, done, _ = env.step(actions)
        replay.add(state, actions, rew, done, obs_rows, n)
        log[it, 0] = rew[:n].mean()
        if replay.size() >= min_batch:
            for _ in range(updates_per_step):
                info = learner.update(replay, min_batch)
            log[it, 1:] = info.double()
            state.copy_(obs_rows)                  # state = next_state (:307)
        elif stale_state_warmup:
            ended = done[:n].bool()                # `break` -> env.reset() -> a fresh state; everyone else keeps the stale one
            state[:, :n][:, ended] = obs_rows[:, :n][:, ended]
        else:
            state.copy_(obs_rows)
        if log_every and (it + 1) % log_every == 0:
            row = log[it].cpu().numpy()
            print(f"iter {it + 1}/{steps}: mean reward {row[0]:.3f} critic loss {row[1]:.4g} mean Q {row[2]:.4g}")
    return log.cpu().numpy()


def _train_collect(env, learner, actor_noise, buffer_size, min_batch, steps, updates_per_step, replay, noise_var, a0,
                   log_every, k):
    n = env.num_envs
    if k < 1:
        raise ValueError("collect_steps must be at least 1")
    replay = replay if replay is not None else ReplayBuffer(buffer_size, 0, device=env.device)
    if n > replay.buffer_size:
        raise ValueError(f"{n} envs add more transitions per step than the replay buffer holds ({replay.buffer_size})")
    env.reset(noise_var=noise_var, a0=a0)
    launches = (steps + k - 1) // k
    log = torch.zeros(launches, 3, dtype=torch.float64, device=env.device)
    rew_sum = env.stats[L.STAT_NAMES.index("sum_reward")]
    done = 0
    for it in range(launches):
        kk = min(k, steps - done)
        before = rew_sum.clone()
        collect(env, learner, actor_noise, replay, kk)
        log[it, 0] = (rew_sum - before) / (kk * n)
        if replay.size() >= min_batch:
            for _ in range(kk * updates_per_step):
                info = learner.update(replay, min_batch)
            log[it, 1:] = info.double()
        done += kk
        if log_every and (it + 1) % log_every == 0:
            row = log[it].cpu().numpy()
            print(f"launch {it + 1}/{launches} ({done} steps): mean reward {row[0]:.3f} critic loss {row[1]:.4g} mean Q {row[2]:.4g}")
    return log.cpu().numpy()


# ---- populations: many independent learners trained in lockstep -------------------------------------------------------
# Member p of a population computes exactly what its solo run computes: DDPGLearner(seed=seeds[p], ...) with its own
# ReplayBuffer, OUNoise(N, seed, env_base=p N) and VecMREnv(N, seed, env_base=p N) (env p N + j of the population's
# VecMREnv(P N, seed) is env j of that solo env).  The difference is the launches: one update launch (one CTA per member)
# and one collect launch for all members, where solo runs take P of each.

def _per_member(name, v, members):
    """A scalar for every member, or one value per member."""
    if np.ndim(v) == 0:
        return [float(v)] * members
    v = [float(x) for x in v]
    if len(v) != members:
        raise ValueError(f"{name} has {len(v)} values for {members} members")
    return v


_HYPER_FIELDS = (("actor_lr", "lr_actor"), ("critic_lr", "lr_critic"), ("tau", "tau"), ("gamma", "gamma"))


def _check_members(members):
    members = int(members)
    if not 1 <= members <= L.DDPG_MAX_MEMBERS:
        raise ValueError(f"members must be in 1..{L.DDPG_MAX_MEMBERS}")
    return members


class PopulationReplay:
    """One replay ring per member, stacked: ``s`` [P, buffer_size, 5], ``a`` [P, buffer_size, 2], ``r`` / ``d``
    [P, buffer_size], ``s2`` [P, buffer_size, 5].  The members fill at the same rate, so ``head`` and ``count`` are shared.
    ``random_seeds`` (a scalar or one per member) plays ReplayBuffer's ``random_seed``."""

    def __init__(self, members, buffer_size, random_seeds=0, device="cuda"):
        self.members = _check_members(members)
        self.random_seeds = [int(s) for s in _per_member("random_seeds", random_seeds, self.members)]
        self.lib = L.load()
        self.device = _cuda_device(device)
        self.buffer_size = int(buffer_size)
        self.count = 0
        self.head = 0
        P, cap = self.members, self.buffer_size
        z = lambda *s: torch.zeros(*s, dtype=torch.float32, device=self.device)
        self.s, self.a, self.r, self.d, self.s2 = z(P, cap, 5), z(P, cap, 2), z(P, cap), z(P, cap), z(P, cap, 5)
        self._c = L.Replay(self.s.data_ptr(), self.a.data_ptr(), self.r.data_ptr(), self.d.data_ptr(), self.s2.data_ptr(), cap)

    def size(self):
        return self.count

    def member(self, p):
        """Member p's ring as a ReplayBuffer whose arrays are views into the stacked rings; head and count are copied
        from the population at this call."""
        rb = ReplayBuffer.__new__(ReplayBuffer)
        rb.lib, rb.device, rb.buffer_size, rb.random_seed = self.lib, self.device, self.buffer_size, self.random_seeds[p]
        rb.count, rb.head = self.count, self.head
        rb.s, rb.a, rb.r, rb.d, rb.s2 = self.s[p], self.a[p], self.r[p], self.d[p], self.s2[p]
        rb._c = L.Replay(rb.s.data_ptr(), rb.a.data_ptr(), rb.r.data_ptr(), rb.d.data_ptr(), rb.s2.data_ptr(), rb.buffer_size)
        return rb

    def clear(self):
        self.count = 0
        self.head = 0


class DDPGPopulation:
    """``members`` independent DDPG learners in stacked storage: ``actor`` / ``actor_target`` [P, actor count], ``critic`` /
    ``critic_target`` [P, critic count], and the Adam moments alike.  Member p starts exactly as
    ``DDPGLearner(seed=seeds[p], actor_lr=..., ...)`` would.  ``actor_lr``, ``critic_lr``, ``tau`` and ``gamma`` are a
    scalar or one value per member; ``action_bound`` is the env's action range, one pair for all.  ``stats`` [P, 8]
    collects each member's episode statistics (``collect_population``)."""

    def __init__(self, members, seeds=None, actor_lr=1e-3, critic_lr=1e-2, tau=1e-3, gamma=0.99,
                 action_bound=(20.0, 2 * math.pi), target_init="independent", device="cuda"):
        P = self.members = _check_members(members)
        self.seeds = list(range(P)) if seeds is None else [int(s) for s in seeds]
        if len(self.seeds) != P:
            raise ValueError(f"seeds has {len(self.seeds)} values for {P} members")
        hp = [_per_member(k, v, P) for k, v in (("actor_lr", actor_lr), ("critic_lr", critic_lr), ("tau", tau), ("gamma", gamma))]
        self.lib = L.load()
        self.device = _cuda_device(device)
        learners = [DDPGLearner(action_bound=action_bound, actor_lr=hp[0][p], critic_lr=hp[1][p], tau=hp[2][p], gamma=hp[3][p],
                                seed=self.seeds[p], device=self.device, target_init=target_init) for p in range(P)]
        stack = lambda get: torch.stack([get(m) for m in learners]).contiguous()
        self.actor, self.actor_target = stack(lambda m: m.actor), stack(lambda m: m.actor_target)
        self.critic, self.critic_target = stack(lambda m: m.critic), stack(lambda m: m.critic_target)
        self._moments = [stack(lambda m, i=i: m._moments[i]) for i in range(4)]
        self._grads = [stack(lambda m, i=i: m._grads[i]) for i in range(2)]
        for p, m in enumerate(learners):             # the members now work on views of the stacked storage
            m.actor, m.actor_target, m.critic, m.critic_target = self.actor[p], self.actor_target[p], self.critic[p], self.critic_target[p]
            m._moments = [t[p] for t in self._moments]
            m._grads = [t[p] for t in self._grads]
            m._c = L.DDPGState(m.actor.data_ptr(), m.actor_target.data_ptr(), m.critic.data_ptr(), m.critic_target.data_ptr(),
                               *[t.data_ptr() for t in m._moments], *[t.data_ptr() for t in m._grads])
        self._learners = learners
        self.action_bound = learners[0].action_bound
        self.hyper = (L.DDPGHyper * P)(*[m.hyper for m in learners])
        state = L.DDPGState(self.actor.data_ptr(), self.actor_target.data_ptr(), self.critic.data_ptr(), self.critic_target.data_ptr(),
                            *[t.data_ptr() for t in self._moments], *[t.data_ptr() for t in self._grads])
        self._c = L.DDPGPopulation(P, state, L.Replay(), self.hyper, None)
        self.updates = 0
        self._info = torch.zeros(P, 2, dtype=torch.float32, device=self.device)
        self.stats = torch.zeros(P, L.STATS_LEN, dtype=torch.float64, device=self.device)
        self.kernel_launches = 0

    def member(self, p):
        """Member p as a DDPGLearner whose tensors are views into the population's storage (predict, actor_params,
        critic_params and a solo update work on it).  Its update count is the population's at this call."""
        m = self._learners[p]
        m.updates = self.updates
        return m

    def hyper_table(self):
        """The hyper-parameters as a [P, 4] float64 array, columns (actor_lr, critic_lr, tau, gamma)."""
        return np.array([[getattr(h, f) for _, f in _HYPER_FIELDS] for h in self.hyper], dtype=np.float64)

    def set_hyper(self, p, actor_lr=None, critic_lr=None, tau=None, gamma=None):
        """Change member p's hyper-parameters (those given); its next update uses them.  ``member(p).hyper`` follows."""
        p = self._index(p)
        for (name, field), v in zip(_HYPER_FIELDS, (actor_lr, critic_lr, tau, gamma)):
            if v is None:
                continue
            if not math.isfinite(float(v)):
                raise ValueError(f"{name} must be finite")
            setattr(self.hyper[p], field, float(v))
            setattr(self._learners[p].hyper, field, float(v))

    def exploit(self, dst, src):
        """Member dst[k] becomes a copy of member src[k]: online and target actor and critic, the four Adam moments (one
        index copy per stacked tensor, all sources read before any destination is written) and the hyper-parameters.
        The destination keeps its sampling seed, replay ring, OU state and envs.  ``dst`` must not repeat a member."""
        dst = [self._index(d) for d in np.atleast_1d(np.asarray(dst, dtype=np.int64))]
        src = [self._index(s) for s in np.atleast_1d(np.asarray(src, dtype=np.int64))]
        if len(dst) != len(src):
            raise ValueError(f"dst has {len(dst)} members, src {len(src)}")
        if len(set(dst)) != len(dst):
            raise ValueError("dst repeats a member")
        if not dst:
            return
        d = torch.tensor(dst, dtype=torch.int64, device=self.device)
        s = torch.tensor(src, dtype=torch.int64, device=self.device)
        for t in (self.actor, self.actor_target, self.critic, self.critic_target, *self._moments):
            t.index_copy_(0, d, t.index_select(0, s))
        rows = [L.DDPGHyper.from_buffer_copy(self.hyper[b]) for b in src]
        for a, h in zip(dst, rows):
            C.memmove(C.byref(self.hyper[a]), C.byref(h), C.sizeof(h))
            C.memmove(C.byref(self._learners[a].hyper), C.byref(h), C.sizeof(h))

    def _index(self, p):
        p = int(p)
        if not 0 <= p < self.members:
            raise ValueError(f"member {p} is not in 0..{self.members - 1}")
        return p

    def update(self, replay, batch_size=64):
        """One update of every member in ONE launch (one CTA per member): member p samples ``batch_size`` rows of its own
        ring, as DDPGLearner.update does with ``seed ^ random_seed``, and takes the single-CTA update (batch 1..4096).
        Returns the device tensor [P, 2] of (critic loss, mean Q)."""
        batch_size = int(batch_size)
        if replay.members != self.members:
            raise ValueError(f"the replay has {replay.members} members, the population {self.members}")
        if not 1 <= batch_size <= 4096:
            raise ValueError("batch_size must be in 1..4096 (the single-CTA update of each member)")
        seeds = (C.c_uint64 * self.members)(*[(s ^ r) & (2**64 - 1) for s, r in zip(self.seeds, replay.random_seeds)])
        self._seeds_c = seeds                      # kept alive for the call
        self._c.ring, self._c.seeds = replay._c, seeds
        self.updates += 1
        with torch.cuda.device(self.device):
            rc = self.lib.mr_ddpg_update_population(C.byref(self._c), replay.count, batch_size, self.updates,
                                                    self._info.data_ptr(), _stream(self.device))
        if rc:
            self.updates -= 1
        L.check(rc, "mr_ddpg_update_population")
        self.kernel_launches += 1
        return self._info


def _member_envs(env, members):
    n = env.num_envs
    if n % members or (n // members) % 128:
        raise ValueError(f"env.num_envs = {n} must be members ({members}) x N with N a multiple of 128")
    return n // members


def collect_population(env, pop, actor_noise, replay, k_steps, **rollout_kw):
    """``collect`` for every member in ONE launch: ``env`` holds members x N envs (N a multiple of 128), env p N + j acts
    with member p's online actor and writes its transitions into member p's ring; one OUNoise covers all envs.  Advances
    ``replay.head`` / ``replay.count`` by K N transitions and ``actor_noise.calls`` by K, and adds each member's episode
    statistics to ``pop.stats[p]``.  Member p's ring, OU rows and envs end exactly as ``collect`` leaves its solo run."""
    k = int(k_steps)
    P = pop.members
    if k < 1:
        raise ValueError("k_steps must be at least 1")
    if replay.members != P:
        raise ValueError(f"the replay has {replay.members} members, the population {P}")
    N = _member_envs(env, P)
    if N > replay.buffer_size:
        raise ValueError(f"{N} envs per member add more transitions per step than a member's replay buffer holds ({replay.buffer_size})")
    if actor_noise.x_prev.shape[0] < env.num_envs:
        raise ValueError(f"the OU noise has {actor_noise.x_prev.shape[0]} processes for {env.num_envs} envs")
    if tuple(pop.action_bound) != (env.params.action_high[0], env.params.action_high[1]):
        raise ValueError("pop.action_bound must equal the env's action_space.high (the in-kernel actor scales by it)")
    c = L.DDPGCollect(actor_noise.x_prev.data_ptr(), actor_noise.theta, actor_noise.mu, actor_noise.sigma, actor_noise.dt,
                      actor_noise.seed & (2**64 - 1), actor_noise.calls, actor_noise.env_base, replay._c, replay.head)
    res = env.rollout(policy=pop.actor, k_steps=k, ddpg_collect=c, ddpg_population=(P, pop.stats), **rollout_kw)
    replay.head = (replay.head + k * N) % replay.buffer_size
    replay.count = min(replay.count + k * N, replay.buffer_size)
    actor_noise.calls += k
    return res


def train_population(env, pop, actor_noise, buffer_size=10000, min_batch=64, steps=1000, updates_per_step=1, replay=None,
                     noise_var=1, a0=1, log_every=0, collect_steps=64, reset=True):
    """``train(collect_steps=K)`` for a population: per launch one ``collect_population`` of K env steps, then
    K * ``updates_per_step`` population updates once the rings hold ``min_batch`` transitions.  Returns the log
    [P, launches, 3]: per member the mean reward of the launch's transitions, and the loss and mean Q of its last update.
    With ``min_batch`` <= 64 member p's run equals its solo ``train(collect_steps=K)`` (above 64 samples the solo update
    takes the data-parallel path, the population the single-CTA one).  ``reset=False`` continues the env's episodes
    instead of resetting it (``noise_var`` and ``a0`` are then unused): two calls of S and T steps, S a multiple of K, then
    equal one call of S + T steps when they share ``replay``."""
    P = pop.members
    k = int(collect_steps)
    if k < 1:
        raise ValueError("collect_steps must be at least 1")
    N = _member_envs(env, P)
    replay = replay if replay is not None else PopulationReplay(P, buffer_size, 0, device=env.device)
    if replay.members != P:
        raise ValueError(f"the replay has {replay.members} members, the population {P}")
    if N > replay.buffer_size:
        raise ValueError(f"{N} envs per member add more transitions per step than a member's replay buffer holds ({replay.buffer_size})")
    if reset:
        env.reset(noise_var=noise_var, a0=a0)
    launches = (steps + k - 1) // k
    log = torch.zeros(P, launches, 3, dtype=torch.float64, device=env.device)
    rew_sum = pop.stats[:, L.STAT_NAMES.index("sum_reward")]
    done = 0
    for it in range(launches):
        kk = min(k, steps - done)
        before = rew_sum.clone()
        collect_population(env, pop, actor_noise, replay, kk)
        log[:, it, 0] = (rew_sum - before) / (kk * N)
        if replay.size() >= min_batch:
            for _ in range(kk * updates_per_step):
                info = pop.update(replay, min_batch)
            log[:, it, 1:] = info.double()
        done += kk
        if log_every and (it + 1) % log_every == 0:
            row = log[:, it].mean(0).cpu().numpy()
            print(f"launch {it + 1}/{launches} ({done} steps), mean over {P} members: reward {row[0]:.3f} "
                  f"critic loss {row[1]:.4g} mean Q {row[2]:.4g}")
    return log.cpu().numpy()


# ---- greedy evaluation and population-based training ------------------------------------------------------------------

@dataclasses.dataclass
class PopulationEvaluation:
    """What ``evaluate_population`` returns.  [P] device tensors, one value per member over its N episodes:
    ``mean_return`` (undiscounted), ``goal_rate`` / ``out_of_bounds_rate`` / ``timeout_rate`` (how the episodes ended),
    ``mean_length`` (steps), ``failed`` (episodes with a status flag) and ``env_steps`` (steps taken).  With ``per_env``
    also the [P, N] rows ``ret`` (float64), ``length`` (int32), ``outcome`` (uint8: 1 goal, 2 out of bounds, 3 timeout)
    and ``status`` (uint8, the sticky ENV_* flags); otherwise those are None."""
    mean_return: torch.Tensor
    goal_rate: torch.Tensor
    out_of_bounds_rate: torch.Tensor
    timeout_rate: torch.Tensor
    mean_length: torch.Tensor
    failed: torch.Tensor
    env_steps: torch.Tensor
    ret: torch.Tensor = None
    length: torch.Tensor = None
    outcome: torch.Tensor = None
    status: torch.Tensor = None


def evaluate_population(env, pop, member_envs, init=None, common_random_numbers=True, offset=0, per_env=False):
    """Every member's greedy policy (its online actor, no exploration noise) on ``member_envs`` = N fresh episodes, in ONE
    launch (mr_ddpg_evaluate_population).  ``env`` (any VecMREnv) supplies the task: storage dtype, noise kind, seed and
    table, a0 / noise_var / is_mismatched, reward mode, bounds, max_timesteps and action bound; its state rows, statistics
    and step index are not touched.  Episode j of every member starts at ``init[j]`` ([N, 2], or one (2,) position for
    all), or at a sample of init_space, and runs to its end (at most max_timesteps + 1 steps).  ``offset`` is the Philox
    step index of the evaluation: the start is drawn at ``offset`` and step k at ``offset + 1 + k``, as a solo env whose
    step index is ``offset`` draws them on ``reset()`` followed by a rollout.  With ``common_random_numbers`` every
    member's episode j draws what env j draws (so members differ only by their policies; a table then needs N columns),
    without it env p N + j draws with key env_base + p N + j (a table needs P N columns).  Returns a PopulationEvaluation;
    the stream is not synchronised.  ``mean_return`` is reduced from the per-env returns, so it does not depend on the
    order of the launch's atomics."""
    return _evaluate(env, pop.actor, pop.members, pop.action_bound, member_envs, init, common_random_numbers, offset, per_env)


def evaluate(env, learner, n_envs, init=None, common_random_numbers=True, offset=0, per_env=False):
    """``evaluate_population`` for one DDPGLearner on ``n_envs`` episodes (a multiple of 128); the result has P = 1."""
    return _evaluate(env, learner.actor.reshape(1, -1), 1, learner.action_bound, n_envs, init, common_random_numbers, offset,
                     per_env)


def _evaluate(env, actors, members, action_bound, member_envs, init, crn, offset, per_env):
    lib = L.load()
    P = _check_members(members)
    N = int(member_envs)
    if N <= 0 or N % 128:
        raise ValueError(f"member_envs = {N} must be a positive multiple of 128")
    if tuple(action_bound) != (env.params.action_high[0], env.params.action_high[1]):
        raise ValueError("the actors' action_bound must equal the env's action_space.high (the in-kernel actor scales by it)")
    if env.per_env_params:
        raise ValueError("the evaluation plays the env's launch parameters: envs with per-env parameter rows are not supported")
    w = actors.to(device=env.device, dtype=torch.float32).contiguous()
    if w.numel() != P * lib.mr_actor_param_count():
        raise ValueError(f"the actors must be [{P}, {lib.mr_actor_param_count()}] (actor.pack_actor per member)")
    init_t = None
    if init is not None:
        init_t = torch.as_tensor(np.asarray(init) if not torch.is_tensor(init) else init).to(device=env.device, dtype=env.dtype)
        if init_t.dim() == 1 and init_t.numel() == 2:
            init_t = init_t.reshape(1, 2).expand(N, 2)
        init_t = init_t.contiguous()
        if tuple(init_t.shape) != (N, 2):
            raise ValueError(f"init must be (2,) or ({N}, 2)")
    cols = 0
    if env.noise_kind == "table":
        cols = env._noise_table.shape[1]
        need = N if crn else P * N
        if cols < need:
            raise ValueError(f"the noise table has {cols} columns; the evaluation reads {need} "
                             f"({'N with' if crn else 'members x N without'} common random numbers)")
    nz = L.Noise.from_buffer_copy(env._noise_for(env.params.noise_var))
    nz.offset, nz.offset_dev = int(offset), None
    dev = env.device
    stats = torch.zeros(P, L.STATS_LEN, dtype=torch.float64, device=dev)
    ret = torch.empty(P, N, dtype=torch.float64, device=dev)
    rows = [torch.empty(P, N, dtype=dt, device=dev) for dt in (torch.int32, torch.uint8, torch.uint8)] if per_env else [None] * 3
    ptr = lambda t: t.data_ptr() if t is not None else None
    ev = L.DDPGEval(w.data_ptr(), P, 1 if crn else 0, N, ptr(init_t), stats.data_ptr(), ret.data_ptr(), *map(ptr, rows), cols)
    with torch.cuda.device(dev):
        rc = lib.mr_ddpg_evaluate_population(C.byref(ev), env._dt, C.byref(env.params), C.byref(nz), C.byref(env._c_tt),
                                             _stream(dev))
    L.check(rc, "mr_ddpg_evaluate_population")
    col = lambda name: stats[:, L.STAT_NAMES.index(name)]
    return PopulationEvaluation(mean_return=ret.mean(1), goal_rate=col("goal") / N, out_of_bounds_rate=col("out_of_bounds") / N,
                                timeout_rate=col("timeout") / N, mean_length=col("sum_length") / N, failed=col("failed"),
                                env_steps=col("env_steps"), ret=ret if per_env else None, length=rows[0], outcome=rows[1],
                                status=rows[2])


def pbt_plan(scores, fraction=0.25, perturb=(0.8, 1.25), rng=None):
    """One exploit / explore decision of population-based training, on the host.  The members are ranked by ``scores``
    (higher is better; equal scores rank by member index, lower first; NaN ranks last).  Each of the bottom
    m = floor(fraction P) members copies a member drawn uniformly from the top m, and then multiplies its actor and critic
    learning rates and tau by factors drawn from ``perturb``.  ``rng``: a numpy Generator or a seed.  Returns
    (dst [m], src [m], factors [m, 3]) with dst in ranking order and factor columns (actor_lr, critic_lr, tau)."""
    s = np.asarray(scores, dtype=np.float64).reshape(-1)
    P = s.size
    if not 0.0 <= float(fraction) <= 0.5:
        raise ValueError("fraction must be in [0, 0.5] (the top and bottom fractions must not overlap)")
    rng = np.random.default_rng(rng)
    m = int(math.floor(float(fraction) * P))
    order = np.lexsort((np.arange(P), -s))          # best first
    dst = order[P - m:].astype(np.int64)
    src = order[:m][rng.integers(0, m, size=m)].astype(np.int64) if m else np.zeros(0, dtype=np.int64)
    factors = rng.choice(np.asarray(perturb, dtype=np.float64), size=(m, 3)) if m else np.zeros((0, 3))
    return dst, src, factors


def pbt_population(env, pop, actor_noise, replay, rounds, steps_per_round, eval_envs, fraction=0.25, perturb=(0.8, 1.25),
                   seed=0, collect_steps=64, min_batch=64, eval_init=None):
    """Population-based training.  Per round: ``train_population`` for ``steps_per_round`` steps (the first round resets
    the env, later rounds continue its episodes and share ``replay``); ``evaluate_population`` with common random numbers
    on ``eval_envs`` episodes per member (start positions ``eval_init`` or samples of init_space), at one Philox offset
    per round drawn from ``seed``; then ``pbt_plan`` on the mean returns, ``pop.exploit(dst, src)`` and the perturbation of
    the copied members' learning rates and tau.  Returns the history {"score": [R, P] mean returns, "hyper": [R, P, 4]
    hyper-parameters the round trained with, "parent": [R, P] the member each member copied after the round (itself if
    none)}.  Raises for the constant reward (every step earns 10, so the return ranks long episodes first) and when any
    evaluation episode failed (as VecMREnv.check_status)."""
    if env.params.reward_mode == L.REWARD_CONST10:
        raise ValueError("population-based training ranks by return: the constant reward (10 per step) would favour "
                         "policies that never reach the goal; use reward_mode='shaped'")
    R, S = int(rounds), int(steps_per_round)
    if R < 1 or S < 1:
        raise ValueError("rounds and steps_per_round must be at least 1")
    P = pop.members
    if replay is None:
        replay = PopulationReplay(P, 10000, 0, device=env.device)
    rng = np.random.default_rng(seed)
    score, hyper = np.zeros((R, P)), np.zeros((R, P, 4))
    parent = np.tile(np.arange(P, dtype=np.int64), (R, 1))
    for r in range(R):
        train_population(env, pop, actor_noise, min_batch=min_batch, steps=S, replay=replay, collect_steps=collect_steps,
                         reset=r == 0)
        res = evaluate_population(env, pop, eval_envs, init=eval_init, common_random_numbers=True,
                                  offset=int(rng.integers(0, 2**62)), per_env=True)
        raise_for_status(res.status.reshape(-1))
        score[r] = res.mean_return.cpu().numpy()
        hyper[r] = pop.hyper_table()
        dst, src, factors = pbt_plan(score[r], fraction, perturb, rng)
        pop.exploit(dst, src)
        table = pop.hyper_table()
        for d, f in zip(dst, factors):
            h = table[d]
            pop.set_hyper(d, actor_lr=h[0] * f[0], critic_lr=h[1] * f[1], tau=h[2] * f[2])
        parent[r, dst] = src
    return {"score": score, "hyper": hyper, "parent": parent}
